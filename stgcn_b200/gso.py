"""Graph shift operators.

Dense preprocessing on the device (SURVEY.md §8f N4): counterparts of the reference's ``calc_gso`` /
``calc_chebynet_gso`` (script/utility.py:6-76), same names and argument meaning, CUDA tensors in and out.

Sparse operators: ``CsrOperator`` holds a graph shift operator as int32 CSR (plus the CSR of its transpose) on a
device.  The graph-convolution layers accept it wherever they take ``gso`` and then contract with a CSR SpMM kernel
instead of the dense ``(N, N)`` product -- for the large, low-degree graphs where a dense operator wastes memory and work.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import _lib as L

GSO_TYPES = {"sym_norm_adj": 0, "sym_renorm_adj": 1, "sym_norm_lap": 2, "sym_renorm_lap": 3,
             "rw_norm_adj": 4, "rw_renorm_adj": 5, "rw_norm_lap": 6, "rw_renorm_lap": 7}


def _build(adj: torch.Tensor, code: int, chebynet: bool):
    if not adj.is_cuda or adj.dtype != torch.float32 or adj.dim() != 2 or adj.shape[0] != adj.shape[1]:
        raise RuntimeError("stgcn_b200.gso: expected a square float32 CUDA tensor")
    adj = adj.contiguous()
    n = adj.shape[0]
    out = torch.empty_like(adj)
    eig = torch.zeros(2, dtype=torch.float32, device=adj.device)
    ws = torch.empty(n * n + 3 * n + 8, dtype=torch.float32, device=adj.device)
    with torch.cuda.device(adj.device):
        L.check(L.lib().stgcn_gso_build(adj.data_ptr(), n, code, int(chebynet), out.data_ptr(), eig.data_ptr(),
                                        ws.data_ptr(), ws.numel(), torch.cuda.current_stream(adj.device).cuda_stream))
    return out, eig


def calc_gso(dir_adj: torch.Tensor, gso_type: str) -> torch.Tensor:
    """utility.py:6-57 on a dense (N, N) adjacency: symmetrise, (re)normalise, optionally form the Laplacian."""
    if gso_type not in GSO_TYPES:
        raise ValueError(f"{gso_type} is not defined.")                                   # utility.py:54
    return _build(dir_adj, GSO_TYPES[gso_type], False)[0]


def calc_chebynet_gso(gso: torch.Tensor, return_eigval: bool = False):
    """utility.py:59-76: 2 L / lambda_max - I (or L - I when lambda_max >= 2), lambda_max = ||L||_2 by power iteration."""
    if not gso.is_cuda or gso.dtype != torch.float32 or gso.dim() != 2 or gso.shape[0] != gso.shape[1]:
        raise RuntimeError("stgcn_b200.gso: expected a square float32 CUDA tensor")
    gso = gso.contiguous()
    n = gso.shape[0]
    lib = L.lib()
    # the rescale alone: feed the operator through the builder's last two stages by treating it as already normalised
    out = torch.empty_like(gso)
    eig = torch.zeros(2, dtype=torch.float32, device=gso.device)
    ws = torch.empty(n * n + 3 * n + 8, dtype=torch.float32, device=gso.device)
    with torch.cuda.device(gso.device):
        L.check(lib.stgcn_gso_rescale(gso.data_ptr(), n, out.data_ptr(), eig.data_ptr(), ws.data_ptr(), ws.numel(),
                                      torch.cuda.current_stream(gso.device).cuda_stream))
    return (out, eig) if return_eigval else out


def build_operator(dir_adj: torch.Tensor, gso_type: str, chebynet: bool) -> torch.Tensor:
    """calc_gso followed (for Chebyshev convolutions, main.py:97-101) by calc_chebynet_gso, in one call."""
    if gso_type not in GSO_TYPES:
        raise ValueError(f"{gso_type} is not defined.")
    return _build(dir_adj, GSO_TYPES[gso_type], chebynet)[0]


# ----------------------------------------------------------------------------------------------
# sparse operators
# ----------------------------------------------------------------------------------------------
def _is_scipy_sparse(obj) -> bool:
    try:
        import scipy.sparse as sp
    except ImportError:                 # without scipy nothing can be a scipy matrix
        return False
    return sp.issparse(obj)


def is_sparse_operator(obj) -> bool:
    """True for what the layers route to the CSR path: a CsrOperator, a torch sparse COO / CSR tensor, a scipy sparse
    matrix.  A dense tensor is not one (it keeps the dense path)."""
    if isinstance(obj, CsrOperator) or _is_scipy_sparse(obj):
        return True
    return torch.is_tensor(obj) and obj.layout in (torch.sparse_coo, torch.sparse_csr)


def _triplets(op):
    """(shape, rows int64, cols int64, values float64) of every stored entry, duplicates included, on the CPU."""
    if _is_scipy_sparse(op):
        m = op.tocoo()
        return (tuple(m.shape), torch.from_numpy(m.row.astype("int64")), torch.from_numpy(m.col.astype("int64")),
                torch.from_numpy(m.data.astype("float64")))
    if not torch.is_tensor(op):
        raise TypeError(f"CsrOperator: expected a scipy sparse matrix or a torch tensor, got {type(op).__name__}")
    t = op.detach().cpu()
    if t.dim() != 2:
        raise ValueError(f"CsrOperator: expected a 2-D operator, got shape {tuple(t.shape)}")
    if t.layout == torch.sparse_coo:
        idx = t._indices()
        return tuple(t.shape), idx[0].long(), idx[1].long(), t._values().double()
    if t.layout == torch.sparse_csr:
        crow = t.crow_indices().long()
        rows = torch.repeat_interleave(torch.arange(t.shape[0]), crow[1:] - crow[:-1])
        return tuple(t.shape), rows, t.col_indices().long(), t.values().double()
    if t.layout != torch.strided:
        raise TypeError(f"CsrOperator: unsupported tensor layout {t.layout}")
    rows, cols = torch.nonzero(t, as_tuple=True)
    return tuple(t.shape), rows, cols, t[rows, cols].double()


def _device(device) -> torch.device:
    """torch.device with the CUDA index made explicit, so that "cuda" and "cuda:0" compare equal."""
    dev = torch.device(device)
    if dev.type == "cuda" and dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    return dev


def _csr(rows: torch.Tensor, cols: torch.Tensor, vals: torch.Tensor, n: int):
    """Row-major int32 CSR of the (already de-duplicated, row-then-column sorted) triplets."""
    counts = torch.bincount(rows, minlength=n)
    row_ptr = torch.zeros(n + 1, dtype=torch.int64)
    row_ptr[1:] = torch.cumsum(counts, 0)
    return row_ptr.int(), cols.int(), vals.float()


class CsrOperator:
    """A graph shift operator in CSR form on one device, for the sparse path of the graph convolutions.

    Built from a scipy sparse matrix (any format), a torch sparse COO / CSR tensor, or -- passed explicitly -- a dense
    torch tensor.  Duplicate entries are summed (in float64, then rounded to float32), columns are sorted within each
    row, and the matrix must be square with indices in range and finite values.  ``row_ptr / col / val`` hold the
    operator, ``t_row_ptr / t_col / t_val`` its transpose (the backward contracts with gso^T); for an exactly symmetric
    operator the transpose arrays are the forward ones.  The conversion runs on the CPU with torch ops; the arrays are
    then copied to ``device``.

    Dense operators are never converted automatically: the dense tcgen05 path is faster for the shipped, 37-52 % dense
    graphs.  Wrap an operator in this class (or hand the layers a sparse tensor / scipy matrix) to take the CSR path."""

    def __init__(self, op, device=None):
        if isinstance(op, CsrOperator):
            src = op
        else:
            src = None
            shape, rows, cols, vals = _triplets(op)
            if len(shape) != 2 or shape[0] != shape[1]:
                raise ValueError(f"CsrOperator: the operator must be square, got shape {shape}")
            n = int(shape[0])
            if n <= 0 or n >= 2 ** 31:
                raise ValueError(f"CsrOperator: unsupported size N = {n}")
            if rows.numel() and (int(rows.min()) < 0 or int(rows.max()) >= n or int(cols.min()) < 0
                                 or int(cols.max()) >= n):
                raise ValueError(f"CsrOperator: an index lies outside [0, {n})")
            if not bool(torch.isfinite(vals).all()):
                raise ValueError("CsrOperator: the operator has non-finite values")
            # sum duplicates, sort (row, col)
            key = rows * n + cols
            uniq, inv = torch.unique(key, sorted=True, return_inverse=True)
            summed = torch.zeros(uniq.numel(), dtype=torch.float64).index_add_(0, inv, vals)
            r, c = uniq // n, uniq % n
            if uniq.numel() >= 2 ** 31:
                raise ValueError("CsrOperator: more than 2^31 - 1 non-zeros")
            fwd = _csr(r, c, summed, n)
            tkey = c * n + r                     # the transpose, sorted by (col, row)
            order = torch.argsort(tkey)
            bwd = _csr(c[order], r[order], summed[order], n)
            symmetric = all(torch.equal(a, b) for a, b in zip(fwd, bwd))
            self.N, self.nnz, self.symmetric = n, int(uniq.numel()), symmetric
            self._arrays = fwd + (fwd if symmetric else bwd)
        if src is not None:
            self.N, self.nnz, self.symmetric = src.N, src.nnz, src.symmetric
            self._arrays = src._arrays
        dev = _device(device) if device is not None else self._arrays[0].device
        self._place(dev)

    def _place(self, dev: torch.device) -> None:
        fwd = tuple(a.to(dev) for a in self._arrays[:3])
        bwd = fwd if self.symmetric else tuple(a.to(dev) for a in self._arrays[3:])
        self._arrays = fwd + bwd
        self.device = dev
        self._c = None

    @property
    def shape(self):
        return (self.N, self.N)

    row_ptr = property(lambda self: self._arrays[0])
    col = property(lambda self: self._arrays[1])
    val = property(lambda self: self._arrays[2])
    t_row_ptr = property(lambda self: self._arrays[3])
    t_col = property(lambda self: self._arrays[4])
    t_val = property(lambda self: self._arrays[5])

    def tensors(self):
        """The device arrays (the transpose's only when they differ), e.g. to watch their addresses."""
        return self._arrays[:3] if self.symmetric else self._arrays

    def to(self, device) -> "CsrOperator":
        """This operator on ``device``: itself when it is already there, else a copy."""
        dev = _device(device)
        if dev == self.device:
            return self
        return CsrOperator(self, device=dev)

    def to_dense(self) -> torch.Tensor:
        """The (N, N) float32 matrix on this operator's device (for tests and comparisons)."""
        rows = torch.repeat_interleave(torch.arange(self.N, device=self.device),
                                       (self.row_ptr[1:] - self.row_ptr[:-1]).long())
        out = torch.zeros((self.N, self.N), dtype=torch.float32, device=self.device)
        out[rows, self.col.long()] = self.val
        return out

    def c_struct(self) -> L.CsrGso:
        """The stgcn_csr_gso the *_csr entry points read (kept alive by this object)."""
        if self._c is None:
            a = self._arrays
            self._c = L.CsrGso(self.N, self.nnz, *[t.data_ptr() if t.numel() else None for t in a])
        return self._c

    def __repr__(self):
        return (f"CsrOperator(N={self.N}, nnz={self.nnz}, symmetric={self.symmetric}, device={self.device})")


def as_operator(gso, device: Optional[torch.device] = None) -> CsrOperator:
    """A sparse ``gso`` (see is_sparse_operator) as a CsrOperator on ``device``."""
    if isinstance(gso, CsrOperator):
        return gso.to(device) if device is not None else gso
    return CsrOperator(gso, device=device)
