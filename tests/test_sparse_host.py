"""CPU-side checks of the sparse graph-shift-operator path: CsrOperator conversion from scipy / torch formats, its
errors, the stgcn_csr_gso ctypes mirror, and the *_csr size queries (no GPU needed)."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from conftest import ROOT
from stgcn_b200.gso import CsrOperator, is_sparse_operator


@pytest.fixture(scope="module")
def L():
    import __graft_entry__ as g
    g.build()
    from stgcn_b200 import _lib
    return _lib


def _random_sparse(n, nnz, seed, symmetric=False):
    rng = np.random.default_rng(seed)
    r, c = rng.integers(0, n, nnz), rng.integers(0, n, nnz)
    v = rng.standard_normal(nnz).astype(np.float32)
    m = sp.coo_matrix((v, (r, c)), shape=(n, n))
    return (m + m.T).tocoo() if symmetric else m


def _dense(m):
    return torch.from_numpy(m.toarray().astype(np.float32))


@pytest.mark.parametrize("fmt", ["scipy_csr", "scipy_coo", "torch_coo", "torch_csr", "dense"])
def test_csr_operator_equals_the_dense_matrix(fmt):
    m = _random_sparse(50, 300, 1)                          # duplicates (summed) and empty rows at this density
    dense = _dense(m)
    src = {"scipy_csr": lambda: m.tocsr(), "scipy_coo": lambda: m,
           "torch_coo": lambda: torch.sparse_coo_tensor(np.vstack([m.row, m.col]), m.data, (50, 50)),
           "torch_csr": lambda: dense.to_sparse_csr(), "dense": lambda: dense}[fmt]()
    op = CsrOperator(src)
    assert op.N == 50 and op.shape == (50, 50) and op.device == torch.device("cpu")
    assert torch.allclose(op.to_dense(), dense, rtol=1e-6, atol=1e-6)
    assert op.row_ptr.dtype == op.col.dtype == torch.int32 and op.val.dtype == torch.float32
    assert int(op.row_ptr[-1]) == op.nnz == op.col.numel()
    for h in range(op.N):                                   # columns sorted within each row, no duplicates
        cols = op.col[op.row_ptr[h]:op.row_ptr[h + 1]]
        assert bool((cols[1:] > cols[:-1]).all())
    assert torch.allclose(op.to_dense(), CsrOperator(op.to_dense()).to_dense())


def test_duplicates_are_summed():
    m = sp.coo_matrix((np.array([1.0, 2.0, 4.0], np.float32), (np.array([0, 0, 1]), np.array([1, 1, 0]))), shape=(3, 3))
    op = CsrOperator(m)
    assert op.nnz == 2
    assert op.to_dense()[0, 1] == 3.0 and op.to_dense()[1, 0] == 4.0
    t = torch.sparse_coo_tensor([[0, 0, 1], [1, 1, 0]], [1.0, 2.0, 4.0], (3, 3))     # uncoalesced torch COO
    assert torch.equal(CsrOperator(t).to_dense(), op.to_dense())


def test_isolated_vertices_have_empty_rows():
    m = sp.coo_matrix((np.ones(2, np.float32), (np.array([1, 3]), np.array([3, 1]))), shape=(6, 6))
    op = CsrOperator(m)
    counts = (op.row_ptr[1:] - op.row_ptr[:-1]).tolist()
    assert counts == [0, 1, 0, 1, 0, 0]
    empty = CsrOperator(sp.csr_matrix((4, 4), dtype=np.float32))
    assert empty.nnz == 0 and empty.row_ptr.tolist() == [0] * 5 and not empty.to_dense().any()


def test_transpose_of_a_non_symmetric_operator():
    m = _random_sparse(40, 200, 2)
    op = CsrOperator(m)
    assert not op.symmetric
    assert op.t_row_ptr.data_ptr() != op.row_ptr.data_ptr()
    rows = torch.repeat_interleave(torch.arange(40), (op.t_row_ptr[1:] - op.t_row_ptr[:-1]).long())
    t = torch.zeros(40, 40)
    t[rows, op.t_col.long()] = op.t_val
    assert torch.equal(t, op.to_dense().T)


def test_symmetric_operator_aliases_its_transpose():
    op = CsrOperator(_random_sparse(40, 200, 3, symmetric=True))
    assert op.symmetric
    for a, b in ((op.row_ptr, op.t_row_ptr), (op.col, op.t_col), (op.val, op.t_val)):
        assert a.data_ptr() == b.data_ptr()
    assert len(op.tensors()) == 3


def test_conversion_errors():
    with pytest.raises(ValueError, match="square"):
        CsrOperator(sp.random(4, 5, density=0.5, format="csr", dtype=np.float32))
    with pytest.raises(ValueError, match="outside"):
        CsrOperator(_out_of_range_coo())
    bad = sp.coo_matrix((np.array([1.0, np.nan], np.float32), (np.array([0, 1]), np.array([1, 0]))), shape=(2, 2))
    with pytest.raises(ValueError, match="non-finite"):
        CsrOperator(bad)
    inf = torch.tensor([[0.0, float("inf")], [1.0, 0.0]])
    with pytest.raises(ValueError, match="non-finite"):
        CsrOperator(inf)
    with pytest.raises(TypeError):
        CsrOperator([[0.0, 1.0], [1.0, 0.0]])


def _out_of_range_coo():
    # torch validates COO indices only on request, so an out-of-range column reaches the converter
    return torch.sparse_coo_tensor(torch.tensor([[0, 1], [1, 7]]), torch.tensor([1.0, 1.0]), (4, 4),
                                   check_invariants=False)


def test_vertex_count_must_match_the_layer():
    from stgcn_b200 import layers
    op = CsrOperator(_random_sparse(20, 60, 4, symmetric=True))
    with pytest.raises(ValueError, match="n_vertex"):
        layers.STConvBlock(3, 3, 21, 1, [8, 4, 8], "glu", "cheb_graph_conv", op, True, 0.0)
    with pytest.raises(ValueError, match="n_vertex"):
        layers.STConvBlock(3, 3, 21, 1, [8, 4, 8], "glu", "graph_conv", _random_sparse(20, 60, 4), True, 0.0)
    blk = layers.STConvBlock(3, 3, 20, 1, [8, 4, 8], "glu", "cheb_graph_conv", op, True, 0.0)
    assert not any("gso" in k for k in blk.state_dict())
    assert is_sparse_operator(op) and is_sparse_operator(sp.eye(3).tocsr())
    assert is_sparse_operator(torch.eye(3).to_sparse()) and not is_sparse_operator(torch.eye(3))


def test_csr_struct_matches_its_ctypes_mirror(L):
    prog = ('#include <stdio.h>\n#include "stgcn_b200.h"\nint main(void){\n'
            'printf("%zu\\n", sizeof(stgcn_csr_gso));\nreturn 0;}\n')
    with tempfile.TemporaryDirectory() as td:
        c = os.path.join(td, "s.c")
        open(c, "w").write(prog)
        exe = os.path.join(td, "s")
        subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe], check=True)
        out = subprocess.run([exe], check=True, capture_output=True, text=True).stdout
    assert C.sizeof(L.CsrGso) == int(out.strip())
    assert C.sizeof(L.CsrGso) == 8 + 6 * C.sizeof(C.c_void_p)


def _fake_op(L, n, nnz=8 * 8192):
    # size queries read shapes only; any non-null address will do for the arrays
    return L.CsrGso(n, nnz, 256, 256, 256, 256, 256, 256)


@pytest.mark.parametrize("prec", ["fp32", "tf32x3", "bf16"])
def test_csr_size_queries_without_gpu(L, prec):
    lib = L.lib()
    n = 8192
    sv, ws, svc, wsc, iw, iwc = (C.c_size_t() for _ in range(6))
    op = _fake_op(L, n)
    st = L.StblockDesc(32, 12, n, 1, 64, 16, 64, 3, 3, 0, 0, 1, 0.0, 1e-12, L.PREC[prec])
    L.check(lib.stgcn_stblock_sizes(C.byref(st), C.byref(sv), C.byref(ws)))
    L.check(lib.stgcn_stblock_sizes_csr(C.byref(st), C.byref(op), C.byref(svc), C.byref(wsc)))
    L.check(lib.stgcn_stblock_infer_sizes(C.byref(st), C.byref(iw)))
    L.check(lib.stgcn_stblock_infer_sizes_csr(C.byref(st), C.byref(op), C.byref(iwc)))
    image = n * ((n + 63) // 64 * 64) * 2                     # the dense bf16 operator image
    assert svc.value > 0 and wsc.value > 0 and iwc.value > 0
    if prec == "bf16":
        assert ws.value - wsc.value >= image, (ws.value, wsc.value)
        assert iw.value - iwc.value >= image
    gd = L.GconvDesc(32, 10, n, 64, 16, 3, 0, 1, 1, L.PREC[prec])
    L.check(lib.stgcn_gconv_sizes(C.byref(gd), C.byref(sv), C.byref(ws)))
    L.check(lib.stgcn_gconv_sizes_csr(C.byref(gd), C.byref(op), C.byref(svc), C.byref(wsc)))
    assert svc.value == sv.value                              # same saved layout: stack planes + output copy
    if prec == "bf16":
        assert ws.value - wsc.value >= image


def test_csr_entry_points_reject_bad_operators_without_gpu(L):
    lib = L.lib()
    sv, ws = C.c_size_t(), C.c_size_t()
    st = L.StblockDesc(4, 12, 100, 1, 8, 4, 8, 3, 3, 0, 0, 0, 0.0, 1e-12, 0)
    gd = L.GconvDesc(4, 10, 100, 4, 4, 3, 0, 0, 1, 0)
    assert lib.stgcn_stblock_sizes_csr(C.byref(st), _fake_op(L, 100, 400), C.byref(sv), C.byref(ws)) == 0
    for op in (L.CsrGso(99, 400, 256, 256, 256, 256, 256, 256),          # N differs from the desc's
               L.CsrGso(100, -1, 256, 256, 256, 256, 256, 256),          # negative nnz
               L.CsrGso(100, 400, 256, None, 256, 256, 256, 256),        # missing columns with nnz > 0
               L.CsrGso(100, 0, None, None, None, None, None, None)):    # missing row offsets
        assert lib.stgcn_stblock_sizes_csr(C.byref(st), C.byref(op), C.byref(sv), C.byref(ws)) == L.E_INVALID
        assert lib.stgcn_gconv_sizes_csr(C.byref(gd), C.byref(op), C.byref(sv), C.byref(ws)) == L.E_INVALID
        assert lib.stgcn_stblock_infer_sizes_csr(C.byref(st), C.byref(op), C.byref(ws)) == L.E_INVALID
    assert b"N" in lib.stgcn_last_error() or b"row offsets" in lib.stgcn_last_error()
    assert lib.stgcn_stblock_sizes_csr(C.byref(st), None, C.byref(sv), C.byref(ws)) == L.E_INVALID
    # a dense gso alongside the CSR operator is rejected before anything is launched
    p = L.StblockParams()
    p.gc.gso = 256
    op = _fake_op(L, 100, 400)
    assert lib.stgcn_stblock_fwd_csr(C.byref(st), 256, C.byref(p), C.byref(op), 256, 256, 256, 1 << 20, 0,
                                     None) == L.E_INVALID
    assert b"dense gso" in lib.stgcn_last_error()
    gp = L.GconvParams(None, None, 256, None, 256)
    assert lib.stgcn_gconv_fwd_csr(C.byref(gd), 256, C.byref(gp), C.byref(op), 256, 256, 256, 1 << 20,
                                   None) == L.E_INVALID
