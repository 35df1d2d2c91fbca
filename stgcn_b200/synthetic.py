"""Synthetic inputs of the BASELINE.json workloads that do not come from a dataset (no network, no dataset files on
the GPU box): the seeded dense operator of the N=2048 roofline sweep (SURVEY.md §8d), seeded sparse k-nearest-neighbour
operators for the CSR path, and default-initialised models."""
from __future__ import annotations

from types import SimpleNamespace

import torch


def knn_operator(n: int, degree: int, seed: int = 0, symmetric: bool = True):
    """Seeded sparse graph shift operator of a k-nearest-neighbour graph, as a scipy CSR float32 matrix: n points
    uniform in the unit square, each joined to its ``degree`` nearest others with Gaussian weights exp(-d^2 / s^2)
    (s = the median neighbour distance).  symmetric: the union graph, D^-1/2 A D^-1/2 (the reference's sym_norm_adj,
    utility.py:21-31), spectrum in [-1, 1]; else the directed graph, D^-1 A (rw_norm_adj, utility.py:33-42)."""
    import numpy as np
    import scipy.sparse as sp
    from scipy.spatial import cKDTree
    rng = np.random.default_rng(seed)
    pts = rng.random((n, 2))
    dist, idx = cKDTree(pts).query(pts, k=degree + 1)
    dist, idx = dist[:, 1:], idx[:, 1:]                        # drop the point itself
    scale = np.median(dist) or 1.0
    w = np.exp(-(dist / scale) ** 2)
    a = sp.csr_matrix((w.reshape(-1), (np.repeat(np.arange(n), degree), idx.reshape(-1))), shape=(n, n))
    if symmetric:
        a = a.maximum(a.T)
        d = np.asarray(a.sum(axis=1)).reshape(-1) ** -0.5
        a = sp.diags(d) @ a @ sp.diags(d)
    else:
        a = sp.diags(1.0 / np.asarray(a.sum(axis=1)).reshape(-1)) @ a
    return sp.csr_matrix(a, dtype=np.float32)


def synthetic_operator(n: int, seed: int = 0, dtype=torch.float32) -> torch.Tensor:
    """Seeded dense symmetric (N, N) operator scaled to spectral norm 1: G = randn, S = (G + G^T) / 2, L = S / ||S||_2
    (the stand-in for a rescaled Laplacian, whose spectrum also lies in [-1, 1]: utility.py:59-76 of the reference)."""
    gen = torch.Generator().manual_seed(seed)
    g = torch.randn(n, n, generator=gen, dtype=torch.float64)
    s = (g + g.T) / 2
    s = s / torch.linalg.matrix_norm(s, ord=2)
    return s.to(dtype)


def build_model(gso: torch.Tensor, kind: str, ks: int, blocks, device, droprate: float = 0.0, seed: int = 0,
                kt: int = 3, n_his: int = 12, act: str = "glu"):
    """The reference's model (models.py:6-103) on this package's layers, default-initialised under ``seed`` the way the
    reference initialises it (kaiming-uniform convolutions and graph weights, unit LayerNorm: layers.py:129-141)."""
    from . import models
    torch.manual_seed(seed)
    args = SimpleNamespace(Kt=kt, Ks=ks, act_func=act, graph_conv_type=kind, gso=gso.to(device), enable_bias=True,
                           droprate=droprate, n_his=n_his)
    cls = models.STGCNChebGraphConv if kind == "cheb_graph_conv" else models.STGCNGraphConv
    return cls(args, blocks, gso.shape[0]).to(device)
