"""CPU oracle for the callers either side of the ST-block path (SURVEY.md §8f N2, N3).  TEST INFRASTRUCTURE ONLY --
imported by tests/ only; nothing under stgcn_b200/ may import it.

numpy restatements of
  * the AdamW update the reference's default optimizer performs (main.py:147-148 builds torch.optim.AdamW; the
    algorithm is PyTorch's documented one -- third-party, pinned torch~=2.2.0 in requirements.txt:5, 2.11.0 installed),
  * the reference's own Lion optimizer (script/opt.py:34-76),
  * data_transform, the window construction (script/dataloader.py:32-48).
Pinned by tests/test_train_oracle.py: AdamW against the installed torch.optim.AdamW, Lion and data_transform against
vectors generated from the UNMODIFIED reference by tests/golden/make_train_golden.py (tests/golden/train_*.npz) and
tests/golden/make_ref_golden.py (tests/golden/ref_windows_small.npz)."""
from __future__ import annotations

import numpy as np


def adamw_step(p, g, m, v, t, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2):
    """One torch.optim.AdamW step (amsgrad=False, maximize=False) on float32 arrays; t = 1-based step number.
    Returns (p, m, v) updated copies."""
    b1, b2 = betas
    p = p.astype(np.float32) * np.float32(1 - lr * weight_decay)          # decoupled weight decay
    m = (m + (g - m) * np.float32(1 - b1)).astype(np.float32)             # exp_avg.lerp_(grad, 1 - beta1)
    v = (v * np.float32(b2) + (g * g) * np.float32(1 - b2)).astype(np.float32)
    bc1, bc2 = 1 - b1 ** t, 1 - b2 ** t
    denom = np.sqrt(v) / np.float32(np.sqrt(bc2)) + np.float32(eps)
    p = (p - np.float32(lr / bc1) * (m / denom)).astype(np.float32)
    return p, m, v


def lion_step(p, g, m, lr=1e-3, betas=(0.9, 0.99), weight_decay=1e-2):
    """One step of the reference's Lion (opt.py:56-74): decay, sign update from the interpolated momentum, momentum
    decay with the second coefficient.  Returns (p, m)."""
    b1, b2 = betas
    p = p.astype(np.float32) * np.float32(1 - lr * weight_decay)          # opt.py:59
    update = m * np.float32(b1) + g * np.float32(1 - b1)                  # opt.py:70
    p = (p - np.float32(lr) * np.sign(update)).astype(np.float32)         # opt.py:72
    m = (m * np.float32(b2) + g * np.float32(1 - b2)).astype(np.float32)  # opt.py:75
    return p, m


def data_transform(data, n_his, n_pred):
    """x[i, 0] = data[i : i + n_his], y[i] = data[i + n_his + n_pred - 1] for i < len - n_his - n_pred
    (dataloader.py:32-48).  float32 out (the reference converts through torch.Tensor)."""
    n_vertex = data.shape[1]
    num = len(data) - n_his - n_pred
    x = np.zeros([num, 1, n_his, n_vertex], dtype=np.float32)
    y = np.zeros([num, n_vertex], dtype=np.float32)
    for i in range(num):
        x[i, 0] = data[i: i + n_his]
        y[i] = data[i + n_his + n_pred - 1]
    return x, y


# ---- graph shift operator (SURVEY.md §8f N4) -------------------------------------------------------------------------
def calc_gso_dense(dir_adj, gso_type):
    """Dense restatement of calc_gso (script/utility.py:6-57) in float64: symmetrise by elementwise max (:18),
    + I for the *_renorm_* types (:20-22), D^-1/2 A D^-1/2 (:24-32) or D^-1 A (:40-47), Laplacian I - (.) (:33-36, :48-51)."""
    a = np.asarray(dir_adj, dtype=np.float64)
    n = a.shape[0]
    a = np.maximum(a, a.T)
    if "renorm" in gso_type:
        a = a + np.eye(n)
    d = a.sum(axis=1)
    if gso_type.startswith("sym_"):
        with np.errstate(divide="ignore"):
            dis = np.power(d, -0.5)
        dis[np.isinf(dis)] = 0.0
        g = dis[:, None] * a * dis[None, :]
    elif gso_type.startswith("rw_"):
        with np.errstate(divide="ignore"):
            di = np.power(d, -1.0)
        di[np.isinf(di)] = 0.0
        g = di[:, None] * a
    else:
        raise ValueError(f"{gso_type} is not defined.")
    if gso_type.endswith("_lap"):
        g = np.eye(n) - g
    return g


def calc_chebynet_gso_dense(gso):
    """calc_chebynet_gso (script/utility.py:59-76): lambda_max = ||gso||_2 (scipy.sparse.linalg.norm(gso, 2) there);
    gso - I when lambda_max >= 2, else 2 gso / lambda_max - I."""
    g = np.asarray(gso, dtype=np.float64)
    lam = np.linalg.norm(g, 2)
    eye = np.eye(g.shape[0])
    return (g - eye if lam >= 2 else 2 * g / lam - eye), lam
