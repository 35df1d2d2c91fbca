"""Pins oracle/train_oracle.py (SURVEY.md §8f N2/N3): AdamW against the installed torch.optim.AdamW, Lion and
data_transform against vectors generated from the unmodified reference (tests/golden/make_train_golden.py)."""
import os

import numpy as np
import torch

from conftest import GOLDEN
from oracle import train_oracle as T


def test_adamw_oracle_matches_torch():
    g = torch.Generator().manual_seed(3)
    p = torch.nn.Parameter(torch.randn(1000, generator=g))
    opt = torch.optim.AdamW([p], lr=2e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.05)
    pn, m, v = p.detach().numpy().copy(), np.zeros(1000, np.float32), np.zeros(1000, np.float32)
    for t in range(1, 6):
        gr = torch.randn(1000, generator=g) * (10.0 ** (-(t % 3)))
        p.grad = gr.clone()
        opt.step()
        pn, m, v = T.adamw_step(pn, gr.numpy(), m, v, t, lr=2e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.05)
        assert np.allclose(pn, p.detach().numpy(), rtol=2e-6, atol=1e-7), t
    st = opt.state[p]
    assert np.allclose(m, st["exp_avg"].numpy(), rtol=1e-6, atol=1e-8)
    assert np.allclose(v, st["exp_avg_sq"].numpy(), rtol=1e-6, atol=1e-10)


def test_lion_oracle_matches_reference_golden():
    z = np.load(os.path.join(GOLDEN, "train_lion.npz"))
    p, m = z["p0"].copy(), np.zeros_like(z["p0"])
    for i in range(z["grads"].shape[0]):
        p, m = T.lion_step(p, z["grads"][i], m, lr=float(z["lr"]), betas=(float(z["b1"]), float(z["b2"])),
                           weight_decay=float(z["wd"]))
        assert np.array_equal(p, z["traj"][i]), i            # sign updates: bit exact
    assert np.allclose(m, z["exp_avg"], rtol=1e-6, atol=1e-8)


def test_data_transform_oracle_matches_reference_golden():
    z = np.load(os.path.join(GOLDEN, "train_windows.npz"))
    x, y = T.data_transform(z["data"], int(z["n_his"]), int(z["n_pred"]))
    assert np.array_equal(x, z["x"]) and np.array_equal(y, z["y"])


def test_data_transform_oracle_matches_reference_small_windows():
    """A second window shape (tests/golden/make_ref_golden.py, ref_windows_small.npz)."""
    z = np.load(os.path.join(GOLDEN, "ref_windows_small.npz"))
    assert np.array_equal(z["data"], np.random.default_rng(5).standard_normal((40, 7)))
    x, y = T.data_transform(z["data"], int(z["n_his"]), int(z["n_pred"]))
    assert np.array_equal(x, z["x"]) and np.array_equal(y, z["y"])


def test_gso_oracle_matches_reference_golden():
    """Dense calc_gso / calc_chebynet_gso restatement against the operators the unmodified reference derived
    (tests/golden/make_train_golden.py --gso); also the committed gso_pemsd7m_*.npy the models are benchmarked on."""
    z = np.load(os.path.join(GOLDEN, "train_gso.npz"))
    for name, types in (("pemsd7m", ("sym_norm_lap", "sym_renorm_adj")),
                        ("rand", ("sym_norm_adj", "sym_renorm_adj", "sym_norm_lap", "sym_renorm_lap"))):
        adj = z[f"adj_{name}"].astype(np.float64)
        for t in types:
            g = T.calc_gso_dense(adj, t)
            assert np.allclose(g, z[f"{name}_{t}"], rtol=1e-6, atol=1e-7), (name, t)
            c, lam = T.calc_chebynet_gso_dense(g)
            assert np.allclose(c, z[f"{name}_{t}_cheb"], rtol=1e-5, atol=2e-6), (name, t, lam)
    cheb = np.load(os.path.join(GOLDEN, "gso_pemsd7m_cheb.npy"))
    c, _ = T.calc_chebynet_gso_dense(T.calc_gso_dense(z["adj_pemsd7m"].astype(np.float64), "sym_norm_lap"))
    assert np.allclose(c, cheb, rtol=1e-5, atol=2e-6)
