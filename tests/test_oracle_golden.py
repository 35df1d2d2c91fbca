"""Pins oracle/stgcn_oracle.py against the reference-generated golden vectors (CPU)."""
import json
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, GoldenCase, golden_case_names, rel_l2
from oracle import stgcn_oracle as O

TOL = 2e-5   # fp32 vs fp32 of the same math, different op fusion/order


@pytest.mark.parametrize("name", golden_case_names())
def test_oracle_matches_reference_vectors(name):
    g = GoldenCase(name)
    params = {k: v.clone().requires_grad_(True) for k, v in g.params.items()}
    x = g.x.clone().requires_grad_(True)
    cfg = g.model_cfg()
    out = O.stgcn_forward(x, params, g.gso, **cfg)
    assert tuple(out.shape) == tuple(g.out.shape)          # shape/index work: exact
    assert rel_l2(out, g.out) < TOL
    loss = torch.nn.functional.mse_loss(out.reshape(x.shape[0], -1), g.y)
    assert abs(loss.item() - g.loss) < 1e-5 * max(1.0, abs(g.loss))
    loss.backward()
    assert rel_l2(x.grad, g.dx) < 1e-4
    for k, gref in g.grads.items():
        assert params[k].grad is not None, k
        assert rel_l2(params[k].grad, gref) < 1e-4, k
    # parameters the reference leaves without gradient (dead align convs) stay without one
    for k in params:
        if k not in g.grads:
            assert params[k].grad is None, k
    # first ST block on its own
    c = g.cfg
    b0 = O.st_conv_block(g.x, g.params, "st_blocks.0.", g.gso, c["Kt"], c["blocks"][1], c["act"], c["kind"])
    assert tuple(b0.shape) == tuple(g.block0_out.shape)
    assert rel_l2(b0, g.block0_out) < TOL


def test_oracle_fp64_is_close_to_fp32_reference():
    g = GoldenCase("tiny_cheb3_glu")
    p64 = {k: v.double() for k, v in g.params.items()}
    out = O.stgcn_forward(g.x.double(), p64, g.gso.double(), **g.model_cfg())
    assert rel_l2(out, g.out) < 1e-5


def test_index_work_bit_exact():
    """Slices/pads/permutes on integer-valued tensors must be exact (SURVEY.md §8c)."""
    x = torch.arange(2 * 3 * 5 * 4, dtype=torch.float32).reshape(2, 3, 5, 4)
    a = O.align_channels(x, 7, None, None)
    assert a.shape == (2, 7, 5, 4)
    assert torch.equal(a[:, :3], x) and torch.count_nonzero(a[:, 3:]) == 0
    assert O.align_channels(x, 3, None, None) is x


def test_oracle_errors_match_reference_behaviour():
    x = torch.zeros(1, 2, 4, 3)
    with pytest.raises(NotImplementedError):
        O.temporal_gated_conv(x, {"t.causal_conv.weight": torch.zeros(2, 2, 2, 1), "t.causal_conv.bias": torch.zeros(2)},
                              "t.", 2, 2, "tanh")
    with pytest.raises(ValueError):
        O.cheb_graph_conv(x, torch.eye(3), torch.zeros(0, 2, 2), None)


def test_oracle_matches_reference_forward_n23():
    """The reference's forward of both model classes on default-initialised weights of a fresh seed
    (tests/golden/make_ref_golden.py, ref_forward_n23.npz)."""
    z = np.load(os.path.join(GOLDEN, "ref_forward_n23.npz"))
    gso = torch.from_numpy(z["gso"])
    assert torch.equal(gso, O.synthetic_gso(23, seed=5))
    blocks = json.loads(str(z["blocks"]))
    for kind in ("cheb_graph_conv", "graph_conv"):
        params = {k[len(kind) + 3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith(f"{kind}/p:")}
        x, ref = torch.from_numpy(z[f"{kind}/x"]), torch.from_numpy(z[f"{kind}/out"])
        got = O.stgcn_forward(x, params, gso, blocks=blocks, kt=3, n_his=12, act="glu", kind=kind)
        assert tuple(got.shape) == tuple(ref.shape)
        assert rel_l2(got, ref) < TOL, kind
