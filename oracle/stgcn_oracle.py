"""CPU oracle for the STGCN ST-block / output-block hot path.  TEST INFRASTRUCTURE ONLY.

This file restates, as plain functions over a flat ``{name: tensor}`` parameter dict,
the arithmetic that hazdzz/STGCN's ``model/layers.py`` performs on the hot path.  It is
imported only by ``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` /
``--impl reference`` legs of ``bench.py``.  Nothing under ``stgcn_b200/`` may import it:
the product path is CUDA-only and fails loudly when the extension is missing.

Parity pinning: the reference ships no golden vectors or tests (SURVEY.md §4, §8c), so
the oracle is pinned against the *reference itself*: ``tests/golden/make_golden.py`` and
``tests/golden/make_ref_golden.py`` import the unmodified reference, run it on seeded
inputs and store inputs/weights/outputs/grads under ``tests/golden/``;
``tests/test_oracle_golden.py`` checks this file against every one of those vectors
(fp32 2e-5 rel), without needing the reference.

All tensors use the reference's layout: activations ``(B, C, T, N)``; every function
works in whatever dtype its inputs carry (fp32 for parity with the reference, fp64 for a
truth value).  Backward comes from torch autograd over these same functions, exactly
as the reference gets its backward (it has no hand-written one).

Each function cites the reference lines (``layers.py:a-b``) it follows.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence

import torch
import torch.nn.functional as F

Tensor = torch.Tensor
Params = Dict[str, Tensor]


# ----------------------------------------------------------------------------------------
# primitive pieces
# ----------------------------------------------------------------------------------------
def align_channels(x: Tensor, c_out: int, w: Optional[Tensor], b: Optional[Tensor]) -> Tensor:
    """Channel adapter (layers.py:14-23): 1x1 conv when shrinking, zero channels appended
    when growing, identity otherwise."""
    c_in = x.shape[1]
    if c_in > c_out:
        return F.conv2d(x, w, b)
    if c_in < c_out:
        bsz, _, t, n = x.shape
        pad = x.new_zeros(bsz, c_out - c_in, t, n)
        return torch.cat((x, pad), dim=1)
    return x


def temporal_gated_conv(x: Tensor, p: Params, prefix: str, kt: int, c_out: int, act: str) -> Tensor:
    """Gated temporal convolution (layers.py:87-120): valid (Kt,1) conv along time
    (layers.py:52-57 with the padding branch dead), residual = channel-aligned input
    cropped to the last T-Kt+1 steps (layers.py:88), then GLU / GTU / relu / silu."""
    res = align_channels(x, c_out, p.get(prefix + "align.align_conv.weight"),
                         p.get(prefix + "align.align_conv.bias"))[:, :, kt - 1:, :]
    z = F.conv2d(x, p[prefix + "causal_conv.weight"], p[prefix + "causal_conv.bias"])
    if act in ("glu", "gtu"):
        lin, gate = z[:, :c_out], z[:, -c_out:]
        if act == "glu":
            return (lin + res) * torch.sigmoid(gate)            # layers.py:105
        return torch.tanh(lin + res) * torch.sigmoid(gate)      # layers.py:109
    if act == "relu":
        return torch.relu(z + res)                              # layers.py:112
    if act == "silu":
        return F.silu(z + res)                                  # layers.py:115
    raise NotImplementedError(f"ERROR: The activation function {act} is not implemented.")


def node_contract(gso: Tensor, x_btnc: Tensor) -> Tensor:
    """out[b,t,h,c] = sum_i gso[h,i] x[b,t,i,c]  ('hi,btij->bthj', layers.py:154)."""
    return torch.einsum("hi,btij->bthj", gso, x_btnc)


def cheb_graph_conv(x: Tensor, gso: Tensor, weight: Tensor, bias: Optional[Tensor]) -> Tensor:
    """Chebyshev graph convolution (layers.py:143-172).  x (B,C,T,N) -> (B,T,N,C_out).
    x_0 = x, x_1 = L x_0, x_k = 2 L x_{k-1} - x_{k-2}; out = sum_k x_k W_k + b."""
    ks = weight.shape[0]
    if ks - 1 < 0:
        raise ValueError(
            f"ERROR: the graph convolution kernel size Ks has to be a positive integer, but received {ks}.")
    h = x.permute(0, 2, 3, 1)
    terms: List[Tensor] = [h]
    if ks >= 2:
        terms.append(node_contract(gso, h))
    for k in range(2, ks):
        terms.append(node_contract(2 * gso, terms[k - 1]) - terms[k - 2])   # layers.py:161
    stacked = torch.stack(terms, dim=2)
    out = torch.einsum("btkhi,kij->bthj", stacked, weight)                   # layers.py:165
    return out if bias is None else out + bias


def first_order_graph_conv(x: Tensor, gso: Tensor, weight: Tensor, bias: Optional[Tensor]) -> Tensor:
    """GCN-style graph convolution (layers.py:194-206): (L x) W + b."""
    h = node_contract(gso, x.permute(0, 2, 3, 1))
    out = torch.einsum("bthi,ij->bthj", h, weight)
    return out if bias is None else out + bias


def graph_conv_layer(x: Tensor, p: Params, prefix: str, gso: Tensor, c_out: int, kind: str) -> Tensor:
    """align -> graph conv -> back to (B,C,T,N) -> + aligned input (layers.py:222-231)."""
    a = align_channels(x, c_out, p.get(prefix + "align.align_conv.weight"),
                       p.get(prefix + "align.align_conv.bias"))
    if kind == "cheb_graph_conv":
        g = cheb_graph_conv(a, gso, p[prefix + "cheb_graph_conv.weight"],
                            p.get(prefix + "cheb_graph_conv.bias"))
    elif kind == "graph_conv":
        g = first_order_graph_conv(a, gso, p[prefix + "graph_conv.weight"],
                                   p.get(prefix + "graph_conv.bias"))
    else:
        raise ValueError(f"unknown graph_conv_type {kind}")
    return g.permute(0, 3, 1, 2) + a


def node_channel_layer_norm(x: Tensor, w: Tensor, b: Tensor, eps: float = 1e-12) -> Tensor:
    """LayerNorm over the joint (N, C) axes of x viewed as (B,T,N,C) (layers.py:246,255);
    returns (B,T,N,C)."""
    h = x.permute(0, 2, 3, 1)
    return F.layer_norm(h, tuple(w.shape), w, b, eps)


def dropout(x: Tensor, p_drop: float, training: bool) -> Tensor:
    return F.dropout(x, p_drop, training)


# ----------------------------------------------------------------------------------------
# blocks
# ----------------------------------------------------------------------------------------
def st_conv_block(x: Tensor, p: Params, prefix: str, gso: Tensor, kt: int, channels: Sequence[int],
                  act: str, kind: str, p_drop: float = 0.0, training: bool = False) -> Tensor:
    """'TGTND' block (layers.py:250-258)."""
    h = temporal_gated_conv(x, p, prefix + "tmp_conv1.", kt, channels[0], act)
    h = graph_conv_layer(h, p, prefix + "graph_conv.", gso, channels[1], kind)
    h = torch.relu(h)
    h = temporal_gated_conv(h, p, prefix + "tmp_conv2.", kt, channels[2], act)
    h = node_channel_layer_norm(h, p[prefix + "tc2_ln.weight"], p[prefix + "tc2_ln.bias"]).permute(0, 3, 1, 2)
    return dropout(h, p_drop, training)


def output_block(x: Tensor, p: Params, prefix: str, ko: int, channels: Sequence[int], act: str,
                 p_drop: float = 0.0, training: bool = False) -> Tensor:
    """'TNFF' block (layers.py:276-284)."""
    h = temporal_gated_conv(x, p, prefix + "tmp_conv1.", ko, channels[0], act)
    h = node_channel_layer_norm(h, p[prefix + "tc1_ln.weight"], p[prefix + "tc1_ln.bias"])
    h = F.linear(h, p[prefix + "fc1.weight"], p.get(prefix + "fc1.bias"))
    h = dropout(torch.relu(h), p_drop, training)
    h = F.linear(h, p[prefix + "fc2.weight"], p.get(prefix + "fc2.bias"))
    return h.permute(0, 3, 1, 2)


def stgcn_forward(x: Tensor, p: Params, gso: Tensor, *, blocks: Sequence[Sequence[int]], kt: int,
                  n_his: int, act: str = "glu", kind: str = "cheb_graph_conv",
                  p_drop: float = 0.0, training: bool = False) -> Tensor:
    """Whole model (models.py:28-53): len(blocks)-3 ST blocks, then the output stage picked
    by Ko = n_his - n_blocks*2*(Kt-1): OutputBlock if Ko>1, two linears if Ko==0, nothing if Ko==1."""
    n_st = len(blocks) - 3
    h = x
    for l in range(n_st):
        h = st_conv_block(h, p, f"st_blocks.{l}.", gso, kt, blocks[l + 1], act, kind, p_drop, training)
    ko = n_his - n_st * 2 * (kt - 1)
    if ko > 1:
        h = output_block(h, p, "output.", ko, blocks[-2], act, p_drop, training)
    elif ko == 0:
        h = F.linear(h.permute(0, 2, 3, 1), p["fc1.weight"], p.get("fc1.bias"))
        h = torch.relu(h)
        h = F.linear(h, p["fc2.weight"], p.get("fc2.bias")).permute(0, 3, 1, 2)
    return h


def mse_step(x: Tensor, y: Tensor, p: Params, gso: Tensor, **cfg) -> Tensor:
    """The training-step body of main.py:166-167: MSE(model(x).view(B,-1), y)."""
    pred = stgcn_forward(x, p, gso, **cfg).reshape(x.shape[0], -1)
    return F.mse_loss(pred, y)


# ----------------------------------------------------------------------------------------
# parameter construction (shapes/names of the reference's state_dict; layers.py:12,80-82,
# 129-141,182-192,246,267-272)
# ----------------------------------------------------------------------------------------
def _kaiming_uniform(shape, fan_in, gen):
    bound = math.sqrt(6.0 / ((1 + 5.0) * fan_in)) if fan_in > 0 else 0.0
    return (torch.rand(shape, generator=gen) * 2 - 1) * bound


def _bias_uniform(shape, fan_in, gen):
    bound = 1.0 / math.sqrt(fan_in) if fan_in > 0 else 0.0
    return (torch.rand(shape, generator=gen) * 2 - 1) * bound


def _tconv_params(p: Params, prefix: str, kt: int, c_in: int, c_out: int, act: str, gen):
    width = 2 * c_out if act in ("glu", "gtu") else c_out
    p[prefix + "align.align_conv.weight"] = _kaiming_uniform((c_out, c_in, 1, 1), c_in, gen)
    p[prefix + "align.align_conv.bias"] = _bias_uniform((c_out,), c_in, gen)
    p[prefix + "causal_conv.weight"] = _kaiming_uniform((width, c_in, kt, 1), c_in * kt, gen)
    p[prefix + "causal_conv.bias"] = _bias_uniform((width,), c_in * kt, gen)


def init_params(*, blocks: Sequence[Sequence[int]], kt: int, ks: int, n_his: int, n_vertex: int,
                act: str = "glu", kind: str = "cheb_graph_conv", bias: bool = True,
                seed: int = 0, dtype=torch.float32) -> Params:
    """A state_dict with the reference's keys and shapes, filled from a seeded generator
    (same distributions as the reference's default init; not the same RNG stream)."""
    gen = torch.Generator().manual_seed(seed)
    p: Params = {}
    n_st = len(blocks) - 3
    for l in range(n_st):
        c_prev = blocks[l][-1]
        c1, c2, c3 = blocks[l + 1]
        pre = f"st_blocks.{l}."
        _tconv_params(p, pre + "tmp_conv1.", kt, c_prev, c1, act, gen)
        p[pre + "graph_conv.align.align_conv.weight"] = _kaiming_uniform((c2, c1, 1, 1), c1, gen)
        p[pre + "graph_conv.align.align_conv.bias"] = _bias_uniform((c2,), c1, gen)
        if kind == "cheb_graph_conv":
            # torch's fan_in for a (Ks, c_in, c_out) tensor is size(1)*receptive = c_in*c_out
            p[pre + "graph_conv.cheb_graph_conv.weight"] = _kaiming_uniform((ks, c2, c2), c2 * c2, gen)
            if bias:
                p[pre + "graph_conv.cheb_graph_conv.bias"] = _bias_uniform((c2,), c2 * c2, gen)
        else:
            p[pre + "graph_conv.graph_conv.weight"] = _kaiming_uniform((c2, c2), c2, gen)
            if bias:
                p[pre + "graph_conv.graph_conv.bias"] = _bias_uniform((c2,), c2, gen)
        _tconv_params(p, pre + "tmp_conv2.", kt, c2, c3, act, gen)
        p[pre + "tc2_ln.weight"] = torch.ones(n_vertex, c3) + 0.1 * torch.randn(n_vertex, c3, generator=gen)
        p[pre + "tc2_ln.bias"] = 0.1 * torch.randn(n_vertex, c3, generator=gen)
    ko = n_his - n_st * 2 * (kt - 1)
    c_last = blocks[-3][-1]
    if ko > 1:
        c0, c1 = blocks[-2]
        _tconv_params(p, "output.tmp_conv1.", ko, c_last, c0, act, gen)
        p["output.fc1.weight"] = _kaiming_uniform((c1, c0), c0, gen)
        p["output.fc2.weight"] = _kaiming_uniform((blocks[-1][0], c1), c1, gen)
        if bias:
            p["output.fc1.bias"] = _bias_uniform((c1,), c0, gen)
            p["output.fc2.bias"] = _bias_uniform((blocks[-1][0],), c1, gen)
        p["output.tc1_ln.weight"] = torch.ones(n_vertex, c0) + 0.1 * torch.randn(n_vertex, c0, generator=gen)
        p["output.tc1_ln.bias"] = 0.1 * torch.randn(n_vertex, c0, generator=gen)
    elif ko == 0:
        c0 = blocks[-2][0]
        p["fc1.weight"] = _kaiming_uniform((c0, c_last), c_last, gen)
        p["fc2.weight"] = _kaiming_uniform((blocks[-1][0], c0), c0, gen)
        if bias:
            p["fc1.bias"] = _bias_uniform((c0,), c_last, gen)
            p["fc2.bias"] = _bias_uniform((blocks[-1][0],), c0, gen)
    return {k: v.to(dtype) for k, v in p.items()}


def synthetic_gso(n: int, seed: int = 0, dtype=torch.float32) -> Tensor:
    """Seeded dense symmetric operator with spectral norm 1 (SURVEY.md §8d, N=2048 sweep)."""
    gen = torch.Generator().manual_seed(seed)
    g = torch.randn(n, n, generator=gen, dtype=torch.float64)
    s = (g + g.T) / 2
    s = s / torch.linalg.matrix_norm(s, ord=2)
    return s.to(dtype)
