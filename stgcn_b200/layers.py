"""Drop-in replacement for hazdzz/STGCN ``model/layers.py`` backed by libstgcn_b200.so.

Same class names, constructor signatures, submodule/parameter names (hence the same
``state_dict`` keys and shapes) and forward semantics as the reference, so the reference's
``model/models.py`` and ``main.py`` load it unchanged (INTEGRATION.md).  Every ``forward``
enqueues hand-written sm_100a CUDA kernels through the C ABI of ``include/stgcn_b200.h``;
there is no PyTorch-op or CPU fallback -- a non-CUDA input raises.

Reference map (``/root/reference/model/layers.py``):
  Align :7-23, CausalConv1d :25-38, CausalConv2d :40-57, TemporalConvLayer :59-120,
  ChebGraphConv :122-172, GraphConv :174-206, GraphConvLayer :208-231,
  STConvBlock :233-258, OutputBlock :260-284.

Tensor layout: module inputs/outputs are ``(B, C, T, N)`` tensors exactly as in the
reference.  Internally activations are channels-last ``(B, T, N, C)`` buffers; an output is
returned as the ``permute(0, 3, 1, 2)`` view of such a buffer (which is also what the
reference's STConvBlock returns, layers.py:255), so chaining blocks never copies.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Dict, Optional, Tuple

import torch
import torch.distributed
import torch.nn as nn
import torch.nn.init as init

from . import _lib as L
from . import gso as G

__all__ = ["Align", "CausalConv1d", "CausalConv2d", "TemporalConvLayer", "ChebGraphConv", "GraphConv",
           "GraphConvLayer", "STConvBlock", "OutputBlock", "set_precision", "get_precision"]

_PRECISION = "fp32"


def set_precision(mode: str) -> None:
    """'fp32': CUDA-core fp32 parity path (<=1e-3 rel of the reference).  'tf32x3': the same fp32 chain with every GEMM
    on tcgen05 (3xTF32 operand splitting, fp32 accumulate) -- the parity gate on the tensor cores.  'bf16': bf16 storage,
    fused tcgen05 kernels (throughput mode)."""
    global _PRECISION
    if mode not in L.PREC:
        raise ValueError(f"precision must be one of {sorted(L.PREC)}")
    _PRECISION = mode


def get_precision() -> str:
    return _PRECISION


# ----------------------------------------------------------------------------------------------
# plumbing: device buffers, pointers, seeds
# ----------------------------------------------------------------------------------------------
_WORKSPACES: Dict[Tuple[int, int], torch.Tensor] = {}
_SEED_COUNTER = 0


def _workspace(device: torch.device, nbytes: int) -> torch.Tensor:
    """Scratch shared by all calls on one (device, stream): calls are stream-ordered."""
    key = (device.index or 0, torch.cuda.current_stream(device).cuda_stream)
    buf = _WORKSPACES.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device)
        _WORKSPACES[key] = buf
    return buf


def _mix64(z: int) -> int:
    """splitmix64 finaliser (the same mixing the kernels apply per element)."""
    z &= 0xFFFFFFFFFFFFFFFF
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & 0xFFFFFFFFFFFFFFFF
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & 0xFFFFFFFFFFFFFFFF
    return z ^ (z >> 31)


def _next_seed() -> int:
    """Seed of one dropout call: (torch seed, data-parallel rank, call counter) hashed, so ranks that set the same manual
    seed (as the reference's set_env does, main.py:27-36) still draw different masks for their shards and successive
    layers / steps are decorrelated.  Under CUDA-graph replay the by-value seed is frozen at capture; graph.GraphedStep
    registers a device-side step counter that the kernels add (stgcn_set_dropout_step)."""
    global _SEED_COUNTER
    _SEED_COUNTER += 1
    rank = 0
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        rank = torch.distributed.get_rank()
    return _mix64(_mix64(torch.initial_seed() + 0x9E3779B97F4A7C15 * (rank + 1)) + 0xD1B54A32D192ED03 * _SEED_COUNTER)


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _stream(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _act_dtype() -> torch.dtype:
    """Storage type of activations crossing the C ABI in the current precision mode."""
    return torch.bfloat16 if _PRECISION == "bf16" else torch.float32


def _require_cuda(x: torch.Tensor, what: str) -> None:
    if not x.is_cuda:
        raise RuntimeError(f"stgcn_b200.{what}: expected a CUDA tensor (this framework has no CPU path), got {x.device}")
    if x.dtype not in (torch.float32, _act_dtype()):
        raise RuntimeError(f"stgcn_b200.{what}: expected float32 (or {_act_dtype()}) input, got {x.dtype}")
    if x.dim() != 4:
        raise RuntimeError(f"stgcn_b200.{what}: expected a 4-D (B, C, T, N) tensor, got shape {tuple(x.shape)}")


def _channels_last(x: torch.Tensor) -> torch.Tensor:
    """(B,C,T,N) tensor -> contiguous (B,T,N,C) buffer in the activation dtype of the current precision mode
    (no copy if x already is a permuted view of such a buffer)."""
    return x.permute(0, 2, 3, 1).to(_act_dtype()).contiguous()


def _as_bctn(y_cl: torch.Tensor) -> torch.Tensor:
    return y_cl.permute(0, 3, 1, 2)


def _f32c(t: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    if t is None:
        return None
    if t.dtype != torch.float32 or not t.is_cuda:
        raise RuntimeError("stgcn_b200: parameters must be float32 CUDA tensors (call .to('cuda'))")
    return t.contiguous()


def _sizes(fn, desc, op: Optional[G.CsrOperator] = None) -> Tuple[int, int]:
    """(saved, workspace) bytes from a *_sizes entry point, or from its *_csr twin when a sparse operator is given."""
    sv, ws = C.c_size_t(0), C.c_size_t(0)
    if op is None:
        L.check(fn(C.byref(desc), C.byref(sv), C.byref(ws)))
    else:
        L.check(fn(C.byref(desc), C.byref(op.c_struct()), C.byref(sv), C.byref(ws)))
    return int(sv.value), int(ws.value)


def _sparse(gso) -> Optional[G.CsrOperator]:
    """The CSR operator when ``gso`` takes the sparse path (the *_csr entry points), else None (dense gso pointer)."""
    return gso if isinstance(gso, G.CsrOperator) else None


def _dense_ptr(gso) -> Optional[int]:
    return None if isinstance(gso, G.CsrOperator) else _ptr(gso)


def _grad_like(p: Optional[torch.Tensor], needed: bool) -> Optional[torch.Tensor]:
    """Buffer the backward kernels write a parameter gradient into.  When the parameter is bound to a flat gradient
    buffer (dist.FlatGradAllReducer.bind) and holds no gradient yet, that is a fresh view of its slot: autograd adopts
    it as ``p.grad`` without a copy, so the data-parallel all-reduce runs on the flat buffer with no pack/unpack."""
    if p is None or not needed:
        return None
    slot = getattr(p, "_stgcn_grad_slot", None)
    if slot is not None and p.grad is None:
        flat, off, n = slot
        return flat.narrow(0, off, n).view_as(p)
    return torch.empty_like(p)


# ----------------------------------------------------------------------------------------------
# autograd functions (one C-ABI call each way)
# ----------------------------------------------------------------------------------------------
class _TconvFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x_cl, dims, conv_w, conv_b, align_w, align_b):
        B, T, N, c_in, c_out, Kt, act = dims
        lib = L.lib()
        desc = L.TconvDesc(B, T, N, c_in, c_out, Kt, act, L.PREC[_PRECISION])
        sv_bytes, ws_bytes = _sizes(lib.stgcn_tconv_sizes, desc)
        dev = x_cl.device
        saved = torch.empty(sv_bytes, dtype=torch.uint8, device=dev)
        ws = _workspace(dev, ws_bytes)
        y = torch.empty((B, T - Kt + 1, N, c_out), dtype=x_cl.dtype, device=dev)
        params = L.TconvParams(_ptr(conv_w), _ptr(conv_b), _ptr(align_w), _ptr(align_b))
        with torch.cuda.device(dev):      # kernels, helper streams and events follow the CUDA current device
            L.check(lib.stgcn_tconv_fwd(C.byref(desc), x_cl.data_ptr(), C.byref(params), y.data_ptr(), saved.data_ptr(),
                                        ws.data_ptr(), ws.numel(), _stream(dev)))
        ctx.desc = desc
        ctx.save_for_backward(x_cl, saved, conv_w, conv_b, align_w, align_b)
        return y

    @staticmethod
    def backward(ctx, dy):
        x_cl, saved, conv_w, conv_b, align_w, align_b = ctx.saved_tensors
        lib = L.lib()
        dev = x_cl.device
        need = ctx.needs_input_grad
        dx = torch.empty_like(x_cl) if need[0] else None
        g = [_grad_like(conv_w, need[2]), _grad_like(conv_b, need[3]), _grad_like(align_w, need[4]),
             _grad_like(align_b, need[5])]
        _, ws_bytes = _sizes(lib.stgcn_tconv_sizes, ctx.desc)
        ws = _workspace(dev, ws_bytes)
        params = L.TconvParams(_ptr(conv_w), _ptr(conv_b), _ptr(align_w), _ptr(align_b))
        grads = L.TconvGrads(*[_ptr(t) for t in g])
        dy = dy.to(x_cl.dtype).contiguous()
        with torch.cuda.device(dev):      # kernels, helper streams and events follow the CUDA current device
            L.check(lib.stgcn_tconv_bwd(C.byref(ctx.desc), x_cl.data_ptr(), saved.data_ptr(), dy.data_ptr(),
                                        C.byref(params), C.byref(grads), _ptr(dx), ws.data_ptr(), ws.numel(), _stream(dev)))
        return (dx, None, *g)


class _GconvFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x_cl, dims, gso, align_w, align_b, w, b):
        B, T, N, c_in, c_out, Ks, gconv, relu, residual = dims
        lib = L.lib()
        desc = L.GconvDesc(B, T, N, c_in, c_out, Ks, gconv, relu, residual, L.PREC[_PRECISION])
        op = _sparse(gso)
        sv_bytes, ws_bytes = _sizes(lib.stgcn_gconv_sizes_csr if op else lib.stgcn_gconv_sizes, desc, op)
        dev = x_cl.device
        saved = torch.empty(sv_bytes, dtype=torch.uint8, device=dev)
        ws = _workspace(dev, ws_bytes)
        y = torch.empty((B, T, N, c_out), dtype=x_cl.dtype, device=dev)
        params = L.GconvParams(_ptr(align_w), _ptr(align_b), _ptr(w), _ptr(b), _dense_ptr(gso))
        with torch.cuda.device(dev):      # kernels, helper streams and events follow the CUDA current device
            if op is None:
                L.check(lib.stgcn_gconv_fwd(C.byref(desc), x_cl.data_ptr(), C.byref(params), y.data_ptr(),
                                            saved.data_ptr(), ws.data_ptr(), ws.numel(), _stream(dev)))
            else:
                L.check(lib.stgcn_gconv_fwd_csr(C.byref(desc), x_cl.data_ptr(), C.byref(params), C.byref(op.c_struct()),
                                                y.data_ptr(), saved.data_ptr(), ws.data_ptr(), ws.numel(), _stream(dev)))
        ctx.desc, ctx.op = desc, op
        ctx.save_for_backward(x_cl, saved, None if op else gso, align_w, align_b, w, b)
        return y

    @staticmethod
    def backward(ctx, dy):
        x_cl, saved, gso, align_w, align_b, w, b = ctx.saved_tensors
        lib = L.lib()
        dev = x_cl.device
        need = ctx.needs_input_grad
        dx = torch.empty_like(x_cl) if need[0] else None
        g = [_grad_like(align_w, need[3]), _grad_like(align_b, need[4]), _grad_like(w, need[5]), _grad_like(b, need[6])]
        op = ctx.op
        _, ws_bytes = _sizes(lib.stgcn_gconv_sizes_csr if op else lib.stgcn_gconv_sizes, ctx.desc, op)
        ws = _workspace(dev, ws_bytes)
        params = L.GconvParams(_ptr(align_w), _ptr(align_b), _ptr(w), _ptr(b), _ptr(gso))
        grads = L.GconvGrads(*[_ptr(t) for t in g])
        dy = dy.to(x_cl.dtype).contiguous()
        with torch.cuda.device(dev):      # kernels, helper streams and events follow the CUDA current device
            if op is None:
                L.check(lib.stgcn_gconv_bwd(C.byref(ctx.desc), x_cl.data_ptr(), saved.data_ptr(), dy.data_ptr(),
                                            C.byref(params), C.byref(grads), _ptr(dx), ws.data_ptr(), ws.numel(),
                                            _stream(dev)))
            else:
                L.check(lib.stgcn_gconv_bwd_csr(C.byref(ctx.desc), x_cl.data_ptr(), saved.data_ptr(), dy.data_ptr(),
                                                C.byref(params), C.byref(op.c_struct()), C.byref(grads), _ptr(dx),
                                                ws.data_ptr(), ws.numel(), _stream(dev)))
        return (dx, None, None, *g)


class _LnormFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x_cl, dims, w, b):
        B, T, N, Cc, training, p_drop, eps = dims
        lib = L.lib()
        desc = L.LnormDesc(B, T, N, Cc, int(training), float(p_drop), float(eps), L.PREC[_PRECISION])
        sv_bytes, _ = _sizes(lib.stgcn_lnorm_sizes, desc)
        dev = x_cl.device
        saved = torch.empty(sv_bytes, dtype=torch.uint8, device=dev)
        y = torch.empty_like(x_cl)
        seed = _next_seed() if (training and p_drop > 0) else 0
        with torch.cuda.device(dev):      # kernels, helper streams and events follow the CUDA current device
            L.check(lib.stgcn_lnorm_fwd(C.byref(desc), x_cl.data_ptr(), w.data_ptr(), b.data_ptr(), y.data_ptr(),
                                        saved.data_ptr(), seed, _stream(dev)))
        ctx.desc, ctx.seed = desc, seed
        ctx.save_for_backward(x_cl, saved, w)
        return y

    @staticmethod
    def backward(ctx, dy):
        x_cl, saved, w = ctx.saved_tensors
        lib = L.lib()
        dev = x_cl.device
        need = ctx.needs_input_grad
        dx = torch.empty_like(x_cl) if need[0] else None
        dw = torch.empty_like(w) if need[2] else None
        db = torch.empty_like(w) if need[3] else None
        dy = dy.to(x_cl.dtype).contiguous()
        with torch.cuda.device(dev):      # kernels, helper streams and events follow the CUDA current device
            L.check(lib.stgcn_lnorm_bwd(C.byref(ctx.desc), x_cl.data_ptr(), saved.data_ptr(), dy.data_ptr(), w.data_ptr(),
                                        _ptr(dw), _ptr(db), _ptr(dx), None, 0, ctx.seed, _stream(dev)))
        return dx, None, dw, db


def _tconv_param_tuple(layer: "TemporalConvLayer"):
    """(conv_w, conv_b, align_w, align_b) with the align conv only when it is live (c_in > c_out)."""
    live = layer.c_in > layer.c_out
    return (_f32c(layer.causal_conv.weight), _f32c(layer.causal_conv.bias),
            _f32c(layer.align.align_conv.weight) if live else None,
            _f32c(layer.align.align_conv.bias) if live else None)


class _STBlockFn(torch.autograd.Function):
    """STConvBlock.forward/backward as one C-ABI call each (layers.py:250-258)."""

    @staticmethod
    def forward(ctx, x_cl, dims, gso, *params):
        (B, T, N, c_in, c1, c2, c3, Kt, Ks, act, gconv, training, p_drop, eps) = dims
        lib = L.lib()
        desc = L.StblockDesc(B, T, N, c_in, c1, c2, c3, Kt, Ks, act, gconv, int(training), float(p_drop), float(eps),
                             L.PREC[_PRECISION])
        op = _sparse(gso)
        sv_bytes, ws_bytes = _sizes(lib.stgcn_stblock_sizes_csr if op else lib.stgcn_stblock_sizes, desc, op)
        dev = x_cl.device
        saved = torch.empty(sv_bytes, dtype=torch.uint8, device=dev)
        ws = _workspace(dev, ws_bytes)
        y = torch.empty((B, T - 2 * (Kt - 1), N, c3), dtype=x_cl.dtype, device=dev)
        seed = _next_seed() if (training and p_drop > 0) else 0
        cparams = _STBlockFn._pack(params, gso)
        with torch.cuda.device(dev):      # kernels, helper streams and events follow the CUDA current device
            if op is None:
                L.check(lib.stgcn_stblock_fwd(C.byref(desc), x_cl.data_ptr(), C.byref(cparams), y.data_ptr(),
                                              saved.data_ptr(), ws.data_ptr(), ws.numel(), seed, _stream(dev)))
            else:
                L.check(lib.stgcn_stblock_fwd_csr(C.byref(desc), x_cl.data_ptr(), C.byref(cparams),
                                                  C.byref(op.c_struct()), y.data_ptr(), saved.data_ptr(), ws.data_ptr(),
                                                  ws.numel(), seed, _stream(dev)))
        ctx.desc, ctx.seed, ctx.ws_bytes, ctx.op = desc, seed, ws_bytes, op
        ctx.save_for_backward(x_cl, saved, None if op else gso, *params)
        return y

    @staticmethod
    def _pack(p, gso):
        (t1w, t1b, t1aw, t1ab, gaw, gab, gw, gb, t2w, t2b, t2aw, t2ab, lw, lb) = p
        return L.StblockParams(L.TconvParams(_ptr(t1w), _ptr(t1b), _ptr(t1aw), _ptr(t1ab)),
                               L.GconvParams(_ptr(gaw), _ptr(gab), _ptr(gw), _ptr(gb), _dense_ptr(gso)),
                               L.TconvParams(_ptr(t2w), _ptr(t2b), _ptr(t2aw), _ptr(t2ab)), _ptr(lw), _ptr(lb))

    @staticmethod
    def backward(ctx, dy):
        x_cl, saved, gso, *params = ctx.saved_tensors
        lib = L.lib()
        dev = x_cl.device
        need = ctx.needs_input_grad
        dx = torch.empty_like(x_cl) if need[0] else None
        g = [_grad_like(p, need[3 + i]) for i, p in enumerate(params)]
        ws = _workspace(dev, ctx.ws_bytes)
        gp = [_ptr(t) for t in g]
        grads = L.StblockGrads(L.TconvGrads(*gp[0:4]), L.GconvGrads(*gp[4:8]), L.TconvGrads(*gp[8:12]), gp[12], gp[13])
        op = ctx.op
        cparams = _STBlockFn._pack(params, gso)
        dy = dy.to(x_cl.dtype).contiguous()
        with torch.cuda.device(dev):      # kernels, helper streams and events follow the CUDA current device
            if op is None:
                L.check(lib.stgcn_stblock_bwd(C.byref(ctx.desc), x_cl.data_ptr(), saved.data_ptr(), dy.data_ptr(),
                                              C.byref(cparams), C.byref(grads), _ptr(dx), ws.data_ptr(), ws.numel(),
                                              ctx.seed, _stream(dev)))
            else:
                L.check(lib.stgcn_stblock_bwd_csr(C.byref(ctx.desc), x_cl.data_ptr(), saved.data_ptr(), dy.data_ptr(),
                                                  C.byref(cparams), C.byref(op.c_struct()), C.byref(grads), _ptr(dx),
                                                  ws.data_ptr(), ws.numel(), ctx.seed, _stream(dev)))
        return (dx, None, None, *g)


class _OutBlockFn(torch.autograd.Function):
    """OutputBlock.forward/backward as one C-ABI call each (layers.py:276-284)."""

    @staticmethod
    def forward(ctx, x_cl, dims, *params):
        (B, T, N, c_in, c0, c1, c_end, Ko, act, training, p_drop, eps) = dims
        lib = L.lib()
        desc = L.OutblockDesc(B, T, N, c_in, c0, c1, c_end, Ko, act, int(training), float(p_drop), float(eps),
                              L.PREC[_PRECISION])
        sv_bytes, ws_bytes = _sizes(lib.stgcn_outblock_sizes, desc)
        dev = x_cl.device
        saved = torch.empty(sv_bytes, dtype=torch.uint8, device=dev)
        ws = _workspace(dev, ws_bytes)
        y = torch.empty((B, T - Ko + 1, N, c_end), dtype=torch.float32, device=dev)
        seed = _next_seed() if (training and p_drop > 0) else 0
        cparams = _OutBlockFn._pack(params)
        with torch.cuda.device(dev):      # kernels, helper streams and events follow the CUDA current device
            L.check(lib.stgcn_outblock_fwd(C.byref(desc), x_cl.data_ptr(), C.byref(cparams), y.data_ptr(), saved.data_ptr(),
                                           ws.data_ptr(), ws.numel(), seed, _stream(dev)))
        ctx.desc, ctx.seed, ctx.ws_bytes = desc, seed, ws_bytes
        ctx.save_for_backward(x_cl, saved, *params)
        return y

    @staticmethod
    def _pack(p):
        (tw, tb, taw, tab, lw, lb, f1w, f1b, f2w, f2b) = p
        return L.OutblockParams(L.TconvParams(_ptr(tw), _ptr(tb), _ptr(taw), _ptr(tab)), _ptr(lw), _ptr(lb),
                                _ptr(f1w), _ptr(f1b), _ptr(f2w), _ptr(f2b))

    @staticmethod
    def backward(ctx, dy):
        x_cl, saved, *params = ctx.saved_tensors
        lib = L.lib()
        dev = x_cl.device
        need = ctx.needs_input_grad
        dx = torch.empty_like(x_cl) if need[0] else None
        g = [_grad_like(p, need[2 + i]) for i, p in enumerate(params)]
        ws = _workspace(dev, ctx.ws_bytes)
        gp = [_ptr(t) for t in g]
        grads = L.OutblockGrads(L.TconvGrads(*gp[0:4]), *gp[4:10])
        cparams = _OutBlockFn._pack(params)
        dy = dy.float().contiguous()
        with torch.cuda.device(dev):      # kernels, helper streams and events follow the CUDA current device
            L.check(lib.stgcn_outblock_bwd(C.byref(ctx.desc), x_cl.data_ptr(), saved.data_ptr(), dy.data_ptr(),
                                           C.byref(cparams), C.byref(grads), _ptr(dx), ws.data_ptr(), ws.numel(), ctx.seed,
                                           _stream(dev)))
        return (dx, None, *g)


# ----------------------------------------------------------------------------------------------
# inference (no autograd node, no backward state: stgcn_*_infer)
# ----------------------------------------------------------------------------------------------
def _no_backward(x: torch.Tensor, params) -> bool:
    """True when autograd will never ask for this block's backward: grad mode is off (torch.no_grad(), inference_mode(),
    evaluate_model / evaluate_metric) or neither the input nor any parameter requires grad."""
    if not torch.is_grad_enabled():
        return True
    return not (x.requires_grad or any(p is not None and p.requires_grad for p in params))


def _stblock_infer(x_cl, dims, gso, params):
    """STConvBlock forward through stgcn_stblock_infer: the result of _STBlockFn.forward, bit for bit, without the
    saved buffer; same workspace cache and dropout-seed rule."""
    (B, T, N, c_in, c1, c2, c3, Kt, Ks, act, gconv, training, p_drop, eps) = dims
    lib = L.lib()
    desc = L.StblockDesc(B, T, N, c_in, c1, c2, c3, Kt, Ks, act, gconv, int(training), float(p_drop), float(eps),
                         L.PREC[_PRECISION])
    ws_bytes = C.c_size_t(0)
    op = _sparse(gso)
    if op is None:
        L.check(lib.stgcn_stblock_infer_sizes(C.byref(desc), C.byref(ws_bytes)))
    else:
        L.check(lib.stgcn_stblock_infer_sizes_csr(C.byref(desc), C.byref(op.c_struct()), C.byref(ws_bytes)))
    dev = x_cl.device
    ws = _workspace(dev, int(ws_bytes.value))
    y = torch.empty((B, T - 2 * (Kt - 1), N, c3), dtype=x_cl.dtype, device=dev)
    seed = _next_seed() if (training and p_drop > 0) else 0
    cparams = _STBlockFn._pack(params, gso)
    with torch.cuda.device(dev):      # kernels, helper streams and events follow the CUDA current device
        if op is None:
            L.check(lib.stgcn_stblock_infer(C.byref(desc), x_cl.data_ptr(), C.byref(cparams), y.data_ptr(),
                                            ws.data_ptr(), ws.numel(), seed, _stream(dev)))
        else:
            L.check(lib.stgcn_stblock_infer_csr(C.byref(desc), x_cl.data_ptr(), C.byref(cparams), C.byref(op.c_struct()),
                                                y.data_ptr(), ws.data_ptr(), ws.numel(), seed, _stream(dev)))
    return y


def _outblock_infer(x_cl, dims, params):
    """OutputBlock forward through stgcn_outblock_infer (see _stblock_infer)."""
    (B, T, N, c_in, c0, c1, c_end, Ko, act, training, p_drop, eps) = dims
    lib = L.lib()
    desc = L.OutblockDesc(B, T, N, c_in, c0, c1, c_end, Ko, act, int(training), float(p_drop), float(eps),
                          L.PREC[_PRECISION])
    ws_bytes = C.c_size_t(0)
    L.check(lib.stgcn_outblock_infer_sizes(C.byref(desc), C.byref(ws_bytes)))
    dev = x_cl.device
    ws = _workspace(dev, int(ws_bytes.value))
    y = torch.empty((B, T - Ko + 1, N, c_end), dtype=torch.float32, device=dev)
    seed = _next_seed() if (training and p_drop > 0) else 0
    cparams = _OutBlockFn._pack(params)
    with torch.cuda.device(dev):      # kernels, helper streams and events follow the CUDA current device
        L.check(lib.stgcn_outblock_infer(C.byref(desc), x_cl.data_ptr(), C.byref(cparams), y.data_ptr(), ws.data_ptr(),
                                         ws.numel(), seed, _stream(dev)))
    return y


# ----------------------------------------------------------------------------------------------
# modules (names, ctor signatures and parameter names of the reference)
# ----------------------------------------------------------------------------------------------
def _act_code(act_func: str) -> int:
    if act_func not in ("glu", "gtu", "relu", "silu"):
        raise NotImplementedError(f"ERROR: The activation function {act_func} is not implemented.")   # layers.py:118
    return L.ACT[act_func]


class Align(nn.Module):
    """Channel adapter (layers.py:7-23).  ``align_conv`` always exists (dead when c_in <= c_out), as in the
    reference, so state_dict keys match."""

    def __init__(self, c_in, c_out):
        super().__init__()
        self.c_in = c_in
        self.c_out = c_out
        self.align_conv = nn.Conv2d(in_channels=c_in, out_channels=c_out, kernel_size=(1, 1))

    def forward(self, x):
        _require_cuda(x, "Align")
        if self.c_in > self.c_out:
            B, _, T, N = x.shape
            dims = (B, T, N, self.c_in, self.c_out, 1, L.ACT["linear"])
            y = _TconvFn.apply(_channels_last(x), dims, _f32c(self.align_conv.weight), _f32c(self.align_conv.bias),
                               None, None)
            return _as_bctn(y)
        if self.c_in < self.c_out:
            B, _, T, N = x.shape                       # pure index work: zero channels appended (layers.py:17-19)
            out = x.new_zeros(B, self.c_out, T, N)
            out[:, : self.c_in] = x
            return out
        return x


class CausalConv1d(nn.Conv1d):
    """Present in the reference (layers.py:25-38) but never called by it; kept importable only."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, enable_padding=False, dilation=1, groups=1,
                 bias=True):
        self._causal_padding = (kernel_size - 1) * dilation if enable_padding else 0
        super().__init__(in_channels, out_channels, kernel_size=kernel_size, stride=stride,
                         padding=self._causal_padding, dilation=dilation, groups=groups, bias=bias)

    def forward(self, input):
        raise NotImplementedError("CausalConv1d is dead code in the reference (no call site) and is outside the "
                                  "B200 hot path; only the class name is provided")


class CausalConv2d(nn.Conv2d):
    """(Kt,1) temporal convolution holder (layers.py:40-57).  The reference always builds it with
    enable_padding=False, i.e. a plain valid convolution along time; that is what the kernels implement."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, enable_padding=False, dilation=1, groups=1,
                 bias=True):
        kernel_size = nn.modules.utils._pair(kernel_size)
        stride = nn.modules.utils._pair(stride)
        dilation = nn.modules.utils._pair(dilation)
        self._enable_padding = bool(enable_padding)
        super().__init__(in_channels, out_channels, kernel_size, stride=stride, padding=0, dilation=dilation,
                         groups=groups, bias=bias)

    def forward(self, input):
        _require_cuda(input, "CausalConv2d")
        if (self._enable_padding or self.kernel_size[1] != 1 or self.stride != (1, 1) or self.dilation != (1, 1)
                or self.groups != 1 or self.bias is None):
            raise NotImplementedError("CausalConv2d: only the configuration the reference uses is implemented "
                                      "(kernel (Kt,1), no padding, stride/dilation/groups 1, bias)")
        B, _, T, N = input.shape
        dims = (B, T, N, self.in_channels, self.out_channels, self.kernel_size[0], L.ACT["linear"])
        y = _TconvFn.apply(_channels_last(input), dims, _f32c(self.weight), _f32c(self.bias), None, None)
        return _as_bctn(y)


class TemporalConvLayer(nn.Module):
    """Gated temporal convolution (layers.py:59-120): x (B,c_in,T,N) -> (B,c_out,T-Kt+1,N)."""

    def __init__(self, Kt, c_in, c_out, n_vertex, act_func):
        super().__init__()
        self.Kt = Kt
        self.c_in = c_in
        self.c_out = c_out
        self.n_vertex = n_vertex
        self.align = Align(c_in, c_out)
        width = 2 * c_out if act_func in ("glu", "gtu") else c_out
        self.causal_conv = CausalConv2d(in_channels=c_in, out_channels=width, kernel_size=(Kt, 1),
                                        enable_padding=False, dilation=1)
        self.relu = nn.ReLU()
        self.silu = nn.SiLU()
        self.act_func = act_func

    def forward(self, x):
        _require_cuda(x, "TemporalConvLayer")
        act = _act_code(self.act_func)
        B, _, T, N = x.shape
        dims = (B, T, N, self.c_in, self.c_out, self.Kt, act)
        return _as_bctn(_TconvFn.apply(_channels_last(x), dims, *_tconv_param_tuple(self)))


def _reset_graph_params(weight, bias):
    init.kaiming_uniform_(weight, a=math.sqrt(5))                     # layers.py:136-141 / 186-192
    if bias is not None:
        fan_in, _ = init._calculate_fan_in_and_fan_out(weight)
        bound = 1 / math.sqrt(fan_in) if fan_in > 0 else 0
        init.uniform_(bias, -bound, bound)


def _gso_device(gso, like: torch.Tensor):
    """The operator a forward on ``like`` (B, C, T, N) uses: a dense tensor on its device, or -- for a CsrOperator, a
    torch sparse tensor or a scipy sparse matrix -- a CsrOperator there (converted once; the caller keeps the result)."""
    if G.is_sparse_operator(gso):
        op = G.as_operator(gso, like.device)
        if op.N != like.shape[-1]:
            raise ValueError(f"gso: a ({op.N}, {op.N}) operator for an input with {like.shape[-1]} vertices")
        return op
    if not torch.is_tensor(gso):
        raise TypeError("gso must be a dense torch tensor (N, N) or a sparse operator (stgcn_b200.gso.CsrOperator, "
                        "a torch sparse COO / CSR tensor or a scipy sparse matrix)")
    if gso.device != like.device or gso.dtype != torch.float32 or not gso.is_contiguous():
        gso = gso.to(device=like.device, dtype=torch.float32).contiguous()
    return gso


class ChebGraphConv(nn.Module):
    """Chebyshev graph convolution (layers.py:122-172): x (B,C,T,N) -> (B,T,N,C_out).  ``gso`` is a plain
    attribute (not a buffer), exactly as in the reference, so it stays out of the state_dict.  A dense tensor takes the
    dense path; a stgcn_b200.gso.CsrOperator, torch sparse tensor or scipy sparse matrix the CSR path (this holds for
    every layer that takes ``gso``)."""

    def __init__(self, c_in, c_out, Ks, gso, bias):
        super().__init__()
        self.c_in = c_in
        self.c_out = c_out
        self.Ks = Ks
        self.gso = gso
        self.weight = nn.Parameter(torch.empty(Ks, c_in, c_out))
        if bias:
            self.bias = nn.Parameter(torch.empty(c_out))
        else:
            self.register_parameter("bias", None)
        self.reset_parameters()

    def reset_parameters(self):
        if self.weight.numel():
            _reset_graph_params(self.weight, self.bias)

    def forward(self, x):
        _require_cuda(x, "ChebGraphConv")
        if self.Ks - 1 < 0:
            raise ValueError(f"ERROR: the graph convolution kernel size Ks has to be a positive integer, "
                             f"but received {self.Ks}.")                                                 # layers.py:148
        if self.c_in != self.c_out:
            raise NotImplementedError("ChebGraphConv: c_in != c_out is never built by the reference (layers.py:218)")
        B, _, T, N = x.shape
        self.gso = _gso_device(self.gso, x)
        dims = (B, T, N, self.c_in, self.c_out, self.Ks, L.GCONV["cheb_graph_conv"], 0, 0)
        return _GconvFn.apply(_channels_last(x), dims, self.gso, None, None, _f32c(self.weight), _f32c(self.bias))


class GraphConv(nn.Module):
    """First-order graph convolution (layers.py:174-206): x (B,C,T,N) -> (B,T,N,C_out)."""

    def __init__(self, c_in, c_out, gso, bias):
        super().__init__()
        self.c_in = c_in
        self.c_out = c_out
        self.gso = gso
        self.weight = nn.Parameter(torch.empty(c_in, c_out))
        if bias:
            self.bias = nn.Parameter(torch.empty(c_out))
        else:
            self.register_parameter("bias", None)
        self.reset_parameters()

    def reset_parameters(self):
        _reset_graph_params(self.weight, self.bias)

    def forward(self, x):
        _require_cuda(x, "GraphConv")
        if self.c_in != self.c_out:
            raise NotImplementedError("GraphConv: c_in != c_out is never built by the reference (layers.py:220)")
        B, _, T, N = x.shape
        self.gso = _gso_device(self.gso, x)
        dims = (B, T, N, self.c_in, self.c_out, 1, L.GCONV["graph_conv"], 0, 0)
        return _GconvFn.apply(_channels_last(x), dims, self.gso, None, None, _f32c(self.weight), _f32c(self.bias))


class GraphConvLayer(nn.Module):
    """align -> graph conv -> + aligned input (layers.py:208-231): (B,c_in,T,N) -> (B,c_out,T,N)."""

    def __init__(self, graph_conv_type, c_in, c_out, Ks, gso, bias):
        super().__init__()
        self.graph_conv_type = graph_conv_type
        self.c_in = c_in
        self.c_out = c_out
        self.align = Align(c_in, c_out)
        self.Ks = Ks
        self.gso = gso
        if self.graph_conv_type == "cheb_graph_conv":
            self.cheb_graph_conv = ChebGraphConv(c_out, c_out, Ks, gso, bias)
        elif self.graph_conv_type == "graph_conv":
            self.graph_conv = GraphConv(c_out, c_out, gso, bias)

    def _inner(self):
        if self.graph_conv_type == "cheb_graph_conv":
            return self.cheb_graph_conv
        if self.graph_conv_type == "graph_conv":
            return self.graph_conv
        raise ValueError(f"unknown graph_conv_type {self.graph_conv_type!r}")

    def _params(self):
        live = self.c_in > self.c_out
        inner = self._inner()
        return (_f32c(self.align.align_conv.weight) if live else None,
                _f32c(self.align.align_conv.bias) if live else None, _f32c(inner.weight), _f32c(inner.bias))

    def forward(self, x, _relu: int = 0):
        _require_cuda(x, "GraphConvLayer")
        inner = self._inner()
        if self.graph_conv_type == "cheb_graph_conv" and self.Ks - 1 < 0:
            raise ValueError(f"ERROR: the graph convolution kernel size Ks has to be a positive integer, "
                             f"but received {self.Ks}.")
        B, _, T, N = x.shape
        self.gso = inner.gso = _gso_device(self.gso, x)
        dims = (B, T, N, self.c_in, self.c_out, max(self.Ks, 1), L.GCONV[self.graph_conv_type], _relu, 1)
        return _as_bctn(_GconvFn.apply(_channels_last(x), dims, self.gso, *self._params()))


class STConvBlock(nn.Module):
    """'TGTND' block (layers.py:233-258): gated temporal conv -> graph conv -> ReLU -> gated temporal conv ->
    LayerNorm([N, C]) -> dropout, as one fused forward and one fused backward call into libstgcn_b200."""

    def __init__(self, Kt, Ks, n_vertex, last_block_channel, channels, act_func, graph_conv_type, gso, bias, droprate):
        super().__init__()
        if G.is_sparse_operator(gso) and tuple(gso.shape) != (n_vertex, n_vertex):
            raise ValueError(f"STConvBlock: a {tuple(gso.shape)} sparse gso for n_vertex = {n_vertex}")
        self.tmp_conv1 = TemporalConvLayer(Kt, last_block_channel, channels[0], n_vertex, act_func)
        self.graph_conv = GraphConvLayer(graph_conv_type, channels[0], channels[1], Ks, gso, bias)
        self.tmp_conv2 = TemporalConvLayer(Kt, channels[1], channels[2], n_vertex, act_func)
        self.tc2_ln = nn.LayerNorm([n_vertex, channels[2]], eps=1e-12)
        self.relu = nn.ReLU()
        self.dropout = nn.Dropout(p=droprate)

    def forward(self, x):
        _require_cuda(x, "STConvBlock")
        t1, gc, t2 = self.tmp_conv1, self.graph_conv, self.tmp_conv2
        act = _act_code(t1.act_func)
        inner = gc._inner()
        if gc.graph_conv_type == "cheb_graph_conv" and gc.Ks - 1 < 0:
            raise ValueError(f"ERROR: the graph convolution kernel size Ks has to be a positive integer, "
                             f"but received {gc.Ks}.")
        B, c_in, T, N = x.shape
        if c_in != t1.c_in or N != t1.n_vertex:
            raise RuntimeError(f"STConvBlock: expected (B, {t1.c_in}, T, {t1.n_vertex}), got {tuple(x.shape)}")
        gc.gso = inner.gso = _gso_device(gc.gso, x)
        dims = (B, T, N, t1.c_in, t1.c_out, gc.c_out, t2.c_out, t1.Kt, max(gc.Ks, 1), act,
                L.GCONV[gc.graph_conv_type], self.training, self.dropout.p, self.tc2_ln.eps)
        params = (*_tconv_param_tuple(t1), *gc._params(), *_tconv_param_tuple(t2),
                  _f32c(self.tc2_ln.weight), _f32c(self.tc2_ln.bias))
        if _no_backward(x, params):
            return _as_bctn(_stblock_infer(_channels_last(x), dims, gc.gso, params))
        return _as_bctn(_STBlockFn.apply(_channels_last(x), dims, gc.gso, *params))


class OutputBlock(nn.Module):
    """'TNFF' block (layers.py:260-284): gated temporal conv(Ko) -> LayerNorm([N,C]) -> fc1 -> ReLU -> dropout -> fc2."""

    def __init__(self, Ko, last_block_channel, channels, end_channel, n_vertex, act_func, bias, droprate):
        super().__init__()
        self.tmp_conv1 = TemporalConvLayer(Ko, last_block_channel, channels[0], n_vertex, act_func)
        self.fc1 = nn.Linear(in_features=channels[0], out_features=channels[1], bias=bias)
        self.fc2 = nn.Linear(in_features=channels[1], out_features=end_channel, bias=bias)
        self.tc1_ln = nn.LayerNorm([n_vertex, channels[0]], eps=1e-12)
        self.relu = nn.ReLU()
        self.dropout = nn.Dropout(p=droprate)

    def forward(self, x):
        _require_cuda(x, "OutputBlock")
        t1 = self.tmp_conv1
        act = _act_code(t1.act_func)
        B, c_in, T, N = x.shape
        if c_in != t1.c_in or N != t1.n_vertex:
            raise RuntimeError(f"OutputBlock: expected (B, {t1.c_in}, T, {t1.n_vertex}), got {tuple(x.shape)}")
        dims = (B, T, N, t1.c_in, t1.c_out, self.fc1.out_features, self.fc2.out_features, t1.Kt, act, self.training,
                self.dropout.p, self.tc1_ln.eps)
        params = (*_tconv_param_tuple(t1), _f32c(self.tc1_ln.weight), _f32c(self.tc1_ln.bias),
                  _f32c(self.fc1.weight), _f32c(self.fc1.bias), _f32c(self.fc2.weight), _f32c(self.fc2.bias))
        if _no_backward(x, params):
            return _as_bctn(_outblock_infer(_channels_last(x), dims, params))
        return _as_bctn(_OutBlockFn.apply(_channels_last(x), dims, *params))
