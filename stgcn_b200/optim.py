"""Optimizer step fused over ONE flat parameter buffer (SURVEY.md §8f N2; the reference's per-tensor optimizers of
``--opt adamw | nadamw | lion``: torch.optim.AdamW, main.py:147-148, torch.optim.NAdam(decoupled_weight_decay=True),
main.py:149-150, and Lion, script/opt.py:34-76 -- FlatAdamW, FlatNAdamW and FlatLion here).

The live parameters of the model are re-pointed at views of one flat fp32 buffer, laid out exactly like the flat
gradient buffer of ``dist.FlatGradAllReducer`` (which the backward kernels write and the all-reduce averages in place), so
one kernel launch updates everything: 1 launch instead of ~28 x 4 per-tensor ones, and capturable in the step's CUDA
graph (``GraphedStep(post_backward=opt.step)``) because the step number and, optionally, the learning rate live in
device memory.  Parameters that never receive a gradient (the reference's dead align convs, layers.py:12) are left
untouched, as torch's optimizers leave parameters whose ``.grad`` is None."""
from __future__ import annotations

import ctypes as C
from typing import List, Optional

import torch

from . import _lib as L
from .dist import FlatGradAllReducer


class _FlatOptimizer:
    def __init__(self, model: torch.nn.Module, reducer: Optional[FlatGradAllReducer] = None, lr: float = 1e-3,
                 weight_decay: float = 1e-2):
        """``reducer``: the model's FlatGradAllReducer, already bound (one backward + ``reducer.bind()`` or one
        ``reducer()`` call), or None to create and bind one here (a first backward must have run)."""
        self.model = model
        self.reducer = reducer if reducer is not None else FlatGradAllReducer(model)
        if self.reducer.live is None:
            self.reducer.bind()
        r = self.reducer
        dev = r.flat.device
        self.flat_params = torch.zeros_like(r.flat)          # the alignment padding between slots stays zero
        with torch.no_grad():
            for p, off, n in zip(r.live, r.offsets, r.sizes):
                view = self.flat_params.narrow(0, off, n).view_as(p)
                view.copy_(p.data)
                p.data = view                    # the module's parameters now ARE slices of the flat buffer
        self.lr, self.weight_decay = float(lr), float(weight_decay)
        self.lr_dev = torch.full((1,), self.lr, dtype=torch.float32, device=dev)
        self.steps_dev = torch.zeros(1, dtype=torch.int64, device=dev)      # completed steps (bias correction uses +1)
        self._lib = L.lib()

    def set_lr(self, lr: float) -> None:
        """StepLR & co. (main.py:158,172): the learning rate lives on the device so a captured step follows it."""
        self.lr = float(lr)
        self.lr_dev.fill_(self.lr)

    def zero_grad(self, set_to_none: bool = True) -> None:
        self.model.zero_grad(set_to_none=set_to_none)

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.flat_params.device).cuda_stream

    def state_tensors(self) -> List[torch.Tensor]:
        """Every device tensor a step reads or writes, apart from the gradients: parameters, learning rate, step count
        and the optimizer's own state (train.WindowTrainer snapshots them around its warm-up)."""
        return [self.flat_params, self.lr_dev, self.steps_dev]


class FlatAdamW(_FlatOptimizer):
    """torch.optim.AdamW semantics (decoupled weight decay, bias-corrected first/second moments) in one launch."""

    def __init__(self, model, reducer=None, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2):
        super().__init__(model, reducer, lr, weight_decay)
        self.betas, self.eps = (float(betas[0]), float(betas[1])), float(eps)
        self.exp_avg = torch.zeros_like(self.flat_params)
        self.exp_avg_sq = torch.zeros_like(self.flat_params)

    @torch.no_grad()
    def step(self, grad_scale: float = 1.0) -> None:
        r = self.reducer
        with torch.cuda.device(self.flat_params.device):
            L.check(self._lib.stgcn_adamw_step(self.flat_params.data_ptr(), r.flat.data_ptr(), self.exp_avg.data_ptr(),
                                               self.exp_avg_sq.data_ptr(), self.flat_params.numel(), C.c_float(self.lr),
                                               C.c_float(self.betas[0]), C.c_float(self.betas[1]), C.c_float(self.eps),
                                               C.c_float(self.weight_decay), C.c_float(grad_scale), 1,
                                               self.steps_dev.data_ptr(), self.lr_dev.data_ptr(), self._stream()))
        self.steps_dev.add_(1)

    def state_tensors(self) -> List[torch.Tensor]:
        return super().state_tensors() + [self.exp_avg, self.exp_avg_sq]


class FlatNAdamW(_FlatOptimizer):
    """torch.optim.NAdam(decoupled_weight_decay=True) semantics (Nesterov momentum with the momentum-cache schedule
    mu_t = b1 (1 - 0.5 * 0.96^(t * momentum_decay)), bias-corrected second moment) in one launch.  The defaults are
    torch NAdam's.  ``mu_products`` holds the float32 product of the momentum caches in two device slots that the kernel
    alternates by step parity (stgcn_nadamw_step); ``mu_product`` is the current one."""

    def __init__(self, model, reducer=None, lr=2e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0,
                 momentum_decay=4e-3):
        super().__init__(model, reducer, lr, weight_decay)
        self.betas, self.eps = (float(betas[0]), float(betas[1])), float(eps)
        self.momentum_decay = float(momentum_decay)
        self.exp_avg = torch.zeros_like(self.flat_params)
        self.exp_avg_sq = torch.zeros_like(self.flat_params)
        self.mu_products = torch.ones(2, dtype=torch.float32, device=self.flat_params.device)

    @property
    def mu_product(self) -> torch.Tensor:
        """The product of the momentum caches after the last step (float32 device tensor [1], no host synchronisation);
        torch keeps the same value as ``state[p]["mu_product"]`` of every parameter."""
        return self.mu_products.index_select(0, self.steps_dev.remainder(2))

    @torch.no_grad()
    def step(self, grad_scale: float = 1.0) -> None:
        r = self.reducer
        with torch.cuda.device(self.flat_params.device):
            L.check(self._lib.stgcn_nadamw_step(self.flat_params.data_ptr(), r.flat.data_ptr(), self.exp_avg.data_ptr(),
                                                self.exp_avg_sq.data_ptr(), self.flat_params.numel(),
                                                C.c_float(self.lr), C.c_float(self.betas[0]), C.c_float(self.betas[1]),
                                                C.c_float(self.eps), C.c_float(self.weight_decay),
                                                C.c_float(grad_scale), 1, self.steps_dev.data_ptr(),
                                                self.lr_dev.data_ptr(), C.c_float(self.momentum_decay),
                                                self.mu_products.data_ptr(), self._stream()))
        self.steps_dev.add_(1)

    def state_tensors(self) -> List[torch.Tensor]:
        return super().state_tensors() + [self.exp_avg, self.exp_avg_sq, self.mu_products]


class FlatLion(_FlatOptimizer):
    """The reference's Lion (script/opt.py:34-76): sign of the interpolated momentum, decoupled weight decay."""

    def __init__(self, model, reducer=None, lr=1e-3, betas=(0.9, 0.99), weight_decay=1e-2):
        super().__init__(model, reducer, lr, weight_decay)
        self.betas = (float(betas[0]), float(betas[1]))
        self.exp_avg = torch.zeros_like(self.flat_params)

    @torch.no_grad()
    def step(self, grad_scale: float = 1.0) -> None:
        r = self.reducer
        with torch.cuda.device(self.flat_params.device):
            L.check(self._lib.stgcn_lion_step(self.flat_params.data_ptr(), r.flat.data_ptr(), self.exp_avg.data_ptr(),
                                              self.flat_params.numel(), C.c_float(self.lr), C.c_float(self.betas[0]),
                                              C.c_float(self.betas[1]), C.c_float(self.weight_decay),
                                              C.c_float(grad_scale), self.lr_dev.data_ptr(), self._stream()))
        self.steps_dev.add_(1)

    def state_tensors(self) -> List[torch.Tensor]:
        return super().state_tensors() + [self.exp_avg]
