"""Validation / test metrics on the device: drop-ins for ``evaluate_model`` / ``evaluate_metric`` (script/utility.py:90-121
of hazdzz/STGCN) and a CUDA-graph evaluator over device-resident windows.

The reference runs ``val()`` every epoch and ``test()`` at the end (main.py:184-203); both pull every batch through the
host (``l.item()``, ``.cpu().numpy()``, a numpy inverse z-score and Python lists).  Here each batch's forward runs with no
autograd state (``stgcn_*_infer``) and its contribution goes into four fp64 device sums (``stgcn_eval_accumulate``); the
host synchronises once, at the end::

    from stgcn_b200.evaluate import evaluate_model, evaluate_metric, WindowEvaluator
    val_loss = evaluate_model(model, loss, val_iter)                  # utility.evaluate_model
    mae, rmse, wmape = evaluate_metric(model, test_iter, zscore)      # utility.evaluate_metric

    ev = WindowEvaluator(model, DeviceWindows(val_series, n_his, n_pred), batch_size, scaler=zscore)
    m = ev.run()              # {"mse", "mae", "rmse", "wmape"}; one graph replay per full batch, one host sync

``scaler`` is anything with the ``mean_`` / ``scale_`` attributes of sklearn's StandardScaler (either may be None, as with
``with_mean`` / ``with_std`` off); they are used rounded to float32, which is what ``inverse_transform`` does on the
float32 arrays the reference hands it.
"""
from __future__ import annotations

import math
from typing import Dict, Optional, Tuple

import numpy as np
import torch
import torch.nn as nn

from . import _lib as L
from . import layers
from .data import DeviceWindows
from .gso import CsrOperator

__all__ = ["eval_accumulate", "evaluate_model", "evaluate_metric", "WindowEvaluator"]


def _scaler_tensors(scaler, device) -> Tuple[Optional[torch.Tensor], Optional[torch.Tensor]]:
    """(mean, scale) of a StandardScaler-like object as float32 device tensors (None where the scaler has none)."""
    def f32(v):
        return None if v is None else torch.from_numpy(np.ascontiguousarray(v, dtype=np.float32).reshape(-1)).to(device)
    if scaler is None:
        return None, None
    return f32(getattr(scaler, "mean_", None)), f32(getattr(scaler, "scale_", None))


def eval_accumulate(pred: torch.Tensor, target: torch.Tensor, acc: torch.Tensor, mean: Optional[torch.Tensor] = None,
                    scale: Optional[torch.Tensor] = None) -> None:
    """Add one batch to ``acc`` (float64 CUDA tensor [4], see stgcn_eval_accumulate): sum (pred - target)^2, and after the
    inverse z-score sum |d|, sum d^2, sum y.  pred / target: (B, N) float32 CUDA tensors."""
    if pred.dim() != 2 or target.shape != pred.shape:
        raise RuntimeError(f"eval_accumulate: expected two (B, N) tensors, got {tuple(pred.shape)} / {tuple(target.shape)}")
    if not (pred.is_cuda and target.is_cuda and acc.is_cuda) or acc.dtype != torch.float64 or acc.numel() != 4:
        raise RuntimeError("eval_accumulate: pred / target / acc must be CUDA tensors, acc float64 [4]")
    B, N = pred.shape
    for v in (mean, scale):
        if v is not None and (v.numel() != N or v.dtype != torch.float32 or not v.is_cuda):
            raise RuntimeError(f"eval_accumulate: mean / scale must be float32 CUDA tensors of {N} entries")
    pred = pred.float().contiguous()
    target = target.float().contiguous()
    dev = pred.device
    with torch.cuda.device(dev):
        L.check(L.lib().stgcn_eval_accumulate(pred.data_ptr(), target.data_ptr(), B, N,
                                              None if mean is None else mean.data_ptr(),
                                              None if scale is None else scale.data_ptr(), acc.data_ptr(),
                                              torch.cuda.current_stream(dev).cuda_stream))


def _model_device(model: nn.Module) -> torch.device:
    return next(model.parameters()).device


def evaluate_model(model: nn.Module, loss, data_iter) -> float:
    """utility.evaluate_model: the mean squared error over every (window, vertex) of ``data_iter`` (batches of CUDA
    tensors).  ``loss`` must be the reference's ``nn.MSELoss()`` (mean reduction), the only loss main.py builds."""
    if not isinstance(loss, nn.MSELoss) or loss.reduction != "mean":
        raise NotImplementedError("evaluate_model: the device accumulation implements nn.MSELoss(reduction='mean')")
    model.eval()
    acc = torch.zeros(4, dtype=torch.float64, device=_model_device(model))
    count = 0
    with torch.no_grad():
        for x, y in data_iter:
            y_pred = model(x).view(len(x), -1)
            eval_accumulate(y_pred, y.view(len(x), -1), acc)
            count += y.numel()
    return float(acc[0].item()) / count


def evaluate_metric(model: nn.Module, data_iter, scaler):
    """utility.evaluate_metric: (MAE, RMSE, WMAPE) of the inverse-z-scored predictions over ``data_iter``."""
    model.eval()
    dev = _model_device(model)
    mean, scale = _scaler_tensors(scaler, dev)
    acc = torch.zeros(4, dtype=torch.float64, device=dev)
    count = 0
    with torch.no_grad():
        for x, y in data_iter:
            y_pred = model(x).view(len(x), -1)
            eval_accumulate(y_pred, y.view(len(x), -1), acc, mean, scale)
            count += y.numel()
    s = acc.tolist()
    return np.float64(s[1] / count), np.float64(math.sqrt(s[2] / count)), np.float64(s[1] / s[3])


class WindowEvaluator:
    """Evaluation of ``model`` over every window of ``windows`` in the reference's unshuffled batch order, as one CUDA
    graph per full batch -- window gather (stgcn_windows) -> no-grad forward -> stgcn_eval_accumulate -> starts += B --
    replayed len(windows) // batch_size times, the partial last batch run eagerly, one host synchronisation per run().
    The graph reads the model's parameters and graph operators by address.  In-place updates (an optimizer step,
    ``load_state_dict``) are seen by the next run(); when a tensor has been replaced instead (e.g. optim.FlatAdamW
    re-binding every parameter into its flat buffer), run() notices the new addresses and captures the graph again."""

    def __init__(self, model: nn.Module, windows: DeviceWindows, batch_size: int, scaler=None, warmup: int = 1):
        self.model, self.windows, self.B = model, windows, int(batch_size)
        if self.B <= 0:
            raise ValueError("WindowEvaluator: batch_size must be positive")
        dev = windows.series.device
        self.device = dev
        self.n = len(windows)
        self.n_full = self.n // self.B
        self.warmup = max(int(warmup), 1)
        self.mean, self.scale = _scaler_tensors(scaler, dev)
        self.acc = torch.zeros(4, dtype=torch.float64, device=dev)
        self.starts = torch.zeros(self.B, dtype=torch.int64, device=dev)
        self.x = torch.empty((self.B, 1, windows.n_his, windows.N), dtype=torch.float32, device=dev)
        self.y = torch.empty((self.B, windows.N), dtype=torch.float32, device=dev)
        self.graph = None
        if self.n_full:
            self.stream = torch.cuda.Stream(device=dev)
            self._capture()

    def _addresses(self):
        """Addresses of every tensor the captured forward reads from the model."""
        gsos = []
        for m in self.model.modules():
            g = getattr(m, "gso", None)
            if torch.is_tensor(g):
                gsos.append(g)
            elif isinstance(g, CsrOperator):           # the CSR arrays the sparse path reads
                gsos.extend(g.tensors())
        return tuple(t.data_ptr() for t in (*self.model.parameters(), *gsos))

    def _capture(self):
        dev = self.device
        self.model.eval()
        self.graph = None
        # warm-up and capture on one stream: the workspace cache (keyed by stream) and the library's helper streams are
        # set up outside the capture
        self.stream.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(self.stream):
            for _ in range(self.warmup):
                self._reset()
                self._body()
        torch.cuda.current_stream(dev).wait_stream(self.stream)
        torch.cuda.synchronize(dev)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=self.stream, capture_error_mode="thread_local"):
            self._body()
        # the captured kernels use the block workspace of the capture stream by address: hold it, so that neither a
        # cache reset nor a larger workspace for the same stream handle frees it while the graph exists
        self.workspace = layers._WORKSPACES[(dev.index or 0, self.stream.cuda_stream)]
        self.graph, self.captured = graph, self._addresses()

    def _reset(self):
        self.acc.zero_()
        torch.arange(self.B, out=self.starts)

    def _body(self):
        self.windows.batch(starts=self.starts, out=(self.x, self.y))
        with torch.no_grad():
            pred = self.model(self.x).view(self.B, -1)
        eval_accumulate(pred, self.y, self.acc, self.mean, self.scale)
        self.starts.add_(self.B)

    def run(self) -> Dict[str, float]:
        """{"mse", "mae", "rmse", "wmape"} over all windows; mae / rmse / wmape on the inverse-z-scored values when a
        scaler was given, mse (evaluate_model's loss) always on the normalised ones."""
        self.model.eval()
        if self.graph is not None and self._addresses() != self.captured:
            self._capture()
        self._reset()
        for _ in range(self.n_full):
            self.graph.replay()
        tail = self.n - self.n_full * self.B
        if tail:
            x, y = self.windows.batch(start=self.n_full * self.B, size=tail)
            with torch.no_grad():
                pred = self.model(x).view(tail, -1)
            eval_accumulate(pred, y, self.acc, self.mean, self.scale)
        s = self.acc.tolist()
        cnt = self.n * self.windows.N
        if cnt == 0:
            raise RuntimeError("WindowEvaluator: no windows to evaluate")
        return {"mse": s[0] / cnt, "mae": s[1] / cnt, "rmse": math.sqrt(s[2] / cnt), "wmape": s[1] / s[3]}
