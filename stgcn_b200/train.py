"""Whole training epochs on the device: the loop of the reference's ``train()`` (main.py:160-182) -- StepLR, early
stopping and the best-epoch checkpoint included -- over device-resident windows and a fused flat optimizer.

The reference synchronises the host every step (``l.item()``, main.py:170) and pulls every batch through a DataLoader.
Here one epoch is one CUDA-graph replay per full batch, with the window gather, the forward, the MSE loss, the backward,
the optimizer step and the loss sum all inside the graph, and the host synchronises once per epoch::

    from stgcn_b200.data import DeviceWindows
    from stgcn_b200.evaluate import WindowEvaluator
    from stgcn_b200.optim import FlatNAdamW
    from stgcn_b200.train import WindowTrainer, fit

    opt = FlatNAdamW(model, lr=args.lr, weight_decay=args.weight_decay_rate)     # after one backward
    trainer = WindowTrainer(model, DeviceWindows(train_series, n_his, n_pred), args.batch_size, opt)
    ev = WindowEvaluator(model, DeviceWindows(val_series, n_his, n_pred), args.batch_size)
    history = fit(trainer, args.epochs, lambda: ev.run()["mse"], step_size=args.step_size, gamma=args.gamma,
                  patience=args.patience, checkpoint_path="STGCN_" + args.dataset + ".pt")
    trainer.close()
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, List, Optional, Union

import numpy as np
import torch
import torch.nn as nn

from . import _lib as L
from . import layers
from .data import DeviceWindows
from .graph import GraphedStep
from .optim import _FlatOptimizer

__all__ = ["WindowTrainer", "fit", "steplr_schedule", "EarlyStopping"]


class _EpochStep(GraphedStep):
    """A GraphedStep (optimizer step as its post_backward) whose captured body then adds ``loss * B`` to the fp64 sum
    ``acc``, advances the window starts by B and gathers the NEXT batch into the static input."""

    def __init__(self, model, windows: DeviceWindows, B: int, acc, starts, optimizer, warmup):
        self.windows, self.acc, self.starts = windows, acc, starts
        super().__init__(model, (B, 1, windows.n_his, windows.N), (B, windows.N), device=acc.device,
                         post_backward=optimizer.step, warmup=warmup)

    def _body(self):
        super()._body()
        B = self.x.shape[0]
        self.acc.add_(self.loss.to(torch.float64), alpha=B)            # l.item() * y.shape[0], exact in fp64
        self.starts.add_(B)
        self.windows.batch(starts=self.starts, out=(self.x, self.y))


class WindowTrainer:
    """One training epoch of ``model`` over every window of ``windows`` per ``run_epoch()``, in the reference's unshuffled
    DataLoader order (main.py:126), as main.py:162-171 runs it: per batch zero_grad -> forward -> nn.MSELoss -> backward
    -> optimizer.step().  ``optimizer`` is one of optim.FlatAdamW / FlatNAdamW / FlatLion, bound to ``model``.

    Each full batch is one replay of a graph.GraphedStep whose captured body ends, after the optimizer step, with
    ``acc += double(loss) * B``, ``starts += B`` and the window gather of the NEXT batch into the step's static input
    (so the first replay needs one gather in front of it).  The ragged last batch of ``len(windows) % batch_size``
    windows runs eagerly: it happens once per epoch, and a second captured graph would cost its own warm-up, capture
    and memory pool for one launch sequence per epoch.  It takes its own optimizer step, enters ``acc`` weighted by its
    own size and advances the dropout step counter, so its masks differ from those of every full batch.

    The warm-up that GraphedStep runs before its capture executes the body, optimizer step included; the optimizer
    state (``optimizer.state_tensors()``) is saved before and restored after it, so construction changes no parameter,
    moment, step count or learning rate.  Single process only: with a multi-rank reducer the all-reduce would have to
    run between the backward and the optimizer step, outside the graph (graph.py)."""

    def __init__(self, model: nn.Module, windows: DeviceWindows, batch_size: int, optimizer: _FlatOptimizer,
                 warmup: int = 1):
        if not isinstance(optimizer, _FlatOptimizer):
            raise TypeError("WindowTrainer: optimizer must be optim.FlatAdamW, FlatNAdamW or FlatLion")
        if optimizer.reducer._world() > 1:
            raise ValueError("WindowTrainer runs in a single process: with a FlatGradAllReducer over more than one rank "
                             "the all-reduce must run between the backward and the optimizer step, outside the CUDA "
                             "graph; use graph.GraphedStep with the reducer and call the optimizer after each step")
        self.model, self.windows, self.opt, self.B = model, windows, optimizer, int(batch_size)
        if self.B <= 0:
            raise ValueError("WindowTrainer: batch_size must be positive")
        self.n = len(windows)
        if self.n == 0:
            raise ValueError("WindowTrainer: no windows to train on")
        self.n_full = self.n // self.B
        self.tail = self.n - self.n_full * self.B
        dev = windows.series.device
        self.device = dev
        self.acc = torch.zeros(1, dtype=torch.float64, device=dev)
        self.starts = torch.zeros(self.B, dtype=torch.int64, device=dev)
        self.tail_loss = torch.zeros(1, dtype=torch.float32, device=dev)
        model.train()
        saved = [t.clone() for t in optimizer.state_tensors()]
        self.step = _EpochStep(model, windows, self.B, self.acc, self.starts, optimizer, warmup)
        with torch.no_grad():
            for t, s in zip(optimizer.state_tensors(), saved):
                t.copy_(s)
        # The captured kernels use the block workspace of the capture stream by address: hold it, so that neither a
        # reset of the workspace cache nor a larger workspace for the same stream frees it while the graph exists.  The
        # saved-state buffers of the captured forward come from the graph's private memory pool, which the graph keeps.
        capture_stream = torch.cuda.graph.default_capture_stream
        self.workspace = layers._WORKSPACES.get((dev.index or 0, capture_stream.cuda_stream))

    def _run_tail(self) -> None:
        x, y = self.windows.batch(start=self.n_full * self.B, size=self.tail)
        self.opt.zero_grad(set_to_none=True)
        pred = self.model(x).reshape(self.tail, -1).float()
        dpred = torch.empty_like(pred)
        dev = self.device
        L.check(L.lib().stgcn_mse_fwd_bwd(pred.data_ptr(), y.data_ptr(), pred.numel(), C.c_float(1.0),
                                          self.tail_loss.data_ptr(), dpred.data_ptr(),
                                          torch.cuda.current_stream(dev).cuda_stream))
        pred.backward(dpred)
        self.opt.step()
        self.acc.add_(self.tail_loss.to(torch.float64), alpha=self.tail)
        self.step.step_counter.add_(1)

    def run_epoch_async(self) -> torch.Tensor:
        """Enqueue one epoch; returns the device fp64 sum of loss_i * B_i over its batches (no host synchronisation)."""
        self.model.train()
        with torch.cuda.device(self.device):
            self.acc.zero_()
            torch.arange(self.B, out=self.starts)
            self.windows.batch(starts=self.starts, out=(self.step.x, self.step.y))
            for _ in range(self.n_full):
                self.step.replay()
            if self.tail:
                self._run_tail()
        return self.acc

    def run_epoch(self) -> float:
        """One epoch; returns l_sum / n, the train loss main.py:170-171 prints."""
        return self.run_epoch_async().item() / self.n

    def close(self) -> None:
        """Release the dropout step counter registration (the trainer must not run afterwards)."""
        self.step.close()


def steplr_schedule(lr: float, step_size: int, gamma: float, epochs: int) -> List[float]:
    """The learning rate of epochs 0 .. epochs-1 under torch.optim.lr_scheduler.StepLR stepped once per epoch
    (main.py:156,172): multiplied by gamma after every step_size-th epoch, by repeated multiplication as StepLR does."""
    out, cur = [], float(lr)
    for e in range(epochs):
        if e > 0 and e % step_size == 0:
            cur = cur * gamma
        out.append(cur)
    return out


class EarlyStopping:
    """The decisions of the reference's EarlyStopping (script/earlystopping.py:27-42) without its file I/O: the first
    call counts as an improvement, ``-val <= best + delta`` does not, and ``early_stop`` is set once ``counter`` reaches
    ``patience``.  The reference compares float32 tensors (val() returns torch.tensor(l_sum / n), main.py:194), so the
    loss, the best score and their sum with delta are rounded to float32 here too."""

    def __init__(self, delta: float = 0.0, patience: int = 7):
        self.delta, self.patience = float(delta), int(patience)
        self.counter = 0
        self.best_score: Optional[np.float32] = None
        self.early_stop = False

    def __call__(self, val_loss: float) -> bool:
        """Record one epoch's validation loss; returns True when it is an improvement (the checkpoint is saved)."""
        score = -np.float32(val_loss)
        if self.best_score is None:
            self.best_score = score
            return True
        if score <= self.best_score + np.float32(self.delta):
            self.counter += 1
            if self.counter >= self.patience:
                self.early_stop = True
            return False
        self.best_score = score
        self.counter = 0
        return True


def fit(trainer: WindowTrainer, epochs: int, val: Callable[[], Union[float, torch.Tensor]], step_size: int = 10,
        gamma: float = 0.95, patience: int = 10, delta: float = 0.0,
        checkpoint_path: Optional[str] = None) -> List[dict]:
    """main.py: train() over ``trainer``: per epoch run_epoch -> StepLR -> ``val()`` -> EarlyStopping, stopping early as
    the reference does.  ``val`` returns the epoch's validation loss, as a float (``lambda: evaluator.run()["mse"]``) or a
    one-element device tensor; the train and validation losses are read back together, once per epoch.

    The learning rate of epoch e is ``steplr_schedule(optimizer.lr, ...)[e]``, pushed with ``optimizer.set_lr``.  On
    every improvement the optimizer's flat parameter buffer is copied into a device snapshot (and ``model.state_dict()``
    written to ``checkpoint_path`` if given, the file the reference's test() loads, main.py:198); when fit returns the
    model holds the parameters of the best epoch.  Parameters outside the flat buffer (the dead align convs) never
    change.  Returns one dict per epoch run: epoch, lr, train_loss, val_loss, improved."""
    opt = trainer.opt
    schedule = steplr_schedule(opt.lr, step_size, gamma, epochs)
    es = EarlyStopping(delta=delta, patience=patience)
    best = torch.empty_like(opt.flat_params)
    history: List[dict] = []
    for epoch in range(epochs):
        opt.set_lr(schedule[epoch])
        train_sum = trainer.run_epoch_async()
        v = val()
        if torch.is_tensor(v):
            train_sum_h, val_loss = torch.cat([train_sum, v.reshape(1).to(train_sum)]).tolist()
        else:
            train_sum_h, val_loss = train_sum.item(), float(v)
        improved = es(val_loss)
        if improved:
            best.copy_(opt.flat_params)
            if checkpoint_path is not None:
                torch.save(trainer.model.state_dict(), checkpoint_path)
        history.append({"epoch": epoch, "lr": schedule[epoch], "train_loss": train_sum_h / trainer.n,
                        "val_loss": val_loss, "improved": improved})
        if es.early_stop:
            break
    if history:
        opt.flat_params.copy_(best)
    return history
