"""Evaluation throughput on one GPU: the reference's val() / test() loop (script/utility.py:90-121: a forward per batch,
then .item() / .cpu().numpy() and numpy metrics on the host) against the device-side drop-in evaluate_metric and the
CUDA-graph WindowEvaluator, plus the forward alone with and without autograd state.  Default PeMSD7-M model (bf16), a
seeded synthetic z-scored series of velocity-like statistics, the unshuffled windows of a PeMSD7-M-sized test split.

    python tools/bench_eval.py [--batches 32,256] [--windows 1900] [--repeats 5] [--precision bf16]

Prints one JSON line per batch size.  Every timed path's metrics are compared with the reference-style loop's, and the
no-grad forward's output with the grad-enabled forward's (bit for bit), on the inputs that are timed.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_identity():
    """Device name and power limit, read in the same run as the measurement."""
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:            # the number is still reported, marked as unattributed
        out = f"nvidia-smi unavailable: {e}"
    return name, out


class Scaler:
    def __init__(self, mean_, scale_):
        self.mean_, self.scale_ = mean_, scale_


def reference_loop(model, loader, scaler):
    """utility.evaluate_model + utility.evaluate_metric as test() runs them (main.py:199-200): two passes."""
    model.eval()
    m32, s32 = np.asarray(scaler.mean_).astype(np.float32), np.asarray(scaler.scale_).astype(np.float32)
    l_sum, n = 0.0, 0
    with torch.no_grad():
        for x, y in loader:
            y_pred = model(x).view(len(x), -1)
            l_sum += torch.nn.functional.mse_loss(y_pred, y).item() * y.shape[0]
            n += y.shape[0]
        mae, sum_y, mse = [], [], []
        for x, y in loader:
            yy = (y.cpu().numpy() * s32 + m32).reshape(-1)
            yp = (model(x).view(len(x), -1).cpu().numpy() * s32 + m32).reshape(-1)
            d = np.abs(yy - yp)
            mae += d.tolist(); sum_y += yy.tolist(); mse += (d ** 2).tolist()
    return (l_sum / n, np.array(mae).mean(), math.sqrt(np.array(mse).mean()), np.sum(np.array(mae)) / np.sum(np.array(sum_y)))


def timed(fn, repeats):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    out = fn()                                               # warm-up (not timed)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(repeats):
        out = fn()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / repeats
    return out, dt, (torch.cuda.max_memory_allocated() - base) / 1e6


def forward_ms(model, x, grad, iters=20):
    model.eval()
    def run():
        if grad:
            return model(x)
        with torch.no_grad():
            return model(x)
    run(); torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        y = run()
        del y
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters, (torch.cuda.max_memory_allocated() - base) / 1e6


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="32,256")
    ap.add_argument("--windows", type=int, default=1900)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--precision", default="bf16")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_eval: needs a CUDA device")
    import __graft_entry__ as g
    g.build()
    import stgcn_b200
    from stgcn_b200 import layers
    from stgcn_b200.data import DeviceWindows
    from stgcn_b200.evaluate import WindowEvaluator, evaluate_metric, evaluate_model
    from stgcn_b200.synthetic import build_model
    dev = torch.device("cuda:0")
    name, smi = gpu_identity()
    stgcn_b200.set_precision(a.precision)
    gso = torch.from_numpy(np.load(os.path.join(ROOT, "tests", "golden", "gso_pemsd7m_cheb.npy")))
    model = build_model(gso, "cheb_graph_conv", 3, [[1], [64, 16, 64], [64, 16, 64], [128, 128], [1]], dev, seed=0)
    rng = np.random.default_rng(0)
    raw = 60.0 + 10.0 * rng.standard_normal((a.windows + 12 + 3, 228)) + rng.uniform(-8, 8, 228)
    mean_, scale_ = raw.mean(axis=0), raw.std(axis=0)
    scaler = Scaler(mean_, scale_)
    win = DeviceWindows(torch.from_numpy(((raw - mean_) / scale_).astype(np.float32)).to(dev), 12, 3)
    for B in [int(b) for b in a.batches.split(",")]:
        loader = [win.batch(start=s, size=B) for s in range(0, len(win), B)]
        ref, t_ref, m_ref = timed(lambda: reference_loop(model, loader, scaler), a.repeats)

        def dropin():
            return (evaluate_model(model, torch.nn.MSELoss(), loader),) + tuple(evaluate_metric(model, loader, scaler))
        new, t_new, m_new = timed(dropin, a.repeats)
        layers._WORKSPACES.clear()
        ev = WindowEvaluator(model, win, B, scaler=scaler)
        evm, t_ev, m_ev = timed(ev.run, a.repeats)
        evt = (evm["mse"], evm["mae"], evm["rmse"], evm["wmape"])
        rel = lambda u, v: max(abs(p - q) / abs(q) for p, q in zip(u, v))
        x = loader[0][0]
        with torch.no_grad():
            y_ng = model.eval()(x)
        y_g = model(x)
        fwd_g, mem_g = forward_ms(model, x, True)
        fwd_ng, mem_ng = forward_ms(model, x, False)
        n = len(win)
        print(json.dumps({
            "metric": "eval_samples_per_s", "gpu": name, "nvidia_smi": smi, "precision": a.precision,
            "model": "PeMSD7-M default (N=228, Kt=Ks=3, blocks 64-16-64 x2, 128-128)", "windows": n, "batch": B,
            "reference_loop": {"samples_per_s": round(n / t_ref, 1), "s_per_eval": t_ref, "peak_mb": round(m_ref, 1),
                               "note": "evaluate_model + evaluate_metric: two passes over the windows, as test() runs them"},
            "dropin": {"samples_per_s": round(n / t_new, 1), "s_per_eval": t_new, "peak_mb": round(m_new, 1),
                       "max_rel_vs_reference": rel(new, ref), "note": "the same two calls"},
            "window_evaluator": {"samples_per_s": round(n / t_ev, 1), "s_per_eval": t_ev, "peak_mb": round(m_ev, 1),
                                 "max_rel_vs_reference": rel(evt, ref), "note": "one pass gives all four metrics"},
            "forward_ms": {"grad": round(fwd_g, 4), "no_grad": round(fwd_ng, 4)},
            "forward_peak_mb": {"grad": round(mem_g, 1), "no_grad": round(mem_ng, 1)},
            "no_grad_equals_grad_forward": bool(torch.equal(y_ng, y_g.detach())),
        }), flush=True)


if __name__ == "__main__":
    main()
