"""Training-epoch throughput on one GPU: the reference's train() loop (main.py:162-171: a per-tensor torch optimizer and
``l.item()`` every step) against graph.GraphedStep with a fused flat optimizer fed by per-step copies into its static
buffers, and against train.WindowTrainer (one graph replay per full batch, window gather and loss sum inside the graph,
one host synchronisation per epoch).  Default PeMSD7-M model, a seeded synthetic z-scored series of the reference's
PeMSD7-M length (12 671 rows; its 70 % train split of 8 871 rows gives 8 856 windows, so B = 32 leaves a ragged last batch
of 24 windows and B = 256 one of 152).

    python tools/bench_train.py [--batches 32,256] [--droprates 0,0.5] [--opts adamw,nadamw] [--epochs 3]

Prints one JSON line.  Every path starts from the same parameters; the first epoch's loss of each is compared with the
eager loop's, which runs twice to measure its own run-to-run spread (the backward accumulates with atomics); the
trainer's must lie within 4x that spread plus 1e-6 (fp32) or 2e-4 (bf16), the bound the GPU tests use.  With
dropout the paths draw different masks, so their losses agree only statistically.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

BLOCKS = [[1], [64, 16, 64], [64, 16, 64], [128, 128], [1]]
LR, WD = 1e-3, 1e-3                 # main.py's defaults (--lr, --weight_decay_rate)


def gpu_identity():
    """Device name and power limit, read in the same run as the measurement."""
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:
        out = f"nvidia-smi unavailable: {e}"
    return name, out


def train_series(dev):
    """PeMSD7-M-shaped series (12 671 x 228), the reference's split (main.py:103-119): first 70 % for training,
    z-scored with the training rows' statistics."""
    rng = np.random.default_rng(0)
    raw = 60.0 + 10.0 * rng.standard_normal((12671, 228)) + rng.uniform(-8, 8, 228)
    n_val = n_test = int(np.floor(12671 * 0.15))
    train = raw[:12671 - n_val - n_test]
    z = (train - train.mean(axis=0)) / train.std(axis=0)
    return torch.from_numpy(z.astype(np.float32)).to(dev)


def timed_epochs(run_epoch, epochs):
    """(first epoch's loss, seconds per epoch over ``epochs`` more).  The first epoch is the warm-up."""
    first = run_epoch()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(epochs):
        run_epoch()
    torch.cuda.synchronize()
    return first, (time.perf_counter() - t0) / epochs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="32,256")
    ap.add_argument("--droprates", default="0,0.5")
    ap.add_argument("--opts", default="adamw,nadamw")
    ap.add_argument("--epochs", type=int, default=3, help="timed epochs per path, after one warm-up epoch")
    ap.add_argument("--precision", default="bf16")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_train: needs a CUDA device")
    import __graft_entry__ as g
    g.build()
    import stgcn_b200
    from stgcn_b200 import optim
    from stgcn_b200.data import DeviceWindows
    from stgcn_b200.graph import GraphedStep
    from stgcn_b200.synthetic import build_model
    from stgcn_b200.train import WindowTrainer
    dev = torch.device("cuda:0")
    name, smi = gpu_identity()
    stgcn_b200.set_precision(a.precision)
    gso = torch.from_numpy(np.load(os.path.join(ROOT, "tests", "golden", "gso_pemsd7m_cheb.npy")))
    win = DeviceWindows(train_series(dev), 12, 3)
    n = len(win)
    # trainer-vs-eager loss bound: 4x the eager loop's own rerun spread plus this floor (tests/test_gpu_trainer.py)
    floor = 1e-6 if a.precision == "fp32" else 2e-4
    results = []
    for B in [int(b) for b in a.batches.split(",")]:
        loader = [win.batch(start=s, size=B) for s in range(0, n, B)]          # main.py's unshuffled DataLoader
        for p in [float(d) for d in a.droprates.split(",")]:
            for opt_name in a.opts.split(","):
                torch.manual_seed(0)
                state0 = {k: v.clone() for k, v in build_model(gso, "cheb_graph_conv", 3, BLOCKS, dev, droprate=p,
                                                                seed=0).state_dict().items()}

                def fresh():
                    m = build_model(gso, "cheb_graph_conv", 3, BLOCKS, dev, droprate=p, seed=0)
                    m.load_state_dict(state0)
                    m.train()
                    return m

                # (a) the reference's loop
                def eager(model, opt):
                    def epoch():
                        model.train()
                        l_sum, cnt = 0.0, 0
                        for x, y in loader:
                            opt.zero_grad()
                            pred = model(x).view(len(x), -1).float()
                            loss = torch.nn.functional.mse_loss(pred, y)
                            loss.backward()
                            opt.step()
                            l_sum += loss.item() * y.shape[0]
                            cnt += y.shape[0]
                        return l_sum / cnt
                    return epoch

                def torch_opt(model):
                    if opt_name == "adamw":
                        return torch.optim.AdamW(model.parameters(), lr=LR, weight_decay=WD)
                    return torch.optim.NAdam(model.parameters(), lr=LR, weight_decay=WD, decoupled_weight_decay=True)

                m = fresh()
                loss_a, t_a = timed_epochs(eager(m, torch_opt(m)), a.epochs)
                m = fresh()
                loss_a2 = eager(m, torch_opt(m))()
                del m

                def flat_opt(model):
                    x, y = loader[0]
                    torch.nn.functional.mse_loss(model(x).view(len(x), -1).float(), y).backward()
                    cls = optim.FlatAdamW if opt_name == "adamw" else optim.FlatNAdamW
                    o = cls(model, lr=LR, weight_decay=WD)
                    model.zero_grad(set_to_none=True)
                    return o

                # (b) GraphedStep, the batch copied into its static buffers every step, the ragged batch eager
                m = fresh()
                o = flat_opt(m)
                saved = [t.clone() for t in o.state_tensors()]
                step = GraphedStep(m, tuple(loader[0][0].shape), tuple(loader[0][1].shape), device=dev,
                                   post_backward=o.step, warmup=1)
                with torch.no_grad():
                    for t, s in zip(o.state_tensors(), saved):
                        t.copy_(s)

                def graphed_epoch():
                    m.train()
                    l_sum, cnt = 0.0, 0
                    for x, y in loader:
                        if len(x) == B:
                            l_sum += step(x, y).item() * B
                        else:
                            o.zero_grad(set_to_none=True)
                            loss = torch.nn.functional.mse_loss(m(x).view(len(x), -1).float(), y)
                            loss.backward()
                            o.step()
                            l_sum += loss.item() * len(x)
                        cnt += len(x)
                    return l_sum / cnt
                loss_b, t_b = timed_epochs(graphed_epoch, a.epochs)
                step.close()
                del step, m, o

                # (c) WindowTrainer
                m = fresh()
                o = flat_opt(m)
                trainer = WindowTrainer(m, win, B, o)
                loss_c, t_c = timed_epochs(trainer.run_epoch, a.epochs)
                trainer.close()
                del trainer, m, o
                torch.cuda.empty_cache()

                noise = abs(loss_a2 - loss_a) / abs(loss_a)
                rel = lambda v: abs(v - loss_a) / abs(loss_a)
                bound = 4 * noise + floor
                results.append({
                    "batch": B, "ragged_last_batch": n % B, "droprate": p, "opt": opt_name,
                    "windows_per_s": {"eager": round(n / t_a, 1), "graphed_step": round(n / t_b, 1),
                                      "window_trainer": round(n / t_c, 1)},
                    "s_per_epoch": {"eager": t_a, "graphed_step": t_b, "window_trainer": t_c},
                    "epoch1_loss": {"eager": loss_a, "eager_rerun": loss_a2, "graphed_step": loss_b,
                                    "window_trainer": loss_c},
                    "epoch1_rel_vs_eager": {"eager_rerun": noise, "graphed_step": rel(loss_b), "window_trainer": rel(loss_c)},
                    "window_trainer_within_bound": rel(loss_c) <= bound, "bound": bound,
                })
                print(json.dumps(results[-1]), file=sys.stderr, flush=True)
    print(json.dumps({
        "metric": "train_windows_per_s", "gpu": name, "nvidia_smi": smi, "precision": a.precision,
        "model": "PeMSD7-M default (N=228, Kt=Ks=3, blocks 64-16-64 x2, 128-128)", "windows": n,
        "lr": LR, "weight_decay": WD, "timed_epochs": a.epochs, "loss_floor": floor,
        "paths": {"eager": "main.py:162-171: torch.optim per tensor, nn.MSELoss, l.item() every step",
                  "graphed_step": "GraphedStep + fused flat optimizer, step(x, y) copies each batch, .item() every step",
                  "window_trainer": "WindowTrainer.run_epoch: gather + step + loss sum in the graph, one sync per epoch"},
        "results": results,
    }), flush=True)


if __name__ == "__main__":
    main()
