#!/usr/bin/env python
"""bench.py -- ST-block (full STGCN) forward+backward throughput, samples/s (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # our CUDA path (one rank per GPU under torchrun)
  python bench.py --impl reference --steps K --warmup W    # the reference's CPU path (oracle port) on host cores

A "step" = zero_grad + forward + MSE loss + backward of the whole model on one synthetic batch (the body of the
reference's main.py:165-168 without the optimizer, as in BASELINE.md §2), plus the gradient all-reduce when N > 1.
Prints ONE JSON line on rank 0 (contract in the task statement; extra keys: roofline, cpu_baseline, clocks, e2e).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from types import SimpleNamespace

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BLOCKS = [[1], [64, 16, 64], [64, 16, 64], [128, 128], [1]]
WORKLOADS = {
    # name: (gso file tag, graph conv kind, Ks, default per-GPU batch, description)
    "pemsd7m": ("pemsd7m", "cheb_graph_conv", 3, 256, "PeMSD7-M N=228 Kt=3 Ks=3 ChebGraphConv T=12"),
    "metrla": ("metrla", "graph_conv", 3, 512, "METR-LA N=207 GraphConv Kt=3 T=12"),
    "pemsbay": ("pemsbay", "cheb_graph_conv", 3, 128, "PEMS-BAY N=325 ChebGraphConv Ks=3 Kt=3 T=12"),
    # BASELINE configs[4] (roofline sweep): seeded dense symmetric operator with spectral norm 1, 64 graph-conv channels.
    # NOT measured in round 1; the node contraction needs STGCN_GSO_KTILED=1 to run on tensor cores (DESIGN.md §7).
    "syn2048": ("syn2048", "cheb_graph_conv", 5, 512, "synthetic N=2048 dense operator ChebGraphConv Ks=5 channels=64 Kt=3 T=12"),
}
WORKLOAD_BLOCKS = {"syn2048": [[1], [64, 64, 64], [64, 64, 64], [128, 128], [1]]}


def workload_blocks(workload):
    return WORKLOAD_BLOCKS.get(workload, BLOCKS)


def load_operator(tag, kind):
    """Dense graph operator of a workload: the reference-derived matrices committed under tests/golden/, or the seeded
    synthetic operator of SURVEY.md §8(d) for the N=2048 sweep."""
    if tag.startswith("syn"):
        from stgcn_b200.synthetic import synthetic_operator
        return synthetic_operator(int(tag[3:]), seed=0)
    return torch.from_numpy(np.load(os.path.join(ROOT, "tests", "golden",
                                                 f"gso_{tag}_{'cheb' if kind == 'cheb_graph_conv' else 'gcn'}.npy")))


# ---- algorithmic work per sample (SURVEY.md §8d closed form; MAC = 2 FLOP) ---------------------------------------
def flops_per_sample(n, kind, ks, blocks=BLOCKS, kt=3, n_his=12):
    """Returns (fwd, fwd+bwd, per-stage dict of fwd+bwd FLOPs)."""
    stages = {}
    fwd = 0.0
    tot = 0.0
    T = n_his
    n_st = len(blocks) - 3
    for l in range(n_st):
        c0 = blocks[l][-1]
        c1, c2, c3 = blocks[l + 1]
        T1, T2 = T - kt + 1, T - 2 * (kt - 1)
        tc1 = 2.0 * (2 * c1) * c0 * kt * T1 * n
        al = 2.0 * c2 * c1 * T1 * n if c1 > c2 else 0.0
        if kind == "cheb_graph_conv":
            nn_ = (ks - 1) * 2.0 * n * n * c2 * T1
            mix = 2.0 * ks * c2 * c2 * T1 * n
        else:
            nn_ = 2.0 * n * n * c2 * T1
            mix = 2.0 * c2 * c2 * T1 * n
        tc2 = 2.0 * (2 * c3) * c2 * kt * T2 * n
        first = l == 0
        # backward: 2x every weight-bearing GEMM (dgrad + wgrad), 1x the node contraction; no dX for block 0's tc1
        f = tc1 + al + nn_ + mix + tc2
        b = (1.0 if first else 2.0) * tc1 + 2 * al + nn_ + 2 * mix + 2 * tc2
        stages[f"st{l}"] = dict(tc1=tc1 * (2 if first else 3), align=3 * al, gso=2 * nn_, mix=3 * mix, tc2=3 * tc2)
        fwd += f
        tot += f + b
        T = T2
    ko = T
    if ko > 1:
        c0, (o0, o1), ce = blocks[-3][-1], blocks[-2], blocks[-1][0]
        tco = 2.0 * (2 * o0) * c0 * ko * n
        fc1 = 2.0 * o0 * o1 * n
        fc2 = 2.0 * o1 * ce * n
        fwd += tco + fc1 + fc2
        tot += 3 * (tco + fc1 + fc2)
        stages["out"] = dict(tc1=3 * tco, fc=3 * (fc1 + fc2))
    return fwd, tot, stages


def bytes_per_sample(n, dtype_bytes, blocks=BLOCKS, kt=3, n_his=12):
    """Compulsory traffic with whole-block fusion + recompute (SURVEY.md §8d): per block |in|+|out| forward,
    |in|+|dout|+|din| backward (no din for block 0)."""
    T = n_his
    total = 0
    n_st = len(blocks) - 3
    sizes = [blocks[0][-1] * T * n]
    for l in range(n_st):
        T -= 2 * (kt - 1)
        sizes.append(blocks[l + 1][-1] * T * n)
    sizes.append(blocks[-1][0] * n)
    for i in range(len(sizes) - 1):
        total += sizes[i] + sizes[i + 1]                 # fwd
        total += sizes[i] + sizes[i + 1] + (sizes[i] if i > 0 else 0)   # bwd
    return total * dtype_bytes


# ---- clocks sampler ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms in the background; `stop()` summarises the samples that
    arrived between `mark_load_begin()` and `mark_load_end()` (the timed regions plus, when those are shorter than a few
    sampling periods, an extra observation window of the same step)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows = []          # (arrival time, line)
        self.proc = None
        self.index = index
        self.t0 = self.t1 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, bufsize=1)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def wait_first_sample(self, timeout=5.0):
        t_end = time.time() + timeout
        while self.proc is not None and not self.rows and time.time() < t_end:
            time.sleep(0.05)

    def mark_load_begin(self):
        self.t0 = time.time()

    def mark_load_end(self):
        self.t1 = time.time()

    def samples_under_load(self):
        lo = self.t0 if self.t0 is not None else 0.0
        hi = self.t1 if self.t1 is not None else float("inf")
        return sum(1 for t, _ in self.rows if lo <= t <= hi)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        lo = self.t0 if self.t0 is not None else 0.0
        hi = self.t1 if self.t1 is not None else float("inf")
        for t, r in self.rows:
            if not (lo <= t <= hi):
                continue
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"], "rows_total": len(self.rows)}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


# ---- CPU reference arm ---------------------------------------------------------------------------------------------
CPU_THREADS = 16        # fixed: on the 128-thread GPU host the reference's step (many small ATen ops) is fastest around 16
                        # threads (all 128 are ~100x slower, profiles/bench_r01_fp32_first.json); a per-run sweep made the
                        # number wander 260-723 samples/s between driver runs


def _reference_modules():
    """The UNMODIFIED reference (model/layers.py, model/models.py) if a copy travels with the repo under baseline/_ref
    (git-ignored; the reference is plain Python without a build, so `pip install --target` has nothing to install --
    DESIGN.md §6); None otherwise.  /root/reference itself does not exist on the GPU box and is never read here."""
    ref = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.exists(os.path.join(ref, "model", "layers.py")):
        return None
    if ref not in sys.path:
        sys.path.insert(0, ref)
    try:
        from model import models as ref_models       # noqa: the reference's own package name
        return ref_models
    except Exception:
        return None


def _make_cpu_step(workload, batch, droprate, device="cpu"):
    """One training-step body (main.py:165-168 without the optimizer) of the reference's arithmetic on `device`:
    the reference's own modules when present, else the oracle's restatement (same ATen ops: conv2d, einsum->bmm,
    layer_norm, autograd).  Returns (step_fn, kind)."""
    from oracle import stgcn_oracle as O
    tag, kind, ks, _, _ = WORKLOADS[workload]
    blocks = workload_blocks(workload)
    gso = load_operator(tag, kind).to(device)
    n = gso.shape[0]
    gen = torch.Generator().manual_seed(0)
    x = torch.randn(batch, 1, 12, n, generator=gen).to(device)
    y = torch.randn(batch, n, generator=gen).to(device)
    ref_models = _reference_modules()
    if ref_models is not None:
        args = SimpleNamespace(Kt=3, Ks=ks, act_func="glu", graph_conv_type=kind, gso=gso, enable_bias=True,
                               droprate=droprate, n_his=12)
        cls = ref_models.STGCNChebGraphConv if kind == "cheb_graph_conv" else ref_models.STGCNGraphConv
        model = cls(args, blocks, n).to(device)
        model.train()

        def step():
            model.zero_grad(set_to_none=True)
            loss = torch.nn.functional.mse_loss(model(x).view(batch, -1), y)
            loss.backward()
            return loss
        return step, "reference"
    params = {k: v.to(device).requires_grad_(True) for k, v in
              O.init_params(blocks=blocks, kt=3, ks=ks, n_his=12, n_vertex=n, kind=kind, seed=0).items()}
    cfg = dict(blocks=blocks, kt=3, n_his=12, act="glu", kind=kind, p_drop=droprate, training=True)

    def step():
        for p in params.values():
            p.grad = None
        loss = O.mse_step(x, y, params, gso, **cfg)
        loss.backward()
        return loss
    return step, "port"


def cpu_reference_run(workload, batch, steps, warmup, droprate, budget_s=None, threads=CPU_THREADS):
    """Times the reference step on the host cores: median of the timed steps at a FIXED thread count.
    Returns dict(samples_per_s, ms_per_step, cores, steps, kind)."""
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    cores = max(1, min(threads, avail))
    torch.set_num_threads(cores)
    step, kind = _make_cpu_step(workload, batch, droprate)
    for _ in range(warmup):
        step()
    times = []
    t_start = time.perf_counter()
    for i in range(steps):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
        if budget_s is not None and time.perf_counter() - t_start > budget_s and i >= 9:
            break
    med = float(np.median(times))
    return dict(samples_per_s=batch / med, ms_per_step=1e3 * med, cores=cores, steps=len(times), batch=batch,
                host_threads_available=avail, kind=kind)


def cuda_eager_baseline(workload, batch, droprate, dev, steps=5, warmup=2):
    """The incumbent on the same box (SURVEY.md §2.2, BASELINE.md §5 item 4): the reference's eager PyTorch path on the
    GPU (cuDNN/cuBLAS kernels behind conv2d / einsum / layer_norm + autograd), same workload and batch, CUDA events.
    A reported baseline: none of this repository's kernels run here."""
    step, kind = _make_cpu_step(workload, batch, droprate, device=dev)
    for _ in range(warmup):
        step()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / steps
    return {"value": batch / (ms / 1e3), "unit": "samples/s", "ms_per_step": ms, "batch": batch, "steps": steps,
            "kind": kind, "what": "reference arithmetic, eager PyTorch CUDA, same B200"}


def _arm_watchdog(seconds, rank):
    """A hung collective or a kernel that never returns must not eat the whole time budget of a measurement pass: after
    `seconds` a daemon thread dumps every Python stack to stderr and ends the process with status 124."""
    if seconds <= 0:
        return
    import faulthandler

    def fire():
        sys.stderr.write(f"[bench watchdog] rank {rank}: not finished after {seconds} s -- stacks follow, exiting 124\n")
        faulthandler.dump_traceback(file=sys.stderr, all_threads=True)
        sys.stderr.flush()
        os._exit(124)

    t = threading.Timer(seconds, fire)
    t.daemon = True
    t.start()


class Runner:
    """One workload on this rank's GPU through the public API: model on stgcn_b200.layers, the whole step (zero_grad +
    forward + MSE + backward [+ gradient all-reduce]) captured in a CUDA graph (stgcn_b200.graph.GraphedStep)."""
    POOL = 4      # distinct input batches cycled through, so no step re-reads a hot input

    def __init__(self, workload, B, precision, dev, rank, world, droprate=0.0, graph=True):
        import stgcn_b200
        from stgcn_b200 import _lib as L
        from stgcn_b200.dist import FlatGradAllReducer
        from stgcn_b200.synthetic import build_model
        self.L, self.lib = L, L.lib()
        self.workload, self.B, self.precision, self.dev, self.world = workload, B, precision, dev, world
        tag, kind, ks, _, self.desc = WORKLOADS[workload]
        self.kind, self.ks = kind, ks
        self.blocks = workload_blocks(workload)
        gso = load_operator(tag, kind)
        self.n = n = gso.shape[0]
        stgcn_b200.set_precision(precision)
        self.model = build_model(gso, kind, ks, self.blocks, dev, droprate=droprate, seed=0)
        self.model.train()
        self.reducer = FlatGradAllReducer(self.model) if world > 1 else None
        gen = torch.Generator().manual_seed(1234 + rank)
        self.xs_host = [torch.randn(B, 1, 12, n, generator=gen).pin_memory() for _ in range(self.POOL)]
        self.ys_host = [torch.randn(B, n, generator=gen).pin_memory() for _ in range(self.POOL)]
        self.xs = [t.to(dev) for t in self.xs_host]
        self.ys = [t.to(dev) for t in self.ys_host]
        self.loss_buf = torch.zeros(1, device=dev)
        self.loss_host = torch.zeros(1).pin_memory()
        self.graphed, self.launches_per_step, self.reduce_mode = None, None, "none" if world == 1 else "after-backward"
        if graph:
            from stgcn_b200.graph import GraphedStep
            n_before = L.launch_count()
            warm = 3
            self.graphed = GraphedStep(self.model, (B, 1, 12, n), (B, n), device=dev, warmup=warm, reducer=self.reducer)
            self.launches_per_step = (L.launch_count() - n_before) // (warm + 1)      # warm-up bodies + 1 capture
            self.loss_buf = self.graphed.loss
            if self.reducer is not None:
                self.reduce_mode = "ncclAvg on the flat gradient buffer the backward kernels write, right behind the graph replay"
        self.x_dev, self.y_dev = torch.empty_like(self.xs[0]), torch.empty_like(self.ys[0])
        self.prefetcher = None
        # (single-process runs only: the multi-GPU legs keep the copy-in-front path they were validated with)
        if self.graphed is not None and world == 1 and os.environ.get("STGCN_BENCH_NO_PREFETCH") is None:
            from stgcn_b200.data import HostBatchPrefetcher
            self.prefetcher = HostBatchPrefetcher(self.xs[0], self.ys[0], dev)

    def eager_step(self, x, y, reduce=True):
        L, B = self.L, self.B
        self.model.zero_grad(set_to_none=True)
        pred = self.model(x).reshape(B, -1)                      # (B,1,1,N) view -> (B,N), main.py:166
        dpred = torch.empty_like(pred)
        L.check(self.lib.stgcn_mse_fwd_bwd(pred.data_ptr(), y.data_ptr(), pred.numel(), 1.0, self.loss_buf.data_ptr(),
                                           dpred.data_ptr(), torch.cuda.current_stream().cuda_stream))
        pred.backward(dpred)
        if reduce and self.reducer is not None:
            self.reducer()

    def step(self, i):
        x, y = self.xs[i % self.POOL], self.ys[i % self.POOL]
        if self.graphed is None:
            self.eager_step(x, y)
        else:
            self.graphed(x, y)                   # device-to-device copy into the static buffers + replay (+ reduce)

    def e2e_step(self, i):
        """Host (pinned) buffers in, loss out, copies inside the timed region, through the public API: every step's inputs
        travel host -> device (stgcn_b200.data.HostBatchPrefetcher: double-buffered on a copy stream, so batch i+1's copy
        overlaps step i's compute; the first step of a timed region requests its own batch inside the region) and the
        loss travels device -> host."""
        if self.graphed is None:
            self.x_dev.copy_(self.xs_host[i % self.POOL], non_blocking=True)
            self.y_dev.copy_(self.ys_host[i % self.POOL], non_blocking=True)
            self.eager_step(self.x_dev, self.y_dev)
        elif self.prefetcher is not None:
            pf, P = self.prefetcher, self.POOL
            if pf.requested != i:                                        # start of a region: nothing in flight for this step
                pf.request(i, self.xs_host[i % P], self.ys_host[i % P])
            x, y = pf.take(i)
            pf.request(i + 1, self.xs_host[(i + 1) % P], self.ys_host[(i + 1) % P])
            self.graphed(x, y)                                           # copy into the graph's static buffers + replay
            pf.release(i)
        else:
            self.graphed(self.xs_host[i % self.POOL], self.ys_host[i % self.POOL])
        self.loss_host.copy_(self.loss_buf, non_blocking=True)

    def timed(self, fn, k):
        import torch.distributed as dist
        dev, world = self.dev, self.world

        def sync_all():
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(k):
            fn(i)
        e1.record()
        sync_all()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    def measure(self, steps, warmup):
        """(samples/s over all ranks, ms/step) of `steps` timed steps after `warmup` untimed ones; max over ranks."""
        for i in range(warmup):
            self.step(i)
        ms = self.timed(self.step, steps)
        return self.B * self.world * steps / (ms / 1e3), ms / steps

    def close(self):
        if self.graphed is not None:
            self.graphed.close()
        if self.reducer is not None:
            self.reducer.unbind()


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(run, out_dir):
    """Writes what the last step of the timed loop handed its caller: the loss and the gradient of every parameter that
    receives one, as float32 ``DIR/loss.npy`` and ``DIR/grad.<parameter name>.npy``.  Inputs and weights are seeded, so
    two builds run with the same arguments can be compared array for array.  Above DUMP_LIMIT_BYTES in all, every array
    is replaced by the same fraction of its elements, flattened, at indices drawn from a fixed seed (the same arguments
    give the same indices, so two builds' samples stay comparable).  Returns the number of bytes written."""
    torch.cuda.synchronize()
    arrays = {"loss": run.loss_buf.reshape(-1)[:1]}
    arrays.update({f"grad.{k}": p.grad for k, p in run.model.named_parameters() if p.grad is not None})
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        frac = (DUMP_LIMIT_BYTES - 4 * len(arrays)) / total        # the max(1, ...) below adds at most one element each
        rng = np.random.default_rng(0)
        arrays = {k: v.reshape(-1)[np.sort(rng.choice(v.size, max(1, int(v.size * frac)), replace=False))]
                  for k, v in arrays.items()}
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), v)
    return sum(v.nbytes for v in arrays.values())


def _short_line(r, value, ms_step, extra=None):
    fwd_f, tot_f, _ = flops_per_sample(r.n, r.kind, r.ks, blocks=r.blocks)
    d = {"workload": f"{r.desc} batch={r.B}/GPU x {r.world} GPU", "precision": r.precision, "value": value,
         "unit": "samples/s", "ms_per_step": ms_step, "tflops_per_gpu": tot_f * value / r.world / 1e12}
    d.update(extra or {})
    return d


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="pemsd7m", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: the workload's BASELINE batch)")
    ap.add_argument("--precision", default=os.environ.get("STGCN_PRECISION", "bf16"), choices=["fp32", "bf16", "tf32x3"],
                    help="bf16 = BASELINE.json configs[1] (fused tcgen05 path); tf32x3 = the 1e-3 parity gate on tensor "
                         "cores; fp32 = the same gate on CUDA cores")
    ap.add_argument("--droprate", type=float, default=0.0,
                    help="dropout p for BOTH arms (0 = the stricter CPU comparison, BASELINE.md §2)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the extra legs of the default line (parity_mode, cuda_baseline, other BASELINE configs)")
    ap.add_argument("--no-graph", action="store_true", help="launch the step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--max-seconds", type=int, default=int(os.environ.get("STGCN_BENCH_MAX_SECONDS", "900")),
                    help="watchdog: dump all Python stacks to stderr and exit 124 if the run has not finished by then")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the loss and parameter gradients of the last timed step as "
                         "float32 DIR/<name>.npy (seeded inputs: two builds can be compared output for output)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    _arm_watchdog(a.max_seconds, rank)
    helper_streams = os.environ.get("STGCN_NO_SIDE_STREAMS") is None
    tag, kind, ks, default_b, desc = WORKLOADS[a.workload]
    B = a.batch or default_b
    steps, warmup = a.steps, max(a.warmup, 3)

    cfg_common = {"workload": f"{desc} batch={B}/GPU fwd+bwd+MSE, dropout {a.droprate}", "per_gpu_batch": B,
                  "global_batch": B * max(world, 1), "droprate": a.droprate}

    # ------------------------------------------------------------------ reference arm (CPU)
    if a.impl == "reference":
        if rank != 0:
            return
        cpu_b = min(B, 32 if a.workload != "syn2048" else 2)       # ~1 GFLOP of conv/bmm per sample-step at N=2048
        r = cpu_reference_run(a.workload, cpu_b, steps, warmup, a.droprate)
        what = "the unmodified reference (baseline/_ref)" if r["kind"] == "reference" else \
            "oracle port of the reference step (same ATen ops)"
        sample = (f"median of {r['steps']} steps of B={cpu_b} (a bounded sample of the B={B} workload: "
                  f"BASELINE configs[0] batch), {what}, {r['cores']} host threads "
                  f"(fixed; {r['host_threads_available']} available)")
        cfg_ref = dict(cfg_common)
        cfg_ref["workload"] = f"{desc} fwd+bwd+MSE, dropout {a.droprate}; CPU sample batch={cpu_b} (GPU arm: batch={B}/GPU)"
        cfg_ref["cpu_sample_batch"] = cpu_b
        line = {"impl": "reference", "metric": "ST-block fwd+bwd samples/sec", "value": r["samples_per_s"],
                "unit": "samples/s", "n_gpus": a.gpus, "steps": r["steps"], "warmup": warmup,
                "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": cfg_ref,
                "cpu_baseline": {"value": r["samples_per_s"], "unit": "samples/s", "cores": r["cores"],
                                 "kind": r["kind"], "sample": sample},
                "e2e": {"value": r["samples_per_s"], "unit": "samples/s", "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line), flush=True)
        return

    # ------------------------------------------------------------------ our arm (CUDA)
    import torch.distributed as dist
    import __graft_entry__ as ge
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if rank == 0:
        ge.build()
    if world > 1:
        dist.barrier()
    from stgcn_b200 import _lib as L

    run = Runner(a.workload, B, a.precision, dev, rank, world, droprate=a.droprate, graph=not a.no_graph)
    n, blocks = run.n, run.blocks

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        sampler.wait_first_sample()
    for i in range(warmup):
        run.step(i)
    sampler.mark_load_begin()
    n0 = L.launch_count()
    ms_total = run.timed(run.step, steps)
    launches = (L.launch_count() - n0) if run.graphed is None else run.launches_per_step * steps
    value = B * world * steps / (ms_total / 1e3)
    if a.dump_outputs and rank == 0:            # before the end-to-end leg overwrites the loss and gradients
        nbytes = dump_outputs(run, a.dump_outputs)
        print(f"[bench] last timed step's loss and gradients: {nbytes} bytes under {a.dump_outputs}", file=sys.stderr)

    for i in range(2):
        run.e2e_step(i)
    ms_e2e = run.timed(run.e2e_step, steps)
    # the pipelined end-to-end step must compute what the device-resident step computes on the same batch
    run.e2e_step(1); torch.cuda.synchronize(); loss_e2e = float(run.loss_host[0])
    run.step(1); torch.cuda.synchronize(); loss_dev = float(run.loss_buf.reshape(-1)[0])
    e2e_ok = abs(loss_e2e - loss_dev) <= 1e-3 * max(abs(loss_dev), 1e-6)
    e2e_pipeline = ("double-buffered pinned-host -> device copies on a copy stream (batch i+1 travels while step i computes; "
                    "stgcn_b200.data.HostBatchPrefetcher)") if getattr(run, "prefetcher", None) is not None \
        else "copy in front of every step"
    if not e2e_ok:
        print(f"[bench] e2e loss {loss_e2e} != device-path loss {loss_dev}", file=sys.stderr)
    # the timed regions last tens of milliseconds, nvidia-smi samples every 100 ms: keep the same step running (untimed,
    # all ranks: it contains the collective) until at least 5 samples have been taken under this load
    obs_rounds = 0
    while obs_rounds < 40:
        need_more = torch.tensor([1 if (rank == 0 and sampler.samples_under_load() < 5 and sampler.proc is not None) else 0],
                                 device=dev)
        if world > 1:
            dist.broadcast(need_more, src=0)
        if int(need_more.item()) == 0:
            break
        for i in range(50):
            run.step(i)
        torch.cuda.synchronize()
        obs_rounds += 1
    sampler.mark_load_end()
    clocks = sampler.stop() if rank == 0 else None
    e2e_value = B * world * steps / (ms_e2e / 1e3)
    h2d = run.xs_host[0].numel() * 4 + run.ys_host[0].numel() * 4

    # live per-kernel CUDA-event profile of the same step (separate short pass so the timed loop is unperturbed)
    roofline, roofline_tc, top = None, None, []
    fwd_f, tot_f, stages = flops_per_sample(n, kind, ks, blocks=blocks)
    peaks = {"hbm_gbs": 6650.0, "bf16_tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        peaks = json.load(open(pk))
        peaks["source"] = "MEASURED_PEAKS.json"
    esize = 2 if a.precision == "bf16" else 4
    if rank == 0 and not a.no_profile:
        psteps = 3
        L.profile_begin()
        for i in range(psteps):
            # eager: the event profiler brackets individual launches.  NO collective here: this pass runs on rank 0 only
            run.eager_step(run.xs[i % run.POOL], run.ys[i % run.POOL], reduce=False)
        prof = L.profile_end()
        tot_ms = sum(v[1] for v in prof.values())
        rows = sorted(prof.items(), key=lambda kv: -kv[1][1])
        top = [{"key": k, "launches_per_step": v[0] / psteps, "ms_per_step": v[1] / psteps,
                "share": v[1] / tot_ms} for k, v in rows[:60]]
        # dominant kernel: algorithmic FLOPs / bytes of the stage it implements over its measured time, against the
        # roof that bounds it (ridge = peak FLOP/s / peak B/s); plus the tcgen05 kernel with the largest share against
        # the TENSOR roof whatever its arithmetic intensity (north_star quotes tensor-pipe utilisation)
        ridge = peaks["bf16_tflops_sustained"] * 1e12 / (peaks["hbm_gbs"] * 1e9)
        for k0, (c0, ms0) in rows:
            work = _kernel_work(k0, n, B, kind, ks, esize, blocks=blocks)
            if not work:
                continue
            fl, by = work
            t_s = ms0 / psteps * 1e-3
            common = {"kernel": k0, "peak_source": peaks["source"], "alg_flops_per_step": fl, "alg_bytes_per_step": by,
                      "launches_per_step": c0 / psteps, "avg_launch_ms": ms0 / c0, "share_of_step": ms0 / tot_ms}
            if roofline is None:
                if by > 0 and fl / by < ridge:
                    ach, peak, bound, unit = by / t_s / 1e9, peaks["hbm_gbs"], "hbm", "GB/s"
                else:
                    ach, peak, bound, unit = fl / t_s / 1e12, peaks["bf16_tflops_sustained"], "tensor", "TFLOP/s"
                roofline = {"bound": bound, "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak,
                            "traffic": _ncu_traffic(k0, a.workload, B, a.precision), **common}
            if roofline_tc is None and "umma" in k0 and fl > 0:
                ach = fl / t_s / 1e12
                roofline_tc = {"bound": "tensor", "achieved": ach, "peak": peaks["bf16_tflops_sustained"],
                               "unit": "TFLOP/s", "frac": ach / peaks["bf16_tflops_sustained"], **common}
            if roofline is not None and roofline_tc is not None:
                break
    step_tflops = tot_f * value / world / 1e12          # per GPU
    roofline_step = {"bound": "tensor", "achieved": step_tflops, "peak": peaks["bf16_tflops_sustained"],
                     "unit": "TFLOP/s", "frac": step_tflops / peaks["bf16_tflops_sustained"],
                     "flops_per_sample": tot_f, "alg_bytes_per_sample": bytes_per_sample(n, esize, blocks=blocks),
                     "peak_source": peaks["source"]}
    reduce_mode = run.reduce_mode
    cuda_graph = run.graphed is not None
    run.close()
    del run
    torch.cuda.empty_cache()

    # ------------------------------------------------------------------ extra legs of the default line
    extras = {}
    default_line = a.workload == "pemsd7m" and not a.batch and a.precision == "bf16" and not a.no_extras and not a.no_graph
    xsteps, xwarm = 10, 3
    if default_line:
        def leg(name, fn):
            try:
                extras[name] = fn()
            except Exception as e:                       # an extra leg must never take the headline down with it
                extras[name] = {"error": f"{type(e).__name__}: {e}"[:300]}
            torch.cuda.synchronize()
            torch.cuda.empty_cache()

        def parity_leg():
            r = Runner("pemsd7m", B, "tf32x3", dev, rank, world, droprate=a.droprate)
            v, ms = r.measure(xsteps, xwarm)
            out = _short_line(r, v, ms, {"what": "the 1e-3 parity gate on tensor cores: fp32 storage, every GEMM tcgen05 "
                                                  "kind::tf32 with 3xTF32 operand splitting (tests/test_gpu_parity.py)"})
            r.close()
            return out

        def config_leg(workload, batch, label):
            r = Runner(workload, batch, "bf16", dev, rank, world, droprate=a.droprate)
            v, ms = r.measure(xsteps, xwarm)
            out = _short_line(r, v, ms, {"baseline_config": label, "global_batch": batch * world})
            r.close()
            return out

        leg("parity_mode", parity_leg)
        if world == 1:
            leg("cfg3_metrla", lambda: config_leg("metrla", 512, "configs[2]: METR-LA N=207 GraphConv batch=512 on 1xB200"))
        else:
            # BASELINE configs[3]: PEMS-BAY, GLOBAL batch 1024 sharded over the ranks (strong scaling: 512/256/128 per GPU)
            leg("cfg4_pemsbay", lambda: config_leg("pemsbay", 1024 // world,
                                                   f"configs[3]: PEMS-BAY N=325 ChebGraphConv Ks=3 global batch=1024 over {world}xB200"))

    cpu_baseline, cuda_baseline = None, None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        r = cpu_reference_run(a.workload, 32 if a.workload != "syn2048" else 2, 40, 3, a.droprate, budget_s=15.0)
        what = "the unmodified reference (baseline/_ref)" if r["kind"] == "reference" else "oracle port of the reference step"
        cpu_baseline = {"value": r["samples_per_s"], "unit": "samples/s", "cores": r["cores"], "kind": r["kind"],
                        "sample": f"median of {r['steps']} steps of B={r['batch']} (BASELINE configs[0] batch), {what} on "
                                  f"{r['cores']} host threads (fixed; {r['host_threads_available']} available), "
                                  f"dropout {a.droprate}"}
        if default_line:
            try:
                # PyTorch's defaults (what the reference's main.py runs with: TF32 allowed in cuDNN convolutions, fp32
                # matmuls) and the strict-fp32 variant
                cuda_baseline = cuda_eager_baseline(a.workload, B, a.droprate, dev)
                cuda_baseline["what"] = "reference arithmetic, eager PyTorch CUDA with PyTorch's default math modes, same B200"
                torch.backends.cuda.matmul.allow_tf32 = False
                torch.backends.cudnn.allow_tf32 = False
                strict = cuda_eager_baseline(a.workload, B, a.droprate, dev)
                cuda_baseline["strict_fp32"] = {"value": strict["value"], "ms_per_step": strict["ms_per_step"]}
            except Exception as e:
                cuda_baseline = {"error": f"{type(e).__name__}: {e}"[:300]}

    if rank == 0:
        line = {"metric": "ST-block fwd+bwd samples/sec", "value": value, "unit": "samples/s", "n_gpus": world,
                "steps": steps, "warmup": warmup, "ms_per_step": ms_total / steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None,
                "dtype": {"fp32": "f32", "bf16": "bf16", "tf32x3": "tf32x3"}[a.precision], "data": "synthetic",
                "config": {**cfg_common, "precision": a.precision,
                           "l2": f"{Runner.POOL} input batches cycled; per-step activation working set exceeds the 126 MB L2",
                           "parallelism": f"dp{world}", "cuda_graph": cuda_graph,
                           "helper_streams": helper_streams,
                           "grad_allreduce": reduce_mode},
                "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                        "ms_per_step": ms_e2e / steps, "loss_matches_device_path": e2e_ok,
                        "input_pipeline": e2e_pipeline},
                "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "roofline_tensor": roofline_tc,
                "roofline_step": roofline_step, "cpu_baseline": cpu_baseline, "cuda_baseline": cuda_baseline,
                **extras, "top_kernels": top}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def _ncu_traffic(key, workload, B, precision):
    """DRAM bytes (read + write) per launch of this kernel from the committed `ncu --set full` captures
    (profiles/r02_traffic.json, then r01_traffic.json; PeMSD7-M, B=256, bf16 only), or None when that kernel was not captured."""
    import re
    if workload != "pemsd7m" or B != 256 or precision != "bf16":
        return None
    tag, kern = key.split(":", 1)
    m = re.search(r"[A-Za-z_][A-Za-z0-9_]*", kern)
    for name in ("r02_traffic.json", "r01_traffic.json"):          # newest capture that has the kernel
        path = os.path.join(ROOT, "profiles", name)
        if not os.path.exists(path):
            continue
        row = json.load(open(path))["kernels"].get(f"{tag}:{m.group(0) if m else kern}")
        if row is not None:
            return row["dram_read_bytes"] + row["dram_write_bytes"]
    return None


def _kernel_work(key, n, B, kind, ks, esize, blocks=BLOCKS, kt=3, n_his=12):
    """Algorithmic (FLOPs, HBM bytes) per step of all launches under one '<stage>.<op>.<dir>:<kernel>' profile key:
    the closed-form GEMM term of the stage the kernel implements (SURVEY.md §8d) and the tensors it must read/write
    once (esize = bytes per activation element).  Returns None for kernels that are not modelled."""
    tag, kern = key.split(":", 1)
    parts = tag.split(".")
    if len(parts) < 3:
        return None
    st, op, direction = parts[0], parts[1], parts[2]
    T = n_his
    dims = {}
    n_st = len(blocks) - 3
    for l in range(n_st):
        c0 = blocks[l][-1]
        c1, c2, c3 = blocks[l + 1]
        dims[f"st{l}"] = dict(c0=c0, c1=c1, c2=c2, c3=c3, T0=T, T1=T - kt + 1, T2=T - 2 * (kt - 1), kt=kt)
        T -= 2 * (kt - 1)
    if T > 1:
        dims["out"] = dict(c0=blocks[-3][-1], c1=blocks[-2][0], c2=blocks[-2][1], c3=blocks[-1][0], T0=T, T1=1, T2=1, kt=T)
    if st not in dims:
        return None
    d = dims[st]
    rows = lambda t: B * t * n
    e = esize
    if op in ("tc1", "tc2"):
        cin, cout = (d["c0"], d["c1"]) if op == "tc1" else (d["c2"], d["c3"])
        tin, tout = (d["T0"], d["T1"]) if op == "tc1" else (d["T1"], d["T2"])
        W = 2 * cout
        gemm = 2.0 * W * cin * d["kt"] * rows(tout)
        if "umma_fb0_kernel" in kern and cin == 1:    # align data gradient + GLU backward + first-conv weight gradient: reads the
            c2 = d["c2"]                         # 16-channel gradient and the model input, writes only the weight gradient
            return gemm + 2.0 * c2 * cout * rows(tout), (rows(tout) * c2 + rows(tin) * cin) * e
        if "umma_fb0_kernel" in kern:     # align data gradient + q-only GLU backward: dX0, Q, H in; dZ out
            c2 = d["c2"]
            return 2.0 * c2 * cout * rows(tout), rows(tout) * (c2 + 2 * cout + W) * e
        if "umma_fb2_kernel" in kern:           # LayerNorm bwd + GLU bwd + data gradient + weight gradient of the second conv:
            return 2.0 * gemm, (3 * rows(tout) * cout + 2 * rows(tin) * cin) * e    # dY, H3, Q, H2 in; dH2 out
        if "ln_bwd_sums_pg" in kern:            # group sums + LayerNorm parameter gradients: one pass over dY and H3
            return 0.0, 2 * rows(tout) * cout * e
        if "umma_tap" in kern or "tapgemm" in kern:
            if direction == "fwd":
                return gemm, (rows(tin) * cin + rows(tout) * (W + cout)) * e
            return gemm, (rows(tout) * W + rows(tin) * cin) * e                      # data gradient
        if "wgrad" in kern and "smallc" not in kern:
            return gemm, (rows(tin) * cin + rows(tout) * W) * e
        if "smallc1" in kern:      # Cin = 1 first layer: z is never stored (recomputed), so only x and h / dh move
            return gemm, (rows(tin) * cin + rows(tout) * cout) * e
        if "smallc_conv" in kern:
            return gemm, (rows(tin) * cin + rows(tout) * (W + cout)) * e
        if "smallc" in kern:                                                         # gate bwd + wgrad fused
            return gemm, (rows(tin) * cin + rows(tout) * (W + cout)) * e
        if "gate" in kern:
            return 0.0, (rows(tout) * (W + cout + W)) * e
    if op == "gc":
        c1, c2, t1 = d["c1"], d["c2"], d["T1"]
        nk = (ks - 1) if kind == "cheb_graph_conv" else 1
        kmix = ks if kind == "cheb_graph_conv" else 1
        if "umma_cheb" in kern:     # fused recurrence + weight GEMMs: fwd reads x0, writes the stack planes and y;
            fl = nk * 2.0 * n * c2 * rows(t1) + 2.0 * kmix * c2 * c2 * rows(t1)     # bwd reads dy, y, writes dG, dx0
            by = rows(t1) * c2 * e * ((1 + nk + 1) if direction == "fwd" else 4)
            return fl, by
        if "gso" in kern:
            return nk * 2.0 * n * n * c2 * rows(t1) / n, nk * 3 * rows(t1) * c2 * e
        if "wgrad" in kern:
            return 2.0 * rows(t1) * c2 * (c1 + kmix * c2), rows(t1) * (c1 + c2 + kmix * c2 + c2) * e
        if "umma_tap" in kern or "tapgemm" in kern:
            fl = 2.0 * rows(t1) * c2 * (c1 + kmix * c2)
            return fl, rows(t1) * (c1 + c2 + kmix * c2 + c2) * e
    if op == "fc":
        return 2.0 * rows(1) * d["c1"] * d["c2"], rows(1) * (d["c1"] + d["c2"]) * e
    if op == "ln":
        c, t = (d["c3"], d["T2"]) if st != "out" else (d["c1"], 1)
        if direction == "bwd" and "gate" in kern and "sums" not in kern:
            return 0.0, rows(t) * (2 * c + 4 * c) * e        # x, dy in; z (2c) in; dz (2c) out
        return 0.0, 2 * rows(t) * c * e
    return None


if __name__ == "__main__":
    main()
