"""Sparse against dense graph shift operators on one GPU: bf16 training steps (forward + backward) of the default STGCN
(Chebyshev, Ks = 3, blocks [[1], [64, 16, 64] x 2, [128, 128], [1]], n_his = 12) at B = 32 on seeded synthetic
k-nearest-neighbour graphs (synthetic.knn_operator, symmetric-normalised union graph, so the mean degree is somewhat
above k), once with a CsrOperator and once with the same operator densified.

    python tools/bench_sparse.py [--cases 2048:8,2048:64,8192:8] [--steps 20] [--warmup 5]
                                 [--parent DIR --rounds 2]

For each case it reports the step time of both paths, the time of the SpMM launches of one step (the library's
CUDA-event profiler, one launch at a time), and their achieved bytes/s over the compulsory bytes computed from shapes:
per launch every input plane read once, the output written once, the aux plane read where the recurrence adds one, and
the CSR arrays read once -- against the data-sheet HBM bandwidth of one B200 (7.7 TB/s).  The planes of one launch
(21-84 MB here) fit in the 126 MB L2, so a rate above what HBM alone allows would be possible; it is reported as
measured.  The dense path runs where its (N, N) operator fits, which on a 180 GB card is every case here.  With
--parent DIR it also runs ``bench.py --gpus 1 --steps K --warmup W`` of the tree in DIR (built) and of this tree,
alternately, ``--rounds`` times each.  Prints one JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

BLOCKS = [[1], [64, 16, 64], [64, 16, 64], [128, 128], [1]]
HBM_PEAK = 7.7e12
B, N_HIS, KT, KS = 32, 12, 3, 3


def gpu_identity():
    """Device name and power limit, read in the same run as the measurement."""
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:
        out = f"nvidia-smi unavailable: {e}"
    return name, out


def step_fn(model, x, y):
    def step():
        model.zero_grad(set_to_none=True)
        loss = torch.nn.functional.mse_loss(model(x).view(B, -1).float(), y)
        loss.backward()
        return loss
    return step


def time_steps(step, steps, warmup):
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        loss = step()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / steps * 1e3, float(loss)


def spmm_bytes(tag, n, nnz, c=16):
    """Compulsory bytes of the SpMM launches of one op tag (st0 / st1, fwd / bwd) in one step, bf16 planes.
    Ks = 3: the forward's two launches read one plane (T_1) and two (T_2, with aux) and write one each; the backward's
    adjoint recurrence reads two and writes one per launch."""
    t1 = N_HIS - (KT - 1) if tag.startswith("st0") else N_HIS - 3 * (KT - 1)
    plane = B * t1 * n * c * 2
    csr = (n + 1) * 4 + nnz * 8
    planes = 5 if tag.endswith(".fwd") else 6
    return planes * plane + 2 * csr


def spmm_profile(step, n, nnz):
    """(SpMM launches, ms, compulsory bytes) of one step, from the library's per-launch event profiler."""
    from stgcn_b200 import _lib as L
    step()
    torch.cuda.synchronize()
    L.profile_begin()
    step()
    prof = L.profile_end()
    launches, ms, nbytes = 0, 0.0, 0
    for key, (cnt, t) in prof.items():
        if "spmm_csr_kernel" in key:
            tag = key.split(":")[0]
            launches += cnt
            ms += t
            nbytes += spmm_bytes(tag, n, nnz)
    return launches, ms, nbytes


def run_case(n, degree, steps, warmup, dev):
    from stgcn_b200.gso import CsrOperator
    from stgcn_b200.synthetic import build_model, knn_operator
    op = CsrOperator(knn_operator(n, degree, seed=0), dev)
    g = torch.Generator().manual_seed(1)
    x = torch.randn(B, 1, N_HIS, n, generator=g).to(dev)
    y = torch.randn(B, n, generator=g).to(dev)
    sparse = build_model(op, "cheb_graph_conv", KS, BLOCKS, dev, seed=0)
    sparse.train()
    s_ms, s_loss = time_steps(step_fn(sparse, x, y), steps, warmup)
    launches, k_ms, k_bytes = spmm_profile(step_fn(sparse, x, y), n, op.nnz)
    res = {"N": n, "k": degree, "nnz": op.nnz, "mean_degree": round(op.nnz / n, 2),
           "sparse_step_ms": round(s_ms, 3), "sparse_loss": s_loss,
           "spmm": {"launches_per_step": launches, "ms_per_step": round(k_ms, 4),
                    "compulsory_bytes_per_step": k_bytes,
                    "achieved_bytes_per_s": k_bytes / (k_ms / 1e3) if k_ms else None,
                    "share_of_hbm_peak": round(k_bytes / (k_ms / 1e3) / HBM_PEAK, 3) if k_ms else None}}
    del sparse
    dense_op = op.to_dense()
    dense = build_model(dense_op, "cheb_graph_conv", KS, BLOCKS, dev, seed=0)
    dense.train()
    d_ms, d_loss = time_steps(step_fn(dense, x, y), steps, warmup)
    res.update(dense_step_ms=round(d_ms, 3), dense_loss=d_loss, dense_over_sparse=round(d_ms / s_ms, 2),
               loss_rel_diff=abs(s_loss - d_loss) / abs(d_loss))
    del dense, dense_op
    torch.cuda.empty_cache()
    return res


def bench_py(tree, steps, warmup):
    cmd = [sys.executable, os.path.join(tree, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup",
           str(warmup), "--no-cpu-baseline", "--no-extras"]
    out = subprocess.run(cmd, capture_output=True, text=True, cwd=tree, timeout=1800)
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    if out.returncode or not lines:
        return {"error": out.stderr[-400:]}
    r = json.loads(lines[-1])
    return {"value": r.get("value"), "unit": r.get("unit")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="2048:8,2048:64,8192:8")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--parent", default=None, help="a built tree of the parent commit: bench.py A/B")
    ap.add_argument("--rounds", type=int, default=2)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sparse.py needs a CUDA device")
    import stgcn_b200
    dev = torch.device("cuda:0")
    stgcn_b200.set_precision("bf16")
    name, smi = gpu_identity()
    cases = []
    for c in a.cases.split(","):
        n, k = (int(v) for v in c.split(":"))
        cases.append(run_case(n, k, a.steps, a.warmup, dev))
        print(json.dumps(cases[-1]), file=sys.stderr, flush=True)
    ab = None
    if a.parent:
        ab = {"parent": [], "branch": []}
        for _ in range(a.rounds):
            ab["parent"].append(bench_py(os.path.abspath(a.parent), 20, 5))
            ab["branch"].append(bench_py(ROOT, 20, 5))
    print(json.dumps({"gpu": name, "nvidia_smi": smi, "precision": "bf16", "batch": B, "model": "STGCNChebGraphConv Ks=3",
                      "steps": a.steps, "warmup": a.warmup, "hbm_peak_bytes_per_s": HBM_PEAK, "cases": cases,
                      "bench_py_ab": ab}), flush=True)


if __name__ == "__main__":
    main()
