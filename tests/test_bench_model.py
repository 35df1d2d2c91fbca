"""Host-side checks of bench.py's work model (no GPU): the closed-form algorithmic FLOPs / bytes of SURVEY.md §8(d),
the per-kernel attribution used for the `roofline` object, and the committed ncu traffic table."""
import json
import os

import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("n,kind,ks,fwd_m,tot_m", [
    (228, "cheb_graph_conv", 3, 206.33, 564.01),      # PeMSD7-M   (SURVEY §8d, = FlopCounterMode on the reference)
    (207, "graph_conv", 3, 157.55, 449.11),           # METR-LA
    (325, "cheb_graph_conv", 3, 326.39, 868.52),      # PEMS-BAY
])
def test_algorithmic_flops_match_survey(n, kind, ks, fwd_m, tot_m):
    fwd, tot, stages = bench.flops_per_sample(n, kind, ks)
    assert abs(fwd / 1e6 - fwd_m) < 0.01
    assert abs(tot / 1e6 - tot_m) < 0.01
    assert abs(sum(sum(v.values()) for v in stages.values()) - tot) < 1.0      # the per-stage split adds up


@pytest.mark.parametrize("n,mb", [(228, 1.763), (207, 1.601), (325, 2.513)])
def test_algorithmic_bytes_match_survey(n, mb):
    assert abs(bench.bytes_per_sample(n, 2) / 1e6 - mb) < 0.001
    assert bench.bytes_per_sample(n, 4) == 2 * bench.bytes_per_sample(n, 2)


def test_kernel_work_model_and_traffic_table():
    r01 = json.load(open(os.path.join(ROOT, "profiles", "r01_traffic.json")))["kernels"]
    r02 = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))["kernels"]
    assert r01 and r02, "empty traffic table"
    for name, table in (("r01", r01), ("r02", r02)):
        for key, row in table.items():
            work = bench._kernel_work(key, 228, 256, "cheb_graph_conv", 3, 2)
            assert work is not None, key                       # every captured kernel is modelled
            fl, by = work
            assert fl >= 0 and by > 0, key
            measured = row["dram_read_bytes"] + row["dram_write_bytes"]
            newest = r02.get(key, row)                         # the round-2 capture wins where both have the kernel
            assert bench._ncu_traffic(key, "pemsd7m", 256, "bf16") == newest["dram_read_bytes"] + newest["dram_write_bytes"]
            # DRAM traffic of one launch never exceeds ~1.3x the algorithmic bytes of its stage (no re-reads); it may be
            # far below when the output stayed in the 126 MB L2 at capture time
            assert measured <= 1.3 * by, (name, key, measured, by)
    assert "st0.tc2.bwd:umma_fb2_kernel" in r02
    assert bench._ncu_traffic("st0.tc2.fwd:umma_tap_kernel<EPI_GATE>", "metrla", 512, "bf16") is None


def test_dump_outputs_full_and_sampled(tmp_path, monkeypatch):
    """--dump-outputs: the loss and every existing gradient as float32 .npy; over the size limit, a seeded sample of
    every array that is the same from run to run and stays within the limit."""
    import types
    import numpy as np
    import torch
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a: None)
    model = torch.nn.Sequential(torch.nn.Linear(300, 200), torch.nn.Linear(200, 3), torch.nn.Linear(3, 3))
    for p in list(model.parameters())[:4]:
        p.grad = torch.randn_like(p)
    run = types.SimpleNamespace(model=model, loss_buf=torch.tensor([0.25]))
    names = {"loss.npy", "grad.0.weight.npy", "grad.0.bias.npy", "grad.1.weight.npy", "grad.1.bias.npy"}
    full = bench.dump_outputs(run, str(tmp_path / "full"))
    assert set(os.listdir(tmp_path / "full")) == names
    assert full == 4 * (1 + 300 * 200 + 200 + 200 * 3 + 3)
    w = np.load(tmp_path / "full" / "grad.0.weight.npy")
    assert w.dtype == np.float32 and np.array_equal(w, model[0].weight.grad.numpy())
    assert np.load(tmp_path / "full" / "loss.npy").tolist() == [0.25]
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", full // 10)
    for d in ("a", "b"):
        assert bench.dump_outputs(run, str(tmp_path / d)) <= full // 10
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype == np.float32 and a.ndim == 1 and np.array_equal(a, b), n
    sample = np.load(tmp_path / "a" / "grad.0.weight.npy")
    assert 0 < sample.size < w.size and np.isin(sample, w).all()


def test_synthetic_sweep_workload_model():
    """BASELINE configs[4] (N=2048, Ks=5, 64 graph-conv channels): FLOPs / bytes of SURVEY.md §8(d) with the workload's
    own block table, and the seeded operator has spectral norm 1 (checked at a small size; same constructor)."""
    import torch
    blocks = bench.workload_blocks("syn2048")
    fwd, tot, _ = bench.flops_per_sample(2048, "cheb_graph_conv", 5, blocks=blocks)
    assert abs(fwd / 1e6 - 37865.65) < 0.01 and abs(tot / 1e6 - 79221.49) < 0.01
    assert abs(bench.bytes_per_sample(2048, 2, blocks=blocks) / 1e6 - 15.835) < 0.001
    op = bench.load_operator("syn96", "cheb_graph_conv")
    assert op.shape == (96, 96) and torch.allclose(op, op.T)
    assert abs(float(torch.linalg.matrix_norm(op.double(), ord=2)) - 1.0) < 1e-5
