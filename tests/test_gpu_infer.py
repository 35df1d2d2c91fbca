"""No-grad inference path (stgcn_*_infer) and device-side evaluation (stgcn_eval_accumulate, stgcn_b200.evaluate) on the
GPU: bit identity with the training forward in every precision, no backward state, dropout, graph capture, and the
metrics of the reference's evaluate_model / evaluate_metric (script/utility.py:90-121)."""
import math
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from conftest import GOLDEN, GoldenCase, golden_case_names, load_gso
import eval_oracle as TO

pytestmark = pytest.mark.gpu

PRECISIONS = ["fp32", "tf32x3", "bf16"]
DEFAULT_BLOCKS = [[1], [64, 16, 64], [64, 16, 64], [128, 128], [1]]


@pytest.fixture(params=PRECISIONS)
def precision(request):
    import stgcn_b200
    stgcn_b200.set_precision(request.param)
    yield request.param
    stgcn_b200.set_precision("fp32")


def _model(kind, ks, blocks, gso, dev, droprate=0.0, seed=0):
    from stgcn_b200.synthetic import build_model
    return build_model(gso, kind, ks, blocks, dev, droprate=droprate, seed=seed)


def _golden_model(g, dev):
    from stgcn_b200 import models
    c = g.cfg
    args = SimpleNamespace(Kt=c["Kt"], Ks=c["Ks"], act_func=c["act"], graph_conv_type=c["kind"], gso=g.gso.to(dev),
                           enable_bias=c["bias"], droprate=0.0, n_his=c["n_his"])
    cls = models.STGCNChebGraphConv if c["kind"] == "cheb_graph_conv" else models.STGCNGraphConv
    m = cls(args, c["blocks"], c["n"]).to(dev)
    m.load_state_dict({k: v for k, v in g.params.items()}, strict=True)
    return m


def _assert_infer_equals_fwd(model, x):
    model.eval()
    ref = model(x)                                   # grad enabled, parameters require grad: the training forward
    assert ref.requires_grad
    with torch.no_grad():
        a = model(x)
    with torch.inference_mode():
        b = model(x)
    assert not a.requires_grad and torch.equal(a, ref.detach())
    assert torch.equal(b, ref.detach())


WORKLOADS = [("pemsd7m", "cheb_graph_conv", 3, DEFAULT_BLOCKS, 256),
             ("metrla", "graph_conv", 3, DEFAULT_BLOCKS, 32),
             ("pemsbay", "cheb_graph_conv", 3, DEFAULT_BLOCKS, 16),
             ("syn2048", "cheb_graph_conv", 5, [[1], [64, 64, 64], [64, 64, 64], [128, 128], [1]], 2)]


@pytest.mark.parametrize("dataset,kind,ks,blocks,B", WORKLOADS, ids=[w[0] for w in WORKLOADS])
def test_no_grad_forward_is_bit_identical(dataset, kind, ks, blocks, B, precision, cuda_device):
    dev = cuda_device
    if dataset == "syn2048":
        from stgcn_b200.synthetic import synthetic_operator
        gso = synthetic_operator(2048, seed=0)
    else:
        gso = load_gso(dataset, "cheb" if kind == "cheb_graph_conv" else "gcn")
    model = _model(kind, ks, blocks, gso, dev)
    x = torch.randn(B, 1, 12, gso.shape[0], generator=torch.Generator().manual_seed(B)).to(dev)
    _assert_infer_equals_fwd(model, x)


@pytest.mark.parametrize("name", golden_case_names())
def test_no_grad_forward_is_bit_identical_golden(name, precision, cuda_device):
    g = GoldenCase(name)
    model = _golden_model(g, cuda_device)
    _assert_infer_equals_fwd(model, g.x.to(cuda_device))


def test_no_grad_forward_keeps_no_backward_state(cuda_device):
    import stgcn_b200
    from stgcn_b200 import _lib, layers
    dev = cuda_device
    stgcn_b200.set_precision("bf16")
    try:
        model = _model("cheb_graph_conv", 3, DEFAULT_BLOCKS, load_gso("pemsd7m", "cheb"), dev).eval()
        x = torch.randn(256, 1, 12, 228, generator=torch.Generator().manual_seed(1)).to(dev)
        layers._WORKSPACES.clear()                   # the inference workspace is allocated (and counted) below
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        n0 = _lib.launch_count()
        with torch.no_grad():
            y = model(x)
        torch.cuda.synchronize()
        n_infer = _lib.launch_count() - n0
        peak = torch.cuda.max_memory_allocated() - base
        assert peak < 687e6, peak                    # the training forward's saved state alone is 687 MB here
        del y
        n0 = _lib.launch_count()
        y = model(x)
        torch.cuda.synchronize()
        n_train = _lib.launch_count() - n0
        assert 0 < n_infer <= n_train, (n_infer, n_train)
    finally:
        stgcn_b200.set_precision("fp32")


def test_no_grad_dropout_in_train_mode(precision, cuda_device):
    from stgcn_b200 import layers
    dev = cuda_device
    torch.manual_seed(0)
    gso = load_gso("pemsd7m", "cheb").to(dev)
    blk = layers.STConvBlock(3, 3, 228, 1, [64, 16, 64], "glu", "cheb_graph_conv", gso, True, 0.5).to(dev).train()
    x = torch.randn(64, 1, 12, 228, device=dev)
    with torch.no_grad():
        y = blk(x)
    frac = (y == 0).float().mean().item()
    assert abs(frac - 0.5) < 0.02, frac


def test_no_grad_dropout_draws_the_training_forward_masks(precision, cuda_device):
    """Train mode, p = 0.5: with the same seeds (call counter reset) the no-grad forward draws exactly the masks of the
    grad-enabled forward in every block, so the outputs are equal bit for bit."""
    from stgcn_b200 import layers
    dev = cuda_device
    model = _model("cheb_graph_conv", 3, DEFAULT_BLOCKS, load_gso("pemsd7m", "cheb"), dev, droprate=0.5).train()
    x = torch.randn(16, 1, 12, 228, generator=torch.Generator().manual_seed(4)).to(dev)
    layers._SEED_COUNTER = 0
    ref = model(x)
    assert ref.requires_grad
    layers._SEED_COUNTER = 0
    with torch.no_grad():
        a = model(x)
    assert torch.equal(a, ref.detach())
    with torch.no_grad():
        b = model(x)                                 # next seeds: other masks
    assert not torch.equal(b, a)


def test_no_grad_forward_graph_capture(precision, cuda_device):
    dev = cuda_device
    model = _model("cheb_graph_conv", 3, DEFAULT_BLOCKS, load_gso("pemsd7m", "cheb"), dev).eval()
    x = torch.randn(32, 1, 12, 228, generator=torch.Generator().manual_seed(2)).to(dev)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s), torch.no_grad():
        eager = model(x).clone()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s), torch.no_grad():
        out = model(x)
    for _ in range(2):
        out.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, eager)


# ------------------------------------------------------------------------------------------ metrics
def _golden_eval():
    return np.load(os.path.join(GOLDEN, "ref_eval_metrics.npz"))


def _acc_of(batches, mean, scale, dev):
    from stgcn_b200.evaluate import eval_accumulate
    acc = torch.zeros(4, dtype=torch.float64, device=dev)
    for p, t in batches:
        eval_accumulate(torch.from_numpy(p).to(dev), torch.from_numpy(t).to(dev), acc, mean, scale)
    return acc


def test_eval_accumulate_matches_reference_metrics(cuda_device):
    z = _golden_eval()
    dev = cuda_device
    bs = int(z["batch_size"])
    mean = torch.from_numpy(z["mean_"].astype(np.float32)).to(dev)
    scale = torch.from_numpy(z["scale_"].astype(np.float32)).to(dev)
    batches = [(z["pred"][i:i + bs], z["target"][i:i + bs]) for i in range(0, len(z["pred"]), bs)]
    acc = _acc_of(batches, mean, scale, dev)
    acc2 = _acc_of(batches, mean, scale, dev)
    assert torch.equal(acc, acc2)                                 # deterministic, bit for bit
    s = acc.cpu().numpy()
    ref = sum(TO.eval_sums(p, t, z["mean_"], z["scale_"]) for p, t in batches)
    assert np.allclose(s, ref, rtol=1e-12, atol=0)
    mse, mae, rmse, wmape = TO.eval_metrics(s, z["pred"].size)
    for got, r in ((mae, z["mae"]), (rmse, z["rmse"]), (wmape, z["wmape"])):
        assert abs(got - r) <= 1e-12 * abs(r), (got, float(r))
    assert abs(mse - z["mse"]) <= 1e-6 * abs(z["mse"])


def test_eval_accumulate_single_element_is_the_float32_inverse(cuda_device):
    z = _golden_eval()
    dev = cuda_device
    p = z["pred"][:1, 5:6].copy()
    t = z["target"][:1, 5:6].copy()
    m32, s32 = z["mean_"][5:6].astype(np.float32), z["scale_"][5:6].astype(np.float32)
    acc = _acc_of([(p, t)], torch.from_numpy(m32).to(dev), torch.from_numpy(s32).to(dev), dev).cpu().numpy()
    y, yp = t * s32 + m32, p * s32 + m32
    assert y.dtype == np.float32
    d = np.abs(y - yp)
    assert acc[3] == float(y[0, 0]) and acc[1] == float(d[0, 0]) and acc[2] == float((d * d)[0, 0])
    # misaligned buffers and a B * N that is not a multiple of 8 take the scalar path; same sums
    pp, tt = torch.from_numpy(z["pred"][:3, :13].copy()).to(dev), torch.from_numpy(z["target"][:3, :13].copy()).to(dev)
    from stgcn_b200.evaluate import eval_accumulate
    a1 = torch.zeros(4, dtype=torch.float64, device=dev)
    buf = torch.empty(2 * 39 + 1, device=dev)
    buf[1:40].copy_(pp.reshape(-1))
    buf[40:79].copy_(tt.reshape(-1))
    eval_accumulate(buf[1:40].view(3, 13), buf[40:79].view(3, 13), a1)
    ref = TO.eval_sums(z["pred"][:3, :13], z["target"][:3, :13])
    assert np.allclose(a1.cpu().numpy(), ref, rtol=1e-12, atol=0)


class _Scaler:
    def __init__(self, mean_, scale_):
        self.mean_, self.scale_ = mean_, scale_


def _eval_setup(dev, n_windows=150):
    from stgcn_b200.data import DeviceWindows
    gso = load_gso("pemsd7m", "cheb")
    model = _model("cheb_graph_conv", 3, DEFAULT_BLOCKS, gso, dev, seed=3)
    rng = np.random.default_rng(11)
    raw = 60.0 + 10.0 * rng.standard_normal((n_windows + 12 + 3, 228))
    mean_, scale_ = raw.mean(axis=0), raw.std(axis=0)
    series = torch.from_numpy(((raw - mean_) / scale_).astype(np.float32)).to(dev)
    return model, DeviceWindows(series, 12, 3), _Scaler(mean_, scale_)


def _host_reference_loop(model, loader, scaler):
    """script/utility.py:90-121 restated on the same model: per-batch .item() / .cpu().numpy(), numpy metrics."""
    model.eval()
    l_sum, n = 0.0, 0
    mae, sum_y, mse = [], [], []
    m32, s32 = np.asarray(scaler.mean_).astype(np.float32), np.asarray(scaler.scale_).astype(np.float32)
    with torch.no_grad():
        for x, y in loader:
            y_pred = model(x).view(len(x), -1)
            l_sum += torch.nn.functional.mse_loss(y_pred, y).item() * y.shape[0]
            n += y.shape[0]
            yy = (y.cpu().numpy() * s32 + m32).reshape(-1)
            yp = (y_pred.cpu().numpy() * s32 + m32).reshape(-1)
            d = np.abs(yy - yp)
            mae += d.tolist(); sum_y += yy.tolist(); mse += (d ** 2).tolist()
    return l_sum / n, np.array(mae).mean(), np.sqrt(np.array(mse).mean()), np.sum(np.array(mae)) / np.sum(np.array(sum_y))


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_drop_ins_and_window_evaluator(prec, cuda_device):
    import stgcn_b200
    from stgcn_b200.evaluate import WindowEvaluator, evaluate_metric, evaluate_model
    dev = cuda_device
    stgcn_b200.set_precision(prec)
    try:
        model, win, scaler = _eval_setup(dev)
        B = 32
        loader = [win.batch(start=s, size=B) for s in range(0, len(win), B)]
        assert loader[-1][0].shape[0] < B                          # partial tail batch
        r_mse, r_mae, r_rmse, r_wmape = _host_reference_loop(model, loader, scaler)
        mse = evaluate_model(model, torch.nn.MSELoss(), loader)
        mae, rmse, wmape = evaluate_metric(model, loader, scaler)
        assert abs(mse - r_mse) <= 1e-6 * abs(r_mse)
        for got, r in ((mae, r_mae), (rmse, r_rmse), (wmape, r_wmape)):
            assert abs(got - r) <= 1e-12 * abs(r), (got, r)
        ev = WindowEvaluator(model, win, B, scaler=scaler)
        m1, m2 = ev.run(), ev.run()
        assert m1 == m2
        assert m1["mae"] == mae and m1["rmse"] == rmse and m1["wmape"] == wmape
        assert m1["mse"] == mse
    finally:
        stgcn_b200.set_precision("fp32")


def test_window_evaluator_survives_cache_reset_and_rebound_parameters(cuda_device):
    """The graph keeps its workspace alive across a reset of the workspace cache, and a parameter re-bound to new
    storage (as optim.FlatAdamW does) makes run() capture again instead of reading the old addresses."""
    from stgcn_b200 import layers
    from stgcn_b200.evaluate import WindowEvaluator
    dev = cuda_device
    model, win, scaler = _eval_setup(dev)
    ev = WindowEvaluator(model, win, 32, scaler=scaler)
    m0 = ev.run()
    ws_lo = ev.workspace.data_ptr()
    ws_hi = ws_lo + ev.workspace.numel()
    layers._WORKSPACES.clear()
    junk = torch.empty_like(ev.workspace)                           # would take the freed block if it were freed
    assert junk.data_ptr() >= ws_hi or junk.data_ptr() + junk.numel() <= ws_lo
    assert ev.run() == m0
    del junk
    g0 = ev.graph
    with torch.no_grad():
        for p in model.parameters():
            p.data = p.data.clone()
    assert ev.run() == m0 and ev.graph is not g0
    with torch.no_grad():
        model.output.fc2.bias.add_(1.0)                             # in-place update: same graph, new result
    g1 = ev.graph
    assert ev.run()["mse"] != m0["mse"] and ev.graph is g1
