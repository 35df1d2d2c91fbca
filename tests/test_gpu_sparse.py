"""GPU checks of the sparse (CSR) graph-shift-operator path: the SpMM node contraction against an fp64 product (isolated
vertices, a hub row of degree N, many CTAs, vector and scalar channel counts), the graph-conv layers and full models
against the same layers with the densified operator, bit-exact no-grad forwards and repeated steps, and the device
trainer / evaluator with a sparse operator."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

from conftest import rel_l2

pytestmark = pytest.mark.gpu

# per-tensor rel-L2 between the CSR path and the same model on the densified operator (DESIGN.md §2 budgets): fp32 and
# tf32x3 differ only in summation order; bf16 contracts with fp32 values where the dense path rounds the operator to bf16
TOL = {"fp32": 1e-5, "tf32x3": 1e-4, "bf16": 3e-2}
TOL_GRAD = {"fp32": 1e-4, "tf32x3": 1e-4, "bf16": 1e-1}


@pytest.fixture
def precision():
    import stgcn_b200
    yield stgcn_b200.set_precision
    stgcn_b200.set_precision("fp32")


def _op_with_hub(n, degree, seed, hub=True, isolated=(), symmetric=False):
    """Random operator: `degree` entries per row, row `hub` full, rows in `isolated` empty."""
    rng = np.random.default_rng(seed)
    rows = np.repeat(np.arange(n), degree)
    cols = rng.integers(0, n, n * degree)
    if hub:
        rows = np.concatenate([rows, np.full(n, n // 3)])
        cols = np.concatenate([cols, np.arange(n)])
    vals = rng.standard_normal(rows.size) / np.sqrt(degree)
    keep = ~np.isin(rows, isolated)
    m = sp.coo_matrix((vals[keep], (rows[keep], cols[keep])), shape=(n, n)).tocsr()
    if symmetric:
        m = (m + m.T) * 0.5
    return sp.csr_matrix(m, dtype=np.float32)


def _knn(n, degree, symmetric=True, seed=0):
    from stgcn_b200.synthetic import knn_operator
    return knn_operator(n, degree, seed=seed, symmetric=symmetric)


# ------------------------------------------------------------------------------------------------ the kernel alone
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("C", [16, 64, 41])
@pytest.mark.parametrize("n,B,T", [(300, 8, 40), (4500, 2, 3)])
def test_node_contraction_matches_fp64(prec, C, n, B, T, precision, cuda_device):
    """Plane 1 of a Ks = 2 ChebGraphConv's saved stack is L x: compared elementwise with an fp64 product, within the
    error bound of a d-term fp32 sum, (d + 2) 2^-24 sum_j |L_hj x_j|, plus the bf16 rounding of the stored result.
    n = 300 spreads G = 320 planes over ~100 CTAs per row tile; n = 4500 puts a degree-4500 hub row in a tile too large
    to stage."""
    from stgcn_b200.gso import CsrOperator
    from stgcn_b200.layers import ChebGraphConv
    dev = cuda_device
    precision(prec)
    m = _op_with_hub(n, 6, seed=n + C, isolated=(0, 7, n - 1))
    op = CsrOperator(m, dev)
    assert (op.row_ptr[1:] - op.row_ptr[:-1]).max().item() == n and op.row_ptr[1].item() == 0
    torch.manual_seed(C)
    layer = ChebGraphConv(C, C, 2, op, bias=False).to(dev)
    x = torch.randn(B, C, T, n, device=dev)
    y = layer(x)
    saved = y.grad_fn.saved_tensors[1]
    dt = torch.float32 if prec == "fp32" else torch.bfloat16
    plane = B * T * n * C
    got = saved.view(dt)[plane:2 * plane].view(B, T, n, C).double()
    x_cl = x.permute(0, 2, 3, 1).to(dt).double()
    a64 = torch.from_numpy(m.toarray()).double().to(dev)
    ref = torch.einsum("hi,btic->bthc", a64, x_cl)
    mag = torch.einsum("hi,btic->bthc", a64.abs(), x_cl.abs())
    deg = (op.row_ptr[1:] - op.row_ptr[:-1]).double().view(1, 1, n, 1)
    bound = (deg + 2) * 2.0 ** -24 * mag + (0 if prec == "fp32" else 2.0 ** -8 * ref.abs())
    excess = ((got - ref).abs() - bound).max().item()
    assert excess <= 0, (excess, rel_l2(got, ref))
    assert torch.equal(got[:, :, [0, 7, n - 1]], torch.zeros_like(got[:, :, [0, 7, n - 1]]))     # isolated rows
    hub = n // 3
    assert rel_l2(got[:, :, hub], ref[:, :, hub]) < (1e-5 if prec == "fp32" else 4e-3)


# ------------------------------------------------------------------------------------------------ layers
def _layer(kind, op, C, seed):
    from stgcn_b200 import layers
    torch.manual_seed(seed)
    if kind == "cheb":
        return layers.ChebGraphConv(C, C, 3, op, True)
    if kind == "gcn":
        return layers.GraphConv(C, C, op, True)
    return layers.GraphConvLayer("cheb_graph_conv" if kind == "layer_cheb" else "graph_conv", 32, C, 3, op, True)


@pytest.mark.parametrize("prec", ["fp32", "tf32x3", "bf16"])
@pytest.mark.parametrize("kind", ["cheb", "gcn", "layer_cheb", "layer_gcn"])
@pytest.mark.parametrize("symmetric", [True, False])
def test_layers_match_the_densified_operator(prec, kind, symmetric, precision, cuda_device):
    """Outputs and every gradient of the layer on the CSR operator against the same layer on its dense matrix.  With a
    non-symmetric operator the input gradient is right only if the backward contracts with gso^T."""
    from stgcn_b200.gso import CsrOperator
    dev = cuda_device
    precision(prec)
    n, C, B, T = 500, 16, 4, 6
    op = CsrOperator(_knn(n, 8, symmetric=symmetric, seed=3), dev)
    assert op.symmetric == symmetric
    c_in = 32 if kind.startswith("layer") else C
    x = torch.randn(B, c_in, T, n, device=dev)
    outs = []
    for gso in (op, op.to_dense()):
        layer = _layer(kind, gso, C, seed=7).to(dev)
        xi = x.clone().requires_grad_(True)
        y = layer(xi)
        w = torch.randn(y.shape, device=dev, generator=torch.Generator(dev).manual_seed(1))
        (y.float() * w).sum().backward()
        outs.append((y.detach().float(), xi.grad.float(), {k: p.grad for k, p in layer.named_parameters()}))
    (ys, dxs, gs), (yd, dxd, gd) = outs
    assert rel_l2(ys, yd) < TOL[prec], rel_l2(ys, yd)
    assert rel_l2(dxs, dxd) < TOL_GRAD[prec], rel_l2(dxs, dxd)
    for k in gd:
        assert gs[k] is not None and rel_l2(gs[k], gd[k]) < TOL_GRAD[prec], (k, rel_l2(gs[k], gd[k]))


def test_layers_accept_torch_and_scipy_sparse(cuda_device):
    """A torch sparse tensor or scipy matrix is converted once on the first forward and kept on the module."""
    from stgcn_b200.gso import CsrOperator
    from stgcn_b200.layers import GraphConv
    dev = cuda_device
    m = _knn(200, 6, seed=5)
    x = torch.randn(2, 16, 4, 200, device=dev)
    ref = GraphConv(16, 16, CsrOperator(m, dev), True).to(dev)
    for src in (m, torch.from_numpy(m.toarray()).to_sparse()):
        layer = GraphConv(16, 16, src, True).to(dev)
        layer.load_state_dict(ref.state_dict())
        y = layer(x)
        assert isinstance(layer.gso, CsrOperator) and layer.gso.device == x.device
        held = layer.gso
        assert torch.equal(layer(x), y) and layer.gso is held
        assert torch.equal(y, ref(x))


# ------------------------------------------------------------------------------------------------ full models
def _models(kind, m, dev, seed=0):
    from stgcn_b200.gso import CsrOperator
    from stgcn_b200.synthetic import build_model
    blocks = [[1], [64, 16, 64], [64, 16, 64], [128, 128], [1]]
    op = CsrOperator(m, dev)
    sparse = build_model(op, kind, 3, blocks, dev, seed=seed)
    dense = build_model(op.to_dense(), kind, 3, blocks, dev, seed=seed)
    dense.load_state_dict(sparse.state_dict())
    return sparse, dense


def _loss_and_grads(model, x, y):
    model.zero_grad(set_to_none=True)
    loss = torch.nn.functional.mse_loss(model(x).view(len(x), -1).float(), y)
    loss.backward()
    # the align convs of a block whose channels do not shrink get no gradient, in the reference too
    return loss.item(), {k: p.grad.detach().clone() for k, p in model.named_parameters() if p.grad is not None}


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("kind", ["cheb_graph_conv", "graph_conv"])
@pytest.mark.parametrize("n", [2048, 8192])
def test_full_model_matches_the_densified_model(prec, kind, n, precision, cuda_device):
    dev = cuda_device
    precision(prec)
    sparse, dense = _models(kind, _knn(n, 8, seed=n), dev)
    g = torch.Generator().manual_seed(9)
    x = torch.randn(2, 1, 12, n, generator=g).to(dev)
    y = torch.randn(2, n, generator=g).to(dev)
    ls, gs = _loss_and_grads(sparse, x, y)
    ld, gd = _loss_and_grads(dense, x, y)
    assert abs(ls - ld) <= TOL[prec] * abs(ld), (ls, ld)
    assert gs.keys() == gd.keys() and len(gd) > 20
    worst = max(rel_l2(gs[k], gd[k]) for k in gd)
    print(f"[sparse-vs-dense {prec} {kind} N={n}] loss {ls:.6f} / {ld:.6f}; worst grad rel-L2 {worst:.2e}")
    assert worst < TOL_GRAD[prec], worst


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_no_grad_forward_and_repeated_steps_are_bit_identical(prec, precision, cuda_device):
    """The no-grad forward (stgcn_stblock_infer_csr) equals the training forward bit for bit; two identical steps give
    identical losses, and a graph conv's output and input gradient -- the SpMM recurrences both ways -- identical bits
    (no atomics).  Parameter gradients are left out: the weight-gradient kernels of the dense layers sum with atomics."""
    from stgcn_b200.gso import CsrOperator
    from stgcn_b200.layers import ChebGraphConv
    dev = cuda_device
    precision(prec)
    m = _knn(2048, 8, seed=1, symmetric=False)
    sparse, _ = _models("cheb_graph_conv", m, dev)
    x = torch.randn(4, 1, 12, 2048, device=dev)
    y = torch.randn(4, 2048, device=dev)
    sparse.eval()
    with torch.no_grad():
        a = sparse(x)
    b = sparse(x)
    assert b.requires_grad and torch.equal(a, b.detach())
    sparse.train()
    assert _loss_and_grads(sparse, x, y)[0] == _loss_and_grads(sparse, x, y)[0]
    layer = ChebGraphConv(16, 16, 3, CsrOperator(m, dev), True).to(dev)
    xg = torch.randn(4, 16, 10, 2048, device=dev)
    runs = []
    for _ in range(2):
        xi = xg.clone().requires_grad_(True)
        out = layer(xi)
        out.float().sum().backward()
        runs.append((out.detach(), xi.grad))
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])


# ------------------------------------------------------------------------------------------------ trainer / evaluator
def _series(dev, length, n, seed=5):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(length, n, generator=g).to(dev)


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_window_trainer_with_a_sparse_operator(prec, precision, cuda_device):
    """WindowTrainer's epoch loss against the eager loop, as in test_gpu_trainer.py, on a model holding a CSR operator."""
    from stgcn_b200 import optim
    from stgcn_b200.data import DeviceWindows
    from stgcn_b200.gso import CsrOperator
    from stgcn_b200.synthetic import build_model
    from stgcn_b200.train import WindowTrainer
    dev = cuda_device
    precision(prec)
    n, B = 300, 8
    op = CsrOperator(_knn(n, 8, seed=2), dev)
    blocks = [[1], [16, 8, 16], [16, 8, 16], [32, 32], [1]]
    windows = DeviceWindows(_series(dev, 45 + 15, n), 12, 3)

    def bound():
        model = build_model(op, "cheb_graph_conv", 3, blocks, dev, seed=4)
        model.train()
        x, y = windows.batch(start=0, size=B)
        torch.nn.functional.mse_loss(model(x).view(B, -1).float(), y).backward()
        opt = optim.FlatAdamW(model, lr=2e-3, weight_decay=1e-2)
        model.zero_grad(set_to_none=True)
        return model, opt

    def eager(model, opt):
        l_sum, cnt = 0.0, 0
        for s in range(0, len(windows), B):
            x, y = windows.batch(start=s, size=B)
            opt.zero_grad(set_to_none=True)
            loss = torch.nn.functional.mse_loss(model(x).view(len(x), -1).float(), y)
            loss.backward()
            opt.step()
            l_sum += loss.item() * y.shape[0]
            cnt += y.shape[0]
        return l_sum / cnt

    e = [eager(*bound()) for _ in range(2)]
    model, opt = bound()
    trainer = WindowTrainer(model, windows, B, opt)
    try:
        got = trainer.run_epoch()
    finally:
        trainer.close()
    noise = abs(e[0] - e[1]) / abs(e[0])
    floor = 1e-6 if prec == "fp32" else 2e-4
    assert abs(got - e[0]) / abs(e[0]) <= 4 * noise + floor, (got, e)


def test_window_evaluator_with_a_sparse_operator(cuda_device):
    """WindowEvaluator equals evaluate_model, and captures again when the operator is replaced."""
    from stgcn_b200.data import DeviceWindows
    from stgcn_b200.evaluate import WindowEvaluator, evaluate_model
    from stgcn_b200.gso import CsrOperator
    from stgcn_b200.synthetic import build_model
    dev = cuda_device
    n = 400
    op = CsrOperator(_knn(n, 8, seed=6), dev)
    model = build_model(op, "cheb_graph_conv", 3, [[1], [16, 8, 16], [16, 8, 16], [32, 32], [1]], dev, seed=3)
    win = DeviceWindows(_series(dev, 100 + 15, n, seed=8), 12, 3)
    B = 32
    loader = [win.batch(start=s, size=B) for s in range(0, len(win), B)]
    ev = WindowEvaluator(model, win, B)
    m0 = ev.run()
    assert m0["mse"] == evaluate_model(model, torch.nn.MSELoss(), loader)
    g0 = ev.graph
    assert ev.run() == m0 and ev.graph is g0
    op2 = CsrOperator(sp.csr_matrix(_knn(n, 8, seed=6) * np.float32(0.5)), dev)
    for blk in model.st_blocks:
        blk.graph_conv.gso = op2
    m1 = ev.run()
    assert ev.graph is not g0 and m1["mse"] != m0["mse"]
    assert m1["mse"] == evaluate_model(model, torch.nn.MSELoss(), loader)
