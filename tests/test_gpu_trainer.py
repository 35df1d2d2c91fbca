"""GPU checks of the device training loop: the fused NAdamW kernel against the numpy oracle and FlatNAdamW against
torch.optim.NAdam(decoupled_weight_decay=True); FlatNAdamW inside a captured step; WindowTrainer against the
reference-style eager loop (ragged last batch, fp32 and bf16), its dropout draws and its warm-up leaving no trace;
train.fit's StepLR, early stopping, best-epoch parameters and checkpoint."""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import rel_l2
from nadamw_oracle import nadamw_step
from oracle import stgcn_oracle as O

pytestmark = pytest.mark.gpu

N_VERTEX, N_HIS, N_PRED = 23, 12, 3
BLOCKS = [[1], [16, 8, 16], [16, 8, 16], [32, 32], [1]]


def _f32(x):
    return float(np.float32(x))


def _tiny_model(dev, seed=0, droprate=0.0):
    from stgcn_b200.synthetic import build_model
    model = build_model(O.synthetic_gso(N_VERTEX, seed=2), "cheb_graph_conv", 3, BLOCKS, dev, droprate=droprate,
                        seed=seed)
    model.train()
    return model


def _series(dev, length, seed=5):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(length, N_VERTEX, generator=g).to(dev)


def _bound(model, windows, B, which, **kw):
    """A model bound to a fresh flat optimizer: one backward on the first batch binds the gradient buffer; no step."""
    from stgcn_b200 import optim
    x, y = windows.batch(start=0, size=B)
    torch.nn.functional.mse_loss(model(x).view(B, -1).float(), y).backward()
    cls = {"adamw": optim.FlatAdamW, "nadamw": optim.FlatNAdamW, "lion": optim.FlatLion}[which]
    opt = cls(model, **kw)
    model.zero_grad(set_to_none=True)
    return opt


def _live(model):
    """Every parameter of the model, flattened in registration order."""
    return torch.cat([p.detach().reshape(-1) for p in model.parameters()])


def _eager_epoch(model, opt, windows, B):
    """main.py:162-171 with the flat optimizer: per-batch l.item(), the unshuffled order, the ragged last batch."""
    model.train()
    l_sum, n = 0.0, 0
    for s in range(0, len(windows), B):
        x, y = windows.batch(start=s, size=B)
        opt.zero_grad(set_to_none=True)
        pred = model(x).view(len(x), -1).float()
        loss = torch.nn.functional.mse_loss(pred, y)
        loss.backward()
        opt.step()
        l_sum += loss.item() * y.shape[0]
        n += y.shape[0]
    return l_sum / n


# ------------------------------------------------------------------------------------------------ the kernel
@pytest.mark.parametrize("path", ["by_value", "device_step_lr", "grad_scale"])
def test_nadamw_kernel_matches_oracle(path, cuda_device):
    from stgcn_b200 import _lib as L
    dev = cuda_device
    n = 100003                                   # not a multiple of 4: exercises the scalar tail
    lr, wd, psi, betas = 1e-3, 1e-2, 4e-3, (0.9, 0.999)
    scale = 0.5 if path == "grad_scale" else 1.0
    g = torch.Generator().manual_seed(1)
    p = torch.randn(n, generator=g)
    pn, m, v, mu = p.numpy().copy(), np.zeros(n, np.float32), np.zeros(n, np.float32), np.float32(1.0)
    pd, md, vd = p.to(dev), torch.zeros(n, device=dev), torch.zeros(n, device=dev)
    mu_d = torch.ones(2, device=dev)
    steps = torch.zeros(1, dtype=torch.int64, device=dev)
    lr_d = torch.full((1,), 3e-3, device=dev)   # the device learning rate overrides the by-value one
    use_dev = path == "device_step_lr"
    lr_eff = 3e-3 if use_dev else lr
    for t in range(1, 6):
        gr = torch.randn(n, generator=g) * 0.3
        # the kernel receives float32 hyper-parameters: give the oracle the same values
        pn, m, v, mu = nadamw_step(pn, gr.numpy() * np.float32(scale), m, v, mu, t, lr=_f32(lr_eff),
                                   betas=(_f32(betas[0]), _f32(betas[1])), eps=1e-8, weight_decay=_f32(wd),
                                   momentum_decay=_f32(psi))
        gd = gr.to(dev)
        L.check(L.lib().stgcn_nadamw_step(pd.data_ptr(), gd.data_ptr(), md.data_ptr(), vd.data_ptr(), n, C.c_float(lr),
                                          C.c_float(betas[0]), C.c_float(betas[1]), C.c_float(1e-8), C.c_float(wd),
                                          C.c_float(scale), t, steps.data_ptr() if use_dev else None,
                                          lr_d.data_ptr() if use_dev else None, C.c_float(psi), mu_d.data_ptr(),
                                          torch.cuda.current_stream().cuda_stream))
        steps.add_(1)
        assert np.allclose(pd.cpu().numpy(), pn, rtol=3e-6, atol=1e-7), t
        got_mu = float(mu_d[t & 1].item())
        assert abs(got_mu - float(mu)) <= 1e-6 * float(mu), (t, got_mu, float(mu))
    assert np.allclose(md.cpu().numpy(), m, rtol=1e-5, atol=1e-7) and np.allclose(vd.cpu().numpy(), v, rtol=1e-4, atol=1e-9)


def test_flat_nadamw_matches_torch_per_tensor(cuda_device):
    """Five steps of the same model twice: torch's per-tensor NAdam(decoupled_weight_decay=True) vs ONE fused launch on
    the flat buffer.  Same gradients by construction, so the parameters agree to fp32 rounding; dead parameters stay
    untouched."""
    import stgcn_b200
    from stgcn_b200.optim import FlatNAdamW
    dev = cuda_device
    stgcn_b200.set_precision("fp32")
    ma, mb = _tiny_model(dev), _tiny_model(dev)
    mb.load_state_dict(ma.state_dict())
    gen = torch.Generator().manual_seed(1)
    x, y = torch.randn(6, 1, 12, N_VERTEX, generator=gen).to(dev), torch.randn(6, N_VERTEX, generator=gen).to(dev)
    before = {k: v.detach().clone() for k, v in ma.named_parameters()}

    def backward(m):
        m.zero_grad(set_to_none=True)
        torch.nn.functional.mse_loss(m(x).view(x.shape[0], -1), y).backward()

    backward(mb)
    opt_b = FlatNAdamW(mb, lr=2e-3, weight_decay=0.05)
    opt_a = torch.optim.NAdam(ma.parameters(), lr=2e-3, weight_decay=0.05, decoupled_weight_decay=True)
    for it in range(5):
        backward(ma)
        if it > 0:
            backward(mb)
        opt_a.step()
        opt_b.step()
        torch.cuda.synchronize()
        pa = dict(ma.named_parameters())
        for k, p in mb.named_parameters():
            assert rel_l2(p.detach().cpu(), pa[k].detach().cpu()) < 2e-6, (it, k)
    live = set(opt_b.reducer.names)
    for k, p in mb.named_parameters():
        if k not in live:
            assert torch.equal(p.detach(), before[k]), k
    assert int(opt_b.steps_dev.item()) == 5


def test_graphed_step_with_fused_nadamw_trains(cuda_device):
    import stgcn_b200
    from stgcn_b200.graph import GraphedStep
    from stgcn_b200.optim import FlatNAdamW
    dev = cuda_device
    stgcn_b200.set_precision("bf16")
    try:
        model = _tiny_model(dev, seed=3)
        gen = torch.Generator().manual_seed(1)
        x, y = torch.randn(6, 1, 12, N_VERTEX, generator=gen).to(dev), torch.randn(6, N_VERTEX, generator=gen).to(dev)
        torch.nn.functional.mse_loss(model(x).view(x.shape[0], -1).float(), y).backward()
        opt = FlatNAdamW(model, lr=5e-3)
        step = GraphedStep(model, tuple(x.shape), tuple(y.shape), device=dev, warmup=2, post_backward=opt.step)
        n0 = int(opt.steps_dev.item())                  # the warm-up steps are real steps here
        losses = [step(x, y).item() for _ in range(30)]
        assert int(opt.steps_dev.item()) == n0 + 30
        # torch's mu_product after the same number of steps (it does not depend on the gradients)
        q = torch.zeros(1, requires_grad=True)
        ref = torch.optim.NAdam([q], lr=5e-3, betas=(_f32(0.9), 0.999), momentum_decay=_f32(4e-3),
                                decoupled_weight_decay=True, foreach=False)
        for _ in range(n0 + 30):
            q.grad = torch.ones(1)
            ref.step()
        want = ref.state[q]["mu_product"].item()
        got = opt.mu_product.item()
        assert abs(got - want) <= 1e-6 * want, (got, want)
        assert losses[-1] < 0.7 * losses[0], losses[::6]
        step.close()
    finally:
        stgcn_b200.set_precision("fp32")


# ------------------------------------------------------------------------------------------------ WindowTrainer
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("which", ["adamw", "nadamw"])
def test_window_trainer_matches_eager_loop(prec, which, cuda_device):
    """Two epochs over 45 windows at B = 8 (5 full batches and a ragged batch of 5) by WindowTrainer and by the
    reference-style eager loop with the same flat optimizer from the same initial state.  The backward sums with
    atomics, so the eager loop runs twice: trainer-vs-eager must stay within 4x eager-vs-eager plus a floor (fp32 1e-6,
    bf16 2e-4, relative): about 10x the largest trainer-vs-eager difference measured on a B200 (fp32 3.5e-8 in the loss,
    2e-8 in the parameters; bf16 2.2e-6 and 2.1e-5), which includes the torch-vs-library MSE loss."""
    import stgcn_b200
    from stgcn_b200.data import DeviceWindows
    from stgcn_b200.train import WindowTrainer
    dev = cuda_device
    B, epochs = 8, 2
    windows = DeviceWindows(_series(dev, 45 + N_HIS + N_PRED), N_HIS, N_PRED)
    assert len(windows) == 45
    kw = dict(lr=2e-3, weight_decay=1e-2)
    floor = 1e-6 if prec == "fp32" else 2e-4
    stgcn_b200.set_precision(prec)
    try:
        runs = []
        for _ in range(2):
            model = _tiny_model(dev, seed=4)
            opt = _bound(model, windows, B, which, **kw)
            losses = [_eager_epoch(model, opt, windows, B) for _ in range(epochs)]
            runs.append((losses, _live(model)))
        model = _tiny_model(dev, seed=4)
        opt = _bound(model, windows, B, which, **kw)
        state0 = [t.clone() for t in opt.state_tensors()]
        trainer = WindowTrainer(model, windows, B, opt)
        for t, t0 in zip(opt.state_tensors(), state0):
            assert torch.equal(t, t0)                   # warm-up and capture leave no trace
        try:
            losses = [trainer.run_epoch() for _ in range(epochs)]
        finally:
            trainer.close()
        assert int(opt.steps_dev.item()) == epochs * -(-45 // B)
        (e1, p1), (e2, p2) = runs
        for k in range(epochs):
            noise = abs(e1[k] - e2[k]) / abs(e1[k])
            assert abs(losses[k] - e1[k]) / abs(e1[k]) <= 4 * noise + floor, (k, losses, e1, e2)
        noise, err = rel_l2(p2, p1), rel_l2(_live(model), p1)
        print(f"[trainer-vs-eager {prec} {which}] losses {losses} eager {e1} rerun {e2}; params rel-L2 {err:.3e} "
              f"(eager rerun {noise:.3e})")
        assert err <= 4 * noise + floor, (err, noise)
    finally:
        stgcn_b200.set_precision("fp32")


def test_window_trainer_dropout_draws_fresh_masks(cuda_device):
    """With lr = 0 the parameters never move, so two epochs differ only by their dropout masks."""
    import stgcn_b200
    from stgcn_b200.data import DeviceWindows
    from stgcn_b200.train import WindowTrainer
    dev = cuda_device
    stgcn_b200.set_precision("fp32")
    windows = DeviceWindows(_series(dev, 45 + N_HIS + N_PRED), N_HIS, N_PRED)
    out = {}
    for p in (0.0, 0.5):
        model = _tiny_model(dev, seed=6, droprate=p)
        opt = _bound(model, windows, 8, "adamw", lr=0.0, weight_decay=0.0)
        trainer = WindowTrainer(model, windows, 8, opt)
        try:
            out[p] = [trainer.run_epoch() for _ in range(2)]
        finally:
            trainer.close()
    assert out[0.0][0] == out[0.0][1], out
    assert out[0.5][0] != out[0.5][1], out


def test_window_trainer_rejects_a_multi_rank_reducer(cuda_device):
    from stgcn_b200.data import DeviceWindows
    from stgcn_b200.train import WindowTrainer
    dev = cuda_device
    windows = DeviceWindows(_series(dev, 45 + N_HIS + N_PRED), N_HIS, N_PRED)
    model = _tiny_model(dev)
    opt = _bound(model, windows, 8, "adamw")
    opt.reducer._world = lambda: 2
    with pytest.raises(ValueError, match="single process"):
        WindowTrainer(model, windows, 8, opt)


# ------------------------------------------------------------------------------------------------ fit
def test_fit_steplr_early_stopping_and_best_parameters(cuda_device, tmp_path):
    import stgcn_b200
    from stgcn_b200.data import DeviceWindows
    from stgcn_b200.train import WindowTrainer, fit, steplr_schedule
    dev = cuda_device
    stgcn_b200.set_precision("fp32")
    windows = DeviceWindows(_series(dev, 45 + N_HIS + N_PRED), N_HIS, N_PRED)
    model = _tiny_model(dev, seed=7)
    opt = _bound(model, windows, 8, "nadamw", lr=1e-3)
    trainer = WindowTrainer(model, windows, 8, opt)
    # decisions: 1.0 T, 0.8 T, 0.9 F, 0.7 T (best: epoch 3), 0.75 F, 0.7 F (tie), 0.71 F -> stop after epoch 6
    scripted = [1.0, 0.8, 0.9, 0.7, 0.75, 0.7, 0.71, 0.5, 0.4]
    snaps, lrs = [], []

    def val():
        e = len(snaps)
        snaps.append(opt.flat_params.clone())
        lrs.append(opt.lr_dev.item())
        return torch.tensor([scripted[e]], dtype=torch.float64, device=dev) if e % 2 else scripted[e]

    ckpt = str(tmp_path / "best.pt")
    try:
        hist = fit(trainer, len(scripted), val, step_size=2, gamma=0.5, patience=3, checkpoint_path=ckpt)
    finally:
        trainer.close()
    assert [h["improved"] for h in hist] == [True, True, False, True, False, False, False]
    assert len(hist) == 7 and [h["val_loss"] for h in hist] == scripted[:7]
    sched = steplr_schedule(1e-3, 2, 0.5, len(scripted))
    assert [h["lr"] for h in hist] == sched[:7]
    assert lrs == [_f32(v) for v in sched[:7]]
    assert all(np.isfinite(h["train_loss"]) for h in hist)
    assert torch.equal(opt.flat_params, snaps[3])
    fresh = _tiny_model(dev, seed=8)
    fresh.load_state_dict(torch.load(ckpt), strict=True)
    for (k, a), b in zip(fresh.state_dict().items(), model.state_dict().values()):
        assert torch.equal(a, b), k
