"""CPU-side checks of the training loop: the NAdamW oracle against torch.optim.NAdam(decoupled_weight_decay=True), the
StepLR schedule against torch's scheduler, the early-stopping decisions of the reference (script/earlystopping.py:27-42)
on scripted losses, and the argument checks of stgcn_nadamw_step (they fail before any device work)."""
import ctypes as C

import numpy as np
import pytest
import torch

from nadamw_oracle import nadamw_step


@pytest.mark.parametrize("weight_decay,momentum_decay", [(0.0, 4e-3), (0.05, 4e-3), (0.01, 2e-2)])
def test_nadamw_oracle_matches_torch(weight_decay, momentum_decay):
    """200 steps, long enough for the float32 momentum-cache product to reach 0."""
    g = torch.Generator().manual_seed(7)
    n = 1031
    p0 = torch.randn(n, generator=g)
    p = p0.clone().requires_grad_(True)
    opt = torch.optim.NAdam([p], lr=2e-3, weight_decay=weight_decay, momentum_decay=momentum_decay,
                            decoupled_weight_decay=True, foreach=False)
    pn, m, v, mu = p0.numpy().copy(), np.zeros(n, np.float32), np.zeros(n, np.float32), np.float32(1.0)
    for t in range(1, 201):
        gr = torch.randn(n, generator=g) * (0.1 + 0.01 * t)
        p.grad = gr.clone()
        opt.step()
        pn, m, v, mu = nadamw_step(pn, gr.numpy(), m, v, mu, t, lr=2e-3, weight_decay=weight_decay,
                                   momentum_decay=momentum_decay)
        st = opt.state[p]
        assert mu == np.float32(st["mu_product"].item()), t          # same float32 products, bit for bit
        # fp32 rounding (torch's lerp / addcmul may fuse what numpy rounds twice): ~1e-7 of the largest element
        for ours, theirs in ((pn, p.detach()), (m, st["exp_avg"]), (v, st["exp_avg_sq"])):
            theirs = theirs.numpy()
            assert np.abs(ours - theirs).max() <= 1e-6 * np.abs(theirs).max(), t
    assert mu == 0.0


@pytest.mark.parametrize("step_size,gamma", [(10, 0.95), (1, 0.9), (3, 0.5), (7, 0.999)])
def test_steplr_schedule_equals_torch(step_size, gamma):
    from stgcn_b200.train import steplr_schedule
    p = torch.zeros(1, requires_grad=True)
    opt = torch.optim.SGD([p], lr=1e-3)
    sched = torch.optim.lr_scheduler.StepLR(opt, step_size=step_size, gamma=gamma)
    want = []
    for _ in range(100):
        want.append(opt.param_groups[0]["lr"])
        opt.step()
        sched.step()
    assert steplr_schedule(1e-3, step_size, gamma, 100) == want


def _decide(losses, patience, delta=0.0):
    from stgcn_b200.train import EarlyStopping
    es = EarlyStopping(delta=delta, patience=patience)
    out = []
    for v in losses:
        out.append(es(v))
        if es.early_stop:
            break
    return out, es.early_stop


def test_early_stopping_first_call_improves_and_patience_stops():
    assert _decide([0.5, 0.6, 0.7], patience=2) == ([True, False, False], True)
    assert _decide([0.5, 0.6, 0.4, 0.45, 0.3], patience=2) == ([True, False, True, False, True], False)


def test_early_stopping_exact_ties_are_not_improvements():
    assert _decide([0.5, 0.5, 0.5], patience=2) == ([True, False, False], True)
    assert _decide([0.5, 0.5, 0.49, 0.49], patience=2) == ([True, False, True, False], False)


def test_early_stopping_ties_after_float32_rounding():
    # 1 - 1e-9 is smaller than 1 in fp64 but rounds to 1 in float32: the reference sees a tie
    assert _decide([1.0, 1.0 - 1e-9, 1.0 - 1e-9], patience=2) == ([True, False, False], True)
    # one float32 ulp below 1 is a real improvement
    assert _decide([1.0, float(np.nextafter(np.float32(1.0), np.float32(0)))], patience=2) == ([True, True], False)


def test_early_stopping_delta():
    # improvement needs -v > -best + delta, i.e. v < best - delta
    assert _decide([1.0, 0.95, 0.85, 0.8], patience=3, delta=0.1) == ([True, False, True, False], False)
    assert _decide([1.0, 0.95, 0.92, 0.91], patience=3, delta=0.1) == ([True, False, False, False], True)


@pytest.fixture(scope="module")
def L():
    import __graft_entry__ as g
    g.build()
    from stgcn_b200 import _lib
    return _lib


def test_nadamw_step_rejects_bad_arguments_without_gpu(L):
    lib = L.lib()
    f = C.c_float

    def call(p=16, g=16, m=16, v=16, n=8, step=1, step_dev=None, mu=16):
        return lib.stgcn_nadamw_step(p, g, m, v, n, f(1e-3), f(0.9), f(0.999), f(1e-8), f(0.0), f(1.0), step, step_dev,
                                     None, f(4e-3), mu, None)

    assert call(p=None) == L.E_INVALID
    assert call(mu=None) == L.E_INVALID
    assert call(n=-1) == L.E_INVALID
    assert call(step=0) == L.E_INVALID                 # step numbers start at 1 unless the device counter is given
    assert b"start at 1" in lib.stgcn_last_error()
    assert call(g=20) == L.E_INVALID                   # not 16-byte aligned
    assert b"aligned" in lib.stgcn_last_error()
    assert call(n=0) == 0                              # nothing to do: no launch
