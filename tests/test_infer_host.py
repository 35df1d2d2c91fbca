"""CPU-side checks of the inference entry points (stgcn_*_infer_sizes): the dry planning pass of the default PeMSD7-M
model's blocks in every precision, the live-set bound of the bf16 plan, and the same errors as the training planner."""
import ctypes as C

import pytest


@pytest.fixture(scope="module")
def L():
    import __graft_entry__ as g
    g.build()
    from stgcn_b200 import _lib
    return _lib


def _blocks(L, prec, B=256, N=228):
    """(name, desc, training sizes fn, inference sizes fn) of the default model: blocks [[1], [64, 16, 64] x 2, [128, 128],
    [1]], Kt = Ks = 3, n_his = 12 (main.py defaults), eval mode."""
    lib = L.lib()
    st = lambda c_in, T: L.StblockDesc(B, T, N, c_in, 64, 16, 64, 3, 3, 0, 0, 0, 0.0, 1e-12, prec)
    return [("st0", st(1, 12), lib.stgcn_stblock_sizes, lib.stgcn_stblock_infer_sizes),
            ("st1", st(64, 8), lib.stgcn_stblock_sizes, lib.stgcn_stblock_infer_sizes),
            ("out", L.OutblockDesc(B, 4, N, 64, 128, 128, 1, 4, 0, 0, 0.0, 1e-12, prec), lib.stgcn_outblock_sizes,
             lib.stgcn_outblock_infer_sizes)]


@pytest.mark.parametrize("prec", ["fp32", "tf32x3", "bf16"])
def test_inference_plan_is_smaller_than_the_saved_state(L, prec):
    for name, d, train_sizes, infer_sizes in _blocks(L, L.PREC[prec]):
        sv, ws, iw = C.c_size_t(), C.c_size_t(), C.c_size_t()
        L.check(train_sizes(C.byref(d), C.byref(sv), C.byref(ws)))
        L.check(infer_sizes(C.byref(d), C.byref(iw)))
        assert 0 < iw.value < sv.value, (prec, name, iw.value, sv.value)


def test_bf16_first_block_inference_plan_is_the_live_set(L):
    _, d, _, infer_sizes = _blocks(L, L.PREC["bf16"])[0]
    iw = C.c_size_t()
    L.check(infer_sizes(C.byref(d), C.byref(iw)))
    # transients h1 75 + x0 18.7 + h2 18.7 + h3 60 MB = 172 MB even without reuse; the plan reuses h1's space for h3
    assert iw.value <= 200e6, iw.value


def test_inference_planner_reports_the_training_planner_errors(L):
    lib = L.lib()
    sv, ws, iw = C.c_size_t(), C.c_size_t(), C.c_size_t()
    bad = L.StblockDesc(2, 3, 20, 1, 8, 4, 8, 3, 3, 0, 0, 0, 0.0, 1e-12, 0)     # time axis too short for two convs
    st = lib.stgcn_stblock_sizes(C.byref(bad), C.byref(sv), C.byref(ws))
    msg = lib.stgcn_last_error()
    assert st == L.E_INVALID and b"Kernel size" in msg
    assert lib.stgcn_stblock_infer_sizes(C.byref(bad), C.byref(iw)) == st and lib.stgcn_last_error() == msg
    bad_o = L.OutblockDesc(2, 3, 20, 8, 8, 8, 1, 4, 0, 0, 0.0, 1e-12, 0)        # Ko > T
    st = lib.stgcn_outblock_sizes(C.byref(bad_o), C.byref(sv), C.byref(ws))
    msg = lib.stgcn_last_error()
    assert st == L.E_INVALID and lib.stgcn_outblock_infer_sizes(C.byref(bad_o), C.byref(iw)) == st
    assert lib.stgcn_last_error() == msg
    bad_p = L.StblockDesc(2, 12, 20, 1, 8, 4, 8, 3, 3, 0, 0, 0, 0.0, 1e-12, 7)    # unknown precision
    assert lib.stgcn_stblock_infer_sizes(C.byref(bad_p), C.byref(iw)) == L.E_UNSUPPORTED


def test_eval_accumulate_rejects_bad_arguments_without_gpu(L):
    lib = L.lib()
    assert lib.stgcn_eval_accumulate(None, None, 4, 8, None, None, None, None) == L.E_INVALID
    assert lib.stgcn_eval_accumulate(16, 16, 4, 0, None, None, 16, None) == L.E_INVALID
    assert lib.stgcn_eval_accumulate(16, 16, 4, 1 << 20, None, None, 16, None) == L.E_UNSUPPORTED
