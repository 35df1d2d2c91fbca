"""Pins the evaluation sums of tests/eval_oracle.py (what stgcn_eval_accumulate computes) against the unmodified
reference's evaluate_model / evaluate_metric (tests/golden/make_eval_golden.py -> ref_eval_metrics.npz)."""
import os

import numpy as np

from conftest import GOLDEN
import eval_oracle as T


def _golden():
    return np.load(os.path.join(GOLDEN, "ref_eval_metrics.npz"))


def test_eval_oracle_matches_reference_metrics():
    z = _golden()
    pred, target, bs = z["pred"], z["target"], int(z["batch_size"])
    assert len(pred) % bs != 0                                   # the golden data end with a partial batch
    acc = np.zeros(4)
    for i in range(0, len(pred), bs):
        acc += T.eval_sums(pred[i:i + bs], target[i:i + bs], z["mean_"], z["scale_"])
    mse, mae, rmse, wmape = T.eval_metrics(acc, pred.size)
    for got, ref in ((mae, z["mae"]), (rmse, z["rmse"]), (wmape, z["wmape"])):
        assert abs(got - ref) <= 1e-12 * abs(ref), (got, float(ref))
    assert abs(mse - z["mse"]) <= 1e-6 * abs(z["mse"])             # the reference sums float32 per-batch losses


def test_eval_oracle_inverse_transform_is_float32():
    z = _golden()
    assert bool(z["inverse_is_f32"]), f"sklearn {z['sklearn_version']}: inverse_transform is not the float32 arithmetic"
    p = z["pred"][:1]
    s = T.eval_sums(p, np.zeros_like(p), z["mean_"], z["scale_"])
    y = (np.zeros_like(p) * z["scale_"].astype(np.float32) + z["mean_"].astype(np.float32)).astype(np.float32)
    assert s[3] == np.sum(y.astype(np.float64))


def test_eval_oracle_without_scaler_is_on_normalised_values():
    rng = np.random.default_rng(0)
    p, t = rng.standard_normal((5, 11)).astype(np.float32), rng.standard_normal((5, 11)).astype(np.float32)
    s = T.eval_sums(p, t)
    d = np.abs(t - p)
    assert s[0] == np.sum(((p - t) ** 2).astype(np.float64)) and s[1] == np.sum(d.astype(np.float64))
    assert s[3] == np.sum(t.astype(np.float64))
