"""CPU oracle of the evaluation sums (TEST INFRASTRUCTURE ONLY -- imported by tests/ only): a numpy restatement of what
stgcn_eval_accumulate adds per batch for the reference's evaluate_model / evaluate_metric (script/utility.py:90-121).
Pinned by tests/test_eval_oracle.py against tests/golden/ref_eval_metrics.npz, which the UNMODIFIED reference computed
(tests/golden/make_eval_golden.py)."""
from __future__ import annotations

import numpy as np


def eval_sums(pred, target, mean=None, scale=None):
    """The four sums stgcn_eval_accumulate adds for one batch of evaluate_model / evaluate_metric (script/utility.py:90-121):
    [sum (pred - target)^2 (evaluate_model's MSELoss, normalised values), sum |d|, sum d^2, sum y] where y / y_pred are
    target / pred after StandardScaler.inverse_transform on float32 arrays (x * float32(scale_), then + float32(mean_),
    each rounded to float32; utility.py:105-106) and d = y - y_pred; |d| and d^2 in float32 (utility.py:107,111), the sums
    in float64 (the reference's lists of Python floats, utility.py:108-111,112-114)."""
    p = np.asarray(pred, dtype=np.float32).reshape(len(pred), -1)
    t = np.asarray(target, dtype=np.float32).reshape(p.shape)
    e = p - t
    y, yp = t.copy(), p.copy()
    if scale is not None:
        s = np.asarray(scale).astype(np.float32)
        y, yp = y * s, yp * s
    if mean is not None:
        m = np.asarray(mean).astype(np.float32)
        y, yp = y + m, yp + m
    d = np.abs(y - yp)
    return np.array([np.sum((e * e).astype(np.float64)), np.sum(d.astype(np.float64)),
                     np.sum((d * d).astype(np.float64)), np.sum(y.astype(np.float64))])


def eval_metrics(acc, count):
    """(MSE, MAE, RMSE, WMAPE) from the summed eval_sums of `count` (window, vertex) elements: evaluate_model's
    l_sum / n (utility.py:97-99) and evaluate_metric's MAE, RMSE, WMAPE (utility.py:112-116)."""
    return acc[0] / count, acc[1] / count, np.sqrt(acc[2] / count), acc[1] / acc[3]
