"""Generates tests/golden/ref_eval_metrics.npz from the UNMODIFIED reference's evaluate_model / evaluate_metric
(script/utility.py:90-121) on seeded data:
    python tests/golden/make_eval_golden.py <reference checkout>

A stub model returns stored predictions batch by batch; the batches are those of DataLoader(shuffle=False) with a partial
last batch; the StandardScaler is fitted on a seeded series with velocity-like statistics (mean ~60, std ~10, N = 37).
The file also records the sklearn version, and whether its float32 inverse_transform equals x * float32(scale_) +
float32(mean_) rounded step by step (the arithmetic stgcn_eval_accumulate implements).
"""
import os
import sys

import numpy as np
import sklearn
import torch
from sklearn.preprocessing import StandardScaler

HERE = os.path.dirname(os.path.abspath(__file__))
N, N_WINDOWS, BATCH = 37, 150, 32


class StoredPredictions(torch.nn.Module):
    """model(x) for the reference's loops: x carries the window indices, the output is the stored prediction."""

    def __init__(self, pred):
        super().__init__()
        self.pred = pred

    def forward(self, x):
        return self.pred[x[:, 0, 0, 0].long()].view(len(x), 1, 1, -1)


def main(ref_root):
    sys.path.insert(0, ref_root)
    from script import utility                                   # noqa: E402  (unmodified reference)

    rng = np.random.default_rng(7)
    series = (60.0 + 10.0 * rng.standard_normal((400, N)) + rng.uniform(-8, 8, N)).astype(np.float64)
    scaler = StandardScaler()
    scaler.fit(series)
    target = scaler.transform(series[:N_WINDOWS]).astype(np.float32)
    pred = (target + 0.3 * rng.standard_normal(target.shape)).astype(np.float32)

    idx = torch.arange(N_WINDOWS, dtype=torch.float32).view(-1, 1, 1, 1).expand(-1, 1, 12, N).contiguous()
    ds = torch.utils.data.TensorDataset(idx, torch.from_numpy(target))
    it = torch.utils.data.DataLoader(ds, batch_size=BATCH, shuffle=False)
    model = StoredPredictions(torch.from_numpy(pred))
    mse = utility.evaluate_model(model, torch.nn.MSELoss(), it)
    mae, rmse, wmape = utility.evaluate_metric(model, it, scaler)

    inv = scaler.inverse_transform(pred.copy())
    f32 = (pred * scaler.scale_.astype(np.float32)).astype(np.float32) + scaler.mean_.astype(np.float32)
    np.savez(os.path.join(HERE, "ref_eval_metrics.npz"), pred=pred, target=target, batch_size=BATCH,
             mean_=scaler.mean_, scale_=scaler.scale_, mse=mse, mae=mae, rmse=rmse, wmape=wmape,
             sklearn_version=sklearn.__version__, inverse_is_f32=bool(np.array_equal(inv, f32)))
    print("written: mse %.9g mae %.9g rmse %.9g wmape %.9g (sklearn %s, float32 inverse %s)"
          % (mse, mae, rmse, wmape, sklearn.__version__, np.array_equal(inv, f32)))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
