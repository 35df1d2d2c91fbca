#!/usr/bin/env python
"""Stores what the UNMODIFIED hazdzz/STGCN computes for the tests that compare against it, so that they run without
it.  Run from the repository root with the path of a checkout of that project:

    python tests/golden/make_ref_golden.py <hazdzz/STGCN checkout>

It writes
  * ``ref_forward_n23.npz``: its model/models.py forward for both graph-conv kinds (N = 23, default-initialised weights
    under torch.manual_seed(123)), with the input, weights and operator it ran on (tests/test_oracle_golden.py);
  * ``ref_windows_small.npz``: its script/dataloader.py data_transform on a seeded 40 x 7 series
    (tests/test_train_oracle.py);
  * ``ref_models_calls.json``: for two golden cases, every layer constructor its model/models.py calls, with the
    arguments, and the submodule path each result ends up under, containers included (tests/test_abi_host.py).
"""
import json
import os
import sys
import types
from types import SimpleNamespace

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))


class _RecordingLayers(types.ModuleType):
    """Stands in for ``model.layers``: builds with the reference's own layer classes and records each call."""

    def __init__(self, inner):
        super().__init__("model.layers")
        self.inner = inner
        self.calls = []

    def __getattr__(self, name):
        cls = getattr(self.inner, name)

        def make(*args, **kwargs):
            module = cls(*args, **kwargs)
            self.calls.append((module, name, args, kwargs))
            return module
        return make


def _import_reference(ref):
    sys.path.insert(0, ref)
    import model                                  # noqa: the reference's own package
    from model import layers as ref_layers
    from script import dataloader                 # noqa
    rec = _RecordingLayers(ref_layers)
    model.layers = rec
    sys.modules["model.layers"] = rec
    from model import models                      # its ``from model import layers`` now resolves to the recorder
    return models, dataloader, rec


def _construction_trace(model, rec, gso):
    """Entries in named_modules() order (parents first): {"path", "container"} for torch.nn containers and
    {"path", "layer", "args"} for the reference's layer calls; the operator argument is stored as the string "gso"."""
    made = {id(m): (name, args, kwargs) for m, name, args, kwargs in rec.calls}
    entries, inside = [], []
    for path, m in model.named_modules():
        if path == "" or any(path.startswith(p + ".") for p in inside):
            continue
        if id(m) in made:
            name, args, kwargs = made[id(m)]
            assert not kwargs, (name, kwargs)
            args = ["gso" if a is gso else a for a in args]
            assert not any(isinstance(a, torch.Tensor) for a in args), name
            entries.append({"path": path, "layer": name, "args": args})
            inside.append(path)
        else:
            assert type(m).__module__.startswith("torch.nn."), (path, type(m))
            entries.append({"path": path, "container": type(m).__name__})
    return entries


def main(ref):
    sys.path.insert(0, ROOT)
    from oracle import stgcn_oracle as O
    models, dataloader, rec = _import_reference(ref)

    # ---- forward of both model classes on a fresh seed
    torch.manual_seed(123)
    n = 23
    gso = O.synthetic_gso(n, seed=5)
    blocks = [[1], [16, 8, 16], [16, 8, 16], [32, 32], [1]]
    out = {"gso": gso.numpy(), "blocks": np.array(json.dumps(blocks))}
    for kind, cls in (("cheb_graph_conv", models.STGCNChebGraphConv), ("graph_conv", models.STGCNGraphConv)):
        args = SimpleNamespace(Kt=3, Ks=3, act_func="glu", graph_conv_type=kind, gso=gso, enable_bias=True,
                               droprate=0.0, n_his=12)
        m = cls(args, blocks, n)
        x = torch.randn(4, 1, 12, n)
        with torch.no_grad():
            y = m(x)
        out[f"{kind}/x"] = x.numpy()
        out[f"{kind}/out"] = y.contiguous().numpy()
        for k, v in m.state_dict().items():
            out[f"{kind}/p:{k}"] = v.numpy()
    np.savez_compressed(os.path.join(HERE, "ref_forward_n23.npz"), **out)

    # ---- sliding windows
    data = np.random.default_rng(5).standard_normal((40, 7))
    x, y = dataloader.data_transform(data, 6, 2, "cpu")
    np.savez(os.path.join(HERE, "ref_windows_small.npz"), data=data, x=x.numpy(), y=y.numpy(), n_his=6, n_pred=2)

    # ---- layer constructor calls of model/models.py
    trace = {}
    for name in ("pemsd7m_cheb3_glu", "tiny_gcn_glu"):
        z = np.load(os.path.join(HERE, f"case_{name}.npz"))
        c = json.loads(str(z["cfg"]))
        g = torch.from_numpy(z["gso"])
        args = SimpleNamespace(Kt=c["Kt"], Ks=c["Ks"], act_func=c["act"], graph_conv_type=c["kind"], gso=g,
                               enable_bias=c["bias"], droprate=0.5, n_his=c["n_his"])
        cls = models.STGCNChebGraphConv if c["kind"] == "cheb_graph_conv" else models.STGCNGraphConv
        rec.calls.clear()
        trace[name] = _construction_trace(cls(args, c["blocks"], c["n"]), rec, g)
    with open(os.path.join(HERE, "ref_models_calls.json"), "w") as f:
        json.dump(trace, f, indent=1)
        f.write("\n")
    for fn in ("ref_forward_n23.npz", "ref_windows_small.npz", "ref_models_calls.json"):
        print(fn, os.path.getsize(os.path.join(HERE, fn)), "bytes")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(os.path.abspath(sys.argv[1]))
