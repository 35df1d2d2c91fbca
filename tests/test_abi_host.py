"""CPU-side checks of the drop-in boundary: the shared library loads, exports every symbol the header declares,
the ctypes mirror has the header's struct layouts, size queries and error reporting work without a GPU, and the
module API keeps the reference's state_dict contract."""
import ctypes as C
import json
import os
import re
import subprocess
import tempfile

import pytest
import torch

from conftest import GOLDEN, ROOT, GoldenCase, golden_case_names

HEADER = os.path.join(ROOT, "include", "stgcn_b200.h")


@pytest.fixture(scope="module")
def L():
    import __graft_entry__ as g
    g.build()
    from stgcn_b200 import _lib
    return _lib


def test_every_declared_symbol_is_exported(L):
    src = open(HEADER).read()
    declared = sorted(set(re.findall(r"\b(stgcn_[a-z0-9_]+)\s*\(", src)))
    assert declared, "no declarations parsed"
    handle = C.CDLL(L.LIB_PATH)
    for name in declared:
        assert hasattr(handle, name), f"{name} declared in the header but not exported"
    assert sorted(L.EXPORTED_SYMBOLS) == declared          # the ctypes table covers exactly the header
    assert L.lib().stgcn_version() == 2


def test_ctypes_structs_match_header_layout(L):
    structs = {"stgcn_tconv_desc": L.TconvDesc, "stgcn_tconv_params": L.TconvParams, "stgcn_tconv_grads": L.TconvGrads,
               "stgcn_gconv_desc": L.GconvDesc, "stgcn_gconv_params": L.GconvParams, "stgcn_gconv_grads": L.GconvGrads,
               "stgcn_lnorm_desc": L.LnormDesc, "stgcn_stblock_desc": L.StblockDesc,
               "stgcn_stblock_params": L.StblockParams, "stgcn_stblock_grads": L.StblockGrads,
               "stgcn_outblock_desc": L.OutblockDesc, "stgcn_outblock_params": L.OutblockParams,
               "stgcn_outblock_grads": L.OutblockGrads}
    prog = '#include <stdio.h>\n#include "stgcn_b200.h"\nint main(void){\n' + "".join(
        f'printf("{n} %zu\\n", sizeof({n}));\n' for n in structs) + "return 0;}\n"
    with tempfile.TemporaryDirectory() as td:
        c = os.path.join(td, "s.c")
        open(c, "w").write(prog)
        exe = os.path.join(td, "s")
        subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe], check=True)
        out = subprocess.run([exe], check=True, capture_output=True, text=True).stdout
    for line in out.strip().splitlines():
        name, size = line.split()
        assert C.sizeof(structs[name]) == int(size), name


def test_size_queries_and_errors_without_gpu(L):
    lib = L.lib()
    sv, ws = C.c_size_t(), C.c_size_t()
    d = L.StblockDesc(256, 12, 228, 1, 64, 16, 64, 3, 3, 0, 0, 0, 0.0, 1e-12, 0)
    assert lib.stgcn_stblock_sizes(C.byref(d), C.byref(sv), C.byref(ws)) == 0
    assert sv.value > 0 and ws.value > 0
    small = L.StblockDesc(1, 12, 228, 1, 64, 16, 64, 3, 3, 0, 0, 0, 0.0, 1e-12, 0)
    sv1, ws1 = C.c_size_t(), C.c_size_t()
    assert lib.stgcn_stblock_sizes(C.byref(small), C.byref(sv1), C.byref(ws1)) == 0
    assert sv1.value < sv.value
    # time axis too short for two temporal convs -> the reference's conv error, here an error status + message
    bad = L.StblockDesc(2, 3, 20, 1, 8, 4, 8, 3, 3, 0, 0, 0, 0.0, 1e-12, 0)
    assert lib.stgcn_stblock_sizes(C.byref(bad), C.byref(sv), C.byref(ws)) == L.E_INVALID
    assert b"Kernel size" in lib.stgcn_last_error()
    with pytest.raises(L.StgcnError):
        L.check(lib.stgcn_stblock_sizes(C.byref(bad), C.byref(sv), C.byref(ws)))
    # unknown activation / Ks < 1 (layers.py:118,148)
    t = L.TconvDesc(2, 6, 20, 4, 4, 3, 9, 0)
    assert lib.stgcn_tconv_sizes(C.byref(t), C.byref(sv), C.byref(ws)) == L.E_UNSUPPORTED
    g = L.GconvDesc(2, 6, 20, 4, 4, 0, 0, 0, 1, 0)
    assert lib.stgcn_gconv_sizes(C.byref(g), C.byref(sv), C.byref(ws)) == L.E_INVALID
    assert b"positive integer" in lib.stgcn_last_error()
    o = L.OutblockDesc(4, 4, 228, 64, 128, 128, 1, 4, 0, 0, 0.0, 1e-12, 0)
    assert lib.stgcn_outblock_sizes(C.byref(o), C.byref(sv), C.byref(ws)) == 0 and sv.value > 0
    # null arguments are rejected, not dereferenced
    assert lib.stgcn_stblock_fwd(None, None, None, None, None, None, 0, 0, None) == L.E_INVALID


def _build(cfg, gso):
    from types import SimpleNamespace
    from stgcn_b200 import models
    args = SimpleNamespace(Kt=cfg["Kt"], Ks=cfg["Ks"], act_func=cfg["act"], graph_conv_type=cfg["kind"], gso=gso,
                           enable_bias=cfg["bias"], droprate=0.5, n_his=cfg["n_his"])
    cls = models.STGCNChebGraphConv if cfg["kind"] == "cheb_graph_conv" else models.STGCNGraphConv
    return cls(args, cfg["blocks"], cfg["n"])


@pytest.mark.parametrize("name", golden_case_names())
def test_state_dict_contract(name):
    """Keys and shapes equal the reference's state_dict (checkpoint compatibility, earlystopping.py:44-47,
    main.py:198); gso stays out of it."""
    g = GoldenCase(name)
    m = _build(g.cfg, g.gso)
    sd = m.state_dict()
    assert list(sd.keys()) == list(g.params.keys())
    for k, v in sd.items():
        assert tuple(v.shape) == tuple(g.params[k].shape), k
    m.load_state_dict(g.params, strict=True)
    assert not any("gso" in k for k in sd)


def test_no_cpu_fallback():
    g = GoldenCase("tiny_cheb3_glu")
    m = _build(g.cfg, g.gso)
    with pytest.raises(RuntimeError, match="no CPU path"):
        m(g.x)


def test_reference_models_py_calls_build_our_layers():
    """The drop-in claim: the layer constructor calls the reference's own model/models.py makes (recorded with their
    arguments and the submodule each result is stored under, tests/golden/make_ref_golden.py), replayed on
    stgcn_b200.layers, build a network with the reference's state_dict."""
    import stgcn_b200.layers as ours
    with open(os.path.join(GOLDEN, "ref_models_calls.json")) as f:
        calls = json.load(f)
    for name in ("pemsd7m_cheb3_glu", "tiny_gcn_glu"):
        g = GoldenCase(name)
        m = torch.nn.Module()
        for e in calls[name]:
            parent, _, attr = e["path"].rpartition(".")
            if "container" in e:
                child = getattr(torch.nn, e["container"])()
            else:
                child = getattr(ours, e["layer"])(*[g.gso if a == "gso" else a for a in e["args"]])
                assert type(child).__module__ == "stgcn_b200.layers"
            m.get_submodule(parent).add_module(attr, child)
        assert list(m.state_dict().keys()) == list(g.params.keys())
        m.load_state_dict(g.params, strict=True)


def _sizes_in_subprocess(env_extra):
    """(saved, workspace) bytes of the default model's two ST blocks and output block in bf16 mode, from a fresh process
    (the library reads its A/B knobs once per process)."""
    import json
    import subprocess
    import sys
    code = r'''
import ctypes as C, json, sys
sys.path.insert(0, %r)
from stgcn_b200 import _lib as L
lib = L.lib()
out = {}
for name, desc in [("st0", L.StblockDesc(256, 12, 228, 1, 64, 16, 64, 3, 3, 0, 0, 1, 0.0, 1e-12, 1)),
                   ("st1", L.StblockDesc(256, 8, 228, 64, 64, 16, 64, 3, 3, 0, 0, 1, 0.0, 1e-12, 1))]:
    sv, ws = C.c_size_t(), C.c_size_t()
    L.check(lib.stgcn_stblock_sizes(C.byref(desc), C.byref(sv), C.byref(ws)))
    out[name] = (sv.value, ws.value)
o = L.OutblockDesc(256, 4, 228, 64, 128, 128, 1, 4, 0, 1, 0.0, 1e-12, 1)
sv, ws = C.c_size_t(), C.c_size_t()
L.check(lib.stgcn_outblock_sizes(C.byref(o), C.byref(sv), C.byref(ws)))
out["out"] = (sv.value, ws.value)
print(json.dumps(out))
''' % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = {k: v for k, v in os.environ.items() if not k.startswith("STGCN_")}
    env.update(env_extra)
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=120)
    assert res.returncode == 0, res.stderr[-800:]
    return json.loads(res.stdout.strip().splitlines()[-1])


def test_bf16_buffer_planning_follows_the_knobs():
    """Sizing (dry) passes of the block-level calls in bf16 mode, on the CPU: both stream configurations plan without
    error; running the weight-gradient kernels on the helper stream keeps their inputs in the non-recycled region, so
    the workspace grows; the saved state does not depend on the stream configuration."""
    base = _sizes_in_subprocess({})
    serial = _sizes_in_subprocess({"STGCN_NO_SIDE_STREAMS": "1"})
    rows1, rows2 = 256 * 10 * 228, 256 * 8 * 228
    # st0 plans (bf16): z1 128ch (reserved; the Cin = 1 kernels recompute it and never touch the buffer) + h1 64ch +
    # stack 3 x 16ch + h2 16ch over T1 steps, gate half Q of tc2 64ch + h3 64ch over T2 steps, LayerNorm statistics; the
    # full 128-channel pre-activation of tc2 would add another 64 channels over T2
    full = (rows1 * (128 + 64 + 48 + 16) + rows2 * (64 + 64)) * 2
    assert full <= base["st0"][0] < full + rows2 * 64 * 2
    for blk in ("st0", "st1", "out"):
        assert base[blk][1] >= serial[blk][1] > 0           # dz & co. move to the keep region
        assert base[blk][0] == serial[blk][0]
