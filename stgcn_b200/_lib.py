"""ctypes binding of libstgcn_b200.so (C ABI declared in include/stgcn_b200.h).

There is deliberately no fallback: if the shared library is missing or fails to load the
import raises, and every entry point raises ``StgcnError`` on a non-zero status.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
# STGCN_B200_LIB: developer knob to A/B another build of the SAME library (tools/build_variants.sh); never a fallback
LIB_PATH = os.environ.get("STGCN_B200_LIB") or os.path.join(_HERE, "lib", "libstgcn_b200.so")

ACT = {"glu": 0, "gtu": 1, "relu": 2, "silu": 3, "linear": 4}
GCONV = {"cheb_graph_conv": 0, "graph_conv": 1}
PREC = {"fp32": 0, "bf16": 1, "tf32x3": 2}

E_INVALID, E_WORKSPACE, E_UNSUPPORTED = 10001, 10002, 10003


class StgcnError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libstgcn_b200 status {code}: {msg}")
        self.code = code


_fp = C.c_void_p   # device pointers travel as integers


class TconvDesc(C.Structure):
    _fields_ = [("B", C.c_int32), ("T", C.c_int32), ("N", C.c_int32), ("c_in", C.c_int32), ("c_out", C.c_int32),
                ("Kt", C.c_int32), ("act", C.c_int32), ("precision", C.c_int32)]


class TconvParams(C.Structure):
    _fields_ = [("conv_w", _fp), ("conv_b", _fp), ("align_w", _fp), ("align_b", _fp)]


TconvGrads = TconvParams


class GconvDesc(C.Structure):
    _fields_ = [("B", C.c_int32), ("T", C.c_int32), ("N", C.c_int32), ("c_in", C.c_int32), ("c_out", C.c_int32),
                ("Ks", C.c_int32), ("gconv", C.c_int32), ("relu", C.c_int32), ("residual", C.c_int32),
                ("precision", C.c_int32)]


class GconvParams(C.Structure):
    _fields_ = [("align_w", _fp), ("align_b", _fp), ("w", _fp), ("b", _fp), ("gso", _fp)]


class GconvGrads(C.Structure):
    _fields_ = [("align_w", _fp), ("align_b", _fp), ("w", _fp), ("b", _fp)]


class LnormDesc(C.Structure):
    _fields_ = [("B", C.c_int32), ("T", C.c_int32), ("N", C.c_int32), ("C", C.c_int32), ("training", C.c_int32),
                ("p_drop", C.c_float), ("eps", C.c_float), ("precision", C.c_int32)]


class StblockDesc(C.Structure):
    _fields_ = [("B", C.c_int32), ("T", C.c_int32), ("N", C.c_int32), ("c_in", C.c_int32), ("c1", C.c_int32),
                ("c2", C.c_int32), ("c3", C.c_int32), ("Kt", C.c_int32), ("Ks", C.c_int32), ("act", C.c_int32),
                ("gconv", C.c_int32), ("training", C.c_int32), ("p_drop", C.c_float), ("eps", C.c_float),
                ("precision", C.c_int32)]


class StblockParams(C.Structure):
    _fields_ = [("tc1", TconvParams), ("gc", GconvParams), ("tc2", TconvParams), ("ln_w", _fp), ("ln_b", _fp)]


class StblockGrads(C.Structure):
    _fields_ = [("tc1", TconvGrads), ("gc", GconvGrads), ("tc2", TconvGrads), ("ln_w", _fp), ("ln_b", _fp)]


class OutblockDesc(C.Structure):
    _fields_ = [("B", C.c_int32), ("T", C.c_int32), ("N", C.c_int32), ("c_in", C.c_int32), ("c0", C.c_int32),
                ("c1", C.c_int32), ("c_end", C.c_int32), ("Ko", C.c_int32), ("act", C.c_int32),
                ("training", C.c_int32), ("p_drop", C.c_float), ("eps", C.c_float), ("precision", C.c_int32)]


class OutblockParams(C.Structure):
    _fields_ = [("tc1", TconvParams), ("ln_w", _fp), ("ln_b", _fp), ("fc1_w", _fp), ("fc1_b", _fp),
                ("fc2_w", _fp), ("fc2_b", _fp)]


class OutblockGrads(C.Structure):
    _fields_ = [("tc1", TconvGrads), ("ln_w", _fp), ("ln_b", _fp), ("fc1_w", _fp), ("fc1_b", _fp),
                ("fc2_w", _fp), ("fc2_b", _fp)]


class CsrGso(C.Structure):
    """stgcn_csr_gso: a sparse graph shift operator, CSR device arrays of gso and of gso^T."""
    _fields_ = [("N", C.c_int32), ("nnz", C.c_int32), ("row_ptr", _fp), ("col", _fp), ("val", _fp),
                ("t_row_ptr", _fp), ("t_col", _fp), ("t_val", _fp)]


# every symbol include/stgcn_b200.h declares: (name, restype, argtypes)
_P = C.POINTER
_sz = C.c_size_t
_SIGNATURES = [
    ("stgcn_version", C.c_int, []),
    ("stgcn_last_error", C.c_char_p, []),
    ("stgcn_launch_count", C.c_uint64, []),
    ("stgcn_set_dropout_step", C.c_int, [_fp]),
    ("stgcn_profile_begin", C.c_int, []),
    ("stgcn_profile_end", C.c_int, [C.c_char_p, _sz, _P(_sz)]),
    ("stgcn_tconv_sizes", C.c_int, [_P(TconvDesc), _P(_sz), _P(_sz)]),
    ("stgcn_tconv_fwd", C.c_int, [_P(TconvDesc), _fp, _P(TconvParams), _fp, _fp, _fp, _sz, _fp]),
    ("stgcn_tconv_bwd", C.c_int, [_P(TconvDesc), _fp, _fp, _fp, _P(TconvParams), _P(TconvGrads), _fp, _fp, _sz, _fp]),
    ("stgcn_gconv_sizes", C.c_int, [_P(GconvDesc), _P(_sz), _P(_sz)]),
    ("stgcn_gconv_fwd", C.c_int, [_P(GconvDesc), _fp, _P(GconvParams), _fp, _fp, _fp, _sz, _fp]),
    ("stgcn_gconv_bwd", C.c_int, [_P(GconvDesc), _fp, _fp, _fp, _P(GconvParams), _P(GconvGrads), _fp, _fp, _sz, _fp]),
    ("stgcn_lnorm_sizes", C.c_int, [_P(LnormDesc), _P(_sz), _P(_sz)]),
    ("stgcn_lnorm_fwd", C.c_int, [_P(LnormDesc), _fp, _fp, _fp, _fp, _fp, C.c_uint64, _fp]),
    ("stgcn_lnorm_bwd", C.c_int, [_P(LnormDesc), _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _sz, C.c_uint64, _fp]),
    ("stgcn_stblock_sizes", C.c_int, [_P(StblockDesc), _P(_sz), _P(_sz)]),
    ("stgcn_stblock_fwd", C.c_int, [_P(StblockDesc), _fp, _P(StblockParams), _fp, _fp, _fp, _sz, C.c_uint64, _fp]),
    ("stgcn_stblock_bwd", C.c_int, [_P(StblockDesc), _fp, _fp, _fp, _P(StblockParams), _P(StblockGrads), _fp, _fp,
                                    _sz, C.c_uint64, _fp]),
    ("stgcn_outblock_sizes", C.c_int, [_P(OutblockDesc), _P(_sz), _P(_sz)]),
    ("stgcn_outblock_fwd", C.c_int, [_P(OutblockDesc), _fp, _P(OutblockParams), _fp, _fp, _fp, _sz, C.c_uint64, _fp]),
    ("stgcn_outblock_bwd", C.c_int, [_P(OutblockDesc), _fp, _fp, _fp, _P(OutblockParams), _P(OutblockGrads), _fp,
                                     _fp, _sz, C.c_uint64, _fp]),
    ("stgcn_stblock_infer_sizes", C.c_int, [_P(StblockDesc), _P(_sz)]),
    ("stgcn_stblock_infer", C.c_int, [_P(StblockDesc), _fp, _P(StblockParams), _fp, _fp, _sz, C.c_uint64, _fp]),
    ("stgcn_outblock_infer_sizes", C.c_int, [_P(OutblockDesc), _P(_sz)]),
    ("stgcn_outblock_infer", C.c_int, [_P(OutblockDesc), _fp, _P(OutblockParams), _fp, _fp, _sz, C.c_uint64, _fp]),
    ("stgcn_gconv_sizes_csr", C.c_int, [_P(GconvDesc), _P(CsrGso), _P(_sz), _P(_sz)]),
    ("stgcn_gconv_fwd_csr", C.c_int, [_P(GconvDesc), _fp, _P(GconvParams), _P(CsrGso), _fp, _fp, _fp, _sz, _fp]),
    ("stgcn_gconv_bwd_csr", C.c_int, [_P(GconvDesc), _fp, _fp, _fp, _P(GconvParams), _P(CsrGso), _P(GconvGrads), _fp,
                                      _fp, _sz, _fp]),
    ("stgcn_stblock_sizes_csr", C.c_int, [_P(StblockDesc), _P(CsrGso), _P(_sz), _P(_sz)]),
    ("stgcn_stblock_fwd_csr", C.c_int, [_P(StblockDesc), _fp, _P(StblockParams), _P(CsrGso), _fp, _fp, _fp, _sz,
                                        C.c_uint64, _fp]),
    ("stgcn_stblock_bwd_csr", C.c_int, [_P(StblockDesc), _fp, _fp, _fp, _P(StblockParams), _P(CsrGso), _P(StblockGrads),
                                        _fp, _fp, _sz, C.c_uint64, _fp]),
    ("stgcn_stblock_infer_sizes_csr", C.c_int, [_P(StblockDesc), _P(CsrGso), _P(_sz)]),
    ("stgcn_stblock_infer_csr", C.c_int, [_P(StblockDesc), _fp, _P(StblockParams), _P(CsrGso), _fp, _fp, _sz,
                                          C.c_uint64, _fp]),
    ("stgcn_eval_accumulate", C.c_int, [_fp, _fp, C.c_int32, C.c_int32, _fp, _fp, _fp, _fp]),
    ("stgcn_umma_selftest", C.c_int, [C.c_int, _fp, _fp, _fp, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_uint32,
                                      C.c_uint32, C.c_uint32, _fp]),
    ("stgcn_debug_timeline", C.c_int, [_fp]),
    ("stgcn_umma_microbench", C.c_int, [C.POINTER(C.c_int32), _fp, _fp]),
    ("stgcn_mse_fwd_bwd", C.c_int, [_fp, _fp, C.c_int64, C.c_float, _fp, _fp, _fp]),
    ("stgcn_adamw_step", C.c_int, [_fp, _fp, _fp, _fp, C.c_int64, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float,
                                   C.c_float, C.c_int64, _fp, _fp, _fp]),
    ("stgcn_nadamw_step", C.c_int, [_fp, _fp, _fp, _fp, C.c_int64, C.c_float, C.c_float, C.c_float, C.c_float,
                                    C.c_float, C.c_float, C.c_int64, _fp, _fp, C.c_float, _fp, _fp]),
    ("stgcn_lion_step", C.c_int, [_fp, _fp, _fp, C.c_int64, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, _fp,
                                  _fp]),
    ("stgcn_gso_build", C.c_int, [_fp, C.c_int32, C.c_int32, C.c_int32, _fp, _fp, _fp, _sz, _fp]),
    ("stgcn_gso_rescale", C.c_int, [_fp, C.c_int32, _fp, _fp, _fp, _sz, _fp]),
    ("stgcn_windows", C.c_int, [_fp, C.c_int64, C.c_int32, C.c_int32, C.c_int32, _fp, C.c_int64, C.c_int32, _fp, _fp,
                                _fp]),
]
EXPORTED_SYMBOLS = [s[0] for s in _SIGNATURES]

_lib: Optional[C.CDLL] = None


def lib() -> C.CDLL:
    """Load (once) and return the shared library; raises if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  stgcn_b200 has no CPU or PyTorch fallback.")
        handle = C.CDLL(LIB_PATH)
        for name, res, args in _SIGNATURES:
            fn = getattr(handle, name)     # AttributeError if the .so does not export it
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(status: int) -> None:
    if status != 0:
        raise StgcnError(status, (lib().stgcn_last_error() or b"").decode(errors="replace"))


def launch_count() -> int:
    return int(lib().stgcn_launch_count())


def profile_begin() -> None:
    check(lib().stgcn_profile_begin())


def profile_end() -> dict:
    """Stop the built-in CUDA-event profiler; returns {"<op tag>:<kernel>": (launches, total_ms)}."""
    cap = 1 << 20
    buf = C.create_string_buffer(cap)
    need = C.c_size_t(0)
    check(lib().stgcn_profile_end(buf, cap, C.byref(need)))
    out = {}
    for line in buf.value.decode().splitlines():
        key, cnt, ms = line.split("\t")
        out[key] = (int(cnt), float(ms))
    return out
