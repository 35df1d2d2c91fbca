"""stgcn_b200 -- B200-native (sm_100a) STGCN ST-block forward/backward behind the reference's layers API.

Importing this package never touches the GPU; the shared library is loaded on first use and there is no
fallback if it is missing (``stgcn_b200._lib.lib()`` raises).
"""
from . import _lib, layers, models, dist, graph, optim, data, gso, synthetic, evaluate
from .layers import (Align, CausalConv1d, CausalConv2d, TemporalConvLayer, ChebGraphConv, GraphConv, GraphConvLayer,
                     STConvBlock, OutputBlock, set_precision, get_precision)
from ._lib import StgcnError, launch_count

__all__ = ["layers", "models", "Align", "CausalConv1d", "CausalConv2d", "TemporalConvLayer", "ChebGraphConv",
           "GraphConv", "GraphConvLayer", "STConvBlock", "OutputBlock", "set_precision", "get_precision",
           "StgcnError", "launch_count"]
