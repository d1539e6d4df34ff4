"""geot_b200 -- B200-native (sm_100a) drop-in for GeoT's segment-reduction operators.

Same Python surface as the reference package (``/root/reference/geot/__init__.py:4-9``) for the hot
path: ``index_scatter``, ``gather_scatter``, ``gather_weight_scatter``, ``mh_spmm``,
``mh_spmm_transposed``, ``csr_gws``, ``coo_to_csr``; plus ``segment_softmax`` (attention weights over the edges of each
dst row, ``gnn.GATConv``), ``gatv2_score`` (the fused GATv2 attention score, ``gnn.GATv2Conv``), ``graph_attention``
(fused dot-product attention, ``gnn.TransformerConv``), ``format_preprocess`` (segment pointers + edge-count partition) and
``dist`` (dst-row sharding over the GPUs of one box).  The operators are ``torch.ops.geot.*``
registered by ``geot_b200/_C.so`` (thin bindings over the C ABI in ``include/geot_b200.h``).

There is no CPU path and no fallback: importing this package without the compiled extension raises.
"""
import os as _os

import torch as _torch

__version__ = "0.1.0"

_HERE = _os.path.dirname(_os.path.abspath(__file__))
LIB_PATH = _os.path.join(_HERE, "lib", "libgeot_b200.so")
EXT_PATH = _os.path.join(_HERE, "_C.so")


def _load():
    if not (_os.path.exists(EXT_PATH) and _os.path.exists(LIB_PATH)):
        raise ImportError(
            "geot_b200: compiled extension not found (%s, %s). Build it with "
            "`make -f geot_b200/csrc/Makefile -j8` (or `python -c 'import __graft_entry__ as g; g.build()'`). "
            "There is no CPU or eager fallback." % (EXT_PATH, LIB_PATH))
    if not hasattr(_torch.ops.geot, "gather_weight_scatter_impl"):
        _torch.ops.load_library(EXT_PATH)


_load()

from .index_scatter import index_scatter  # noqa: E402
from .gather_scatter import gather_scatter  # noqa: E402
from .gather_weight_scatter import gather_weight_scatter  # noqa: E402
from .mh_spmm import mh_spmm, mh_spmm_transposed  # noqa: E402
from .softmax import segment_softmax  # noqa: E402
from .gatv2 import gatv2_score  # noqa: E402
from .attention import graph_attention  # noqa: E402
from .gather_weight_scatter import sddmm_coo_impl  # noqa: E402
from .csr_gws import csr_gws, coo_to_csr  # noqa: E402
from .format_preprocess import format_preprocess, Plan, clear_plan_cache  # noqa: E402
from . import fake as _fake  # noqa: E402,F401  (register_fake for the C++-registered operators)
from .match_replace import pattern_transform  # noqa: E402
from . import dist  # noqa: E402

__all__ = ["index_scatter", "gather_scatter", "gather_weight_scatter", "mh_spmm", "mh_spmm_transposed", "csr_gws",
           "coo_to_csr", "sddmm_coo_impl", "pattern_transform", "format_preprocess", "Plan", "clear_plan_cache", "dist",
           "segment_softmax", "gatv2_score", "graph_attention"]
