"""gno_b200 — host side of the B200-native GNN aggregation path.

`_lib` binds lib/libgno_b200.so (C-ABI in include/gno_b200.h); `plan` builds and
caches dst-sorted CSR plans; `ops` holds the operators with torch_scatter /
torch_sparse semantics; `attention` the graph-attention ops (GATv2 logits, segment softmax,
multi-head attention-weighted aggregation, and all three fused in `gatv2_attention`); `multiagg` several aggregators with degree scalers in
one pass (PNAConv.aggregate).  There is no CPU fallback: importing this package
without the built CUDA library raises.
"""
from . import _lib, attention, autograd, dist, graph, host, multiagg, ops, plan  # noqa: F401
from ._lib import GnoError, launch_count  # noqa: F401
from .attention import attention_aggregate, gatv2_attention, gatv2_logits, softmax  # noqa: F401
from .multiagg import multi_aggregate  # noqa: F401
from .ops import (clear_caches, coalesce, gather_coo, gather_csr, gather_scatter, index_add,  # noqa: F401
                  index_select, scatter, segment_coo, segment_csr, segment_reduce, sort, sort_pairs, spmm,
                  spmm_csr, transpose)
from .plan import CSRPlan, build_plan, plan_cache, plan_from_rowptr  # noqa: F401
