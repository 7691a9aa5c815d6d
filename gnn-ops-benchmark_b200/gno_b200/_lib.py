"""ctypes binding of the C-ABI in include/gno_b200.h (lib/libgno_b200.so).

There is no fallback: if the library is missing or a symbol is absent the
import fails loudly — the product path is the CUDA library or nothing.
"""
import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_double, c_int, c_int64, c_size_t, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "lib", "libgno_b200.so")

GNO_F32, GNO_F16, GNO_BF16 = 0, 1, 2
GNO_SUM, GNO_MEAN, GNO_MUL, GNO_MIN, GNO_MAX = 0, 1, 2, 3, 4
REDUCE_IDS = {"sum": GNO_SUM, "add": GNO_SUM, "mean": GNO_MEAN, "mul": GNO_MUL,
              "min": GNO_MIN, "max": GNO_MAX}


class GnoError(RuntimeError):
    pass


class gno_csr(Structure):
    _fields_ = [
        ("N", c_int64),
        ("E", c_int64),
        ("rowptr", c_void_p),
        ("erow", c_void_p),
        ("gidx", c_void_p),
        ("eid", c_void_p),
        ("chunk_len", c_int64),
        ("n_span", c_int64),
        ("srow", c_void_p),
        ("n_empty", c_int64),
        ("zrow", c_void_p),
    ]


# name -> (restype, argtypes); must list every function declared in gno_b200.h
PROTOTYPES = {
    "gno_abi_version": (c_int, []),
    "gno_last_error": (c_char_p, []),
    "gno_launch_count": (c_int64, []),
    "gno_transpose_batched": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int, c_void_p]),
    "gno_sort_pairs_workspace": (c_int, [c_int64, c_int, c_int, POINTER(c_size_t)]),
    "gno_sort_pairs": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int,
                               c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "gno_sort_f32_workspace": (c_int, [c_int64, c_int64, c_int64, POINTER(c_size_t)]),
    "gno_sort_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int,
                             c_void_p, c_size_t, c_void_p]),
    "gno_plan_workspace": (c_int, [c_int64, c_int64, POINTER(c_size_t)]),
    "gno_plan_build": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_void_p, c_void_p,
                               c_void_p, c_void_p, c_size_t, c_void_p]),
    "gno_plan_from_rowptr": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_void_p,
                                     c_void_p]),
    "gno_plan_lists_workspace": (c_int, [c_int64, POINTER(c_size_t)]),
    "gno_plan_lists": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_size_t,
                               c_void_p]),
    "gno_permute_i64_to_i32": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "gno_narrow_i64_to_i32": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "gno_permute_rows": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p]),
    "gno_segment_reduce_workspace": (c_int, [POINTER(gno_csr), c_int64, c_int, c_int, c_int,
                                             POINTER(c_size_t)]),
    "gno_segment_reduce": (c_int, [POINTER(gno_csr), c_void_p, c_int64, c_int64, c_void_p,
                                   c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int, c_int,
                                   c_int, c_void_p, c_size_t, c_void_p]),
    "gno_segment_reduce_two": (c_int, [POINTER(gno_csr), c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p,
                                       c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int, c_int,
                                       c_int, c_void_p, c_size_t, c_void_p]),
    "gno_segment_reduce_heads": (c_int, [POINTER(gno_csr), c_void_p, c_int64, c_void_p, c_int64, c_void_p,
                                         c_int64, c_int, c_void_p, c_size_t, c_void_p]),
    "gno_edge_head_dot": (c_int, [POINTER(gno_csr), c_void_p, c_int64, c_void_p, c_int64, c_int64, c_void_p,
                                  c_int, c_void_p]),
    "gno_segment_softmax_workspace": (c_int, [POINTER(gno_csr), c_int64, POINTER(c_size_t)]),
    "gno_segment_softmax": (c_int, [POINTER(gno_csr), c_void_p, c_void_p, c_int64, c_int64, c_double, c_void_p,
                                    c_int, c_void_p, c_size_t, c_void_p]),
    "gno_segment_softmax_backward": (c_int, [POINTER(gno_csr), c_void_p, c_void_p, c_void_p, c_int64, c_int64,
                                             c_void_p, c_int, c_void_p, c_size_t, c_void_p]),
    "gno_gatv2_logits": (c_int, [POINTER(gno_csr), c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_int64,
                                 c_double, c_void_p, c_int, c_void_p]),
    "gno_gatv2_logits_backward_workspace": (c_int, [POINTER(gno_csr), c_int64, c_int64, c_int, c_int,
                                                    POINTER(c_size_t)]),
    "gno_gatv2_logits_backward": (c_int, [POINTER(gno_csr), c_void_p, c_void_p, c_int64, c_void_p, c_void_p,
                                          c_int64, c_int64, c_double, c_void_p, c_void_p, c_int, c_void_p,
                                          c_size_t, c_void_p]),
    "gno_gatv2_attention_workspace": (c_int, [POINTER(gno_csr), c_int64, c_int64, POINTER(c_size_t)]),
    "gno_gatv2_attention": (c_int, [POINTER(gno_csr), c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_int64,
                                    c_double, c_double, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_size_t,
                                    c_void_p]),
    "gno_gatv2_attention_backward_workspace": (c_int, [POINTER(gno_csr), c_int64, c_int64, c_int, c_int,
                                                       POINTER(c_size_t)]),
    "gno_gatv2_attention_backward": (c_int, [POINTER(gno_csr), c_void_p, c_int64, c_void_p, c_void_p, c_void_p,
                                             c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_double, c_void_p,
                                             c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_size_t, c_void_p]),
    "gno_multi_aggregate_workspace": (c_int, [POINTER(gno_csr), c_int64, c_int64, c_void_p, c_int,
                                              POINTER(c_size_t)]),
    "gno_multi_aggregate": (c_int, [POINTER(gno_csr), c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int,
                                    c_void_p, c_int, c_double, c_double, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_int64, c_int, c_void_p, c_size_t, c_void_p]),
    "gno_multi_aggregate_backward": (c_int, [POINTER(gno_csr), c_void_p, c_int64, c_int64, c_int64, c_void_p,
                                             c_int, c_void_p, c_int, c_double, c_double, c_void_p, c_void_p,
                                             c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "gno_multi_aggregate_coeffs": (c_int, [POINTER(gno_csr), c_int64, c_int64, c_void_p, c_int, c_void_p, c_int,
                                           c_double, c_double, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                           c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "gno_segment_reduce_int": (c_int, [POINTER(gno_csr), c_void_p, c_int64, c_void_p, c_int64, c_void_p,
                                       c_int64, c_int64, c_int, c_int, c_int, c_void_p]),
    "gno_segment_reduce_lastdim": (c_int, [POINTER(gno_csr), c_void_p, c_int64, c_int64, c_int64,
                                           c_void_p, c_int64, c_void_p, c_int64, c_int, c_int,
                                           c_int, c_void_p]),
    "gno_pad_rows": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int64, c_void_p]),
    "gno_push_rows": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int, POINTER(c_void_p),
                              POINTER(c_int64), POINTER(c_int64), c_int64, c_int64, c_int, c_void_p]),
    "gno_push_set_chunk": (c_int, [c_int]),
    "gno_gather_rows": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p,
                                c_void_p]),
    "gno_scatter_elementwise_workspace": (c_int, [c_int64, c_int64, c_int64, c_int64, c_int, c_int,
                                                  POINTER(c_size_t)]),
    "gno_scatter_elementwise": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p,
                                        c_void_p, c_int64, c_int, c_int, c_int, c_void_p, c_size_t,
                                        c_void_p]),
    "gno_scatter_planned_layout": (c_int, [c_int64, c_int64, c_int64, c_int64, c_int, POINTER(c_int),
                                           POINTER(c_int)]),
    "gno_scatter_planned_ok": (c_int, [c_int64, c_int64, c_int64, c_int64, c_int]),
    "gno_scatter_planned": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p,
                                    c_void_p, c_int64, c_int, c_int, c_int, c_void_p]),
    "gno_coalesce_workspace": (c_int, [c_int64, c_int64, c_int64, c_int64, c_int,
                                       POINTER(c_size_t)]),
    "gno_coalesce": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int64, c_int64,
                             c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                             c_void_p, c_size_t, c_void_p]),
    "gno_coo_order_check": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
}


def _load():
    if not os.path.exists(LIB_PATH):
        raise GnoError(
            f"{LIB_PATH} is missing: build it with `python __graft_entry__.py` "
            "(nvcc, sm_100a). There is no CPU fallback.")
    import torch  # noqa: F401  (loads libcudart.so.12 first so the soname resolves)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.gno_abi_version() != 3:
        raise GnoError("libgno_b200.so ABI version mismatch")
    return lib


lib = _load()


def check(rc):
    if rc != 0:
        msg = lib.gno_last_error()
        raise GnoError(f"gno_b200 error {rc}: {msg.decode() if msg else ''}")


def launch_count():
    return int(lib.gno_launch_count())

