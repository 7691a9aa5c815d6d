"""Operator layer: torch tensors in, C-ABI calls out (include/gno_b200.h).

Semantics follow torch-scatter 2.0.9 / torch-sparse 0.6.12 as the reference
scripts call them (op_bm_scripts/benchmark_scatter_*.py:15-19,
benchmark_sparse_coalesce.py:35-37) and the native torch ops they time
(benchmark_native_index_add_.py:13-16, benchmark_native_sort.py:28-30,
benchmark_sparse_spmm.py:12-14).  Everything runs on the CUDA library; CPU
tensors are rejected (there is no fallback).
"""
import collections
import ctypes
import os

import torch

from . import _lib
from ._lib import (GNO_BF16, GNO_F16, GNO_F32, GNO_MAX, GNO_MEAN, GNO_MIN, GNO_MUL, GNO_SUM,
                   REDUCE_IDS, GnoError, check, lib)
from .plan import (CSRPlan, _on_device, _ptr, _stream, _workspace, build_plan, plan_cache,
                   plan_from_rowptr)

_DTYPES = {torch.float32: GNO_F32, torch.float16: GNO_F16, torch.bfloat16: GNO_BF16}


def _dtype_id(t):
    try:
        return _DTYPES[t.dtype]
    except KeyError:
        raise GnoError(f"gno_b200: unsupported dtype {t.dtype} (float32/float16/bfloat16 only)")


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise GnoError("gno_b200 has no CPU path: tensors must live on a CUDA device")


def _reduce_id(reduce):
    try:
        return REDUCE_IDS[reduce]
    except KeyError:
        raise ValueError(f"unknown reduce '{reduce}'")


_memo_store = collections.OrderedDict()
_pad_store = collections.OrderedDict()   # padded copies of x (_pad_for_gather): at most two


def _memo(kind, t, extra, builder, capacity=32):
    """Small LRU keyed on a tensor's identity/version (keeps the tensor alive)."""
    key = (kind, t.data_ptr(), t._version, tuple(t.shape), t.stride(), t.dtype, t.device) + tuple(extra)
    hit = _memo_store.get(key)
    if hit is not None:
        _memo_store.move_to_end(key)
        return hit[0]
    val = builder()
    _memo_store[key] = (val, t)
    while len(_memo_store) > capacity:
        _memo_store.popitem(last=False)
    return val


def _check_range(ids, limit, what):
    """Upstream raises on an out-of-range gather index (index error on CPU, device assert on CUDA);
    the kernels would read out of bounds.  One min/max reduction + host read per index tensor,
    memoised on its identity like the plan."""
    if ids.numel() == 0:
        return
    lo, hi = _memo("idx_range", ids, (), lambda: (int(ids.min()), int(ids.max())))
    if lo < 0 or hi >= limit:
        raise IndexError(f"{what}: index out of range (min {lo}, max {hi}, size {limit})")


def clear_caches():
    plan_cache.clear()
    _memo_store.clear()
    _pad_store.clear()
    _fast_calls.clear()
    from . import attention  # imports this module: bound at call time
    attention._sorted_alpha.clear()


# ------------------------------------------------------------ segment reduce --
def segment_reduce(plan, x, reduce, *, gidx=None, eid=None, weights=None, out=None,
                   accumulate=False, want_arg=False, arg_fill=None, x2=None):
    """out[i, :] = reduce_{k in row i} weights[k] * x[gidx[k], :]   (x is 2-D).

    gidx/eid: int32 [E] tensors or None (identity).  Returns out or (out, arg).
    x2: second gather buffer (same dtype, width and row stride as x): ids >= x.size(0) read row
    id - x.size(0) of x2 (gno_segment_reduce_two).
    """
    _need_cuda(x, gidx, eid, weights, out, x2)
    if x.dim() != 2:
        raise ValueError("segment_reduce expects a 2-D x")
    if x.stride(1) != 1 and x.size(1) > 1:
        x = x.contiguous()
    red = _reduce_id(reduce)
    dt = _dtype_id(x)
    N, F = plan.N, x.size(1)
    dev = x.device
    if out is None:
        out = torch.empty((N, F), dtype=x.dtype, device=dev)
    elif out.dtype != x.dtype or out.dim() != 2 or out.size(0) != N or out.size(1) != F or \
            (out.stride(1) != 1 and F > 1):
        raise ValueError("segment_reduce: bad out tensor")
    arg = None
    if want_arg:
        arg = torch.empty((N, F), dtype=torch.int64, device=dev)
    if arg_fill is None:
        arg_fill = plan.E
    if weights is not None:
        weights = weights.to(x.dtype).contiguous()
    if x2 is not None:
        if x2.dtype != x.dtype or x2.dim() != 2 or x2.size(1) != F or not x.is_contiguous() or \
                not x2.is_contiguous() or (F * x.element_size()) % 16:
            raise ValueError("segment_reduce: x2 must match x (dtype, width), both contiguous with 16-byte rows")
    else:
        x = _pad_for_gather(x, plan)
    csr = plan.csr(gidx, eid if want_arg else None)
    nbytes = ctypes.c_size_t()
    check(lib.gno_segment_reduce_workspace(ctypes.byref(csr), F, dt, red, 1 if want_arg else 0,
                                           ctypes.byref(nbytes)))
    ws = _workspace(nbytes.value, dev) if nbytes.value else None
    ldx = x.stride(0) if x.size(0) > 1 else max(F, 1)
    ldo = out.stride(0) if N > 1 else max(F, 1)
    with _on_device(dev):
        check(lib.gno_segment_reduce_two(ctypes.byref(csr), _ptr(x), x.size(0), ldx, _ptr(x2),
                                         x2.size(0) if x2 is not None else 0, _ptr(weights),
                                         _ptr(out), ldo, _ptr(arg), int(arg_fill), F, dt, red,
                                         1 if accumulate else 0, _ptr(ws), nbytes.value, _stream(dev)))
    return (out, arg) if want_arg else out


def _pad_for_gather(x, plan):
    """Rows whose byte length is not a multiple of 16 (F=602: 2408 B fp32, 1204 B bf16) would be
    gathered with 8/4-byte loads.  When the gather volume dwarfs x (E >> rows), copy x once into a
    scratch whose row stride is a multiple of 16 bytes; the kernel then reads whole 128-bit
    vectors and drops the padding columns on output."""
    es = x.element_size()
    row_bytes = x.size(1) * es
    if row_bytes % 16 == 0 or row_bytes < 64 or plan.E_valid < 4 * x.size(0):
        return x
    if (x.stride(0) * es) % 16 == 0 and x.stride(0) * es >= (row_bytes + 15) // 16 * 16 \
            and x.data_ptr() % 16 == 0:
        return x  # caller already padded
    ld = ((row_bytes + 15) // 16 * 16) // es

    def build():
        xp = torch.empty((x.size(0), ld), dtype=x.dtype, device=x.device)
        with _on_device(x.device):
            check(lib.gno_pad_rows(_ptr(x), x.size(0), row_bytes, x.stride(0) * es, _ptr(xp), ld * es,
                                   _stream(x.device)))
        return xp
    # memoised on the tensor's identity + version like the plan (a benchmark loop, or a layer
    # evaluated twice, re-uses the padded copy; an in-place update of x bumps the version);
    # only while the copy is small enough to keep around
    if x.numel() * es > (1 << 30):
        return build()[:, :x.size(1)]
    key = (x.data_ptr(), x._version, tuple(x.shape), x.stride(), x.dtype, x.device)
    hit = _pad_store.get(key)
    if hit is None:
        hit = (build(), x)                      # keeps x alive, so the pointer cannot be recycled
        _pad_store[key] = hit
        while len(_pad_store) > 2:              # activations change every layer: never hoard copies
            _pad_store.popitem(last=False)
    else:
        _pad_store.move_to_end(key)
    return hit[0][:, :x.size(1)]


def _segment_reduce_lastdim(plan, x2d, reduce, gidx, eid, out2d, accumulate, want_arg, arg_fill):
    red = _reduce_id(reduce)
    dt = _dtype_id(x2d)
    dev = x2d.device
    B, L = x2d.shape
    arg = torch.empty((B, plan.N), dtype=torch.int64, device=dev) if want_arg else None
    csr = plan.csr(gidx, eid if want_arg else None)
    with _on_device(dev):
        check(lib.gno_segment_reduce_lastdim(ctypes.byref(csr), _ptr(x2d), B, L, x2d.stride(0) if B > 1 else L,
                                             _ptr(out2d), out2d.stride(0) if B > 1 else plan.N,
                                             _ptr(arg), int(arg_fill), dt, red,
                                             1 if accumulate else 0, _stream(dev)))
    return arg


# -------------------------------------------------------------------- scatter --
def _index_as_1d(index, src, dim):
    """Return the 1-D index if `index` is 1-D or a stride-0 broadcast of one, else None."""
    if index.dim() == 1:
        return index if (src.dim() == 1 or index.numel() == src.size(dim)) else None
    if index.dim() != src.dim():
        return None
    for d in range(index.dim()):
        if d != dim and index.size(d) > 1 and index.stride(d) != 0:
            return None
    if index.size(dim) != src.size(dim):
        return None
    return index.as_strided((index.size(dim),), (index.stride(dim),), index.storage_offset())


# Prepared launches of the full-shape form, keyed on everything that decides them (index identity +
# version, shapes, strides, dtype, dim, dim_size, reduce).  A hit skips the argument analysis and
# the three memo lookups of the general path: what is left per call is the output allocation and
# one C call — the reference scripts' timeit(100) loops on 0.1-4 MB inputs are host-bound
# (profiles/ref_scripts/: 60-88 us per call in round 1, 19-28 us through the general path).
_fast_calls = collections.OrderedDict()


def _fast_key(src, index, dim, dim_size, reduce, return_arg):
    return (index.data_ptr(), index._version, index.shape, index.stride(), src.shape, src.stride(), src.dtype,
            dim, dim_size, reduce, return_arg)


def _fast_put(key, index, fn):
    _fast_calls[key] = (fn, index)   # the key holds a raw pointer: keep the index tensor alive
    while len(_fast_calls) > 16:
        _fast_calls.popitem(last=False)


def scatter(src, index, dim=-1, out=None, dim_size=None, reduce="sum", return_arg=False):
    """torch_scatter.scatter semantics; returns out or (out, arg) for min/max with return_arg."""
    if out is None and _fast_calls:
        hit = _fast_calls.get(_fast_key(src, index, dim, dim_size, reduce, return_arg))
        if hit is not None:
            return hit[0](src)
    _need_cuda(src, index, out)
    src_in, index_in, dim_in = src, index, dim
    red = _reduce_id(reduce)
    if index.dtype != torch.int64:
        raise ValueError("index must be int64")
    if dim < 0:
        dim += src.dim()
    if dim < 0 or dim >= src.dim():
        raise IndexError("dim out of range")
    want_arg = return_arg and red in (GNO_MIN, GNO_MAX)

    if 1 < index.dim() < src.dim():
        # upstream's broadcast(index, src, dim): missing trailing dims are unsqueezed, then the
        # index is expanded to src's shape (pytorch_scatter utils.py)
        index = index.reshape(tuple(index.shape) + (1,) * (src.dim() - index.dim())).expand(src.shape)
    idx1d = _index_as_1d(index, src, dim)
    if idx1d is None:
        if index.dim() != src.dim():
            raise ValueError("index must be 1-D or have as many dims as src")
        if tuple(index.shape) != tuple(src.shape):
            if any(i > s for i, s in zip(index.shape, src.shape)):
                raise ValueError("index is larger than src")
            src = src[tuple(slice(0, s) for s in index.shape)]
    if dim_size is not None:
        N = int(dim_size)
    elif out is not None:
        N = out.size(dim)
    elif index.numel() == 0:
        N = 0
    else:
        # host sync, as upstream — once per index tensor (identity + version), like the plan
        N = _memo("dim_size", index, (), lambda: int(index.max()) + 1, capacity=16)

    src = src.contiguous()
    shape = list(src.shape)
    E = shape[dim]
    B = 1
    for s in shape[:dim]:
        B *= s
    K = 1
    for s in shape[dim + 1:]:
        K *= s
    out_shape = shape[:dim] + [N] + shape[dim + 1:]
    accumulate = out is not None
    if accumulate:
        if list(out.shape) != out_shape or not out.is_contiguous() or out.dtype != src.dtype:
            raise ValueError("out has the wrong shape/dtype or is not contiguous")
    else:
        out = torch.empty(out_shape, dtype=src.dtype, device=src.device)
    arg = None

    if E > _MAX_PLAN_EDGES and idx1d is not None:
        return _scatter_chunked(src, idx1d, dim, out if accumulate else None, N, reduce, red, want_arg, E)
    if not src.is_floating_point():
        return _scatter_int(src, idx1d, dim, out, accumulate, N, B, E, K, out_shape, reduce, red, want_arg)
    if idx1d is not None:
        plan = plan_cache.get(idx1d.contiguous() if not idx1d.is_contiguous() else idx1d, N)
        # torch_scatter's out= forms: sum/mul accumulate in the kernel; mean = (out + sum) / count;
        # min/max start from out and keep it (arg = sentinel) unless an element beats it strictly
        prev = out if (accumulate and red in (GNO_MIN, GNO_MAX)) else None
        kacc = accumulate and prev is None
        kred = "sum" if (accumulate and red == GNO_MEAN) else reduce
        if prev is not None:
            out = torch.empty(out_shape, dtype=src.dtype, device=src.device)
        karg = want_arg or prev is not None
        if K == 1 and B > 1:
            arg2 = _segment_reduce_lastdim(plan, src.view(B, E), kred, plan.perm, plan.perm,
                                           out.view(B, N), kacc, karg, E)
            if karg:
                arg = arg2.view(out_shape)
        else:
            s3, o3 = src.view(B, E, K), out.view(B, N, K)
            args = []
            for b in range(B):
                r = segment_reduce(plan, s3[b], kred, gidx=plan.perm, eid=plan.perm, out=o3[b],
                                   accumulate=kacc, want_arg=karg, arg_fill=E)
                if karg:
                    args.append(r[1])
            if karg:
                arg = (args[0] if B == 1 else torch.stack(args)).view(out_shape)
        if accumulate and red == GNO_MEAN:
            cnt = (plan.rowptr[1:] - plan.rowptr[:-1]).clamp_(min=1).to(out.dtype)
            out.div_(cnt.view([1] * dim + [N] + [1] * (len(out_shape) - dim - 1)))
        if prev is not None:
            win = (arg != E) & ((out > prev) if red == GNO_MAX else (out < prev))
            prev.copy_(torch.where(win, out, prev))
            out = prev
            arg = torch.where(win, arg, torch.full_like(arg, E)) if want_arg else None
    else:
        index = index.contiguous()
        dt = _dtype_id(src)
        if want_arg:
            arg = torch.empty(out_shape, dtype=torch.int64, device=src.device)
        fs = _full_shape_plan(index, dim, N, B, E, K, dt)
        if fs is not None:
            with _on_device(src.device):
                check(lib.gno_scatter_planned(_ptr(src), _ptr(fs[0]), _ptr(fs[1]), B, E, K, _ptr(out), _ptr(arg),
                                              N, dt, red, 1 if accumulate else 0, _stream(src.device)))
            if not accumulate and index is index_in and src is src_in:
                order_p, ptr_p, dev, dtype = _ptr(fs[0]), _ptr(fs[1]), src.device, src.dtype

                def fast(s_, _keep=fs):
                    o_ = torch.empty(out_shape, dtype=dtype, device=dev)
                    a_ = torch.empty(out_shape, dtype=torch.int64, device=dev) if want_arg else None
                    with _on_device(dev):
                        check(lib.gno_scatter_planned(_ptr(s_), order_p, ptr_p, B, E, K, _ptr(o_), _ptr(a_), N, dt,
                                                      red, 0, _stream(dev)))
                    return (o_, a_) if want_arg else o_
                _fast_put(_fast_key(src_in, index_in, dim_in, dim_size, reduce, return_arg), index_in, fast)
            return (out, arg) if want_arg else out
        nbytes = ctypes.c_size_t()
        check(lib.gno_scatter_elementwise_workspace(B, E, N, K, dt, red, ctypes.byref(nbytes)))
        ws = _workspace(nbytes.value, src.device) if nbytes.value else None
        with _on_device(src.device):
            check(lib.gno_scatter_elementwise(_ptr(src), _ptr(index), B, E, K, _ptr(out), _ptr(arg),
                                              N, dt, red, 1 if accumulate else 0, _ptr(ws), nbytes.value,
                                              _stream(src.device)))
    return (out, arg) if want_arg else out


# Plans index edges with 32 bits.  Longer inputs (benchmark_scatter_multiply.py:52-58 sweeps a
# 2.4 G-element 1-D tensor) are reduced in slices along the scatter dim, each slice on its own
# plan, combined through the out= forms (sum / mul accumulate, mean divides once at the end,
# min / max keep the earlier winner unless a later slice beats it strictly — the sequential order).
_MAX_PLAN_EDGES = int(os.environ.get("GNO_MAX_PLAN_EDGES", str((1 << 31) - 2)))


def _scatter_chunked(src, idx1d, dim, out, N, reduce, red, want_arg, E):
    if red in (GNO_MIN, GNO_MAX) and not src.is_floating_point():
        raise NotImplementedError("gno_b200: integer scatter_min/max beyond 2^31 elements is not supported")
    step = _MAX_PLAN_EDGES
    lead = [slice(None)] * dim
    total, arg = out, None
    inner = "sum" if red == GNO_MEAN else reduce
    for e0 in range(0, E, step):
        e1 = min(E, e0 + step)
        part_src = src[tuple(lead + [slice(e0, e1)])]
        part_idx = idx1d[e0:e1]
        if total is None:
            r = scatter(part_src, part_idx, dim, None, N, inner, return_arg=red in (GNO_MIN, GNO_MAX))
        else:
            r = scatter(part_src, part_idx, dim, total, N, inner, return_arg=red in (GNO_MIN, GNO_MAX))
        if red in (GNO_MIN, GNO_MAX):
            val, a = r
            a = torch.where(a == (e1 - e0), torch.full_like(a, E), a + e0)   # slice positions -> positions along dim
            if arg is None:
                arg = a
                # empty bins of the first slice hold 0: later slices must beat the dtype's init, not 0
                none = a == E
                init = torch.finfo(val.dtype).min if red == GNO_MAX else torch.finfo(val.dtype).max
                val = torch.where(none, torch.full_like(val, init), val) if src.is_floating_point() else val
            else:
                arg = torch.where(a == E, arg, a)                              # a slice that won reports its own position
            total = val
        else:
            total = r
    if red in (GNO_MIN, GNO_MAX):
        if src.is_floating_point():
            total = torch.where(arg == E, torch.zeros_like(total), total)
        return (total, arg) if want_arg else total
    if red == GNO_MEAN:
        cnt = torch.bincount(idx1d[(idx1d >= 0) & (idx1d < N)], minlength=N)[:N].clamp_(min=1)
        shape = [1] * total.dim()
        shape[dim] = N
        total = total / cnt.view(shape).to(total.dtype) if src.is_floating_point() else \
            torch.div(total, cnt.view(shape), rounding_mode="floor")
    return total


_FS_PLAN = os.environ.get("GNO_FS_PLAN", "1") != "0"


def blocked_output_ids(idx3, N, kb):
    """Blocked output id of every element of a full-shape index viewed as [B, E, K] — the sort key of
    gno_scatter_planned's plan (include/gno_b200.h): ob = (((b*ncb + cb)*N + n) << kb) + kk with
    k = cb*2^kb + kk, ncb = ceil(K / 2^kb); out-of-range destinations get `total` (they sort to the
    tail and are dropped).  Returns (ids flattened in element order, total).  Device-agnostic."""
    B, E, K = idx3.shape
    dev = idx3.device
    ncb = (K + (1 << kb) - 1) >> kb
    total = (B * ncb * N) << kb
    k = torch.arange(K, device=dev)
    blk = (torch.arange(B, device=dev).view(B, 1, 1) * ncb + (k >> kb).view(1, 1, K)) * N   # (b*ncb + cb)*N
    o = ((blk + idx3) << kb) + (k & ((1 << kb) - 1)).view(1, 1, K)
    o = torch.where((idx3 >= 0) & (idx3 < N), o, torch.full_like(o, total)).reshape(-1)
    return o, total


def _full_shape_plan(index, dim, N, B, E, K, dt):
    """(order, ptr) of a full-shape index in the blocked layout of gno_scatter_planned
    (include/gno_b200.h), or None.  The first call on an index tensor takes the one-launch atomic
    path (no preparation); from the second call on — the reference scripts' timeit loops, a GNN
    layer reusing its graph — the index is sorted once into a plan cached on the tensor's
    identity + version, and every later call is atomic-free."""
    if not _FS_PLAN or B * E * K == 0:
        return None
    kb_c, ob_c = ctypes.c_int(), ctypes.c_int()
    if not lib.gno_scatter_planned_layout(B, E, K, N, dt, ctypes.byref(kb_c), ctypes.byref(ob_c)):
        return None
    kb, order_bytes = kb_c.value, ob_c.value
    seen = _memo("fs_seen", index, (dim, N), lambda: [0])
    seen[0] += 1
    if seen[0] < 2:
        return None

    def build():
        dev = index.device
        o, total = blocked_output_ids(index.view(B, E, K), N, kb)
        iota = torch.arange(o.numel(), dtype=torch.int32, device=dev)
        skey, perm = sort_pairs(o, iota, 0, max(1, int(total).bit_length()))
        order = (torch.div(perm, K, rounding_mode="floor") % E).to(torch.int16 if order_bytes == 2 else torch.int32)
        ptr = torch.zeros(total + 1, dtype=torch.int64, device=dev)
        counts = torch.bincount(o[o < total], minlength=total)
        torch.cumsum(counts, 0, out=ptr[1:])
        return order.contiguous(), ptr.to(torch.int32)
    return _memo("fs_plan", index, (dim, N, kb, order_bytes), build)


def _scatter_int(src, idx1d, dim, out, accumulate, N, B, E, K, out_shape, reduce, red, want_arg):
    """Integer values (PyG's bookkeeping: scatter_add of ones over the batch vector): exact int64
    accumulation on the cached plan.  1-D / broadcast index only."""
    if idx1d is None:
        raise NotImplementedError("gno_b200: integer scatter covers a 1-D (or broadcast) index")
    if accumulate and red in (GNO_MIN, GNO_MAX):
        raise NotImplementedError("gno_b200: integer scatter_min/max with out= is not supported")
    kind = src.dtype
    if kind not in (torch.int32, torch.int64):
        if kind in (torch.int8, torch.int16, torch.uint8, torch.bool):
            src = src.to(torch.int64)
            if accumulate:
                raise NotImplementedError("gno_b200: out= needs int32 / int64 values")
            out = torch.empty(out_shape, dtype=torch.int64, device=src.device)
        else:
            raise GnoError(f"gno_b200: unsupported dtype {kind}")
    plan = plan_cache.get(idx1d.contiguous(), N)
    arg = torch.empty(out_shape, dtype=torch.int64, device=src.device) if want_arg else None
    csr = plan.csr(plan.perm, plan.perm)
    es = src.element_size()
    s3, o3 = src.view(B, E, K), out.view(B, N, K)
    a3 = arg.view(B, N, K) if want_arg else None
    with _on_device(src.device):
        for b in range(B):
            check(lib.gno_segment_reduce_int(ctypes.byref(csr), _ptr(s3[b]), K, _ptr(o3[b]), K,
                                             _ptr(a3[b]) if want_arg else None, E, K, es, red,
                                             1 if accumulate else 0, _stream(src.device)))
    if kind not in (torch.int32, torch.int64) and kind != torch.bool:
        out = out.to(kind)
    return (out, arg) if want_arg else out


def gather_scatter(x, src_ids, dst_ids, dim_size, reduce="sum", return_arg=False, out=None):
    """Fused message passing: scatter(x.index_select(0, src_ids), dst_ids, 0, dim_size, reduce)
    without materialising the [E, F] messages (the C2/C3 hot path)."""
    _need_cuda(x, src_ids, dst_ids)
    red = _reduce_id(reduce)
    want_arg = return_arg and red in (GNO_MIN, GNO_MAX)
    plan = plan_cache.get(dst_ids, dim_size)
    _check_range(src_ids, x.size(0), "gather_scatter: src_ids")
    gidx = plan.sorted_ids(src_ids)
    x2 = x if x.dim() == 2 else x.reshape(x.size(0), -1)
    r = segment_reduce(plan, x2, reduce, gidx=gidx, eid=plan.perm, want_arg=want_arg,
                       arg_fill=plan.E, out=out, accumulate=out is not None)
    if x.dim() == 2:
        return r
    tail = list(x.shape[1:])
    if want_arg:
        return r[0].view([dim_size] + tail), r[1].view([dim_size] + tail)
    return r.view([dim_size] + tail)


def index_add(input, dim, index, source, inplace=False):
    """Tensor.index_add_(dim, index, source) / torch.index_add on 2-D tensors, dim 0 or 1."""
    _need_cuda(input, index, source)
    if dim < 0:
        dim += input.dim()
    if input.dim() != 2 or source.dim() != 2 or dim not in (0, 1):
        raise NotImplementedError("gno_b200.index_add covers 2-D tensors, dim 0/1")
    out = input if inplace else input.clone()
    if not out.is_contiguous():
        raise ValueError("index_add_: input must be contiguous")
    source = source.contiguous()
    _check_range(index, out.size(dim), "index_add_")  # native torch raises on an out-of-range index
    plan = plan_cache.get(index, out.size(dim))
    if dim == 0:
        segment_reduce(plan, source, "sum", gidx=plan.perm, out=out, accumulate=True)
    else:
        _segment_reduce_lastdim(plan, source, "sum", plan.perm, None, out, True, False, 0)
    return out


def index_select(input, dim, index):
    """torch.index_select on 2-D tensors (dim 0: vectorised row gather; dim 1: last-dim gather)."""
    _need_cuda(input, index)
    if index.dtype != torch.int64 or index.dim() != 1:
        raise ValueError("index must be a 1-D int64 tensor")
    if dim < 0:
        dim += input.dim()
    input = input.contiguous()
    if input.dim() == 2:
        _check_range(index, input.size(dim), "index_select")
    if input.dim() == 2 and dim == 0:
        out = torch.empty((index.numel(), input.size(1)), dtype=input.dtype, device=input.device)
        index = index.contiguous()
        with _on_device(input.device):
            check(lib.gno_gather_rows(_ptr(input), input.size(0), input.size(1) * input.element_size(),
                                      _ptr(index), index.numel(), _ptr(out),
                                      _stream(input.device)))
        return out
    if input.dim() == 2 and dim == 1:
        # out[b, i] = input[b, index[i]]: a segment reduce with one edge per row
        n = index.numel()
        rowptr = _memo("iota_ptr", index, (), lambda: torch.arange(n + 1, dtype=torch.int64, device=index.device))
        plan = _memo("rowptr_plan", rowptr, (n,), lambda: plan_from_rowptr(rowptr, n))
        gidx = _memo("narrow", index, (), lambda: index.to(torch.int32))
        out = torch.empty((input.size(0), n), dtype=input.dtype, device=input.device)
        _segment_reduce_lastdim(plan, input, "sum", gidx, None, out, False, False, 0)
        return out
    raise NotImplementedError("gno_b200.index_select covers 2-D tensors, dim 0/1")


# ----------------------------------------------------------------- segment_csr --
def _csr_plan(indptr, n_elems):
    """Plan of a 1-D indptr over a dim of n_elems elements, plus the element range it covers.
    Upstream lets indptr cover a sub-range [indptr[0], indptr[-1]) of the dim and ignores the
    rest; the plan is built over that range (one host read of the two end pointers per indptr
    tensor — memoised on its identity like every plan)."""
    def build():
        lo, hi = (int(v) for v in indptr[[0, -1]].tolist())
        if lo < 0 or hi < lo or hi > n_elems:
            raise ValueError(f"indptr covers [{lo}, {hi}) but the segment dim has {n_elems} elements")
        ptr = indptr.to(torch.int64)
        if lo:
            ptr = ptr - lo
        return plan_from_rowptr(ptr, hi - lo), lo, hi
    return _memo("csr_plan", indptr, (int(n_elems),), build)


def _csr_nd(src, indptr):
    """Normalise an N-D indptr (torch_scatter: its leading dims broadcast against src, segments run
    along dim = indptr.dim() - 1).  Returns (src3 [B, E, K] contiguous, ptr2 [B or 1, M+1], dim)."""
    dim = indptr.dim() - 1
    if dim >= src.dim():
        raise ValueError("indptr has more dims than src")
    for d in range(dim):
        if indptr.size(d) not in (1, src.size(d)):
            raise ValueError("indptr is not broadcastable to src")
    B = 1
    for s_ in src.shape[:dim]:
        B *= s_
    E = src.size(dim)
    shared = all(indptr.size(d) == 1 for d in range(dim))
    if shared:
        ptr2 = indptr.reshape(1, -1)
    else:
        ptr2 = indptr.expand(list(src.shape[:dim]) + [indptr.size(-1)]).reshape(B, -1)
    return src.contiguous().view(B, E, -1), ptr2, dim


def _flat_rowptr(ptr2, B, E):
    """Per-batch pointers [B, M+1] as ONE rowptr over the flattened [B*E] elements — valid when every
    batch covers its whole dim (ptr[b, 0] == 0, ptr[b, M] == E).  Returns None otherwise."""
    def build():
        ends = ptr2[:, [0, -1]]
        if not bool(((ends[:, 0] == 0) & (ends[:, 1] == E)).all()):
            return (None,)
        off = torch.arange(B, device=ptr2.device, dtype=torch.int64).view(-1, 1) * E
        flat = torch.cat([(ptr2[:, :-1].to(torch.int64) + off).reshape(-1),
                          torch.full((1,), B * E, dtype=torch.int64, device=ptr2.device)])
        return (flat.contiguous(),)
    return _memo("flat_rowptr", ptr2, (B, E), build)[0]


def _segment_ids(ptr2, B, E):
    """Generic per-batch pointers: the segment of every element as a COO index into [B*M]
    (elements outside their batch's pointer range get B*M and are dropped by the plan)."""
    M = ptr2.size(1) - 1
    e = torch.arange(E, device=ptr2.device, dtype=torch.int64).view(1, -1).expand(B, E).contiguous()
    p = ptr2.to(torch.int64).contiguous()
    seg = torch.searchsorted(p, e, right=True) - 1
    ok = (e >= p[:, :1]) & (e < p[:, -1:])
    seg = seg + torch.arange(B, device=ptr2.device, dtype=torch.int64).view(-1, 1) * M
    return torch.where(ok, seg, torch.full_like(seg, B * M)).reshape(-1)


def segment_csr(src, indptr, out=None, reduce="sum", return_arg=False):
    """torch_scatter.segment_csr: segments [indptr[..., m], indptr[..., m+1]) along
    dim = indptr.dim() - 1 of src; the leading dims of indptr broadcast against src
    (upstream docstring: src [10, 6, 64], indptr [1, 4] -> out [10, 3, 64])."""
    _need_cuda(src, indptr, out)
    red = _reduce_id(reduce)
    want_arg = return_arg and red in (GNO_MIN, GNO_MAX)
    if indptr.dim() < 1 or indptr.size(-1) < 1:
        raise ValueError("indptr needs at least one pointer along its last dim")
    if out is not None:
        raise NotImplementedError("gno_b200.segment_csr: out= is not supported")
    if indptr.dim() == 1:
        E = src.size(0)
        plan, lo, hi = _csr_plan(indptr, E)
        x2 = src.contiguous().view(E, -1)[lo:hi]
        r = segment_reduce(plan, x2, reduce, want_arg=want_arg, arg_fill=E)
        shape = [plan.N] + list(src.shape[1:])
        if want_arg:
            arg = r[1]
            if lo:  # positions are along the whole dim, the sentinel stays src.size(dim)
                arg = torch.where(arg == E, arg, arg + lo)
            return r[0].view(shape), arg.view(shape)
        return r.view(shape)
    src3, ptr2, dim = _csr_nd(src, indptr)
    B, E, K = src3.shape
    M = ptr2.size(1) - 1
    out_shape = list(src.shape[:dim]) + [M] + list(src.shape[dim + 1:])
    if ptr2.size(0) == 1 and B > 1:
        # one pointer row for every batch: move the segment dim first ([E, B*K] rows), reduce with the
        # 1-D kernel, move back
        xt = src3.permute(1, 0, 2).reshape(E, B * K)
        r = segment_csr(xt, ptr2[0], None, reduce, return_arg=want_arg)
        if want_arg:
            return (r[0].view(M, B, K).permute(1, 0, 2).reshape(out_shape),
                    r[1].view(M, B, K).permute(1, 0, 2).reshape(out_shape))
        return r.view(M, B, K).permute(1, 0, 2).reshape(out_shape)
    flat = _flat_rowptr(ptr2, B, E) if B > 0 else None
    x2 = src3.view(B * E, K)
    if flat is not None:
        plan = _memo("rowptr_plan", flat, (B * E,), lambda: plan_from_rowptr(flat, B * E))
        r = segment_reduce(plan, x2, reduce, want_arg=want_arg, arg_fill=B * E)
    else:
        ids = _memo("segment_ids", ptr2, (B, E), lambda: _segment_ids(ptr2, B, E))
        plan = plan_cache.get(ids, B * M)
        r = segment_reduce(plan, x2, reduce, gidx=plan.perm, eid=plan.perm, want_arg=want_arg,
                           arg_fill=B * E)
    if want_arg:
        val, arg = r
        # flat positions b*E + e -> e along the dim; sentinel -> E
        arg = torch.where(arg == B * E, torch.full_like(arg, E), arg % max(E, 1))
        return val.view(out_shape), arg.view(out_shape)
    return r.view(out_shape)


def gather_csr(src, indptr):
    """torch_scatter.gather_csr: out[..., e, :] = src[..., m, :] for e in segment m, along
    dim = indptr.dim() - 1; the output has indptr[..., -1] elements along that dim."""
    _need_cuda(src, indptr)
    if indptr.dim() == 1:
        M = indptr.numel() - 1
        if src.size(0) != M:
            raise ValueError("src must have indptr.numel() - 1 rows")
        total = _memo("ptr_last", indptr, (), lambda: int(indptr[-1]))
        plan, lo, hi = _csr_plan(indptr, total)
        rows = _memo("erow64", plan.rowptr, (), lambda: plan.erow.to(torch.int64))
        body = index_select(src.contiguous().view(M, -1), 0, rows)
        if lo:  # elements before the first pointer belong to no segment: zeros, as upstream's empty init
            body = torch.cat([body.new_zeros((lo, body.size(1))), body])
        return body.view([total] + list(src.shape[1:]))
    src3, ptr2, dim = _csr_nd(src, indptr)
    B, M, K = src3.shape
    if ptr2.size(1) - 1 != M:
        raise ValueError("src must have indptr.size(-1) - 1 elements along the segment dim")
    total = _memo("ptr_last_max", indptr, (), lambda: int(indptr[..., -1].max()))
    if ptr2.size(0) == 1:
        r = gather_csr(src3.permute(1, 0, 2).reshape(M, B * K), ptr2[0])
        return r.view(total, B, K).permute(1, 0, 2).reshape(list(src.shape[:dim]) + [total] + list(src.shape[dim + 1:]))
    ids = _memo("segment_ids", ptr2, (B, total), lambda: _segment_ids(ptr2, B, total))
    valid = ids < B * M
    rows = torch.where(valid, ids, torch.zeros_like(ids))
    body = index_select(src3.reshape(B * M, K), 0, rows)
    body = torch.where(valid.view(-1, 1), body, torch.zeros_like(body))
    return body.view(list(src.shape[:dim]) + [total] + list(src.shape[dim + 1:]))


def segment_coo(src, index, out=None, dim_size=None, reduce="sum", return_arg=False):
    """torch_scatter.segment_coo: `index` is sorted along its last dim and addresses dim
    index.dim()-1 of src.  A sorted index is a special case of scatter's: the plan's stable
    dst-sort leaves it in place, so the segment reduce reads src rows in order."""
    _need_cuda(src, index, out)
    if index.dim() < 1 or index.dim() > src.dim():
        raise ValueError("index must have between 1 and src.dim() dims")
    dim = index.dim() - 1
    for d in range(dim):
        if index.size(d) not in (1, src.size(d)):
            raise ValueError("index is not broadcastable to src")
    if index.size(dim) != src.size(dim):
        raise ValueError("index and src differ along the segment dim")
    if index.dim() > 1:
        index = index.reshape(list(index.shape) + [1] * (src.dim() - index.dim())).expand_as(src)
    if dim_size is None and out is None:
        dim_size = int(index.max()) + 1 if index.numel() > 0 else 0  # host sync, as upstream
    return scatter(src, index, dim, out, dim_size, reduce, return_arg=return_arg)


def gather_coo(src, index):
    """torch_scatter.gather_coo: out[..., e, :] = src[..., index[..., e], :] along dim index.dim()-1."""
    _need_cuda(src, index)
    if index.dim() < 1 or index.dim() > src.dim():
        raise ValueError("index must have between 1 and src.dim() dims")
    dim = index.dim() - 1
    lead = list(src.shape[:dim])
    B = 1
    for s in lead:
        B *= s
    n_seg, E = src.size(dim), index.size(dim)
    tail = list(src.shape[dim + 1:])
    src2 = src.contiguous().view(B * n_seg, -1)
    if dim == 0:
        rows = index
    else:
        idx = index.expand(lead + [E]).reshape(B, E)
        rows = (idx + torch.arange(B, device=index.device).unsqueeze(1) * n_seg).reshape(-1)
    return index_select(src2, 0, rows).view(lead + [E] + tail)


# ------------------------------------------------------------------------ spmm --
def spmm(index, value, m, n, matrix, reduce="sum"):
    """torch_sparse.spmm(index, value, m, n, matrix): COO [2, nnz] × dense [n, F] → [m, F]."""
    _need_cuda(index, value, matrix)
    squeeze = matrix.dim() == 1
    mat = matrix.unsqueeze(-1) if squeeze else matrix
    row, col = index[0], index[1]
    plan = plan_cache.get(row, m)
    _check_range(col, mat.size(0), "spmm: column index")
    gidx = plan.sorted_ids(col)
    w = None
    if value is not None:
        v = value.to(mat.dtype).contiguous()

        def _permute():
            o = torch.empty_like(v)
            with _on_device(v.device):
                check(lib.gno_permute_rows(_ptr(v), _ptr(plan.perm), _ptr(o), v.numel(),
                                           v.element_size(), _stream(v.device)))
            return o
        w = _memo("perm_val", value, (plan.rowptr.data_ptr(), str(mat.dtype)), _permute)
    out = segment_reduce(plan, mat.contiguous(), reduce, gidx=gidx, weights=w)
    return out.squeeze(-1) if squeeze else out


def spmm_csr(rowptr, col, value, matrix, reduce="sum", return_arg=False):
    """torch_sparse.matmul(SparseTensor(rowptr, col, value), matrix, reduce) on a given CSR."""
    _need_cuda(rowptr, col, value, matrix)
    red = _reduce_id(reduce)
    want_arg = return_arg and red in (GNO_MIN, GNO_MAX)
    nnz = col.numel()
    plan, lo, hi = _csr_plan(rowptr, nnz)
    if lo != 0 or hi != nnz:
        raise ValueError(f"rowptr covers [{lo}, {hi}) but col has {nnz} entries")

    def _narrow():
        o = torch.empty(nnz, dtype=torch.int32, device=col.device)
        c = col.contiguous()
        with _on_device(col.device):
            check(lib.gno_narrow_i64_to_i32(_ptr(c), _ptr(o), nnz, _stream(col.device)))
        return o
    _check_range(col, matrix.size(0), "spmm_csr: col")
    gidx = col if col.dtype == torch.int32 else _memo("narrow", col, (), _narrow)
    w = None if value is None else value.to(matrix.dtype).contiguous()
    return segment_reduce(plan, matrix.contiguous(), reduce, gidx=gidx, weights=w,
                          want_arg=want_arg, arg_fill=nnz)


def csr_rows(rowptr, nnz):
    """Row id of every CSR entry (int64 [nnz]); memoised with the rowptr's plan."""
    plan, lo, hi = _csr_plan(rowptr, nnz)
    return _memo("erow64", plan.rowptr, (), lambda: plan.erow.to(torch.int64))


def spmm_csr_t(rowptr, col, value, grad, n_cols):
    """Transposed CSR product  out[c, :] = sum_{k: col[k] = c} value[k] * grad[row[k], :]  — the
    backward of spmm_csr w.r.t. the dense matrix.  Same segment-reduce kernel; the plan (sorted by
    column id) is cached on `col`, like upstream caches csr2csc."""
    _need_cuda(rowptr, col, value, grad)
    row = csr_rows(rowptr, col.numel())
    plan = plan_cache.get(col, n_cols)
    gidx = plan.sorted_ids(row)
    w = None
    if value is not None:
        v = value.detach().to(grad.dtype).contiguous()

        def _permute():
            o = torch.empty_like(v)
            with _on_device(v.device):
                check(lib.gno_permute_rows(_ptr(v), _ptr(plan.perm), _ptr(o), v.numel(),
                                           v.element_size(), _stream(v.device)))
            return o
        w = _memo("perm_val", value, (plan.rowptr.data_ptr(), str(grad.dtype)), _permute)
    return segment_reduce(plan, grad.contiguous(), "sum", gidx=gidx, weights=w)


# ------------------------------------------------------- coalesce / transpose --
def coo_order(index, n):
    """(#inversions, #adjacent duplicates) of key=row*n+col — one host sync."""
    status = torch.empty(2, dtype=torch.int64, device=index.device)
    row, col = index[0].contiguous(), index[1].contiguous()
    with _on_device(index.device):
        check(lib.gno_coo_order_check(_ptr(row), _ptr(col), row.numel(), int(n), _ptr(status),
                                      _stream(index.device)))
    inv, dup = status.tolist()
    return int(inv), int(dup)


def _coalesce_impl(row, col, value, m, n, op, flags):
    dev = row.device
    E = row.numel()
    red = _reduce_id(op)
    K, dt, v2 = 0, GNO_F32, None
    if value is not None:
        v2 = value.contiguous().view(E, -1)
        K, dt = v2.size(1), _dtype_id(v2)
    out_row = torch.empty(E, dtype=torch.int64, device=dev)
    out_col = torch.empty(E, dtype=torch.int64, device=dev)
    out_val = torch.empty_like(v2) if v2 is not None else None
    nnz = torch.zeros(1, dtype=torch.int64, device=dev)
    nbytes = ctypes.c_size_t()
    check(lib.gno_coalesce_workspace(E, m, n, K, dt, ctypes.byref(nbytes)))
    ws = _workspace(nbytes.value, dev)
    row, col = row.contiguous(), col.contiguous()
    with _on_device(dev):
        check(lib.gno_coalesce(_ptr(row), _ptr(col), _ptr(v2), K, dt, E,
                               int(m), int(n), red, flags, _ptr(out_row), _ptr(out_col),
                               _ptr(out_val), _ptr(nnz), _ptr(ws), ws.numel(), _stream(dev)))
    cnt = int(nnz.item())  # output size is data dependent: one sync, as upstream
    index = torch.stack([out_row[:cnt], out_col[:cnt]])
    if value is None:
        return index, None
    return index, out_val[:cnt].view([cnt] + list(value.shape[1:]))


def coalesce(index, value, m, n, op="add"):
    """torch_sparse.coalesce(index, value, m, n, op) → (index, value)."""
    _need_cuda(index, value)
    if index.dim() != 2 or index.size(0) != 2 or index.dtype != torch.int64:
        raise ValueError("index must be an int64 [2, nnz] tensor")
    if index.size(1) <= 1:
        return index, value
    inv, dup = coo_order(index, n)
    if inv == 0 and dup == 0:
        return index, value  # upstream early exit: already sorted and unique
    return _coalesce_impl(index[0], index[1], value, m, n, op, 0)


def sort_coo(index, value, m, n):
    """Entries of a COO matrix in (row, col) order, duplicates kept — what torch_sparse's
    SparseStorage does on construction (storage.py: argsort of row*n+col, no merge)."""
    _need_cuda(index, value)
    if index.size(1) <= 1:
        return index, value
    inv, _ = coo_order(index, n)
    if inv == 0:
        return index, value
    return _coalesce_impl(index[0], index[1], value, m, n, "add", 2)


def transpose(index, value, m, n, coalesced=True):
    """torch_sparse.transpose(index, value, m, n, coalesced) → (index, value) of the n×m matrix."""
    _need_cuda(index, value)
    row, col = index[0], index[1]
    if not coalesced:
        return torch.stack([col, row]), value
    if index.size(1) == 0:
        return torch.stack([col, row]), value
    # A (row, col)-sorted input is already ascending in the transposed minor key:
    # a stable sort on the new major key alone finishes the job.
    inv, _ = coo_order(index, n)
    flags = 1 if (inv == 0 and n <= (1 << 32)) else 0
    return _coalesce_impl(col, row, value, n, m, "add", flags)


# ------------------------------------------------------------------------ sort --
def _transpose_batched(t, outer, rows, cols):
    """[outer, rows, cols] → [outer, cols, rows] (contiguous, 4- or 8-byte elements)."""
    out = torch.empty(t.numel(), dtype=t.dtype, device=t.device)
    with _on_device(t.device):
        check(lib.gno_transpose_batched(_ptr(t), _ptr(out), outer, rows, cols, t.element_size(),
                                        _stream(t.device)))
    return out


def sort(input, dim=-1, descending=False, stable=True):
    """torch.sort for float32 (always stable); returns (values, int64 indices)."""
    _need_cuda(input)
    if input.dtype != torch.float32:
        raise GnoError("gno_b200.sort: float32 only")
    if input.dim() == 0:
        return input.clone(), torch.zeros((), dtype=torch.int64, device=input.device)
    if dim < 0:
        dim += input.dim()
    x = input.contiguous()
    outer = 1
    for s in x.shape[:dim]:
        outer *= s
    inner = 1
    for s in x.shape[dim + 1:]:
        inner *= s
    length = x.shape[dim]
    if inner > 1 and x.numel() > 0:
        # Sorting along an inner dim scatters its results with a stride of `inner` elements;
        # moving the sorted dim last through a tiled transpose (and the two results back) halves
        # the time of a (20000, 20000) dim-0 sort.
        xt = _transpose_batched(x, outer, length, inner)
        v, i = sort(xt.view(outer * inner, length), -1, descending, stable)
        return (_transpose_batched(v, outer, inner, length).view(x.shape),
                _transpose_batched(i, outer, inner, length).view(x.shape))
    vals = torch.empty_like(x)
    idx = torch.empty(x.shape, dtype=torch.int64, device=x.device)
    nbytes = ctypes.c_size_t()
    check(lib.gno_sort_f32_workspace(outer, length, inner, ctypes.byref(nbytes)))
    ws = _workspace(nbytes.value, x.device)
    with _on_device(x.device):
        check(lib.gno_sort_f32(_ptr(x), _ptr(vals), _ptr(idx), outer, length, inner,
                               1 if descending else 0, _ptr(ws), ws.numel(), _stream(x.device)))
    return vals, idx


def sort_pairs(keys, values=None, begin_bit=0, end_bit=None):
    """Stable ascending radix sort of int32/int64 keys (as unsigned) with optional payload."""
    _need_cuda(keys, values)
    kb = keys.element_size()
    if kb not in (4, 8):
        raise ValueError("keys must be 4 or 8 bytes wide")
    vb = 0 if values is None else values.element_size()
    n = keys.numel()
    keys = keys.contiguous()
    values = values.contiguous() if values is not None else None
    out_k = torch.empty_like(keys)
    out_v = torch.empty_like(values) if values is not None else None
    nbytes = ctypes.c_size_t()
    check(lib.gno_sort_pairs_workspace(n, kb, vb, ctypes.byref(nbytes)))
    ws = _workspace(nbytes.value, keys.device)
    with _on_device(keys.device):
        check(lib.gno_sort_pairs(_ptr(keys), _ptr(out_k), _ptr(values),
                                 _ptr(out_v), n, kb, vb, begin_bit, kb * 8 if end_bit is None else end_bit,
                                 _ptr(ws), ws.numel(), _stream(keys.device)))
    return (out_k, out_v) if values is not None else out_k
