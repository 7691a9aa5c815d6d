"""Graph attention on the fused path: the attention logits of a GATv2 layer, the segment softmax of
torch_geometric.utils.softmax and the multi-head attention-weighted aggregation (GATv2REG,
SURVEY.md §3), forward and backward, on the CUDA library (include/gno_b200.h: gno_gatv2_logits*,
gno_segment_softmax, gno_segment_reduce_heads, gno_edge_head_dot).

A GATv2 layer computes per-edge, per-head logits [E, H] with `gatv2_logits`, normalises them over
each destination's incoming edges with `softmax`, and aggregates
    out[i, h, :] = sum_{e: dst[e] = i} alpha[e, h] * x[src[e], h, :]
with `attention_aggregate`, without materialising the [E, H, C] messages.  `gatv2_attention` is
the same three steps in one pass (gno_gatv2_attention*): the logits and alpha are never stored.
All these ops use the cached dst-sorted plan of the destination index; the backward passes that
scatter to source nodes run on the cached src-sorted plan, so a training step builds two plans
once and reuses them.
"""
import collections
import ctypes

import torch

from . import ops
from ._lib import GNO_SUM, check, lib
from .plan import _on_device, _ptr, _stream, _workspace, plan_cache

EPS = 1e-16  # PyG 2.0.2's softmax: out / (out_sum + 1e-16)


def _softmax_launch(plan, a, b, index, out, backward):
    """One forward (a = logits) or backward (a = y, b = grad of y) pass over [E, H] tensors."""
    E, H = a.shape
    dev = a.device
    csr = plan.csr(None, plan.perm)
    nbytes = ctypes.c_size_t()
    check(lib.gno_segment_softmax_workspace(ctypes.byref(csr), H, ctypes.byref(nbytes)))
    ws = _workspace(nbytes.value, dev) if nbytes.value else None
    dt = ops._dtype_id(a)
    with _on_device(dev):
        if backward:
            check(lib.gno_segment_softmax_backward(ctypes.byref(csr), _ptr(a), _ptr(b), _ptr(index), E, H,
                                                   _ptr(out), dt, _ptr(ws), nbytes.value, _stream(dev)))
        else:
            check(lib.gno_segment_softmax(ctypes.byref(csr), _ptr(a), _ptr(index), E, H, EPS, _ptr(out), dt,
                                          _ptr(ws), nbytes.value, _stream(dev)))
    return out


class _Softmax(torch.autograd.Function):
    @staticmethod
    def forward(ctx, src, plan, index):
        y = _softmax_launch(plan, src, None, index, torch.empty_like(src), False)
        ctx.plan, ctx.index = plan, index
        ctx.save_for_backward(y)
        return y

    @staticmethod
    def backward(ctx, grad_y):
        (y,) = ctx.saved_tensors
        g = grad_y.to(y.dtype).contiguous()
        return _softmax_launch(ctx.plan, y, g, ctx.index, torch.empty_like(y), True), None, None


def softmax(src, index=None, ptr=None, num_nodes=None, dim=0):
    """torch_geometric.utils.softmax (PyG 2.0.2): softmax of `src` [E] or [E, *] over the groups
    that `index` (or the CSR pointer `ptr`) assigns along dim 0; trailing dims are heads.  The group
    maximum follows torch_scatter's rule (NaN never wins, a group whose every entry is -inf gets
    0 after the eps of 1e-16).  Differentiable."""
    ops._need_cuda(src, index, ptr)
    if dim < 0:
        dim += src.dim()
    if dim != 0:
        raise NotImplementedError("gno_b200.softmax: groups along dim 0 only")
    ops._dtype_id(src)
    E = src.size(0)
    H = 1
    for s in src.shape[1:]:
        H *= s
    if E == 0 or H == 0:
        return src.clone()
    src2 = src.contiguous().view(E, H)
    if ptr is not None:
        plan, lo, hi = ops._csr_plan(ptr, E)
        if lo != 0 or hi != E:
            raise ValueError(f"ptr covers [{lo}, {hi}) but src has {E} entries along dim 0")
        idx = None
    elif index is not None:
        if index.dtype != torch.int64 or index.dim() != 1 or index.numel() != E:
            raise ValueError(f"index must be a 1-D int64 tensor of {E} entries")
        if num_nodes is None:  # host sync, as upstream's maybe_num_nodes: once per index tensor
            num_nodes = ops._memo("dim_size", index, (), lambda: int(index.max()) + 1, capacity=16)
        idx = index.contiguous()
        plan = plan_cache.get(idx, int(num_nodes))
    else:
        raise NotImplementedError("gno_b200.softmax needs index or ptr")
    return _Softmax.apply(src2, plan, idx).view(src.shape)


# alpha reordered into a plan's sorted order (one head): at most two entries, like ops._pad_store —
# every layer and step brings a new alpha, so the store must not hoard [E] tensors.
_sorted_alpha = collections.OrderedDict()


def _alpha_sorted(plan, alpha):
    """alpha[:, 0][plan.perm] — the per-sorted-edge weight slab of the weighted segment reduce.
    Memoised on alpha's identity + version and the plan, so repeated calls with one alpha permute
    once; the entry keeps alpha alive so its pointer cannot be recycled."""
    key = (alpha.data_ptr(), alpha._version, alpha.numel(), alpha.dtype, alpha.device, plan.perm.data_ptr())
    hit = _sorted_alpha.get(key)
    if hit is not None:
        _sorted_alpha.move_to_end(key)
        return hit[0]
    w = torch.empty(alpha.size(0), dtype=alpha.dtype, device=alpha.device)
    with _on_device(alpha.device):
        check(lib.gno_permute_rows(_ptr(alpha), _ptr(plan.perm), _ptr(w), alpha.size(0), alpha.element_size(),
                                   _stream(alpha.device)))
    _sorted_alpha[key] = (w, alpha, plan.perm)
    while len(_sorted_alpha) > 2:
        _sorted_alpha.popitem(last=False)
    return w


def _aggregate(plan, gidx, x, alpha, H, n_rows):
    """out[i, h*C:(h+1)*C] = sum over the plan's row i of alpha[eid, h] * x[gidx, h*C:(h+1)*C]."""
    if H == 1:
        # One head is the existing weighted segment reduce with alpha in sorted order: a coalesced
        # weight slab and the full-occupancy kernel, where the per-head mode would gather every
        # weight through eid (a 32-byte sector per edge).  Same arithmetic in the same order.
        return ops.segment_reduce(plan, x, "sum", gidx=gidx, weights=_alpha_sorted(plan, alpha))
    F = x.size(1)
    dev = x.device
    out = torch.empty((n_rows, F), dtype=x.dtype, device=dev)
    csr = plan.csr(gidx, plan.perm)
    dt = ops._dtype_id(x)
    nbytes = ctypes.c_size_t()
    check(lib.gno_segment_reduce_workspace(ctypes.byref(csr), F, dt, GNO_SUM, 0, ctypes.byref(nbytes)))
    ws = _workspace(nbytes.value, dev) if nbytes.value else None
    with _on_device(dev):
        check(lib.gno_segment_reduce_heads(ctypes.byref(csr), _ptr(x), x.size(0), _ptr(alpha), H, _ptr(out), F, dt,
                                           _ptr(ws), nbytes.value, _stream(dev)))
    return out


def _kept_edges(dst, n_rows):
    """(dst with dropped entries pointed at row 0, mask of the kept edges) — the transposed
    aggregation gathers grad_out[dst], so an edge the forward dropped must read a valid row and
    carry weight 0.  Memoised on dst like its plan."""
    def build():
        keep = (dst >= 0) & (dst < n_rows)
        return torch.where(keep, dst, torch.zeros_like(dst)), keep
    return ops._memo("attn_kept", dst, (n_rows,), build)


class _AttentionAggregate(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, alpha, src, dst, dim_size):
        ops._check_range(src, x.size(0), "attention_aggregate: src")
        plan = plan_cache.get(dst, dim_size)
        out = _aggregate(plan, plan.sorted_ids(src), x, alpha, alpha.size(1), dim_size)
        ctx.dim_size = dim_size
        ctx.save_for_backward(x, alpha, src, dst)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        x, alpha, src, dst = ctx.saved_tensors
        g = grad_out.to(x.dtype).contiguous()
        N, H = ctx.dim_size, alpha.size(1)
        plan = plan_cache.get(dst, N)
        grad_x = grad_alpha = None
        if ctx.needs_input_grad[0]:
            # transposed aggregation: grad_x[s, h, :] = sum_{e: src[e] = s} alpha[e, h] * g[dst[e], h, :]
            a_t, d_t = alpha, dst
            if plan.n_dropped:
                d_t, keep = _kept_edges(dst, N)
                a_t = alpha.masked_fill(~keep.unsqueeze(1), 0)
            if N == 0:
                grad_x = torch.zeros_like(x)
            else:
                plan_t = plan_cache.get(src, x.size(0))
                grad_x = _aggregate(plan_t, plan_t.sorted_ids(d_t), g, a_t, H, x.size(0))
        if ctx.needs_input_grad[1]:
            grad_alpha = torch.zeros_like(alpha)  # dropped edges keep 0
            if plan.E_valid and x.size(1):
                csr = plan.csr(plan.sorted_ids(src), plan.perm)
                with _on_device(x.device):
                    check(lib.gno_edge_head_dot(ctypes.byref(csr), _ptr(x), x.size(0), _ptr(g), H, x.size(1),
                                                _ptr(grad_alpha), ops._dtype_id(x), _stream(x.device)))
        return grad_x, grad_alpha, None, None, None


def attention_aggregate(x, alpha, src, dst, dim_size):
    """out[i, h, :] = sum_{e: dst[e] = i} alpha[e, h] * x[src[e], h, :] — GATv2's message passing
    (PyG: x_j * alpha.unsqueeze(-1), then a scatter-sum) without the [E, H, C] messages.

    x [N_src, H, C] or [N_src, H*C]; alpha [E, H] ([E] for one head), cast to x's dtype;
    src / dst int64 [E].  Returns [dim_size, H, C].  An out-of-range src raises IndexError; edges
    whose dst lies outside [0, dim_size) are dropped with a warning.  Differentiable w.r.t. x and
    alpha."""
    ops._need_cuda(x, alpha, src, dst)
    ops._dtype_id(x)
    for name, t in (("src", src), ("dst", dst)):
        if t.dtype != torch.int64 or t.dim() != 1:
            raise ValueError(f"attention_aggregate: {name} must be a 1-D int64 tensor")
    E = src.numel()
    if dst.numel() != E:
        raise ValueError("attention_aggregate: src and dst differ in length")
    H = alpha.size(1) if alpha.dim() == 2 else 1
    if alpha.dim() > 2 or alpha.size(0) != E or H == 0:
        raise ValueError(f"attention_aggregate: alpha must be [E, H] with E = {E}")
    if x.dim() == 3:
        if x.size(1) != H:
            raise ValueError(f"attention_aggregate: x has {x.size(1)} heads, alpha {H}")
        C = x.size(2)
    elif x.dim() == 2:
        if x.size(1) % H:
            raise ValueError(f"attention_aggregate: {x.size(1)} columns do not split into {H} heads")
        C = x.size(1) // H
    else:
        raise ValueError("attention_aggregate: x must be [N, H, C] or [N, H*C]")
    dim_size = int(dim_size)
    x2 = x.reshape(x.size(0), H * C).contiguous()
    a2 = alpha.reshape(E, H).to(x.dtype).contiguous()
    out = _AttentionAggregate.apply(x2, a2, src.contiguous(), dst.contiguous(), dim_size)
    return out.view(dim_size, H, C)


def _gatv2_backward(plan, gidx, own, other, att, g, H, slope, grad_own, grad_att):
    """One backward pass of the logits along `plan`: grad_own (or None) and fp32 grad_att (or None)."""
    F = own.size(1)
    dev = own.device
    csr = plan.csr(gidx, plan.perm)
    nbytes = ctypes.c_size_t()
    check(lib.gno_gatv2_logits_backward_workspace(ctypes.byref(csr), H, F, grad_own is not None,
                                                  grad_att is not None, ctypes.byref(nbytes)))
    ws = _workspace(nbytes.value, dev)
    with _on_device(dev):
        check(lib.gno_gatv2_logits_backward(ctypes.byref(csr), _ptr(own), _ptr(other), other.size(0), _ptr(att),
                                            _ptr(g), H, F, slope, _ptr(grad_own), _ptr(grad_att),
                                            ops._dtype_id(own), _ptr(ws), nbytes.value, _stream(dev)))


class _GATv2Logits(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x_l, x_r, att, src, dst, H, slope):
        E, F = src.numel(), x_l.size(1)
        ctx.H, ctx.slope = H, slope
        ctx.save_for_backward(x_l, x_r, att, src, dst)
        if E == 0 or F == 0:  # nothing to sum: zeros, and zero gradients below
            return torch.zeros((E, H), dtype=x_l.dtype, device=x_l.device)
        out = torch.empty((E, H), dtype=x_l.dtype, device=x_l.device)
        plan = plan_cache.get(dst, x_r.size(0))
        csr = plan.csr(plan.sorted_ids(src), plan.perm)
        with _on_device(x_l.device):
            check(lib.gno_gatv2_logits(ctypes.byref(csr), _ptr(x_l), x_l.size(0), _ptr(x_r), _ptr(att), H, F, slope,
                                       _ptr(out), ops._dtype_id(x_l), _stream(x_l.device)))
        return out

    @staticmethod
    def backward(ctx, grad_logits):
        x_l, x_r, att, src, dst = ctx.saved_tensors
        need_l, need_r, need_att = ctx.needs_input_grad[:3]
        g = grad_logits.to(x_l.dtype).contiguous()
        H, slope = ctx.H, ctx.slope
        empty = src.numel() == 0 or x_l.size(1) == 0
        new = torch.zeros_like if empty else torch.empty_like
        grad_l = new(x_l) if need_l else None
        grad_r = new(x_r) if need_r else None
        grad_att = new(att, dtype=torch.float32) if need_att else None
        if not empty and (need_r or need_att):
            plan = plan_cache.get(dst, x_r.size(0))
            _gatv2_backward(plan, plan.sorted_ids(src), x_r, x_l, att, g, H, slope, grad_r, grad_att)
        if not empty and need_l:
            plan_t = plan_cache.get(src, x_l.size(0))
            _gatv2_backward(plan_t, plan_t.sorted_ids(dst), x_l, x_r, att, g, H, slope, grad_l, None)
        if grad_att is not None:
            grad_att = grad_att.to(att.dtype)
        return grad_l, grad_r, grad_att, None, None, None, None


def _heads_view(t, name, H, C, fn):
    """[N, H, C] or [N, H*C] -> [N, H*C] (checks H and C against att's)."""
    if t.dim() == 3:
        if t.size(1) != H or t.size(2) != C:
            raise ValueError(f"{fn}: {name} is [N, {t.size(1)}, {t.size(2)}], att [{H}, {C}]")
    elif t.dim() != 2 or t.size(1) != H * C:
        raise ValueError(f"{fn}: {name} must be [N, {H}, {C}] or [N, {H * C}], got {tuple(t.shape)}")
    return t.reshape(t.size(0), H * C).contiguous()


def _gatv2_args(fn, x_l, x_r, att, src, dst):
    """The input conventions of gatv2_logits and gatv2_attention: checks, then (x_l [N_src, H*C],
    x_r [N_dst, H*C], att [H*C] in x_l's dtype, src, dst, H, C)."""
    ops._need_cuda(x_l, x_r, att, src, dst)
    ops._dtype_id(x_l)
    if x_r.dtype != x_l.dtype:
        raise ValueError(f"{fn}: x_l is {x_l.dtype}, x_r {x_r.dtype}")
    for name, t in (("src", src), ("dst", dst)):
        if t.dtype != torch.int64 or t.dim() != 1:
            raise ValueError(f"{fn}: {name} must be a 1-D int64 tensor")
    E = src.numel()
    if dst.numel() != E:
        raise ValueError(f"{fn}: src and dst differ in length")
    if att.dim() == 3 and att.size(0) == 1:
        H, C = att.size(1), att.size(2)
    elif att.dim() == 2:
        H, C = att.shape
    elif att.dim() == 1 and (x_l.dim() == 3 or x_r.dim() == 3):
        H, C = (x_l if x_l.dim() == 3 else x_r).shape[1:]
    elif att.dim() == 1:
        raise ValueError(f"{fn}: a flat att needs x_l or x_r as [N, H, C] to know the heads")
    else:
        raise ValueError(f"{fn}: att must be [H, C], [1, H, C] or [H*C], got {tuple(att.shape)}")
    if H == 0 or att.numel() != H * C:
        raise ValueError(f"{fn}: att has {att.numel()} entries for {H} heads of {C}")
    xl2 = _heads_view(x_l, "x_l", H, C, fn)
    xr2 = _heads_view(x_r, "x_r", H, C, fn)
    ops._check_range(src, xl2.size(0), f"{fn}: src")
    ops._check_range(dst, xr2.size(0), f"{fn}: dst")
    a2 = att.reshape(H * C).to(x_l.dtype).contiguous()
    return xl2, xr2, a2, src.contiguous(), dst.contiguous(), H, C


def gatv2_logits(x_l, x_r, att, src, dst, negative_slope=0.2):
    """logits[e, h] = sum_c att[h, c] * leaky_relu(x_l[src[e], h, c] + x_r[dst[e], h, c], negative_slope)
    — PyG 2.0.2 GATv2Conv.message (x_i + x_j, leaky_relu, (x * att).sum(-1)) without the [E, H, C]
    messages.

    x_l [N_src, H, C] or [N_src, H*C]; x_r [N_dst, H, C] or [N_dst, H*C] (N_src != N_dst allowed);
    att [H, C], [1, H, C] (GATv2Conv's parameter) or [H*C], cast to x_l's dtype; src / dst int64 [E].
    Returns [E, H] in x_l's dtype, in the original edge order (what `softmax` consumes).  The sum
    x_l + x_r is formed in fp32 from the stored values; fp32 math, one rounding.  An out-of-range
    src or dst raises IndexError.  Differentiable w.r.t. x_l, x_r and att (x_l and x_r may be the
    same tensor); the backward recomputes the sums and saves no [E, ...] tensor."""
    xl2, xr2, a2, src, dst, H, _ = _gatv2_args("gatv2_logits", x_l, x_r, att, src, dst)
    return _GATv2Logits.apply(xl2, xr2, a2, src, dst, H, float(negative_slope))


class _GATv2Attention(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x_l, x_r, att, src, dst, H, slope):
        N, F, dev = x_r.size(0), x_l.size(1), x_l.device
        ctx.H, ctx.slope = H, slope
        if src.numel() == 0 or F == 0:  # nothing to aggregate: zeros, and zero gradients below
            out = torch.zeros((N, H, F // H), dtype=x_l.dtype, device=dev)
            ctx.save_for_backward(x_l, x_r, att, src, dst, out, None, None)
            return out
        plan = plan_cache.get(dst, N)
        csr = plan.csr(plan.sorted_ids(src), plan.perm)
        out = torch.empty((N, H, F // H), dtype=x_l.dtype, device=dev)
        m = torch.empty((N, H), dtype=torch.float32, device=dev)
        s = torch.empty((N, H), dtype=torch.float32, device=dev)
        nbytes = ctypes.c_size_t()
        check(lib.gno_gatv2_attention_workspace(ctypes.byref(csr), H, F, ctypes.byref(nbytes)))
        ws = _workspace(nbytes.value, dev)
        with _on_device(dev):
            check(lib.gno_gatv2_attention(ctypes.byref(csr), _ptr(x_l), x_l.size(0), _ptr(x_r), _ptr(att), H, F,
                                          slope, EPS, _ptr(out), _ptr(m), _ptr(s), ops._dtype_id(x_l), _ptr(ws),
                                          nbytes.value, _stream(dev)))
        ctx.save_for_backward(x_l, x_r, att, src, dst, out, m, s)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        x_l, x_r, att, src, dst, out, m, s = ctx.saved_tensors
        need_l, need_r, need_att = ctx.needs_input_grad[:3]
        H, slope = ctx.H, ctx.slope
        E, F, dev = src.numel(), x_l.size(1), x_l.device
        if E == 0 or F == 0:
            return (torch.zeros_like(x_l) if need_l else None, torch.zeros_like(x_r) if need_r else None,
                    torch.zeros_like(att) if need_att else None, None, None, None, None)
        g = grad_out.to(x_l.dtype).reshape(-1, F).contiguous()
        grad_l = grad_r = grad_att = da = alpha = None
        if need_r:
            grad_r = torch.empty_like(x_r)
        if need_att:
            grad_att = torch.empty(F, dtype=torch.float32, device=dev)
        if need_l:
            da = torch.empty((E, H), dtype=x_l.dtype, device=dev)
            alpha = torch.empty((E, H), dtype=x_l.dtype, device=dev)
        # destination pass: grad_x_r, grad_att, and da / alpha for the source pass
        plan = plan_cache.get(dst, x_r.size(0))
        csr = plan.csr(plan.sorted_ids(src), plan.perm)
        nbytes = ctypes.c_size_t()
        check(lib.gno_gatv2_attention_backward_workspace(ctypes.byref(csr), H, F, need_r, need_att,
                                                         ctypes.byref(nbytes)))
        ws = _workspace(nbytes.value, dev)
        with _on_device(dev):
            check(lib.gno_gatv2_attention_backward(ctypes.byref(csr), _ptr(x_l), x_l.size(0), _ptr(x_r), _ptr(att),
                                                   _ptr(out), _ptr(m), _ptr(s), _ptr(g), H, F, slope, _ptr(grad_r),
                                                   _ptr(grad_att), _ptr(da), _ptr(alpha), ops._dtype_id(x_l),
                                                   _ptr(ws), nbytes.value, _stream(dev)))
        if need_l:
            # source pass: the logit part through da, plus the transposed aggregation sum alpha * g[dst]
            plan_t = plan_cache.get(src, x_l.size(0))
            dst_t = plan_t.sorted_ids(dst)
            grad_l = torch.empty_like(x_l)
            _gatv2_backward(plan_t, dst_t, x_l, x_r, att, da, H, slope, grad_l, None)
            grad_l += _aggregate(plan_t, dst_t, g, alpha, H, x_l.size(0))
        if grad_att is not None:
            grad_att = grad_att.to(att.dtype)
        return grad_l, grad_r, grad_att, None, None, None, None


def gatv2_attention(x_l, x_r, att, src, dst, negative_slope=0.2):
    """A GATv2 layer's message passing in one op:
        out[i, h, :] = sum_{e: dst[e] = i} alpha[e, h] * x_l[src[e], h, :]
    with alpha = softmax over each destination (PyG 2.0.2: exp(a - max) / (sum exp + 1e-16), the
    maximum by torch_scatter's rule as in `softmax`) of the logits
        a[e, h] = sum_c att[h, c] * leaky_relu(x_l[src[e], h, c] + x_r[dst[e], h, c], negative_slope),
    i.e. attention_aggregate(x_l, softmax(gatv2_logits(x_l, x_r, att, src, dst), dst,
    num_nodes=N_dst), src, dst, N_dst), in one pass over the edges: each gathered x_l row serves
    the logit and the weighted sum, and neither the [E, H] logits nor alpha are stored.  The
    logits, the softmax statistics and the sum stay in fp32 and the output is rounded once, where
    the three-op composition rounds the logits and alpha to a 16-bit dtype on the way.

    Inputs as in `gatv2_logits`: x_l [N_src, H, C] or [N_src, H*C]; x_r [N_dst, H, C] or
    [N_dst, H*C]; att [H, C], [1, H, C] or [H*C]; src / dst int64 [E]; fp32, fp16 or bf16.
    Returns [N_dst, H, C] in x_l's dtype; destinations without an edge get 0.  An out-of-range
    src or dst raises IndexError.  Differentiable w.r.t. x_l, x_r and att (x_l may be x_r); the
    backward keeps no [E, ...] tensor from the forward, only out and fp32 [N_dst, H] statistics,
    and builds the src-sorted plan only when x_l needs a gradient.

    Not covered: attention dropout, return_attention_weights and edge features (GATv2Conv's
    edge_dim).  Callers that need them use the three ops above, whose alpha is an explicit
    tensor."""
    xl2, xr2, a2, src, dst, H, C = _gatv2_args("gatv2_attention", x_l, x_r, att, src, dst)
    return _GATv2Attention.apply(xl2, xr2, a2, src, dst, H, float(negative_slope))
