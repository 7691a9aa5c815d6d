"""Differentiable wrappers (SURVEY §8f rank 2): OpProfiler profiles a training step
(graph_benchmark/profile/OpProfiler.py:277-292), so the aggregation needs a backward.

Backward formulas are torch-scatter 2.0.9's (csrc/scatter.cpp ScatterSum/ScatterMean/ScatterMin/
ScatterMax/ScatterMul::backward):
    sum   grad_src = grad_out gathered by index
    mean  grad_src = (grad_out / clamp(count, 1)) gathered by index
    min/max  grad_src = scatter of grad_out to the arg positions (no collisions)
    mul   grad_src = (grad_out * out) gathered by index / src
For the fused gather→scatter the backward w.r.t. x is the transposed aggregation — the same
segment-reduce kernel on a plan sorted by the SOURCE ids (cached like the forward plan).
"""
import torch

from . import ops
from .plan import plan_cache


def _div_count(g, cnt, dim, dtype=None):
    """g / max(cnt, 1), a 1-D cnt broadcast along dim: in fp32 from the exact integer count, rounded
    once to `dtype` (default g's).  A 16-bit count is already wrong above 256 in bf16 and 2048 in
    fp16, and inf above 65504."""
    if cnt.dim() == 1:
        shape = [1] * g.dim()
        shape[dim] = -1
        cnt = cnt.view(shape)
    return (g.to(torch.float32) / cnt.clamp(min=1).to(torch.float32)).to(dtype or g.dtype)


def _row_counts(index, n):
    """Entries of a 1-D index per row in [0, n) (int64; out-of-range entries, which the forward
    drops, are not counted): the cached forward plan's rowptr, so no extra pass."""
    if index.numel() > ops._MAX_PLAN_EDGES:
        return torch.bincount(index[(index >= 0) & (index < n)], minlength=n)
    rowptr = plan_cache.get(index, n).rowptr
    return rowptr[1:] - rowptr[:-1]


def _in_range(index, n):
    """(index, keep): keep is None when every entry lies in [0, n); otherwise the entries the forward
    dropped are replaced by 0 (n > 0) and keep marks the others.  The range is memoised per index
    tensor, so the common case costs one host read per index."""
    if index.numel() == 0:
        return index, None
    lo, hi = ops._memo("idx_range", index, (), lambda: (int(index.min()), int(index.max())))
    if lo >= 0 and hi < n:
        return index, None
    keep = (index >= 0) & (index < n)
    return torch.where(keep, index, torch.zeros_like(index)), keep


def _gather_dim(t, dim, index, like):
    """t gathered along dim by a 1-D or full-shape index, shaped like `like`."""
    if index.dim() == 1 and t.dim() == 2 and dim == 0:
        return ops.index_select(t, 0, index)
    if index.dim() == 1:
        return t.index_select(dim, index)
    if index.shape != like.shape:
        index = index.expand_as(like)
    return t.gather(dim, index)


class _Scatter(torch.autograd.Function):
    @staticmethod
    def forward(ctx, src, index, dim, dim_size, reduce):
        if dim < 0:
            dim += src.dim()
        ctx.dim, ctx.reduce, ctx.shape = dim, reduce, src.shape
        if reduce in ("min", "max"):
            out, arg = ops.scatter(src, index, dim, None, dim_size, reduce, return_arg=True)
            ctx.save_for_backward(arg)
            ctx.mark_non_differentiable(arg)
            return out, arg
        out = ops.scatter(src, index, dim, None, dim_size, reduce)
        if reduce == "mul":
            ctx.save_for_backward(index, src, out)
        else:
            ctx.save_for_backward(index)
        return out

    @staticmethod
    def backward(ctx, grad_out, *unused):
        dim, reduce = ctx.dim, ctx.reduce
        grad_out = grad_out.contiguous()
        if reduce in ("min", "max"):
            (arg,) = ctx.saved_tensors
            shape = list(ctx.shape)
            shape[dim] += 1  # sentinel row for empty outputs, trimmed below
            g = grad_out.new_zeros(shape).scatter_(dim, arg, grad_out)
            return g.narrow(dim, 0, shape[dim] - 1), None, None, None, None
        saved = ctx.saved_tensors
        index, n = saved[0], grad_out.size(dim)
        if grad_out.numel() == 0 or index.numel() == 0:
            # no output rows (every entry dropped) or no entries: nothing reaches src
            return grad_out.new_zeros(ctx.shape), None, None, None, None
        like = grad_out.new_empty(ctx.shape)
        if reduce == "mean":
            if index.dim() == 1:
                cnt = _row_counts(index, n)
            else:  # full-shape index: count in fp32 (exact to 2^24), not with 16-bit ones
                ones = torch.ones(like.shape, dtype=torch.float32, device=like.device)
                cnt = ops.scatter(ones, index, dim, None, n, "sum")
            grad_out = _div_count(grad_out, cnt, dim)
        elif reduce == "mul":
            out = saved[2]
            grad_out = grad_out.to(torch.float32) * out.to(torch.float32)
        # entries the forward dropped get zero gradient; the native gathers never see them
        index, keep = _in_range(index, n)
        g = _gather_dim(grad_out, dim, index, like)
        if reduce == "mul":
            g = (g / saved[1].to(torch.float32)).to(like.dtype)
            g.masked_fill_(g.isnan(), 0)
        if keep is not None:
            if keep.dim() == 1 and g.dim() > 1:
                shape = [1] * g.dim()
                shape[dim] = -1
                keep = keep.view(shape)
            g = g.masked_fill(~keep, 0)
        return g, None, None, None, None


class _GatherScatter(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, src_ids, dst_ids, dim_size, reduce):
        ctx.reduce, ctx.n_src, ctx.dim_size, ctx.dtype = reduce, x.size(0), dim_size, x.dtype
        if reduce in ("min", "max"):
            out, arg = ops.gather_scatter(x, src_ids, dst_ids, dim_size, reduce, return_arg=True)
            ctx.save_for_backward(src_ids, arg)
            ctx.mark_non_differentiable(arg)
            return out, arg
        out = ops.gather_scatter(x, src_ids, dst_ids, dim_size, reduce)
        ctx.save_for_backward(src_ids, dst_ids)
        return out

    @staticmethod
    def backward(ctx, grad_out, *unused):
        reduce = ctx.reduce
        grad_out = grad_out.contiguous()
        src_ids = ctx.saved_tensors[0]
        if grad_out.numel() == 0 or src_ids.numel() == 0:
            return grad_out.new_zeros((ctx.n_src,) + tuple(grad_out.shape[1:])), None, None, None, None
        if reduce in ("min", "max"):
            src_ids, arg = ctx.saved_tensors
            E = src_ids.numel()
            # row of x that won each output element (sentinel -> dropped by the range check)
            winner = torch.cat([src_ids, src_ids.new_full((1,), -1)])[arg.clamp(max=E)]
            g = ops.scatter(grad_out, winner, 0, None, ctx.n_src, "sum")  # full-shape index, collisions
            return g, None, None, None, None
        src_ids, dst_ids = ctx.saved_tensors
        plan = plan_cache.get(dst_ids, ctx.dim_size)      # the forward's plan
        if reduce == "mean":
            # fp32 gradient into the transposed aggregation: divided and summed, rounded once
            grad_out = _div_count(grad_out, plan.rowptr[1:] - plan.rowptr[:-1], 0, torch.float32)
        elif reduce != "sum":
            raise NotImplementedError("gather_scatter backward: sum/mean/min/max")
        if plan.n_dropped:
            # edges the forward dropped read a zero row appended to the gradient
            n = ctx.dim_size
            dst_ids = ops._memo("dst_in_range", dst_ids, (n,),
                                lambda: torch.where((dst_ids >= 0) & (dst_ids < n), dst_ids, torch.full_like(dst_ids, n)))
            grad_out = torch.cat([grad_out, grad_out.new_zeros((1,) + tuple(grad_out.shape[1:]))])
        # transposed aggregation: grad_x[s] = sum over edges with source s of grad_out[dst]
        g = ops.gather_scatter(grad_out, dst_ids, src_ids, ctx.n_src, "sum")
        return g.to(ctx.dtype), None, None, None, None


class _SegmentCSR(torch.autograd.Function):
    """torch_scatter.segment_csr (1-D indptr) with upstream's backward (csrc/segment_csr.cpp):
    sum -> gather_csr(grad), mean -> gather_csr(grad / count), min/max -> grad scattered to arg."""

    @staticmethod
    def forward(ctx, src, indptr, reduce):
        ctx.reduce, ctx.shape = reduce, src.shape
        if reduce in ("min", "max"):
            out, arg = ops.segment_csr(src, indptr, None, reduce, return_arg=True)
            ctx.save_for_backward(arg)
            ctx.mark_non_differentiable(arg)
            return out, arg
        ctx.save_for_backward(indptr)
        return ops.segment_csr(src, indptr, None, reduce)

    @staticmethod
    def backward(ctx, grad_out, *unused):
        grad_out = grad_out.contiguous()
        E = ctx.shape[0]
        if grad_out.numel() == 0 or E == 0:
            return grad_out.new_zeros(ctx.shape), None, None
        if ctx.reduce in ("min", "max"):
            (arg,) = ctx.saved_tensors
            g = grad_out.new_zeros([E + 1] + list(ctx.shape[1:])).scatter_(0, arg, grad_out)
            return g[:E], None, None
        (indptr,) = ctx.saved_tensors
        if ctx.reduce == "mean":
            grad_out = _div_count(grad_out, indptr[1:] - indptr[:-1], 0)
        g = ops.gather_csr(grad_out, indptr)            # rows [0, indptr[-1]); zeros before indptr[0]
        if g.size(0) < E:                                # elements past the last pointer get no gradient
            g = torch.cat([g, g.new_zeros([E - g.size(0)] + list(g.shape[1:]))])
        return g, None, None


class _SpmmCSR(torch.autograd.Function):
    """torch_sparse.matmul(SparseTensor, dense, reduce) on a CSR: backward w.r.t. the dense matrix
    is the TRANSPOSED aggregation (same segment-reduce kernel, plan on the column ids, cached);
    w.r.t. the edge values it is one dot product per edge."""

    @staticmethod
    def forward(ctx, rowptr, col, value, mat, reduce):
        ctx.reduce, ctx.n_src = reduce, mat.size(0)
        ctx.has_value = value is not None
        if reduce in ("min", "max"):
            out, arg = ops.spmm_csr(rowptr, col, value, mat, reduce, return_arg=True)
            ctx.save_for_backward(col, arg, value if value is not None else col.new_empty(0), mat)
            ctx.mark_non_differentiable(arg)
            return out, arg
        ctx.save_for_backward(rowptr, col, value if value is not None else col.new_empty(0), mat)
        return ops.spmm_csr(rowptr, col, value, mat, reduce)

    @staticmethod
    def backward(ctx, grad_out, *unused):
        grad_out = grad_out.contiguous()
        need_mat, need_val = ctx.needs_input_grad[3], ctx.needs_input_grad[2] and ctx.has_value
        dtype = grad_out.dtype
        if ctx.reduce in ("min", "max"):
            col, arg, value, mat = ctx.saved_tensors
        else:
            rowptr, col, value, mat = ctx.saved_tensors
        nnz = col.numel()
        if nnz == 0 or grad_out.numel() == 0:
            return (None, None, torch.zeros_like(value) if need_val else None,
                    torch.zeros_like(mat) if need_mat else None, None)
        if ctx.reduce in ("min", "max"):
            safe = arg.clamp(max=nnz - 1)
            hit = arg < nnz
            g_mat = g_val = None
            # products and collisions in fp32, rounded once
            g32 = grad_out.to(torch.float32)
            if need_mat:
                w = g32 if not ctx.has_value else g32 * value[safe].to(torch.float32)
                winner = torch.where(hit, col[safe], torch.full_like(arg, -1))
                g_mat = ops.scatter(w.contiguous(), winner, 0, None, ctx.n_src, "sum").to(dtype)
            if need_val:
                picked = mat[col[safe], torch.arange(mat.size(1), device=mat.device)].to(torch.float32)
                contrib = torch.where(hit, g32 * picked, torch.zeros_like(g32))
                g_val = torch.zeros(nnz + 1, dtype=torch.float32, device=grad_out.device)
                g_val.index_add_(0, arg.reshape(-1).clamp(max=nnz), contrib.reshape(-1))
                g_val = g_val[:nnz].to(value.dtype)
            return None, None, g_val, g_mat, None
        if ctx.reduce == "mean":
            # fp32 gradient into the transposed product: divided and summed, rounded once
            grad_out = _div_count(grad_out, rowptr[1:] - rowptr[:-1], 0, torch.float32)
        elif ctx.reduce not in ("sum", "add"):
            raise NotImplementedError("spmm backward: sum / mean / min / max")
        g_mat = None
        if need_mat:
            g_mat = ops.spmm_csr_t(rowptr, col, value if ctx.has_value else None, grad_out, ctx.n_src).to(dtype)
        g_val = None
        if need_val:
            row = ops.csr_rows(rowptr, nnz)
            g_val = (grad_out.index_select(0, row).to(torch.float32) *
                     mat.index_select(0, col).to(torch.float32)).sum(-1).to(value.dtype)
        return None, None, g_val, g_mat, None


def segment_csr(src, indptr, reduce="sum"):
    """Differentiable torch_scatter.segment_csr (1-D indptr). min/max return (out, arg)."""
    if indptr.dim() != 1:
        raise NotImplementedError("gno_b200: segment_csr gradients cover a 1-D indptr")
    return _SegmentCSR.apply(src, indptr, reduce)


def spmm_csr(rowptr, col, value, mat, reduce="sum"):
    """Differentiable CSR spmm (w.r.t. mat and value). min/max return (out, arg)."""
    return _SpmmCSR.apply(rowptr, col, value, mat, reduce)


def scatter(src, index, dim=-1, dim_size=None, reduce="sum"):
    """Differentiable torch_scatter.scatter (no out=). min/max return (out, arg)."""
    if dim_size is None:
        dim_size = int(index.max()) + 1 if index.numel() else 0
    return _Scatter.apply(src, index, dim, dim_size, reduce)


def gather_scatter(x, src_ids, dst_ids, dim_size, reduce="sum"):
    """Differentiable fused message passing. min/max return (out, arg)."""
    return _GatherScatter.apply(x, src_ids, dst_ids, dim_size, reduce)
