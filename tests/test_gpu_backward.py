"""Backward of the core aggregation ops against fp64 on the device, in fp32, bf16 and fp16.

Covered: torch_scatter.scatter (1-D index, full-shape index, dims 0 / 1 / -1 and a 3-D middle
dim), gno_b200.autograd.gather_scatter, torch_scatter.segment_csr, SparseTensor.matmul,
torch_sparse.spmm, the composites, the torch.ops.torch_scatter / torch.ops.torch_sparse entries
(directly and under TorchScript), a training loop, the value-permutation memo and one full-size
case per op family.

The reference is native torch in fp64: index_add_ / scatter_reduce restatements of the forward
and their autograd.  max / min route the whole gradient to the arg, lowest edge position first
(upstream's rule; torch's amax splits ties evenly), so their reference gradient is the upstream
gradient scattered to the arg the CPU oracle computes.  Tolerances:

* exact gradients (sum: copies of the upstream gradient; max / min routing without collisions)
  are compared bit for bit;
* a mean gradient with a 1-D index is one division: |got - ref| <= ulp/2 + 1e-5 |ref|;
* accumulated gradients (the transposed aggregation, winner collisions):
  |got - ref| <= ulp/2 + 1e-5 sum|terms| in bf16 / fp16, 1e-5 sum|terms| in fp32.

The ulp/2 term is what "fp32 accumulate, one rounding" (DESIGN.md §2) allows a 16-bit result; a
second rounding (a 16-bit count, a 16-bit intermediate) fails it.  Destination hubs of 301, 3001
and 70001 entries cross the counts bf16 (256) and fp16 (2048) hold exactly and fp16's largest
finite value (65504).
"""
import pytest
import torch

import oracle

pytestmark = pytest.mark.gpu

DTYPES = [torch.float32, torch.bfloat16, torch.float16]
WIDTHS = [1, 3, 8, 33, 128, 602]      # 33: narrow-vector path; 602: padded gather
_MANT = {torch.float32: 23, torch.bfloat16: 7, torch.float16: 10}
_VIEW = {torch.float32: torch.int32, torch.bfloat16: torch.int16, torch.float16: torch.int16}


def _dt(dtype):
    return str(dtype).split(".")[-1]


# ---- tolerances ----------------------------------------------------------------------------------
def _ulp(ref, dtype):
    """Spacing of `dtype` at |ref| (fp64 tensor); subnormals get the subnormal spacing."""
    _, e = torch.frexp(ref.abs().clamp(min=torch.finfo(dtype).tiny))
    return torch.ldexp(torch.ones_like(ref), (e - 1 - _MANT[dtype]).to(torch.float64))


def _report(got, ref, bound, what):
    err = (got.double() - ref).abs()
    bad = ~(err <= bound)                       # NaN fails
    if bad.any():
        i = int(torch.nonzero(bad.reshape(-1))[0])
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements out of bound; first at "
                             f"flat {i}: got {got.reshape(-1)[i].item()!r}, ref {ref.reshape(-1)[i].item()!r}, "
                             f"bound {bound.reshape(-1)[i].item():.3e}")


def _exact(got, ref, what):
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    _report(got, ref, torch.zeros_like(ref), what)


def _div(got, ref, dtype, what):
    """One division rounded once."""
    assert got.shape == ref.shape and got.dtype == dtype, (what, got.shape, got.dtype)
    _report(got, ref, 0.5 * _ulp(ref, dtype) + 1e-5 * ref.abs(), what)


def _acc(got, ref, mag, dtype, what):
    """An fp32-accumulated sum rounded once to dtype; mag = sum of |terms|."""
    assert got.shape == ref.shape and got.dtype == dtype, (what, got.shape, got.dtype)
    bound = 1e-5 * torch.maximum(mag, ref.abs()) + 1e-30
    if dtype != torch.float32:
        bound = bound + 0.5 * _ulp(ref, dtype)
    _report(got, ref, bound, what)


# ---- inputs --------------------------------------------------------------------------------------
def _hubs(F):
    return (301, 3001, 70001) if F <= 8 else (301, 3001)


def _hub_index(n, hubs, extra, g, n_empty=3):
    """1-D destination index over n rows: row i < len(hubs) gets exactly hubs[i] entries, `extra`
    entries land uniformly on the rows before the last n_empty, which stay empty; shuffled."""
    parts = [torch.full((h,), i, dtype=torch.int64) for i, h in enumerate(hubs)]
    parts.append(torch.randint(len(hubs), n - n_empty, (extra,), generator=g))
    idx = torch.cat(parts)
    return idx[torch.randperm(idx.numel(), generator=g)]


def _upstream(N, F, dtype, g, scale=16):
    """Upstream gradient, |g| in [scale, 2 scale): 16 keeps g / 70001 a normal fp16 number; sums
    into a source hub take scale 1, so that thousands of same-sign terms stay below fp16's 65504."""
    s = torch.where(torch.rand(N, F, generator=g) < 0.5, -1.0, 1.0)
    return (s * (1 + torch.rand(N, F, generator=g)) * scale).to(dtype)


def _values(shape, dtype, g, coarse):
    """Values on a coarse grid (ties in max / min) or continuous ones."""
    if coarse:
        return (torch.randint(-8, 9, shape, generator=g).double() / 4).to(dtype)
    return (torch.rand(shape, generator=g) * 4 - 2).to(dtype)


def _mul_values(shape, dtype, g):
    """Powers of two, never 0: products and quotients are exact in fp32."""
    pick = torch.tensor([1.0, 1.0, -1.0, 2.0, 0.5])
    return pick[torch.randint(0, 5, shape, generator=g)].to(dtype)


def _extreme_grad(grad, arg, dim, size):
    """Upstream's min / max backward in fp64: grad scattered to arg along dim (sentinel = size)."""
    shape = list(grad.shape)
    shape[dim] = size + 1
    out = torch.zeros(shape, dtype=torch.float64, device=grad.device)
    return out.scatter_(dim, arg.to(grad.device), grad.double()).narrow(dim, 0, size)


def _native_ref(src, index, dim, N, reduce, grad):
    """fp64 autograd of scatter_reduce(include_self=False); entries outside [0, N) dropped."""
    s = src.double().requires_grad_()
    idx = index
    if index.dim() == 1 and src.dim() > 1:
        shape = [1] * src.dim()
        shape[dim] = -1
        idx = index.view(shape).expand_as(src)
    idx = torch.where((idx >= 0) & (idx < N), idx, torch.full_like(idx, N))   # spare row, trimmed
    size = list(src.shape)
    size[dim] = N + 1
    red = {"sum": "sum", "mean": "mean", "mul": "prod"}[reduce]
    base = torch.ones if reduce == "mul" else torch.zeros
    out = base(size, dtype=torch.float64, device=src.device).scatter_reduce(dim, idx, s, red, include_self=False)
    out.narrow(dim, 0, N).backward(grad.double())
    return s.grad


def _check_scatter_grad(got, src, index, dim, N, reduce, grad, dtype, what):
    if reduce in ("min", "max"):
        _, arg = oracle.scatter(src.cpu(), index.cpu(), dim, N, reduce)
        _exact(got, _extreme_grad(grad, arg, dim, src.size(dim)), what)
        return
    ref = _native_ref(src, index, dim, N, reduce, grad)
    if reduce == "sum":
        _exact(got, ref, what)
    else:  # mean: one division; mul: an exact fp32 product of powers of two, rounded once
        _div(got, ref, dtype, what)


@pytest.mark.parametrize("dtype", DTYPES, ids=_dt)
def test_scatter_out_mean_divides_by_the_exact_count(cuda, dtype):
    """The out= mean, (out + sum) / count: the division uses the exact count past 256 / 2048 / 65504."""
    import torch_scatter
    g = torch.Generator().manual_seed(90)
    N, F = 8, 3
    index = _hub_index(N, (301, 3001, 70001), 50, g)
    # +1 / -1 alternating within each row: every row sums to 0 or 1, so out + sum is exact in any
    # dtype and the division is the only rounding
    order = torch.sort(index, stable=True).indices
    start = torch.cat([torch.zeros(1, dtype=torch.int64), torch.bincount(index, minlength=N).cumsum(0)])
    rank = torch.empty_like(index)
    rank[order] = torch.arange(index.numel()) - start[index[order]]
    src = (1.0 - 2.0 * (rank % 2).double()).view(-1, 1).expand(-1, F)
    out = torch.randint(1, 4, (N, F), generator=g).double()
    got = torch_scatter.scatter(src.to(dtype).to(cuda), index.to(cuda), 0, out=out.to(dtype).to(cuda), reduce="mean")
    cnt = torch.bincount(index, minlength=N).clamp(min=1).double().view(-1, 1)
    ref = (out + torch.zeros(N, F, dtype=torch.float64).index_add_(0, index, src)) / cnt
    _div(got, ref.to(cuda), dtype, f"out= mean {dtype}")


# ---- torch_scatter.scatter -----------------------------------------------------------------------
@pytest.mark.parametrize("dtype", DTYPES, ids=_dt)
@pytest.mark.parametrize("F", WIDTHS)
@pytest.mark.parametrize("reduce", ["sum", "mean", "mul", "min", "max"])
def test_scatter_1d_index(cuda, dtype, F, reduce):
    import torch_scatter
    g = torch.Generator().manual_seed(100 + F)
    if reduce == "mul":
        N = 300
        index = _hub_index(N, (), 1500, g)                      # products of at most a few dozen factors
        src = _mul_values((index.numel(), F), dtype, g)
    else:
        N = 400
        index = _hub_index(N, _hubs(F), 2000, g)
        src = _values((index.numel(), F), dtype, g, coarse=reduce in ("min", "max"))
    grad = _upstream(N, F, dtype, g).to(cuda)
    a = src.to(cuda).requires_grad_()
    out = torch_scatter.scatter(a, index.to(cuda), 0, dim_size=N, reduce=reduce)
    out.backward(grad)
    _check_scatter_grad(a.grad, src.to(cuda), index.to(cuda), 0, N, reduce, grad, dtype,
                        f"scatter {reduce} F={F} {dtype}")


@pytest.mark.parametrize("dtype", DTYPES, ids=_dt)
@pytest.mark.parametrize("F", [1, 3, 8, 33, 128])
@pytest.mark.parametrize("reduce", ["sum", "mean", "mul", "min", "max"])
def test_scatter_full_shape_index(cuda, dtype, F, reduce):
    """Every column has its own index (its own hubs); first call on the atomic path, second on the
    cached plan."""
    import torch_scatter
    g = torch.Generator().manual_seed(200 + F)
    N = 300
    if reduce == "mul":
        cols = [_hub_index(N, (), 1200, g) for _ in range(F)]
    else:
        cols = [_hub_index(N, (301, 3001), 1200, g) for _ in range(F)]
    index = torch.stack(cols, 1).to(cuda)
    E = index.size(0)
    src = (_mul_values((E, F), dtype, g) if reduce == "mul" else
           _values((E, F), dtype, g, coarse=reduce in ("min", "max"))).to(cuda)
    grad = _upstream(N, F, dtype, g).to(cuda)
    for call in range(2):
        a = src.clone().requires_grad_()
        out = torch_scatter.scatter(a, index, 0, dim_size=N, reduce=reduce)
        out.backward(grad)
        _check_scatter_grad(a.grad, src, index, 0, N, reduce, grad, dtype,
                            f"full-shape scatter {reduce} F={F} {dtype} call {call}")


# (src shape, dim, position of the edge dim in the shape)
_DIM_CASES = {"dim0": ((None, 5), 0), "dim1": ((6, None), 1), "dim-1": ((2, 3, None), -1),
              "3d-middle": ((3, None, 4), 1)}


@pytest.mark.parametrize("dtype", DTYPES, ids=_dt)
@pytest.mark.parametrize("case", list(_DIM_CASES))
@pytest.mark.parametrize("reduce", ["sum", "mean", "mul", "min", "max"])
def test_scatter_dims(cuda, dtype, case, reduce):
    import torch_scatter
    g = torch.Generator().manual_seed(300)
    shape_t, dim = _DIM_CASES[case]
    N = 200
    if reduce == "mul":
        index = _hub_index(N, (), 900, g)
    else:
        index = _hub_index(N, (301, 3001), 900, g)
    shape = [index.numel() if s is None else s for s in shape_t]
    src = (_mul_values(shape, dtype, g) if reduce == "mul" else
           _values(shape, dtype, g, coarse=reduce in ("min", "max"))).to(cuda)
    oshape = list(shape)
    oshape[dim] = N
    grad = _upstream(int(torch.tensor(oshape).prod()), 1, dtype, g).view(oshape).to(cuda)
    a = src.clone().requires_grad_()
    out = torch_scatter.scatter(a, index.to(cuda), dim, dim_size=N, reduce=reduce)
    out.backward(grad)
    d = dim % src.dim()
    _check_scatter_grad(a.grad, src, index.to(cuda), d, N, reduce, grad, dtype,
                        f"scatter {reduce} {case} {dtype}")


# ---- gather_scatter --------------------------------------------------------------------------------
def _gs_graph(F, g, n_src=500, N=400):
    """dst with destination hubs and empty rows; src with a source hub of 5000 out-edges, so the
    transposed plan has a row spanning many chunks."""
    dst = _hub_index(N, _hubs(F), 6000, g)
    E = dst.numel()
    src = torch.randint(1, n_src, (E,), generator=g)
    src[torch.randperm(E, generator=g)[:5000]] = 0
    src[src == n_src - 1] = n_src - 2          # source n_src - 1 has no out-edge: zero gradient
    return src, dst, n_src, N


def _gs_ref(x, src, dst, N, reduce, grad, valid=None):
    """fp64 autograd of index_add_(x[src]) (/ count), and the sum of |terms| of the gradient."""
    if valid is not None:
        src, dst = src[valid], dst[valid]
    x64 = x.double().requires_grad_()
    out = torch.zeros(N, x.size(1), dtype=torch.float64, device=x.device).index_add(0, dst, x64[src])
    g64 = grad.double()
    if reduce == "mean":
        cnt = torch.bincount(dst, minlength=N).clamp(min=1).double().view(-1, 1)
        out = out / cnt
        g64 = g64 / cnt
    out.backward(grad.double())
    mag = torch.zeros_like(x64).index_add_(0, src, g64.abs()[dst])
    return x64.grad, mag


def _gs_extreme_ref(x, src, dst, N, reduce, grad):
    _, arg = oracle.gather_scatter(x.cpu(), src.cpu(), dst.cpu(), N, reduce)
    arg = arg.to(x.device)
    n = x.size(0)
    winner = torch.cat([src, src.new_full((1,), n)])[arg]
    ref = torch.zeros(n + 1, x.size(1), dtype=torch.float64, device=x.device)
    mag = torch.zeros_like(ref)
    ref.scatter_add_(0, winner, grad.double())
    mag.scatter_add_(0, winner, grad.double().abs())
    return ref[:n], mag[:n]


@pytest.mark.parametrize("dtype", DTYPES, ids=_dt)
@pytest.mark.parametrize("F", WIDTHS)
@pytest.mark.parametrize("reduce", ["sum", "mean", "min", "max"])
def test_gather_scatter(cuda, dtype, F, reduce):
    from gno_b200 import autograd as ag
    g = torch.Generator().manual_seed(400 + F)
    src, dst, n, N = _gs_graph(F, g)
    x = _values((n, F), dtype, g, coarse=reduce in ("min", "max")).to(cuda)
    src, dst = src.to(cuda), dst.to(cuda)
    grad = _upstream(N, F, dtype, g, scale=16 if reduce == "mean" else 1).to(cuda)
    a = x.clone().requires_grad_()
    out = ag.gather_scatter(a, src, dst, N, reduce)
    out = out[0] if isinstance(out, tuple) else out
    out.backward(grad)
    if reduce in ("min", "max"):
        ref, mag = _gs_extreme_ref(x, src, dst, N, reduce, grad)
    else:
        ref, mag = _gs_ref(x, src, dst, N, reduce, grad)
    _acc(a.grad, ref, mag, dtype, f"gather_scatter {reduce} F={F} {dtype}")


# ---- segment_csr -----------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", DTYPES, ids=_dt)
@pytest.mark.parametrize("F", WIDTHS)
@pytest.mark.parametrize("reduce", ["sum", "mean", "min", "max"])
def test_segment_csr(cuda, dtype, F, reduce):
    """indptr covers a sub-range [7, hi) of the dim, with empty and long segments; elements
    outside it get no gradient."""
    import torch_scatter
    g = torch.Generator().manual_seed(500 + F)
    lens = [0, 5, *_hubs(F), 0, 17, 1, 0, 40]
    lens += torch.randint(0, 12, (60,), generator=g).tolist()
    lo = 7
    indptr = torch.tensor([lo] + lens).cumsum(0)
    hi = int(indptr[-1])
    E = hi + 11
    M = len(lens)
    src = _values((E, F), dtype, g, coarse=reduce in ("min", "max")).to(cuda)
    grad = _upstream(M, F, dtype, g).to(cuda)
    a = src.clone().requires_grad_()
    out = torch_scatter.segment_csr(a, indptr.to(cuda), reduce=reduce)
    out.backward(grad)
    seg = torch.repeat_interleave(torch.arange(M), torch.tensor(lens)).to(cuda)
    what = f"segment_csr {reduce} F={F} {dtype}"
    if reduce in ("min", "max"):
        _, arg = oracle.scatter(src[lo:hi].cpu(), seg.cpu(), 0, M, reduce)
        arg = torch.where(arg == hi - lo, torch.full_like(arg, E), arg + lo)
        _exact(a.grad, _extreme_grad(grad, arg, 0, E), what)
        return
    ref = torch.zeros(E, F, dtype=torch.float64, device=cuda)
    ref[lo:hi] = _native_ref(src[lo:hi], seg, 0, M, reduce, grad)
    if reduce == "sum":
        _exact(a.grad, ref, what)
    else:
        _div(a.grad, ref, dtype, what)


# ---- SparseTensor.matmul / torch_sparse.spmm ----------------------------------------------------
def _csr_graph(F, g, m=300, n=400):
    """(row, col) sorted by row * n + col (so SparseTensor keeps the input order), with destination
    hubs, a source hub (column 0, 4000 entries), empty rows and duplicate entries."""
    row = _hub_index(m, _hubs(F), 5000, g)
    col = torch.randint(1, n, (row.numel(),), generator=g)
    col[torch.randperm(row.numel(), generator=g)[:4000]] = 0
    key = row * n + col
    order = torch.sort(key, stable=True).indices
    return row[order], col[order], m, n


def _spmm_ref(row, col, value, mat, m, reduce, grad):
    """fp64 reference gradients w.r.t. mat and value (value may be None) and their sums of |terms|."""
    mat64 = mat.double().requires_grad_()
    v64 = value.double().requires_grad_() if value is not None else None
    msgs = mat64[col] * (v64.view(-1, 1) if v64 is not None else 1.0)
    out = torch.zeros(m, mat.size(1), dtype=torch.float64, device=mat.device).index_add(0, row, msgs)
    g64 = grad.double()
    if reduce == "mean":
        cnt = torch.bincount(row, minlength=m).clamp(min=1).double().view(-1, 1)
        out = out / cnt
        g64 = g64 / cnt
    out.backward(grad.double())
    gr = g64.abs()[row]
    vabs = value.double().abs().view(-1, 1) if value is not None else 1.0
    mag_mat = torch.zeros_like(mat64).index_add_(0, col, gr * vabs)
    mag_val = (gr * mat.double().abs()[col]).sum(1)
    return mat64.grad, mag_mat, (v64.grad if v64 is not None else None), mag_val


def _spmm_extreme_ref(rowptr, col, value, mat, reduce, grad):
    _, arg = oracle.spmm_csr(rowptr.cpu(), col.cpu(), value.cpu() if value is not None else None,
                             mat.cpu(), reduce)
    arg = arg.to(mat.device)
    nnz, n, F = col.numel(), mat.size(0), mat.size(1)
    hit = arg < nnz
    safe = torch.where(hit, arg, torch.zeros_like(arg))
    g64 = torch.where(hit, grad.double(), torch.zeros((), dtype=torch.float64, device=mat.device))
    v = value.double()[safe] if value is not None else torch.ones_like(g64)
    winner = torch.where(hit, col[safe], torch.full_like(arg, n))
    g_mat = torch.zeros(n + 1, F, dtype=torch.float64, device=mat.device)
    mag_mat = torch.zeros_like(g_mat)
    g_mat.scatter_add_(0, winner, g64 * v)
    mag_mat.scatter_add_(0, winner, (g64 * v).abs())
    cols = torch.arange(F, device=mat.device).view(1, -1)
    contrib = g64 * mat.double()[col[safe], cols]
    g_val = torch.zeros(nnz + 1, dtype=torch.float64, device=mat.device)
    mag_val = torch.zeros_like(g_val)
    slot = torch.where(hit, arg, torch.full_like(arg, nnz)).reshape(-1)
    g_val.index_add_(0, slot, contrib.reshape(-1))
    mag_val.index_add_(0, slot, contrib.abs().reshape(-1))
    return g_mat[:n], mag_mat[:n], g_val[:nnz], mag_val[:nnz]


@pytest.mark.parametrize("dtype", DTYPES, ids=_dt)
@pytest.mark.parametrize("F", WIDTHS)
@pytest.mark.parametrize("reduce", ["sum", "mean", "min", "max"])
@pytest.mark.parametrize("with_value", [False, True], ids=["novalue", "value"])
def test_sparse_matmul(cuda, dtype, F, reduce, with_value):
    import torch_sparse
    g = torch.Generator().manual_seed(600 + F)
    row, col, m, n = _csr_graph(F, g)
    row, col = row.to(cuda), col.to(cuda)
    ext = reduce in ("min", "max")
    mat = _values((n, F), dtype, g, coarse=ext).to(cuda)
    if ext:
        value = _mul_values((row.numel(),), dtype, g).abs().to(cuda)     # products exact: ties are real ties
    else:
        value = (torch.rand(row.numel(), generator=g) + 0.5).to(dtype).to(cuda)
    grad = _upstream(m, F, dtype, g, scale=16 if reduce == "mean" else 1).to(cuda)
    va = value.clone().requires_grad_() if with_value else None
    ma = mat.clone().requires_grad_()
    adj = torch_sparse.SparseTensor(row=row, col=col, value=va, sparse_sizes=(m, n))
    out = adj.matmul(ma, reduce=reduce)
    out.backward(grad)
    what = f"SparseTensor.matmul {reduce} F={F} {dtype} value={with_value}"
    v = value if with_value else None
    if ext:
        rowptr = torch.zeros(m + 1, dtype=torch.int64, device=cuda)
        rowptr[1:] = torch.bincount(row, minlength=m).cumsum(0)
        g_mat, mag_mat, g_val, mag_val = _spmm_extreme_ref(rowptr, col, v, mat, reduce, grad)
    else:
        g_mat, mag_mat, g_val, mag_val = _spmm_ref(row, col, v, mat, m, reduce, grad)
    _acc(ma.grad, g_mat, mag_mat, dtype, what + " d/dmat")
    if with_value:
        _acc(va.grad, g_val, mag_val, dtype, what + " d/dvalue")


@pytest.mark.parametrize("dtype", DTYPES, ids=_dt)
@pytest.mark.parametrize("F", WIDTHS)
def test_spmm_functional(cuda, dtype, F):
    import torch_sparse
    g = torch.Generator().manual_seed(700 + F)
    row, col, m, n = _csr_graph(F, g)
    perm = torch.randperm(row.numel(), generator=g)          # unsorted COO input
    row, col = row[perm].to(cuda), col[perm].to(cuda)
    mat = _values((n, F), dtype, g, coarse=False).to(cuda)
    value = (torch.rand(row.numel(), generator=g) + 0.5).to(dtype).to(cuda)
    grad = _upstream(m, F, dtype, g, scale=1).to(cuda)
    va, ma = value.clone().requires_grad_(), mat.clone().requires_grad_()
    out = torch_sparse.spmm(torch.stack([row, col]), va, m, n, ma)
    out.backward(grad)
    g_mat, mag_mat, g_val, mag_val = _spmm_ref(row, col, value, mat, m, "sum", grad)
    _acc(ma.grad, g_mat, mag_mat, dtype, f"spmm F={F} {dtype} d/dmat")
    _acc(va.grad, g_val, mag_val, dtype, f"spmm F={F} {dtype} d/dvalue")


# ---- composites (bf16) ----------------------------------------------------------------------------
def _ref_softmax(src, index, n):
    mx = torch.zeros(n, src.size(1), dtype=src.dtype, device=src.device).scatter_reduce(
        0, index.view(-1, 1).expand_as(src), src.detach(), "amax", include_self=False)
    e = (src - mx.index_select(0, index)).exp()
    s = torch.zeros(n, src.size(1), dtype=src.dtype, device=src.device).index_add(0, index, e)
    return e / s.index_select(0, index), mx, s


@pytest.mark.parametrize("fn", ["softmax", "log_softmax", "logsumexp", "std"])
def test_composites_bf16(cuda, fn):
    """bf16 at the project tolerance (1e-2), against fp64 autograd of the same composition."""
    import torch_scatter
    g = torch.Generator().manual_seed(800)
    N, F = 60, 7
    index = _hub_index(N, (301,), 900, g, n_empty=0).to(cuda)
    E = index.numel()
    src = torch.randn(E, F, generator=g).to(torch.bfloat16).to(cuda)
    w = torch.randn(E if fn in ("softmax", "log_softmax") else N, F, generator=g).to(torch.bfloat16).to(cuda)
    a = src.clone().requires_grad_()
    b = src.double().requires_grad_()
    if fn == "softmax":
        out, ref = torch_scatter.scatter_softmax(a, index, dim=0), _ref_softmax(b, index, N)[0]
    elif fn == "log_softmax":
        out, ref = torch_scatter.scatter_log_softmax(a, index, dim=0), _ref_softmax(b, index, N)[0].log()
    elif fn == "logsumexp":
        out = torch_scatter.scatter_logsumexp(a, index, dim=0, dim_size=N)
        _, mx, s = _ref_softmax(b, index, N)
        ref = (s + 1e-12).log() + mx
    else:
        out = torch_scatter.scatter_std(a, index, dim=0, dim_size=N)
        cnt = torch.bincount(index, minlength=N).double().view(-1, 1)
        mean = torch.zeros(N, F, dtype=torch.float64, device=cuda).index_add(0, index, b) / cnt.clamp(min=1)
        d = b - mean.index_select(0, index)
        ref = (torch.zeros(N, F, dtype=torch.float64, device=cuda).index_add(0, index, d * d)
               / ((cnt - 1).clamp(min=1) + 1e-6)).sqrt()
    (out * w).sum().backward()
    (ref * w.double()).sum().backward()
    for got, want, what in ((out.detach(), ref.detach(), "value"), (a.grad, b.grad, "grad")):
        err = (got.double() - want).abs()
        bound = 1e-2 * (want.abs() + want.abs().max())
        assert (err <= bound).all(), f"{fn} {what}: max err {err.max().item():.3e}"


# ---- dispatcher entries and TorchScript -----------------------------------------------------------
@pytest.mark.parametrize("dtype", DTYPES, ids=_dt)
def test_dispatcher_and_torchscript_gradients(cuda, dtype):
    """Gradients through torch.ops.torch_scatter.* / torch.ops.torch_sparse.*, called directly and
    from a scripted function, are bit-identical to the Python path's."""
    import torch_scatter
    import torch_sparse
    ts, sp = torch.ops.torch_scatter, torch.ops.torch_sparse
    g = torch.Generator().manual_seed(900)
    N, F = 50, 8
    index = _hub_index(N, (301, 3001), 700, g).to(cuda)
    E = index.numel()
    src = _values((E, F), dtype, g, coarse=True).to(cuda)
    gs = _upstream(N, F, dtype, g).to(cuda)
    lens = torch.bincount(index, minlength=N)
    indptr = torch.cat([lens.new_zeros(1), lens.cumsum(0)])
    # unique columns: no two max winners share a source row, so the mat gradient has no collisions
    m, n, nnz = 40, 4000, 3000
    row = torch.sort(torch.randint(0, m - 2, (nnz,), generator=g)).values.to(cuda)
    col = torch.randperm(n, generator=g)[:nnz].to(cuda)
    rowptr = torch.cat([row.new_zeros(1), torch.bincount(row, minlength=m).cumsum(0)])
    value = (torch.rand(nnz, generator=g) + 0.5).to(dtype).to(cuda)
    mat = _values((n, F), dtype, g, coarse=True).to(cuda)
    gm = _upstream(m, F, dtype, g).to(cuda)

    @torch.jit.script
    def ts_scatter(s: torch.Tensor, i: torch.Tensor, n: int, red: str) -> torch.Tensor:
        if red == "sum":
            return torch.ops.torch_scatter.scatter_sum(s, i, 0, None, n)
        if red == "mean":
            return torch.ops.torch_scatter.scatter_mean(s, i, 0, None, n)
        return torch.ops.torch_scatter.scatter_max(s, i, 0, None, n)[0]

    @torch.jit.script
    def ts_segment(s: torch.Tensor, p: torch.Tensor, red: str) -> torch.Tensor:
        if red == "sum":
            return torch.ops.torch_scatter.segment_sum_csr(s, p, None)
        if red == "mean":
            return torch.ops.torch_scatter.segment_mean_csr(s, p, None)
        return torch.ops.torch_scatter.segment_max_csr(s, p, None)[0]

    @torch.jit.script
    def ts_spmm(rp: torch.Tensor, c: torch.Tensor, v: torch.Tensor, x: torch.Tensor, red: str) -> torch.Tensor:
        if red == "sum":
            return torch.ops.torch_sparse.spmm_sum(None, rp, c, v, None, None, x)
        if red == "mean":
            return torch.ops.torch_sparse.spmm_mean(None, rp, c, v, None, None, None, x)
        return torch.ops.torch_sparse.spmm_max(rp, c, v, x)[0]

    def grads(fn, inputs, upstream):
        leaves = [t.clone().requires_grad_() for t in inputs]
        torch.autograd.backward(fn(*leaves), upstream)
        return [t.grad for t in leaves]

    def same(a, b, what):
        for x, y in zip(a, b):
            assert torch.equal(x.view(_VIEW[dtype]), y.view(_VIEW[dtype])), what

    for red in ("sum", "mean", "max"):
        py = grads(lambda s: torch_scatter.scatter(s, index, 0, dim_size=N, reduce=red), [src], gs)
        same(py, grads(lambda s: getattr(ts, "scatter_" + red)(s, index, 0, None, N), [src], gs)
             if red != "max" else grads(lambda s: ts.scatter_max(s, index, 0, None, N)[0], [src], gs),
             f"scatter_{red} dispatcher")
        same(py, grads(lambda s: ts_scatter(s, index, N, red), [src], gs), f"scatter_{red} script")

        py = grads(lambda s: torch_scatter.segment_csr(s, indptr, reduce=red), [src], gs)
        direct = (lambda s: ts.segment_max_csr(s, indptr, None)[0]) if red == "max" else \
            (lambda s: getattr(ts, f"segment_{red}_csr")(s, indptr, None))
        same(py, grads(direct, [src], gs), f"segment_{red}_csr dispatcher")
        same(py, grads(lambda s: ts_segment(s, indptr, red), [src], gs), f"segment_{red}_csr script")

        py = grads(lambda v, x: torch_sparse.SparseTensor(rowptr=rowptr, col=col, value=v, sparse_sizes=(m, n))
                   .matmul(x, reduce=red), [value, mat], gm)
        if red == "sum":
            direct = lambda v, x: sp.spmm_sum(None, rowptr, col, v, None, None, x)      # noqa: E731
        elif red == "mean":
            direct = lambda v, x: sp.spmm_mean(None, rowptr, col, v, None, None, None, x)  # noqa: E731
        else:
            direct = lambda v, x: sp.spmm_max(rowptr, col, v, x)[0]                     # noqa: E731
        same(py, grads(direct, [value, mat], gm), f"spmm_{red} dispatcher")
        same(py, grads(lambda v, x: ts_spmm(rowptr, col, v, x, red), [value, mat], gm), f"spmm_{red} script")


# ---- a training loop ------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", DTYPES, ids=_dt)
def test_training_loop(cuda, dtype):
    """Three steps on a fixed graph with changing features, run twice: sum / mean gradients are
    bit-identical across the repeats, no plan is built after step 1, and a non-contiguous upstream
    gradient gives the same result as its contiguous copy."""
    import gno_b200
    import torch_scatter
    import torch_sparse
    from gno_b200 import autograd as ag
    g = torch.Generator().manual_seed(1000)
    F = 33
    src, dst, n, N = _gs_graph(F, g)
    src, dst = src.to(cuda), dst.to(cuda)
    adj = torch_sparse.SparseTensor(row=dst, col=src, sparse_sizes=(N, n))
    sidx = dst[:n].clone()          # a 1-D index over the features themselves
    feats = [_values((n, F), dtype, g, coarse=True).to(cuda) for _ in range(3)]
    ups = [_upstream(N, F, dtype, g).to(cuda) for _ in range(3)]
    ops = {
        "gather_scatter sum": lambda x: ag.gather_scatter(x, src, dst, N, "sum"),
        "gather_scatter mean": lambda x: ag.gather_scatter(x, src, dst, N, "mean"),
        "matmul sum": lambda x: adj.matmul(x, "sum"),
        "matmul mean": lambda x: adj.matmul(x, "mean"),
        "scatter mean": lambda x: torch_scatter.scatter(x, sidx, 0, dim_size=N, reduce="mean"),
    }

    def step(op, t, upstream=None):
        x = feats[t].clone().requires_grad_()
        out = op(x)
        out.backward(ups[t] if upstream is None else upstream)
        return x.grad

    runs = []
    misses = []
    for rep in range(2):
        res = {}
        for t in range(3):
            m0 = gno_b200.plan_cache.misses
            for name, op in ops.items():
                res[(name, t)] = step(op, t)
            misses.append(gno_b200.plan_cache.misses - m0)
        runs.append(res)
    assert misses[1:] == [0] * 5, f"plans built after step 1: {misses}"
    for key, got in runs[0].items():
        assert torch.equal(got.view(_VIEW[dtype]), runs[1][key].view(_VIEW[dtype])), f"{key} not reproducible"

    for name, op in ops.items():
        x = feats[0].clone().requires_grad_()
        op(x).sum().backward()                                   # expanded (stride-0) upstream gradient
        want = step(op, 0, torch.ones(N, F, dtype=dtype, device=cuda))
        assert torch.equal(x.grad.view(_VIEW[dtype]), want.view(_VIEW[dtype])), f"{name}: expanded gradient"
        gt = ups[1].t().contiguous().t()                         # transposed view
        assert not gt.is_contiguous()
        assert torch.equal(step(op, 0, gt).view(_VIEW[dtype]), step(op, 0, ups[1]).view(_VIEW[dtype])), \
            f"{name}: transposed gradient"

    # max / min: the backward scatters to the winners through the full-shape scatter, whose first call
    # on an index takes the atomic path; collisions make it reproducible only up to the bound
    for reduce in ("max", "min"):
        for t in range(3):
            x = feats[t].clone().requires_grad_()
            ag.gather_scatter(x, src, dst, N, reduce)[0].backward(ups[t])
            ref, mag = _gs_extreme_ref(feats[t], src, dst, N, reduce, ups[t])
            _acc(x.grad, ref, mag, dtype, f"gather_scatter {reduce} step {t}")


# ---- the value-permutation memo -------------------------------------------------------------------
def test_value_permutation_memo_follows_the_plan(cuda):
    """Permuted edge values are memoised per (value, plan).  Cycle one value tensor through more index
    tensors of identical shape than the plan cache holds, then revisit the first ones: an evicted
    plan's freed rowptr may be handed to the next plan, which must not inherit its permutation."""
    import gno_b200
    import torch_sparse
    gno_b200.clear_caches()
    g = torch.Generator().manual_seed(1100)
    m, n, nnz, F = 64, 80, 3000, 8
    k = gno_b200.plan_cache.capacity + 2
    value = (torch.rand(nnz, generator=g) + 0.5).to(cuda)
    mat = torch.randn(n, F, generator=g).to(cuda)
    grad = torch.randn(m, F, generator=g).to(cuda)
    coo = [torch.stack([torch.randint(0, m, (nnz,), generator=g),
                        torch.randint(0, n, (nnz,), generator=g)]).to(cuda) for _ in range(k)]

    def check_spmm(i):
        out = torch_sparse.spmm(coo[i], value, m, n, mat)
        ref = torch.zeros(m, F, dtype=torch.float64, device=cuda).index_add(
            0, coo[i][0], mat.double()[coo[i][1]] * value.double().view(-1, 1))
        mag = torch.zeros_like(ref).index_add(0, coo[i][0], (mat.double()[coo[i][1]] * value.double().view(-1, 1)).abs())
        _acc(out, ref, mag, torch.float32, f"spmm on index {i}")

    for i in list(range(k)) + [0, 1, 2]:
        check_spmm(i)

    # the backward's transposed product memoises the same way on the column plan
    gno_b200.clear_caches()
    rowptr = torch.cat([torch.zeros(1, dtype=torch.int64), torch.full((m,), nnz // m).cumsum(0)]).to(cuda)
    rowptr[-1] = nnz
    row = torch.repeat_interleave(torch.arange(m, device=cuda), rowptr[1:] - rowptr[:-1])
    cols = [torch.randint(0, n, (nnz,), generator=g).to(cuda) for _ in range(k)]

    def check_matmul(i):
        ma = mat.clone().requires_grad_()
        adj = torch_sparse.SparseTensor(rowptr=rowptr, col=cols[i], value=value, sparse_sizes=(m, n))
        adj.matmul(ma).backward(grad)
        ref, mag, _, _ = _spmm_ref(row, cols[i], value, mat, m, "sum", grad)
        _acc(ma.grad, ref, mag, torch.float32, f"matmul backward on column set {i}")

    for i in list(range(k)) + [0, 1, 2]:
        check_matmul(i)


# ---- empty inputs and dropped entries -----------------------------------------------------------
@pytest.mark.parametrize("reduce", ["sum", "mean", "mul", "min", "max"])
def test_empty_inputs(cuda, reduce):
    """E = 0, N = 0 and F = 0 give zero (or empty) gradients of the right shape on every op."""
    import torch_scatter
    import torch_sparse
    from gno_b200 import autograd as ag
    i64 = dict(dtype=torch.int64, device=cuda)
    for E, N, F in ((0, 5, 4), (0, 0, 4), (6, 5, 0)):
        index = torch.arange(E, **i64) % max(N, 1)
        a = torch.ones(E, F, device=cuda, requires_grad=True)
        out = torch_scatter.scatter(a, index, 0, dim_size=N, reduce=reduce)
        out.backward(torch.ones_like(out))
        assert a.grad.shape == (E, F), ("scatter", reduce, E, N, F)
        if reduce == "mul":
            continue
        x = torch.ones(3, F, device=cuda, requires_grad=True)
        out = ag.gather_scatter(x, index % 3, index, N, reduce)
        out = out[0] if isinstance(out, tuple) else out
        out.backward(torch.ones_like(out))
        assert x.grad.shape == (3, F) and not x.grad.any(), ("gather_scatter", reduce, E, N, F)
        s = torch.ones(E, F, device=cuda, requires_grad=True)
        indptr = torch.zeros(N + 1, **i64)
        indptr[1:] = E // max(N, 1) * torch.arange(1, N + 1, **i64)
        if N:
            indptr[-1] = E
        out = torch_scatter.segment_csr(s, indptr, reduce=reduce)
        out.backward(torch.ones_like(out))
        assert s.grad.shape == (E, F), ("segment_csr", reduce, E, N, F)
        # a CSR matrix without entries, with and without values
        for with_value in (False, True):
            mat = torch.ones(4, F, device=cuda, requires_grad=True)
            v = torch.ones(0, device=cuda, requires_grad=True) if with_value else None
            adj = torch_sparse.SparseTensor(rowptr=torch.zeros(N + 1, **i64), col=torch.zeros(0, **i64),
                                            value=v, sparse_sizes=(N, 4))
            out = adj.matmul(mat, reduce=reduce)
            out.backward(torch.ones_like(out))
            assert mat.grad.shape == (4, F) and not mat.grad.any(), ("matmul", reduce, E, N, F, with_value)
            if with_value:
                assert v.grad is None or v.grad.shape == (0,)


@pytest.mark.filterwarnings("ignore:gno_b200")
@pytest.mark.parametrize("dtype", DTYPES, ids=_dt)
@pytest.mark.parametrize("reduce", ["sum", "mean", "mul", "min", "max"])
def test_dropped_entries(cuda, dtype, reduce):
    """Entries outside [0, dim_size) are dropped by the forward and get zero gradient, on every
    backward path: 1-D index along dim 0 and along the last dim, full-shape index, gather_scatter."""
    import torch_scatter
    from gno_b200 import autograd as ag
    g = torch.Generator().manual_seed(1200)
    N, F = 120, 8
    index = _hub_index(N, () if reduce == "mul" else (301,), 800, g)   # a 301-factor product overflows fp16
    index[::7] = N + 3
    index = index.to(cuda)
    E = index.numel()
    mk = (lambda shape: _mul_values(shape, dtype, g)) if reduce == "mul" else \
        (lambda shape: _values(shape, dtype, g, coarse=reduce in ("min", "max")))
    grad = _upstream(N, F, dtype, g).to(cuda)
    cases = [("dim 0", mk((E, F)).to(cuda), index, 0),
             ("last dim", mk((F, E)).to(cuda), index, 1)]
    full = index.view(-1, 1).repeat(1, F)
    full[torch.randperm(E, generator=g)[:E // 5].to(cuda), 3] = N + 5
    cases.append(("full-shape", mk((E, F)).to(cuda), full, 0))
    for what, src, idx, dim in cases:
        a = src.clone().requires_grad_()
        out = torch_scatter.scatter(a, idx, dim, dim_size=N, reduce=reduce)
        up = grad if dim == 0 else grad.t().contiguous()
        out.backward(up)
        # the reference gives dropped entries exactly zero gradient
        _check_scatter_grad(a.grad, src, idx, dim, N, reduce, up, dtype, f"dropped {what} {reduce} {dtype}")
    if reduce == "mul":
        return
    n = 90
    x = _values((n, F), dtype, g, coarse=reduce in ("min", "max")).to(cuda)
    src_ids = torch.randint(0, n, (E,), generator=g).to(cuda)
    a = x.clone().requires_grad_()
    out = ag.gather_scatter(a, src_ids, index, N, reduce)
    out = out[0] if isinstance(out, tuple) else out
    out.backward(grad)
    keep = index < N
    if reduce in ("min", "max"):
        ref, mag = _gs_extreme_ref(x, src_ids, index, N, reduce, grad)
    else:
        ref, mag = _gs_ref(x, src_ids, index, N, reduce, grad, valid=keep)
    _acc(a.grad, ref, mag, dtype, f"dropped gather_scatter {reduce} {dtype}")


# ---- full size (products-shaped graph) ------------------------------------------------------------
def _products(dev):
    import bench as B
    n, e, F, _, ex, off = B.WORKLOADS["products"]
    src, dst = B.make_graph(n, n, e, ex, off, dev, 42)
    return n, F, src, dst


def _transposed_ref(g64, src, dst, n, step=4_000_000):
    """fp64 sum over edges of g64[dst[e]] into row src[e], and the sum of |terms|, over edge slices."""
    ref = torch.zeros(n, g64.size(1), dtype=torch.float64, device=g64.device)
    mag = torch.zeros_like(ref)
    for a in range(0, dst.numel(), step):
        t = g64[dst[a:a + step]]
        ref.index_add_(0, src[a:a + step], t)
        mag.index_add_(0, src[a:a + step], t.abs_())
        del t
    return ref, mag


def test_fullsize_products(cuda):
    """Products-shaped graph (2.45M nodes, 61.9M edges, F=100): gather_scatter sum / mean backward in
    bf16 and fp32, max backward by conservation, SparseTensor.matmul(sum) backward in bf16."""
    import torch_sparse
    from gno_b200 import autograd as ag
    n, F, src, dst = _products(cuda)
    gen = torch.Generator(device=cuda).manual_seed(7)
    cnt = torch.bincount(dst, minlength=n).clamp(min=1).double().view(-1, 1)
    for dtype in (torch.bfloat16, torch.float32):
        x = torch.randn(n, F, device=cuda, generator=gen).to(dtype)
        grad = torch.randn(n, F, device=cuda, generator=gen).to(dtype)
        for reduce in ("sum", "mean"):
            a = x.clone().requires_grad_()
            ag.gather_scatter(a, src, dst, n, reduce).backward(grad)
            g64 = grad.double() / cnt if reduce == "mean" else grad.double()
            ref, mag = _transposed_ref(g64, src, dst, n)
            del g64
            _acc(a.grad, ref, mag, dtype, f"products gather_scatter {reduce} {dtype}")
            del a, ref, mag
        del x, grad
    # max: every row's gradient lands on the source of its arg edge
    x = torch.randn(n, F, device=cuda, generator=gen)
    grad = torch.randn(n, F, device=cuda, generator=gen)
    a = x.clone().requires_grad_()
    out, arg = ag.gather_scatter(a, src, dst, n, "max")
    out.backward(grad)
    E = src.numel()
    live = arg < E
    winner = torch.where(live, src[arg.clamp(max=E - 1)], torch.full_like(arg, n))
    flat = (winner * F + torch.arange(F, device=cuda)).view(-1)
    g64 = torch.where(live, grad.double(), torch.zeros((), dtype=torch.float64, device=cuda)).view(-1)
    ref = torch.zeros((n + 1) * F, dtype=torch.float64, device=cuda).index_add_(0, flat, g64)
    mag = torch.zeros_like(ref).index_add_(0, flat, g64.abs())
    _acc(a.grad, ref[:n * F].view(n, F), mag[:n * F].view(n, F), torch.float32, "products gather_scatter max")
    del x, a, out, arg, live, winner, flat, g64, ref, mag
    # SparseTensor.matmul(sum) backward w.r.t. mat, bf16
    adj = torch_sparse.SparseTensor(row=dst, col=src, sparse_sizes=(n, n))
    mat = torch.randn(n, F, device=cuda, generator=gen).to(torch.bfloat16).requires_grad_()
    grad = torch.randn(n, F, device=cuda, generator=gen).to(torch.bfloat16)
    adj.matmul(mat).backward(grad)
    ref, mag = _transposed_ref(grad.double(), src, dst, n)
    _acc(mat.grad, ref, mag, torch.bfloat16, "products matmul sum bf16")
