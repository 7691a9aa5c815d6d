"""Graph attention on the GPU: gno_b200.softmax (torch_geometric.utils.softmax, PyG 2.0.2) and
gno_b200.attention_aggregate (GATv2's multi-head weighted aggregation), forward and backward.

The reference is fp64 torch on the same inputs: PyG's formulas with torch_scatter's max rule (start
at the dtype's lowest finite value, strictly greater wins, NaN never wins, no winner -> 0)."""
import warnings

import pytest
import torch

import gno_b200

pytestmark = pytest.mark.gpu

DTYPES = [torch.float32, torch.float16, torch.bfloat16]
TOL = {torch.float32: 1e-5, torch.float16: 1e-2, torch.bfloat16: 1e-2}


def ref_softmax(a, index, N, lowest):
    """PyG softmax in fp64 over a [E, H] (differentiable; the max is a constant).  Edges whose
    index lies outside [0, N) get 0."""
    a = a.double()
    E, H = a.shape
    keep = (index >= 0) & (index < N)
    idx = torch.where(keep, index, torch.zeros_like(index))
    masked = torch.where(torch.isnan(a) | ~keep.unsqueeze(1), torch.full_like(a, float("-inf")), a).detach()
    m = torch.full((N, H), lowest, dtype=torch.float64, device=a.device)
    if N:
        m = m.scatter_reduce(0, idx.view(-1, 1).expand(E, H), masked, "amax", include_self=True)
    m = torch.where(m == lowest, torch.zeros_like(m), m)
    mi = m[idx] if N else torch.zeros_like(a)
    ex = torch.where(keep.unsqueeze(1), torch.exp(a - mi), torch.zeros_like(a))
    s = torch.zeros((N, H), dtype=torch.float64, device=a.device).index_add(0, idx, ex)
    return torch.where(keep.unsqueeze(1), ex / ((s[idx] if N else 0) + 1e-16), torch.zeros_like(a))


def ref_aggregate(x, alpha, src, dst, N):
    """fp64 out[i, h, :] = sum_{e: dst[e] = i} alpha[e, h] x[src[e], h, :] and the sum of |terms|."""
    msg = x.double()[src] * alpha.double().unsqueeze(-1)
    out = torch.zeros((N,) + tuple(x.shape[1:]), dtype=torch.float64, device=x.device).index_add(0, dst, msg)
    mag = torch.zeros_like(out).index_add(0, dst, msg.abs())
    return out, mag


def graph(dev, N, E, hub_len=0, seed=0):
    """Random edges plus one hub row of hub_len edges (spans several chunks); edge order shuffled."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    dst = torch.randint(0, N, (E - hub_len,), generator=g)
    dst = torch.cat([dst, torch.full((hub_len,), N // 2, dtype=torch.int64)])
    dst = dst[torch.randperm(E, generator=g)]
    src = torch.randint(0, N, (E,), generator=g)
    return src.to(dev), dst.to(dev)


def lowest(dtype):
    return torch.finfo(dtype).min


def check_softmax(y, ref, tol, index, N):
    # below the dtype's normal range only the subnormal spacing is representable (fp16: 6e-8)
    floor = max(1e-30, torch.finfo(y.dtype).tiny * torch.finfo(y.dtype).eps)
    err = (y.double() - ref).abs()
    bad = err > tol * ref.abs() + floor
    assert not bad.any(), f"max rel err {(err / (ref.abs() + 1e-30)).max().item():.3e}"
    E, H = ref.shape
    rows = torch.zeros((N, H), dtype=torch.float64, device=y.device).index_add(0, index, y.double())
    live = torch.bincount(index, minlength=N) > 0
    assert ((rows[live] - 1).abs() <= 2 * tol).all(), "a row's softmax does not sum to 1"


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("H", [1, 3, 8])
@pytest.mark.parametrize("form", ["index", "ptr"])
def test_softmax_forward(cuda, dtype, H, form):
    N, E, extra = 300, 5001, 37                       # odd E, num_nodes beyond the largest index
    src, dst = graph(cuda, N, E, hub_len=1000, seed=H)
    if form == "ptr":
        dst = dst.sort().values                       # a CSR input: edges already grouped by row
    g = torch.Generator(device=cuda).manual_seed(1)
    a = (torch.randn((E, H), generator=g, device=cuda) * 3).to(dtype)
    a_in = a.view(E) if H == 1 else a
    plan = gno_b200.plan_cache.get(dst, N + extra)
    assert plan.max_len > 4 * plan.chunk_len
    if form == "index":
        y = gno_b200.softmax(a_in, dst, num_nodes=N + extra)
    else:
        ptr = torch.zeros(N + extra + 1, dtype=torch.int64, device=cuda)
        ptr[1:] = torch.cumsum(torch.bincount(dst, minlength=N + extra), 0)
        y = gno_b200.softmax(a_in, ptr=ptr)
    assert y.shape == a_in.shape and y.dtype == dtype
    ref = ref_softmax(a, dst, N + extra, lowest(dtype))
    check_softmax(y.view(E, H), ref, TOL[dtype], dst, N + extra)
    if form == "index" and dtype == torch.float32:   # num_nodes defaults to max(index) + 1
        assert torch.equal(gno_b200.softmax(a_in, dst), y)


def test_softmax_non_finite(cuda):
    N, H = 6, 2
    dst = torch.tensor([0, 0, 0, 1, 1, 2, 2, 3, 3, 3, 5], device=cuda)
    E = dst.numel()
    a = torch.randn(E, H, device=cuda)
    a[dst == 1] = float("-inf")                      # a fully -inf row
    a[5, 0] = float("nan")                           # row 2, head 0
    a[1, 1] = float("inf")                           # row 0, head 1: PyG's exp(inf - inf) is NaN
    y = gno_b200.softmax(a, dst, num_nodes=N)
    assert (y[dst == 1] == 0).all()
    assert torch.isnan(y[dst == 2][:, 0]).all() and not torch.isnan(y[dst == 2][:, 1]).any()
    assert torch.isnan(y[dst == 0][:, 1]).all() and not torch.isnan(y[dst == 0][:, 0]).any()
    nan_expected = torch.zeros(E, H, dtype=torch.bool, device=cuda)
    nan_expected[dst == 2, 0] = True
    nan_expected[dst == 0, 1] = True
    assert torch.equal(torch.isnan(y), nan_expected)
    assert torch.equal(torch.isnan(ref_softmax(a, dst, N, lowest(torch.float32))), nan_expected)
    finite = (dst != 0) & (dst != 1) & (dst != 2)
    check_softmax(y[finite].clone(), ref_softmax(a, dst, N, lowest(torch.float32))[finite], 1e-5, dst[finite], N)
    # a destination outside [0, num_nodes) is dropped: 0, with the plan cache's warning
    bad = dst.clone()
    bad[-1] = N + 4
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        y2 = gno_b200.softmax(torch.randn(E, H, device=cuda), bad, num_nodes=N)
    assert any(issubclass(x.category, RuntimeWarning) for x in w)
    assert (y2[-1] == 0).all() and (y2[:-1] > 0).any()


def test_softmax_bitwise_reproducible(cuda):
    N, E, H = 2000, 300_001, 4
    src, dst = graph(cuda, N, E, hub_len=50_000, seed=3)
    a = torch.randn(E, H, device=cuda).to(torch.bfloat16)
    y1 = gno_b200.softmax(a, dst, num_nodes=N)
    y2 = gno_b200.softmax(a, dst, num_nodes=N)
    assert torch.equal(y1.view(torch.int16), y2.view(torch.int16))
    check_softmax(y1, ref_softmax(a, dst, N, lowest(torch.bfloat16)), 1e-2, dst, N)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("H", [1, 2, 8])
@pytest.mark.parametrize("C", [1, 3, 16, 64])
def test_aggregate_forward(cuda, dtype, H, C):
    N, E = 400, 6001
    src, dst = graph(cuda, N, E, hub_len=700, seed=C)
    dst = torch.where(dst % 7 == 3, (dst + 1) % N, dst)   # every row with id % 7 == 3 stays empty
    g = torch.Generator(device=cuda).manual_seed(H * 100 + C)
    x = torch.randn((N, H, C), generator=g, device=cuda).to(dtype)
    alpha = torch.rand((E, H), generator=g, device=cuda).to(dtype)
    out = gno_b200.attention_aggregate(x, alpha, src, dst, N + 5)
    assert out.shape == (N + 5, H, C) and out.dtype == dtype
    ref, mag = ref_aggregate(x, alpha, src, dst, N + 5)
    err = (out.double() - ref).abs()
    assert (err <= TOL[dtype] * mag + 1e-30).all(), f"max err {(err / (mag + 1e-30)).max().item():.3e}"
    empty = torch.bincount(dst, minlength=N + 5) == 0
    assert empty.sum() > 50 and (out[empty] == 0).all()
    out2 = gno_b200.attention_aggregate(x.view(N, H * C), alpha, src, dst, N + 5)
    assert torch.equal(out2, out)


@pytest.mark.parametrize("dtype", DTYPES)
def test_aggregate_exact_with_powers_of_two(cuda, dtype):
    N, E, H, C = 500, 8001, 4, 24
    src, dst = graph(cuda, N, E, hub_len=1500, seed=5)
    g = torch.Generator(device=cuda).manual_seed(5)
    x = (2.0 ** -torch.randint(0, 4, (N, H, C), generator=g, device=cuda)) * \
        (torch.randint(0, 2, (N, H, C), generator=g, device=cuda) * 2 - 1)
    alpha = 2.0 ** -torch.randint(0, 4, (E, H), generator=g, device=cuda)
    out = gno_b200.attention_aggregate(x.to(dtype), alpha.to(dtype), src, dst, N)
    ref, _ = ref_aggregate(x, alpha, src, dst, N)
    assert torch.equal(out, ref.to(dtype))


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("C", [1, 3, 16, 64])
def test_aggregate_one_head_is_weighted_segment_reduce(cuda, dtype, C):
    N, E = 700, 9001
    src, dst = graph(cuda, N, E, hub_len=2000, seed=C + 1)
    g = torch.Generator(device=cuda).manual_seed(C)
    x = torch.randn((N, C), generator=g, device=cuda).to(dtype)
    alpha = torch.rand((E, 1), generator=g, device=cuda).to(dtype)
    out = gno_b200.attention_aggregate(x, alpha, src, dst, N)
    plan = gno_b200.plan_cache.get(dst, N)
    want = gno_b200.segment_reduce(plan, x, "sum", gidx=plan.sorted_ids(src),
                                   weights=alpha[:, 0][plan.perm.long()])
    assert torch.equal(out.view(N, C), want)


def test_aggregate_empty_inputs(cuda):
    x = torch.randn(5, 2, 3, device=cuda)
    none = torch.empty(0, dtype=torch.int64, device=cuda)
    out = gno_b200.attention_aggregate(x, torch.empty(0, 2, device=cuda), none, none, 4)
    assert out.shape == (4, 2, 3) and (out == 0).all()
    out = gno_b200.attention_aggregate(x, torch.empty(0, 2, device=cuda), none, none, 0)
    assert out.shape == (0, 2, 3)
    assert gno_b200.softmax(torch.empty(0, 3, device=cuda), none).shape == (0, 3)
    with pytest.raises(IndexError):
        gno_b200.attention_aggregate(x, torch.ones(1, 2, device=cuda), torch.tensor([5], device=cuda),
                                     torch.tensor([0], device=cuda), 4)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_softmax_backward(cuda, dtype):
    N, E, H = 300, 5001, 3
    src, dst = graph(cuda, N, E, hub_len=1200, seed=7)
    g = torch.Generator(device=cuda).manual_seed(7)
    a = torch.randn((E, H), generator=g, device=cuda).to(dtype).requires_grad_()
    w = torch.randn((E, H), generator=g, device=cuda).to(dtype)
    y = gno_b200.softmax(a, dst, num_nodes=N)
    (y.float() * w.float()).sum().backward()
    a64 = a.detach().double().requires_grad_()
    y64 = ref_softmax(a64, dst, N, lowest(dtype))
    (y64 * w.double()).sum().backward()
    dot = torch.zeros(N, H, dtype=torch.float64, device=cuda).index_add(0, dst, (w.double() * y64).abs())
    mag = y64.detach() * (w.double().abs() + dot[dst])
    tol = 1e-4 if dtype == torch.float32 else 3e-2
    err = (a.grad.double() - a64.grad).abs()
    assert (err <= tol * mag + 1e-30).all(), f"max err {(err / (mag + 1e-30)).max().item():.3e}"


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("H,C", [(1, 16), (4, 3), (8, 16)])
def test_aggregate_backward(cuda, dtype, H, C):
    N, E = 350, 7001
    src, dst = graph(cuda, N, E, hub_len=1500, seed=11)
    g = torch.Generator(device=cuda).manual_seed(11)
    x = torch.randn((N, H, C), generator=g, device=cuda).to(dtype).requires_grad_()
    alpha = torch.rand((E, H), generator=g, device=cuda).to(dtype).requires_grad_()
    w = torch.randn((N, H, C), generator=g, device=cuda).to(dtype)
    out = gno_b200.attention_aggregate(x, alpha, src, dst, N)
    (out.float() * w.float()).sum().backward()
    x64 = x.detach().double().requires_grad_()
    a64 = alpha.detach().double().requires_grad_()
    ref, _ = ref_aggregate(x64, a64, src, dst, N)
    (ref * w.double()).sum().backward()
    tol = 1e-5 if dtype == torch.float32 else 1e-2
    mag_x = torch.zeros_like(x64).index_add(0, src, (a64.detach().abs().unsqueeze(-1) * w.double().abs()[dst]))
    err = (x.grad.double() - x64.grad).abs()
    assert (err <= tol * mag_x + 1e-30).all()
    mag_a = (w.double().abs()[dst] * x64.detach().abs()[src]).sum(-1)
    err = (alpha.grad.double() - a64.grad).abs()
    assert (err <= tol * mag_a + 1e-30).all()


def test_aggregate_backward_with_dropped_destinations(cuda):
    N, E, H, C = 50, 801, 2, 8
    src, dst = graph(cuda, N, E, seed=13)
    dst = dst.clone()
    dst[::9] = N + 3
    x = torch.randn(N, H, C, device=cuda, requires_grad=True)
    alpha = torch.rand(E, H, device=cuda, requires_grad=True)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        out = gno_b200.attention_aggregate(x, alpha, src, dst, N)
    out.sum().backward()
    keep = dst < N
    x64 = x.detach().double().requires_grad_()
    a64 = alpha.detach().double().requires_grad_()
    ref, _ = ref_aggregate(x64, a64 * keep.unsqueeze(1), src, torch.where(keep, dst, 0), N)
    ref.sum().backward()
    assert torch.allclose(out.double(), ref, rtol=1e-5, atol=1e-5)
    assert torch.allclose(x.grad.double(), x64.grad, rtol=1e-5, atol=1e-5)
    assert torch.allclose(alpha.grad.double(), a64.grad, rtol=1e-5, atol=1e-5)
    assert (alpha.grad[~keep] == 0).all()


def _gatv2(x, edge_index, params, H, C, fused):
    """A GATv2-style layer: logits from torch ops, then softmax and aggregation."""
    W_l, W_r, att = params
    N = x.size(0)
    src, dst = edge_index[0], edge_index[1]
    x_l = (x @ W_l).view(N, H, C)
    x_r = (x @ W_r).view(N, H, C)
    e = torch.nn.functional.leaky_relu(x_l[src] + x_r[dst], 0.2)
    logits = (e * att).sum(-1)                                       # [E, H]
    if fused:
        alpha = gno_b200.softmax(logits, dst, num_nodes=N)
        return gno_b200.attention_aggregate(x_l, alpha, src, dst, N)
    m = torch.full((N, H), torch.finfo(logits.dtype).min, device=x.device, dtype=logits.dtype)
    m = m.scatter_reduce(0, dst.view(-1, 1).expand(-1, H), logits.detach(), "amax", include_self=True)
    ex = (logits - m[dst]).exp()
    s = torch.zeros_like(m).index_add(0, dst, ex)
    alpha = ex / (s[dst] + 1e-16)
    return torch.zeros(N, H, C, device=x.device).index_add(0, dst, x_l[src] * alpha.unsqueeze(-1))


def test_gatv2_layer_matches_native_torch(cuda):
    torch.manual_seed(0)
    N, E, Fin, H, C = 600, 9001, 32, 4, 8
    src, dst = graph(cuda, N, E, hub_len=900, seed=17)
    edge_index = torch.stack([src, dst])
    x = torch.randn(N, Fin, device=cuda)
    params = [torch.randn(Fin, H * C, device=cuda) * 0.2, torch.randn(Fin, H * C, device=cuda) * 0.2,
              torch.randn(H, C, device=cuda)]
    w = torch.randn(N, H, C, device=cuda)
    grads = {}
    gno_b200.clear_caches()
    for fused in (True, True, False):
        ps = [p.clone().requires_grad_() for p in params]
        xx = x.clone().requires_grad_()
        misses = gno_b200.plan_cache.misses
        out = _gatv2(xx, edge_index, ps, H, C, fused)
        (out * w).sum().backward()
        if fused:
            built = gno_b200.plan_cache.misses - misses
            assert built == (2 if "fused" not in grads else 0), f"{built} plans built"
        grads["fused" if fused else "native"] = [out.detach()] + [t.grad for t in [xx] + ps]
    for got, want in zip(grads["fused"], grads["native"]):
        assert torch.allclose(got, want, rtol=1e-4, atol=1e-5), (got - want).abs().max()


def test_fullsize_products_bf16(cuda):
    """products-shaped graph (bench.WORKLOADS), H = 8, C = 16, bf16: forward and grad_x against
    fp64 index_add_ over edge slices, |err| <= 1e-2 * sum|terms|."""
    import bench as B
    n, e, _, _, ex, off = B.WORKLOADS["products"]
    src, dst = B.make_graph(n, n, e, ex, off, cuda, 42)
    H, C = 8, 16
    g = torch.Generator(device=cuda).manual_seed(3)
    x = torch.randn((n, H, C), generator=g, device=cuda).to(torch.bfloat16).requires_grad_()
    alpha = torch.rand((e, H), generator=g, device=cuda).to(torch.bfloat16)
    gout = torch.randn((n, H, C), generator=g, device=cuda).to(torch.bfloat16)
    out = gno_b200.attention_aggregate(x, alpha, src, dst, n)
    out.backward(gout)
    step = 4_000_000

    def sliced(gather_rows, scatter_rows, values):
        ref = torch.zeros((n, H, C), dtype=torch.float64, device=cuda)
        mag = torch.zeros_like(ref)
        for a in range(0, e, step):
            b = min(e, a + step)
            m = values[gather_rows[a:b]].double() * alpha[a:b].double().unsqueeze(-1)
            ref.index_add_(0, scatter_rows[a:b], m)
            mag.index_add_(0, scatter_rows[a:b], m.abs_())
            del m
        return ref, mag

    for got, (ref, mag) in ((out.detach(), sliced(src, dst, x.detach())), (x.grad, sliced(dst, src, gout))):
        err = (got.double() - ref).abs()
        assert (err <= 1e-2 * mag + 1e-30).all(), f"max err {(err / (mag + 1e-30)).max().item():.3e}"
        del ref, mag, err
