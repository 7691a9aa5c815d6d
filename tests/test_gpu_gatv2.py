"""GATv2 attention logits on the GPU: gno_b200.gatv2_logits (PyG 2.0.2 GATv2Conv.message: x_i + x_j,
leaky_relu, (x * att).sum(-1)), forward and backward.

The reference is fp64 torch on the same stored values.  Every bound is |err| <= tol * sum|terms|,
the sum of the magnitudes of the terms the result adds up."""
import itertools

import pytest
import torch
import torch.nn.functional as Fn

import gno_b200

pytestmark = pytest.mark.gpu

DTYPES = [torch.float32, torch.float16, torch.bfloat16]
TOL = {torch.float32: 1e-5, torch.float16: 1e-2, torch.bfloat16: 1e-2}
SLOPE = 0.2


def bigraph(dev, n_src, n_dst, E, hub_len, seed):
    """Random edges plus one hub destination of hub_len edges (spans several chunks).  Destinations
    with id % 7 == 3 get no edge and sources with id % 5 == 2 are never used; edge order shuffled."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    dst = torch.randint(0, n_dst, (E - hub_len,), generator=g)
    dst = torch.where(dst % 7 == 3, (dst + 1) % n_dst, dst)
    dst = torch.cat([dst, torch.full((hub_len,), n_dst // 2 if (n_dst // 2) % 7 != 3 else 0, dtype=torch.int64)])
    dst = dst[torch.randperm(E, generator=g)]
    src = torch.randint(0, n_src, (E,), generator=g)
    src = torch.where(src % 5 == 2, (src + 1) % n_src, src)
    return src.to(dev), dst.to(dev)


def ref_terms(x_l, x_r, att, src, dst):
    """fp64 att * leaky_relu(x_l[src] + x_r[dst]) as [E, H, C], and z."""
    z = x_l.double()[src] + x_r.double()[dst]
    return att.double() * Fn.leaky_relu(z, SLOPE), z


def check(got, ref, mag, tol, what):
    err = (got.double() - ref).abs()
    assert (err <= tol * mag + 1e-30).all(), f"{what}: max err {(err / (mag + 1e-30)).max().item():.3e}"


def inputs(dev, dtype, n_src, n_dst, H, C, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    x_l = torch.randn((n_src, H, C), generator=g, device=dev).to(dtype)
    x_r = torch.randn((n_dst, H, C), generator=g, device=dev).to(dtype)
    att = torch.randn((H, C), generator=g, device=dev).to(dtype)
    return x_l, x_r, att


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("H", [1, 2, 4, 8])
@pytest.mark.parametrize("C", [1, 3, 8, 16, 33])
def test_logits_forward(cuda, dtype, H, C):
    n_src, n_dst, E = 530, 400, 6001
    src, dst = bigraph(cuda, n_src, n_dst, E, hub_len=1500, seed=H * 10 + C)
    plan = gno_b200.plan_cache.get(dst, n_dst)
    assert plan.max_len > 4 * plan.chunk_len and plan.n_empty > 50
    x_l, x_r, att = inputs(cuda, dtype, n_src, n_dst, H, C, seed=H * 100 + C)
    out = gno_b200.gatv2_logits(x_l, x_r, att, src, dst)
    assert out.shape == (E, H) and out.dtype == dtype
    terms, _ = ref_terms(x_l, x_r, att, src, dst)
    check(out, terms.sum(-1), terms.abs().sum(-1), TOL[dtype], "logits")
    # flat feature rows, PyG's [1, H, C] parameter and a flat att give the same bits
    flat = gno_b200.gatv2_logits(x_l.view(n_src, H * C), x_r.view(n_dst, H * C), att.view(1, H, C), src, dst)
    assert torch.equal(flat, out)
    assert torch.equal(gno_b200.gatv2_logits(x_l, x_r, att.view(H * C), src, dst), out)


def test_logits_negative_slope(cuda):
    src, dst = bigraph(cuda, 300, 200, 3001, hub_len=400, seed=1)
    x_l, x_r, att = inputs(cuda, torch.float32, 300, 200, 4, 8, seed=1)
    out = gno_b200.gatv2_logits(x_l, x_r, att, src, dst, negative_slope=0.01)
    z = x_l.double()[src] + x_r.double()[dst]
    terms = att.double() * Fn.leaky_relu(z, 0.01)
    check(out, terms.sum(-1), terms.abs().sum(-1), 1e-5, "logits")


def ref_grads(x_l, x_r, att, src, dst, g):
    """fp64 autograd of the native formula, and sum|terms| bounds for each gradient."""
    xl = x_l.detach().double().requires_grad_()
    xr = x_r.detach().double().requires_grad_()
    a = att.detach().double().requires_grad_()
    z = xl[src] + xr[dst]
    (Fn.leaky_relu(z, SLOPE) * a).sum(-1).mul(g.double()).sum().backward()
    z = z.detach()
    d = torch.where(z > 0, torch.ones_like(z), torch.full_like(z, SLOPE))
    t = (g.double().unsqueeze(-1) * a.detach() * d).abs()
    mag_l = torch.zeros_like(xl).index_add(0, src, t)
    mag_r = torch.zeros_like(xr).index_add(0, dst, t)
    mag_a = (g.double().unsqueeze(-1) * Fn.leaky_relu(z, SLOPE)).abs().sum(0)
    return (xl.grad, mag_l), (xr.grad, mag_r), (a.grad, mag_a)


SUBSETS = [s for n in (1, 2, 3) for s in itertools.combinations(("x_l", "x_r", "att"), n)]


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("need", SUBSETS, ids=["+".join(s) for s in SUBSETS])
def test_logits_backward(cuda, dtype, need):
    n_src, n_dst, E, H, C = 450, 350, 7001, 4, 8
    src, dst = bigraph(cuda, n_src, n_dst, E, hub_len=1500, seed=11)
    x_l, x_r, att = inputs(cuda, dtype, n_src, n_dst, H, C, seed=11)
    g = torch.randn((E, H), device=cuda).to(dtype)
    ts = {"x_l": x_l, "x_r": x_r, "att": att}
    for name in need:
        ts[name].requires_grad_()
    gno_b200.clear_caches()
    out = gno_b200.gatv2_logits(x_l, x_r, att, src, dst)
    misses = gno_b200.plan_cache.misses
    out.backward(g)
    # the src-sorted plan is built only for grad_x_l
    assert gno_b200.plan_cache.misses - misses == (1 if "x_l" in need else 0)
    refs = dict(zip(("x_l", "x_r", "att"), ref_grads(x_l, x_r, att, src, dst, g)))
    for name, t in ts.items():
        if name not in need:
            assert t.grad is None
            continue
        assert t.grad.dtype == dtype and t.grad.shape == t.shape
        check(t.grad, *refs[name], TOL[dtype], f"grad {name}")
    if "x_r" in need:   # destinations without an edge get exactly 0
        empty = torch.bincount(dst, minlength=n_dst) == 0
        assert empty.sum() > 30 and (x_r.grad[empty] == 0).all()


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("H,C", [(1, 3), (2, 33), (8, 16)])
def test_logits_backward_shapes(cuda, dtype, H, C):
    n, E = 380, 6001
    src, dst = bigraph(cuda, n, n, E, hub_len=1200, seed=H + C)
    x_l, x_r, att = inputs(cuda, dtype, n, n, H, C, seed=H + C)
    g = torch.randn((E, H), device=cuda).to(dtype)
    for t in (x_l, x_r, att):
        t.requires_grad_()
    gno_b200.gatv2_logits(x_l, x_r, att, src, dst).backward(g)
    for t, ref in zip((x_l, x_r, att), ref_grads(x_l, x_r, att, src, dst, g)):
        check(t.grad, *ref, TOL[dtype], "grad")


def test_logits_shared_weights(cuda):
    """x_l is x_r (GATv2Conv(share_weights=True)): autograd adds the two gradients."""
    n, E, H, C = 400, 6001, 4, 8
    src, dst = bigraph(cuda, n, n, E, hub_len=1000, seed=5)
    x, _, att = inputs(cuda, torch.float32, n, n, H, C, seed=5)
    x.requires_grad_()
    att.requires_grad_()
    g = torch.randn((E, H), device=cuda)
    out = gno_b200.gatv2_logits(x, x, att, src, dst)
    out.backward(g)
    terms, _ = ref_terms(x, x, att, src, dst)
    check(out, terms.sum(-1), terms.abs().sum(-1), 1e-5, "logits")
    (gl, ml), (gr, mr), (ga, ma) = ref_grads(x, x, att, src, dst, g)
    check(x.grad, gl + gr, ml + mr, 1e-5, "grad x")
    check(att.grad, ga, ma, 1e-5, "grad att")


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_logits_bitwise_reproducible(cuda, dtype):
    # 2.9 M edges in chunks of 128: 1416 (bf16) / 2832 (fp32) groups of chunks, more than the
    # backward grid's 148 * 8 CTAs at most, so every CTA's grad_att partial spans several groups
    n, E, H, C = 30_000, 2_900_001, 8, 16
    src, dst = bigraph(cuda, n, n, E, hub_len=200_000, seed=3)
    x_l, x_r, att = inputs(cuda, dtype, n, n, H, C, seed=3)
    g = torch.randn((E, H), device=cuda).to(dtype)
    runs = []
    for _ in range(2):
        ts = [t.detach().clone().requires_grad_() for t in (x_l, x_r, att)]
        out = gno_b200.gatv2_logits(*ts, src, dst)
        out.backward(g)
        runs.append([out.detach()] + [t.grad for t in ts])
    for a, b in zip(*runs):
        assert torch.equal(a, b)


def test_logits_non_finite_match_native(cuda):
    n, E, H, C = 60, 901, 2, 8
    src, dst = bigraph(cuda, n, n, E, hub_len=200, seed=9)
    x_l, x_r, att = inputs(cuda, torch.float32, n, n, H, C, seed=9)
    j, i = int(src[0]), int(dst[0])
    x_l[j, 0, 1] = float("nan")
    x_l[j, 1, 2] = float("inf")
    x_r[i, 0, 3] = float("-inf")
    x_r[i, 1, 2] = float("-inf")      # with x_l[j, 1, 2] = +inf: inf - inf on an edge j -> i
    x_r[i, 1, 5] = float("nan")
    g = torch.randn((E, H), device=cuda)
    results = []
    for fused in (True, False):
        ts = [t.detach().clone().requires_grad_() for t in (x_l, x_r, att)]
        if fused:
            out = gno_b200.gatv2_logits(*ts, src, dst)
        else:
            out = (Fn.leaky_relu(ts[0][src] + ts[1][dst], SLOPE) * ts[2]).sum(-1)
        out.backward(g)
        results.append([out.detach()] + [t.grad for t in ts])
    for got, want in zip(*results):
        assert torch.equal(torch.isnan(got), torch.isnan(want))
        assert torch.equal(torch.isposinf(got), torch.isposinf(want))
        assert torch.equal(torch.isneginf(got), torch.isneginf(want))
    assert torch.isnan(results[0][0]).any() and torch.isinf(results[0][0]).any()
    assert torch.isnan(results[0][3]).any()


def test_logits_errors_and_empty(cuda):
    n, H, C = 10, 2, 4
    x_l, x_r, att = inputs(cuda, torch.float32, n, n + 3, H, C, seed=0)
    src = torch.tensor([0, 1, 9], device=cuda)
    dst = torch.tensor([1, 12, 2], device=cuda)
    gno_b200.gatv2_logits(x_l, x_r, att, src, dst)
    with pytest.raises(IndexError):
        gno_b200.gatv2_logits(x_l, x_r, att, torch.tensor([0, 1, n], device=cuda), dst)
    with pytest.raises(IndexError):
        gno_b200.gatv2_logits(x_l, x_r, att, src, torch.tensor([1, n + 3, 2], device=cuda))
    with pytest.raises(IndexError):
        gno_b200.gatv2_logits(x_l, x_r, att, src, torch.tensor([1, -1, 2], device=cuda))
    with pytest.raises(ValueError):
        gno_b200.gatv2_logits(x_l, x_r, torch.randn(4, C, device=cuda), src, dst)       # heads
    with pytest.raises(ValueError):
        gno_b200.gatv2_logits(x_l, x_r.view(n + 3, H * C)[:, :6], att, src, dst)      # width
    with pytest.raises(ValueError):
        gno_b200.gatv2_logits(x_l, x_r.half(), att, src, dst)                         # dtype
    none = torch.empty(0, dtype=torch.int64, device=cuda)
    xl = x_l.clone().requires_grad_()
    out = gno_b200.gatv2_logits(xl, x_r, att, none, none)
    assert out.shape == (0, H)
    out.sum().backward()
    assert (xl.grad == 0).all()


def _layer(x, edge_index, params, H, C, fused):
    """A GATv2-style layer: logits, softmax over each destination, aggregation of x_l."""
    W_l, W_r, att = params
    N = x.size(0)
    src, dst = edge_index[0], edge_index[1]
    x_l = (x @ W_l).view(N, H, C)
    x_r = (x @ W_r).view(N, H, C)
    if fused:
        logits = gno_b200.gatv2_logits(x_l, x_r, att, src, dst)
        alpha = gno_b200.softmax(logits, dst, num_nodes=N)
        return gno_b200.attention_aggregate(x_l, alpha, src, dst, N)
    logits = (Fn.leaky_relu(x_l[src] + x_r[dst], SLOPE) * att).sum(-1)
    m = torch.full((N, H), torch.finfo(logits.dtype).min, device=x.device, dtype=logits.dtype)
    m = m.scatter_reduce(0, dst.view(-1, 1).expand(-1, H), logits.detach(), "amax", include_self=True)
    ex = (logits - m[dst]).exp()
    s = torch.zeros_like(m).index_add(0, dst, ex)
    alpha = ex / (s[dst] + 1e-16)
    return torch.zeros(N, H, C, device=x.device).index_add(0, dst, x_l[src] * alpha.unsqueeze(-1))


def test_gatv2_layer_with_fused_logits_matches_native_torch(cuda):
    torch.manual_seed(0)
    N, E, Fin, H, C = 600, 9001, 32, 4, 8
    src, dst = bigraph(cuda, N, N, E, hub_len=900, seed=17)
    edge_index = torch.stack([src, dst])
    x = torch.randn(N, Fin, device=cuda)
    params = [torch.randn(Fin, H * C, device=cuda) * 0.2, torch.randn(Fin, H * C, device=cuda) * 0.2,
              torch.randn(1, H, C, device=cuda)]
    w = torch.randn(N, H, C, device=cuda)
    grads = {}
    gno_b200.clear_caches()
    for step, fused in enumerate((True, True, False)):
        ps = [p.clone().requires_grad_() for p in params]
        xx = x.clone().requires_grad_()
        misses = gno_b200.plan_cache.misses
        out = _layer(xx, edge_index, ps, H, C, fused)
        (out * w).sum().backward()
        if fused:
            built = gno_b200.plan_cache.misses - misses
            assert built == (2 if step == 0 else 0), f"{built} plans built"
        grads["fused" if fused else "native"] = [out.detach()] + [t.grad for t in [xx] + ps]
    for got, want in zip(grads["fused"], grads["native"]):
        assert torch.allclose(got, want, rtol=1e-4, atol=1e-5), (got - want).abs().max()


def test_fullsize_products_bf16(cuda):
    """products-shaped graph (bench.WORKLOADS), H = 8, C = 16, bf16: logits and the gradients of
    x_l, x_r and att against fp64 over edge slices, |err| <= 1e-2 * sum|terms|."""
    import bench as B
    n, e, _, _, ex, off = B.WORKLOADS["products"]
    src, dst = B.make_graph(n, n, e, ex, off, cuda, 42)
    H, C = 8, 16
    x_l, x_r, att = inputs(cuda, torch.bfloat16, n, n, H, C, seed=3)
    for t in (x_l, x_r, att):
        t.requires_grad_()
    g = torch.randn((e, H), device=cuda).to(torch.bfloat16)
    out = gno_b200.gatv2_logits(x_l, x_r, att, src, dst)
    out.backward(g)
    out = out.detach()
    a = att.detach().double()
    ref_l = torch.zeros((n, H, C), dtype=torch.float64, device=cuda)
    mag_l, ref_r, mag_r = torch.zeros_like(ref_l), torch.zeros_like(ref_l), torch.zeros_like(ref_l)
    ref_a = torch.zeros((H, C), dtype=torch.float64, device=cuda)
    mag_a = torch.zeros_like(ref_a)
    step = 4_000_000
    for lo in range(0, e, step):
        hi = min(e, lo + step)
        s, d = src[lo:hi], dst[lo:hi]
        z = x_l.detach()[s].double() + x_r.detach()[d].double()
        lr = Fn.leaky_relu(z, SLOPE)
        t = a * lr
        check(out[lo:hi], t.sum(-1), t.abs().sum(-1), 1e-2, "logits")
        gg = g[lo:hi].double().unsqueeze(-1)
        t = gg * lr
        ref_a += t.sum(0)
        mag_a += t.abs_().sum(0)
        t = gg * a * torch.where(z > 0, 1.0, SLOPE)
        ref_l.index_add_(0, s, t)
        ref_r.index_add_(0, d, t)
        t.abs_()
        mag_l.index_add_(0, s, t)
        mag_r.index_add_(0, d, t)
        del z, lr, t, gg
    check(att.grad, ref_a, mag_a, 1e-2, "grad att")
    check(x_l.grad, ref_l, mag_l, 1e-2, "grad x_l")
    check(x_r.grad, ref_r, mag_r, 1e-2, "grad x_r")
