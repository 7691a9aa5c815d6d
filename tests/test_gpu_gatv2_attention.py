"""The fused GATv2 message passing on the GPU: gno_b200.gatv2_attention (logits, edge softmax and
attention-weighted aggregation in one pass), forward and backward.

The reference is fp64 torch on the same stored values.  Every bound is |err| <= tol * sum|terms|,
tol 1e-5 in fp32 and 1e-2 in 16-bit dtypes.  For the output out[i] = sum_e alpha_e x_e (x_e the
gathered x_l row, e over row i's edges) the terms are

    sum_e alpha_e * (|x_e| + |x_e - out_i| * A_e),    A_e = sum_c |att * leaky_relu(z_e)|:

the products alpha_e x_e, plus the error of a logit, which is at most tol * A_e and moves the
output by alpha_e * da_e * (x_e - out_i) through the exponential and the normalisation.  The
gradients are sums of da_e = alpha_e * g_i . (x_e - out_i) times att * leaky_relu'(z) (x_l, x_r)
or leaky_relu(z) (att), plus alpha_e * g_i for x_l; |da_e| is bounded by
M_e = alpha_e * sum_c |g_i| (|x_e| + |out_i|) * (1 + A_e), which again carries a logit's error
through the exponential, and the terms use M_e and (1 + A_e) alpha_e |g_i| in their place."""
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


def inputs(dev, dtype, n_src, n_dst, H, C, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    x_l = torch.randn((n_src, H, C), generator=g, device=dev).to(dtype)
    x_r = torch.randn((n_dst, H, C), generator=g, device=dev).to(dtype)
    att = torch.randn((H, C), generator=g, device=dev).to(dtype)
    return x_l, x_r, att


def check(got, ref, mag, tol, what):
    err = (got.double() - ref).abs()
    assert (err <= tol * mag + 1e-30).all(), f"{what}: max err {(err / (mag + 1e-30)).max().item():.3e}"


def reference(x_l, x_r, att, src, dst, n_dst, g=None, slope=SLOPE, step=1 << 62):
    """fp64 output and bound of the docstring, and with g (grad of out) the three gradients and
    their bounds, over edge slices of `step` edges."""
    xl, xr = x_l.detach().double(), x_r.detach().double()
    H, C = xl.shape[1], xl.shape[2]
    a = att.detach().double().reshape(H, C)
    E, dev = src.numel(), xl.device
    slices = [(lo, min(E, lo + step)) for lo in range(0, E, step)]

    def edges(lo, hi):
        s, d = src[lo:hi], dst[lo:hi]
        z = xl[s] + xr[d]
        lr = Fn.leaky_relu(z, slope)
        t = a * lr
        return s, d, z, lr, t.sum(-1), t.abs().sum(-1)

    m = torch.full((n_dst, H), float("-inf"), dtype=torch.float64, device=dev)
    for lo, hi in slices:
        _, d, _, _, lg, _ = edges(lo, hi)
        m.scatter_reduce_(0, d.view(-1, 1).expand(-1, H), lg, "amax")
    m = torch.where(torch.isinf(m), torch.zeros_like(m), m)
    den = torch.zeros_like(m)
    for lo, hi in slices:
        _, d, _, _, lg, _ = edges(lo, hi)
        den.index_add_(0, d, (lg - m[d]).exp())
    den += 1e-16
    out = torch.zeros((n_dst, H, C), dtype=torch.float64, device=dev)
    for lo, hi in slices:
        s, d, _, _, lg, _ = edges(lo, hi)
        out.index_add_(0, d, ((lg - m[d]).exp() / den[d]).unsqueeze(-1) * xl[s])
    mag = torch.zeros_like(out)
    for lo, hi in slices:
        s, d, _, _, lg, A = edges(lo, hi)
        al = ((lg - m[d]).exp() / den[d]).unsqueeze(-1)
        mag.index_add_(0, d, al * (xl[s].abs() + (xl[s] - out[d]).abs() * A.unsqueeze(-1)))
    if g is None:
        return out, mag
    gg = g.detach().double()
    D = (gg * out).sum(-1)
    grads = [torch.zeros_like(xl), torch.zeros_like(xr), torch.zeros_like(a)]
    mags = [torch.zeros_like(xl), torch.zeros_like(xr), torch.zeros_like(a)]
    for lo, hi in slices:
        s, d, z, lr, lg, A = edges(lo, hi)
        al = (lg - m[d]).exp() / den[d]
        gd = gg[d]
        da = (al * ((gd * xl[s]).sum(-1) - D[d])).unsqueeze(-1)
        M = (al * (gd.abs() * (xl[s].abs() + out[d].abs())).sum(-1) * (1 + A)).unsqueeze(-1)
        dz = torch.where(z > 0, 1.0, slope)
        t = da * a * dz
        grads[0].index_add_(0, s, t + al.unsqueeze(-1) * gd)
        grads[1].index_add_(0, d, t)
        grads[2] += (da * lr).sum(0)
        t = M * a.abs() * dz
        mags[0].index_add_(0, s, t + (al * (1 + A)).unsqueeze(-1) * gd.abs())
        mags[1].index_add_(0, d, t)
        mags[2] += (M * lr.abs()).sum(0)
        del z, lr, t, gd, da, M, dz
    return out, mag, list(zip(grads, mags))


def native(x_l, x_r, att, src, dst, n_dst, slope=SLOPE):
    """PyG 2.0.2's GATv2Conv message passing in plain torch (differentiable)."""
    H, C = x_l.shape[1], x_l.shape[2]
    logits = (Fn.leaky_relu(x_l[src] + x_r[dst], slope) * att.reshape(H, C)).sum(-1)
    m = torch.full((n_dst, H), torch.finfo(logits.dtype).min, device=x_l.device, dtype=logits.dtype)
    m = m.scatter_reduce(0, dst.view(-1, 1).expand(-1, H), logits.detach(), "amax", include_self=True)
    ex = (logits - m[dst]).exp()
    s = torch.zeros_like(m).index_add(0, dst, ex)
    alpha = ex / (s[dst] + 1e-16)
    return torch.zeros(n_dst, H, C, device=x_l.device, dtype=x_l.dtype).index_add(
        0, dst, x_l[src] * alpha.unsqueeze(-1))


def composition(x_l, x_r, att, src, dst, n_dst, slope=SLOPE):
    logits = gno_b200.gatv2_logits(x_l, x_r, att, src, dst, negative_slope=slope)
    alpha = gno_b200.softmax(logits, dst, num_nodes=n_dst)
    return gno_b200.attention_aggregate(x_l, alpha, src, dst, n_dst)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("H", [1, 2, 4, 8])
@pytest.mark.parametrize("C", [1, 3, 8, 16, 33, 64])
def test_forward(cuda, dtype, H, C):
    n_src, n_dst, E = 530, 400, 6001
    src, dst = bigraph(cuda, n_src, n_dst, E, hub_len=1500, seed=H * 10 + C)
    plan = gno_b200.plan_cache.get(dst, n_dst)
    assert plan.max_len > 4 * plan.chunk_len and plan.n_empty > 50
    x_l, x_r, att = inputs(cuda, dtype, n_src, n_dst, H, C, seed=H * 100 + C)
    out = gno_b200.gatv2_attention(x_l, x_r, att, src, dst)
    assert out.shape == (n_dst, H, C) and out.dtype == dtype
    ref, mag = reference(x_l, x_r, att, src, dst, n_dst)
    check(out, ref, mag, TOL[dtype], "out")
    empty = torch.bincount(dst, minlength=n_dst) == 0
    assert (out[empty] == 0).all()
    # flat feature rows, PyG's [1, H, C] parameter and a flat att give the same bits
    flat = gno_b200.gatv2_attention(x_l.view(n_src, H * C), x_r.view(n_dst, H * C), att.view(1, H, C), src, dst)
    assert torch.equal(flat, out)
    assert torch.equal(gno_b200.gatv2_attention(x_l, x_r, att.view(H * C), src, dst), out)


def test_negative_slope_and_shared_input(cuda):
    n, E, H, C = 300, 3001, 4, 8
    src, dst = bigraph(cuda, n, n, E, hub_len=400, seed=1)
    x_l, x_r, att = inputs(cuda, torch.float32, n, n, H, C, seed=1)
    out = gno_b200.gatv2_attention(x_l, x_r, att, src, dst, negative_slope=0.01)
    ref, mag = reference(x_l, x_r, att, src, dst, n, slope=0.01)
    check(out, ref, mag, 1e-5, "out")
    out = gno_b200.gatv2_attention(x_l, x_l, att, src, dst)        # x_l is x_r
    ref, mag = reference(x_l, x_l, att, src, dst, n)
    check(out, ref, mag, 1e-5, "out")


SUBSETS = [s for n in (1, 2, 3) for s in itertools.combinations(("x_l", "x_r", "att"), n)]


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("need", SUBSETS, ids=["+".join(s) for s in SUBSETS])
def test_backward(cuda, dtype, need):
    n_src, n_dst, E, H, C = 450, 350, 7001, 4, 8
    src, dst = bigraph(cuda, n_src, n_dst, E, hub_len=1500, seed=11)
    x_l, x_r, att = inputs(cuda, dtype, n_src, n_dst, H, C, seed=11)
    g = torch.randn((n_dst, H, C), device=cuda).to(dtype)
    ts = {"x_l": x_l, "x_r": x_r, "att": att}
    for name in need:
        ts[name].requires_grad_()
    gno_b200.clear_caches()
    out = gno_b200.gatv2_attention(x_l, x_r, att, src, dst)
    misses = gno_b200.plan_cache.misses
    out.backward(g)
    # the src-sorted plan is built only for grad_x_l
    assert gno_b200.plan_cache.misses - misses == (1 if "x_l" in need else 0)
    _, _, refs = reference(x_l, x_r, att, src, dst, n_dst, g)
    # the analytic fp64 gradients of `reference` are fp64 autograd of the native formula (the sums
    # cancel: sum_e alpha_e (x_e - out_i) = 0, so the comparison is against the magnitudes)
    leaves = [t.detach().double().requires_grad_() for t in (x_l, x_r, att)]
    native(*leaves, src, dst, n_dst).backward(g.double())
    for (r, mag), leaf in zip(refs, leaves):
        check(leaf.grad, r, mag, 1e-7, "fp64 autograd vs analytic")
    for name, (ref, mag) in zip(("x_l", "x_r", "att"), refs):
        t = ts[name]
        if name not in need:
            assert t.grad is None
            continue
        assert t.grad.dtype == dtype and t.grad.shape == t.shape
        check(t.grad, ref, mag, TOL[dtype], f"grad {name}")
    if "x_r" in need:   # destinations without an edge get exactly 0
        empty = torch.bincount(dst, minlength=n_dst) == 0
        assert empty.sum() > 30 and (x_r.grad[empty] == 0).all()


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("H,C", [(1, 3), (2, 33), (8, 16), (3, 64)])
def test_backward_shapes(cuda, dtype, H, C):
    n, E = 380, 6001
    src, dst = bigraph(cuda, n, n, E, hub_len=1200, seed=H + C)
    x_l, x_r, att = inputs(cuda, dtype, n, n, H, C, seed=H + C)
    g = torch.randn((n, H, C), device=cuda).to(dtype)
    for t in (x_l, x_r, att):
        t.requires_grad_()
    gno_b200.gatv2_attention(x_l, x_r, att, src, dst).backward(g)
    _, _, refs = reference(x_l, x_r, att, src, dst, n, g)
    for t, (ref, mag) in zip((x_l, x_r, att), refs):
        check(t.grad, ref, mag, TOL[dtype], "grad")


def test_shared_input_backward(cuda):
    """x_l is x_r (GATv2Conv(share_weights=True)): autograd adds the two gradients."""
    n, E, H, C = 400, 6001, 4, 8
    src, dst = bigraph(cuda, n, n, E, hub_len=1000, seed=5)
    x, _, att = inputs(cuda, torch.float32, n, n, H, C, seed=5)
    x.requires_grad_()
    att.requires_grad_()
    g = torch.randn((n, H, C), device=cuda)
    gno_b200.gatv2_attention(x, x, att, src, dst).backward(g)
    _, _, ((gl, ml), (gr, mr), (ga, ma)) = reference(x, x, att, src, dst, n, g)
    check(x.grad, gl + gr, ml + mr, 1e-5, "grad x")
    check(att.grad, ga, ma, 1e-5, "grad att")


def test_agrees_with_composition_fp32(cuda):
    n_src, n_dst, E, H, C = 700, 500, 20001, 4, 16
    src, dst = bigraph(cuda, n_src, n_dst, E, hub_len=3000, seed=21)
    x_l, x_r, att = inputs(cuda, torch.float32, n_src, n_dst, H, C, seed=21)
    g = torch.randn((n_dst, H, C), device=cuda)
    res = []
    for fused in (True, False):
        ts = [t.detach().clone().requires_grad_() for t in (x_l, x_r, att)]
        out = (gno_b200.gatv2_attention(*ts, src, dst) if fused else composition(*ts, src, dst, n_dst))
        out.backward(g)
        res.append([out.detach()] + [t.grad for t in ts])
    ref, mag, grads = reference(x_l, x_r, att, src, dst, n_dst, g)
    for got, want, m in zip(res[0], res[1], [mag] + [mg for _, mg in grads]):
        check(got, want.double(), 2 * m, 1e-5, "fused vs composition")


def test_bf16_error_no_larger_than_composition(cuda):
    """Normwise error against fp64 at a mid-size graph: the fused op rounds once, the composition
    rounds the logits and alpha to bf16 on the way."""
    n, E, H, C = 20_000, 400_001, 8, 16
    src, dst = bigraph(cuda, n, n, E, hub_len=20_000, seed=7)
    x_l, x_r, att = inputs(cuda, torch.bfloat16, n, n, H, C, seed=7)
    x_l, x_r = x_l * 2, x_r * 2                     # logits of several units: exp is sensitive
    ref, _ = reference(x_l, x_r, att, src, dst, n)
    err = {}
    for name, out in (("fused", gno_b200.gatv2_attention(x_l, x_r, att, src, dst)),
                      ("composition", composition(x_l, x_r, att, src, dst, n))):
        err[name] = ((out.double() - ref).norm() / ref.norm()).item()
    assert err["fused"] <= err["composition"], err


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_bitwise_reproducible(cuda, dtype):
    # 1 M edges in chunks of 128: more groups of chunks than the backward grid has CTAs, so every
    # CTA's grad_att partial spans several groups
    n, E, H, C = 30_000, 1_000_001, 8, 16
    src, dst = bigraph(cuda, n, n, E, hub_len=100_000, seed=3)
    x_l, x_r, att = inputs(cuda, dtype, n, n, H, C, seed=3)
    g = torch.randn((n, H, C), device=cuda).to(dtype)
    runs = []
    for _ in range(2):
        ts = [t.detach().clone().requires_grad_() for t in (x_l, x_r, att)]
        out = gno_b200.gatv2_attention(*ts, src, dst)
        out.backward(g)
        runs.append([out.detach()] + [t.grad for t in ts])
    for a, b in zip(*runs):
        assert torch.equal(a, b)


def test_non_finite_rows_match_composition(cuda):
    n, E, H, C = 60, 901, 2, 8
    src, dst = bigraph(cuda, n, n, E, hub_len=200, seed=9)
    x_l, x_r, att = inputs(cuda, torch.float32, n, n, H, C, seed=9)
    j, i = int(src[0]), int(dst[0])
    x_l[j, 0, 1] = float("nan")
    x_l[j, 1, 2] = float("inf")
    x_r[i, 0, 3] = float("-inf")
    x_r[int(dst[5]), 1, 5] = float("nan")
    x_l[int(src[9]), 1, 0] = float("-inf")
    fused = gno_b200.gatv2_attention(x_l, x_r, att, src, dst)
    comp = composition(x_l, x_r, att, src, dst, n)
    assert torch.isnan(comp).any()
    assert torch.equal(torch.isnan(fused).any(-1), torch.isnan(comp).any(-1))


def test_errors_and_empty(cuda):
    n, H, C = 10, 2, 4
    x_l, x_r, att = inputs(cuda, torch.float32, n, n + 3, H, C, seed=0)
    src = torch.tensor([0, 1, 9], device=cuda)
    dst = torch.tensor([1, 12, 2], device=cuda)
    gno_b200.gatv2_attention(x_l, x_r, att, src, dst)
    with pytest.raises(IndexError):
        gno_b200.gatv2_attention(x_l, x_r, att, torch.tensor([0, 1, n], device=cuda), dst)
    with pytest.raises(IndexError):
        gno_b200.gatv2_attention(x_l, x_r, att, src, torch.tensor([1, n + 3, 2], device=cuda))
    with pytest.raises(IndexError):
        gno_b200.gatv2_attention(x_l, x_r, att, src, torch.tensor([1, -1, 2], device=cuda))
    with pytest.raises(ValueError):
        gno_b200.gatv2_attention(x_l, x_r, torch.randn(4, C, device=cuda), src, dst)       # heads
    with pytest.raises(ValueError):
        gno_b200.gatv2_attention(x_l, x_r.view(n + 3, H * C)[:, :6], att, src, dst)      # width
    with pytest.raises(ValueError):
        gno_b200.gatv2_attention(x_l, x_r.half(), att, src, dst)                         # dtype
    none = torch.empty(0, dtype=torch.int64, device=cuda)
    xl = x_l.clone().requires_grad_()
    xr = x_r.clone().requires_grad_()
    out = gno_b200.gatv2_attention(xl, xr, att, none, none)
    assert out.shape == (n + 3, H, C) and (out == 0).all()
    out.sum().backward()
    assert (xl.grad == 0).all() and (xr.grad == 0).all()


def test_saves_no_edge_sized_tensor(cuda):
    n_src, n_dst, E, H, C = 300, 200, 5003, 4, 8
    src, dst = bigraph(cuda, n_src, n_dst, E, hub_len=500, seed=2)
    x_l, x_r, att = inputs(cuda, torch.float32, n_src, n_dst, H, C, seed=2)
    x_l.requires_grad_()
    out = gno_b200.gatv2_attention(x_l, x_r, att, src, dst)
    saved = [t for t in out.grad_fn.saved_tensors if t is not None]
    big = [t for t in saved if t.dim() > 0 and t.size(0) == E]
    assert len(big) == 2
    assert {t.data_ptr() for t in big} == {src.data_ptr(), dst.data_ptr()}


def _layer(x, edge_index, params, H, C, fused):
    """A GATv2 layer: x @ W_l, x @ W_r, then the message passing."""
    W_l, W_r, att = params
    N = x.size(0)
    src, dst = edge_index[0], edge_index[1]
    x_l = (x @ W_l).view(N, H, C)
    x_r = (x @ W_r).view(N, H, C)
    if fused:
        return gno_b200.gatv2_attention(x_l, x_r, att, src, dst)
    return native(x_l, x_r, att, src, dst, N)


def test_gatv2_layer_matches_native_torch(cuda):
    """A GATv2 layer on the fused op in fp32 against the same layer in native torch.  The reference
    is native torch in fp64: the weight gradients are sums over all rows of terms up to ~100, so two
    fp32 runs (the native one accumulates with atomics, in a different order every run) differ from
    each other and from the exact value by a few 1e-5.  Each fp32 layer, fused and native, must lie
    within 1e-5 * max|ref| of it, element by element (both measure ~6e-7 * max|ref|)."""
    torch.manual_seed(0)
    N, E, Fin, H, C = 600, 9001, 32, 4, 8
    src, dst = bigraph(cuda, N, N, E, hub_len=900, seed=17)
    edge_index = torch.stack([src, dst])
    x = torch.randn(N, Fin, device=cuda)
    params = [torch.randn(Fin, H * C, device=cuda) * 0.2, torch.randn(Fin, H * C, device=cuda) * 0.2,
              torch.randn(1, H, C, device=cuda)]
    w = torch.randn(N, H, C, device=cuda)
    results = {}
    gno_b200.clear_caches()
    for step, (name, fused, dtype) in enumerate((("fused", True, torch.float32), ("fused", True, torch.float32),
                                                  ("native", False, torch.float32),
                                                  ("exact", False, torch.float64))):
        ps = [p.to(dtype).clone().requires_grad_() for p in params]
        xx = x.to(dtype).clone().requires_grad_()
        misses = gno_b200.plan_cache.misses
        out = _layer(xx, edge_index, ps, H, C, fused)
        (out * w.to(dtype)).sum().backward()
        if fused:
            built = gno_b200.plan_cache.misses - misses
            assert built == (2 if step == 0 else 0), f"{built} plans built"
        results[name] = [out.detach()] + [t.grad for t in [xx] + ps]
    for what in ("fused", "native"):
        for i, (got, ref) in enumerate(zip(results[what], results["exact"])):
            assert got.dtype == torch.float32
            err = (got.double() - ref).abs().max().item()
            assert err <= 1e-5 * ref.abs().max().item(), f"{what} tensor {i}: max err {err:.3e}"


def test_fullsize_products_bf16(cuda):
    """products-shaped graph (bench.WORKLOADS), H = 8, C = 16, bf16: the output and the gradients of
    x_l, x_r and att against fp64 over edge slices, within 1e-2 of the bounds above."""
    import bench as B
    n, e, _, _, ex, off = B.WORKLOADS["products"]
    src, dst = B.make_graph(n, n, e, ex, off, cuda, 42)
    H, C = 8, 16
    x_l, x_r, att = inputs(cuda, torch.bfloat16, n, n, H, C, seed=3)
    for t in (x_l, x_r, att):
        t.requires_grad_()
    g = torch.randn((n, H, C), device=cuda).to(torch.bfloat16)
    out = gno_b200.gatv2_attention(x_l, x_r, att, src, dst)
    out.backward(g)
    ref, mag, refs = reference(x_l, x_r, att, src, dst, n, g, step=2_000_000)
    check(out.detach(), ref, mag, 1e-2, "out")
    for name, t, (r, m) in zip(("x_l", "x_r", "att"), (x_l, x_r, att), refs):
        check(t.grad, r, m, 1e-2, f"grad {name}")
