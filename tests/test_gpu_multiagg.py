"""multi_aggregate on the GPU (PNAConv.aggregate's aggregators and degree scalers in one pass),
message and gather form, forward and backward.

The reference restates the contract in fp64 torch on the same stored values.  Bounds: sum within
tol * sum|m|, mean within tol * sum|m| / d, var within tol * sum(m^2) / d, std through
|std^2 - std_ref^2| (the same bound on var), each scaled by its scaler, plus tol * |ref| for the
output rounding.  min / max and their winners are bit-identical to gno_b200.scatter /
gather_scatter with return_arg=True."""
import math

import pytest
import torch

import gno_b200
from gno_b200 import multiagg

pytestmark = pytest.mark.gpu

DTYPES = [torch.float32, torch.float16, torch.bfloat16]
TOL = {torch.float32: 1e-5, torch.float16: 1e-2, torch.bfloat16: 1e-2}
AGGS = ("sum", "mean", "min", "max", "var", "std")
SCALERS = ("identity", "amplification", "attenuation", "linear", "inverse_linear")
AVG = {"lin": 7.5, "log": 1.9}


def graph(dev, n_src, n_dst, E, hub_len, seed, n_drop=0):
    """Random edges plus one hub destination of hub_len edges (spans several chunks).  Destinations
    with id % 7 == 3 get no edge; n_drop edges point past n_dst (dropped); order shuffled."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    dst = torch.randint(0, n_dst, (E - hub_len,), generator=g)
    dst = torch.where(dst % 7 == 3, (dst + 1) % n_dst, dst)
    dst = torch.cat([dst, torch.full((hub_len,), 5, dtype=torch.int64)])
    dst[:n_drop] = n_dst + 3
    perm = torch.randperm(E, generator=g)
    dst = dst[perm]
    src = torch.randint(0, n_src, (E,), generator=g)
    return src.to(dev), dst.to(dev)


def scale(name, d):
    return {"identity": torch.ones_like(d), "amplification": torch.log(d + 1) / AVG["log"],
            "attenuation": AVG["log"] / torch.log(d + 1), "linear": d / AVG["lin"],
            "inverse_linear": AVG["lin"] / d}[name]


def ref_stats(m, dst, N, args=None):
    """fp64 per-row statistics of messages m [E, W]: dict of [N, W] tensors and d [N, 1].  With
    args = (argmin, argmax) (edge ids, E = none), min / max are the winners' messages, so their
    gradient goes to the winning edge as the contract says (torch's amin splits ties)."""
    keep = (dst >= 0) & (dst < N)
    won = None
    if args is not None:
        m_ext = torch.cat([m, m.new_zeros((1, m.size(1)))])
        won = [m_ext.gather(0, a) for a in args]
    m, dst = m[keep], dst[keep]
    W = m.size(1)
    deg = torch.bincount(dst, minlength=N).double()
    d = deg.clamp(min=1).view(N, 1)
    z = m.new_zeros((N, W))
    s = z.index_add(0, dst, m)
    sa = z.index_add(0, dst, m.abs())
    sq = z.index_add(0, dst, m * m)
    idx = dst.view(-1, 1).expand_as(m)
    mn = z.scatter_reduce(0, idx, m, "amin", include_self=False)
    mx = z.scatter_reduce(0, idx, m, "amax", include_self=False)
    if won is not None:
        mn, mx = won
    mean = s / d
    var = sq / d - mean * mean
    std = torch.sqrt(torch.relu(var) + 1e-5)
    vals = {"sum": s, "mean": mean, "min": mn, "max": mx, "var": var, "std": std}
    mag = {"sum": sa, "mean": sa / d, "min": mn.abs(), "max": mx.abs(), "var": sq / d, "std": sq / d}
    return vals, mag, d


def ref_output(m, dst, N, T, F, aggs, scalers, args=None):
    """fp64 restatement: [N, T, S*A*F] (differentiable w.r.t. m)."""
    vals, _, d = ref_stats(m, dst, N, args)
    blocks = [vals[a].view(N, T, F) * scale(s, d).view(N, 1, 1) for s in scalers for a in aggs]
    return torch.cat(blocks, -1)


def check_forward(out, m64, dst, N, T, F, aggs, scalers, tol):
    vals, mag, d = ref_stats(m64, dst, N)
    A = len(aggs)
    o = out.double().view(N, T, len(scalers) * A, F)
    for si, s in enumerate(scalers):
        sc = scale(s, d).view(N, 1, 1)
        for ai, a in enumerate(aggs):
            got = o[:, :, si * A + ai] / sc
            ref, bound = vals[a].view(N, T, F), mag[a].view(N, T, F)
            if a == "std":
                err = (got - ref).abs() * (got + ref)
                lim = tol * (bound + ref * ref) + 1e-6 * tol
            else:
                err = (got - ref).abs()
                lim = tol * (bound + ref.abs()) + 1e-30
            bad = ~(err <= lim)
            assert not bad.any(), f"{a} x {s}: {int(bad.sum())} elements, max err {(err - lim).max().item():.3e}"


def messages(dev, dtype, rows, T, F, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    return torch.randn((rows, T, F), generator=g, device=dev).to(dtype)


def run(x, src, dst, N, T, F, aggs, scalers, gather):
    xin = x if T > 1 else x.view(x.size(0), F)
    out = gno_b200.multi_aggregate(xin, dst, N, aggs, scalers, AVG, src=src if gather else None)
    assert out.shape == ((N, T, len(aggs) * len(scalers) * F) if T > 1 else (N, len(aggs) * len(scalers) * F))
    assert out.dtype == x.dtype
    m = (x[src] if gather else x).double().reshape(-1, T * F)
    return out, m


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("F", [1, 3, 8, 33, 64, 100])
@pytest.mark.parametrize("T", [1, 4])
@pytest.mark.parametrize("gather", [False, True], ids=["message", "gather"])
def test_forward_all_aggregators_and_scalers(cuda, dtype, F, T, gather):
    n_src, N, E = 700, 400, 5001
    src, dst = graph(cuda, n_src, N, E, hub_len=1500, seed=F * 10 + T, n_drop=7)
    plan = gno_b200.plan_cache.get(dst, N)
    assert plan.max_len > 4 * plan.chunk_len and plan.n_empty > 40 and plan.n_dropped == 7
    x = messages(cuda, dtype, n_src if gather else E, T, F, seed=F + 100 * T)
    out, m = run(x, src, dst, N, T, F, AGGS, SCALERS, gather)
    check_forward(out, m, dst, N, T, F, AGGS, SCALERS, TOL[dtype])


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("agg", AGGS)
def test_forward_each_aggregator_alone(cuda, dtype, agg):
    N, E, F = 300, 4000, 33
    src, dst = graph(cuda, 500, N, E, hub_len=900, seed=3)
    for gather in (False, True):
        x = messages(cuda, dtype, 500 if gather else E, 1, F, seed=4)
        out, m = run(x, src, dst, N, 1, F, (agg,), ("identity",), gather)
        check_forward(out, m, dst, N, 1, F, (agg,), ("identity",), TOL[dtype])


@pytest.mark.parametrize("scaler", SCALERS)
def test_forward_each_scaler(cuda, scaler):
    N, E, F = 300, 4000, 8
    src, dst = graph(cuda, 500, N, E, hub_len=900, seed=5)
    x = messages(cuda, torch.float32, E, 1, F, seed=6)
    out, m = run(x, src, dst, N, 1, F, ("mean", "std"), (scaler,), False)
    check_forward(out, m, dst, N, 1, F, ("mean", "std"), (scaler,), 1e-5)


def test_duplicates_and_unusual_orders(cuda):
    N, E, F = 250, 3000, 16
    src, dst = graph(cuda, 400, N, E, hub_len=700, seed=7)
    x = messages(cuda, torch.bfloat16, E, 2, F, seed=8)
    aggs = ("std", "max", "sum", "max", "var", "min", "mean", "std")
    scalers = ("linear", "identity", "linear", "attenuation")
    out, m = run(x, src, dst, N, 2, F, aggs, scalers, False)
    check_forward(out, m, dst, N, 2, F, aggs, scalers, 1e-2)
    # each block is the same bits as the block computed alone
    o = out.view(N, 2, len(scalers) * len(aggs), F)
    alone = gno_b200.multi_aggregate(x, dst, N, ("max",), ("linear",), AVG).view(N, 2, 1, F)
    assert torch.equal(o[:, :, 1], alone[:, :, 0]) and torch.equal(o[:, :, 3], alone[:, :, 0])
    assert torch.equal(o[:, :, 2 * 8 + 1], alone[:, :, 0])


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("gather", [False, True], ids=["message", "gather"])
def test_extremes_bit_identical_to_scatter(cuda, dtype, gather):
    """Ties, +-0.0 and NaN: values and winners equal scatter / gather_scatter's with return_arg."""
    n_src, N, E, F = 600, 300, 6000, 24
    src, dst = graph(cuda, n_src, N, E, hub_len=2000, seed=9, n_drop=5)
    g = torch.Generator(device=cuda).manual_seed(10)
    x = torch.randint(-3, 4, (n_src if gather else E, F), generator=g, device=cuda).to(dtype)
    x[torch.rand(x.shape, generator=g, device=cuda) < 0.1] = float("nan")
    x[torch.rand(x.shape, generator=g, device=cuda) < 0.1] = -0.0
    x[torch.rand(x.shape, generator=g, device=cuda) < 0.05] = 0.0
    spec, _ = multiagg._prepare(x, dst, N, ("min", "max"), ("identity",), None, src if gather else None)
    out, state = multiagg._run_forward(x, dst, src if gather else None, N, spec, True)
    for i, red in enumerate(("min", "max")):
        if gather:
            want, arg = gno_b200.gather_scatter(x, src, dst, N, red, return_arg=True)
        else:
            want, arg = gno_b200.scatter(x, dst, 0, None, N, red, return_arg=True)
        got = out[:, i * F:(i + 1) * F]
        assert torch.equal(got.view(torch.int16) if dtype != torch.float32 else got.view(torch.int32),
                           want.view(torch.int16) if dtype != torch.float32 else want.view(torch.int32))
        assert torch.equal(state["amin" if red == "min" else "amax"].long(), arg)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("gather", [False, True], ids=["message", "gather"])
def test_small_integer_sums_are_exact(cuda, dtype, gather):
    n_src, N, E, F = 500, 200, 8000, 40
    src, dst = graph(cuda, n_src, N, E, hub_len=3000, seed=11)
    g = torch.Generator(device=cuda).manual_seed(12)
    x = torch.randint(-4, 5, (n_src if gather else E, F), generator=g, device=cuda).to(dtype)
    out = gno_b200.multi_aggregate(x, dst, N, ("sum",), ("identity",), src=src if gather else None)
    want = torch.zeros((N, F), dtype=torch.float64, device=cuda).index_add_(
        0, dst, (x[src] if gather else x).double())
    # the fp32 sum is exact; 16-bit outputs are that sum rounded once
    assert torch.equal(out, want.to(dtype))


def _grad_check(x, src, dst, N, T, F, aggs, scalers, gather, tol, seed):
    xr = x.detach().clone().requires_grad_(True)
    xin = xr if T > 1 else xr.view(xr.size(0), F)
    out = gno_b200.multi_aggregate(xin, dst, N, aggs, scalers, AVG, src=src if gather else None)
    g = torch.randn(out.shape, generator=torch.Generator(device=x.device).manual_seed(seed),
                    device=x.device).to(x.dtype)
    (gx,) = torch.autograd.grad(out, xr, g)
    msg = (x.detach()[src] if gather else x.detach()).reshape(-1, T * F)
    args = [gno_b200.scatter(msg, dst, 0, None, N, r, return_arg=True)[1] for r in ("min", "max")]
    x64 = x.detach().double().requires_grad_(True)
    m = (x64[src] if gather else x64).reshape(-1, T * F)
    ref = ref_output(m, dst, N, T, F, aggs, scalers, args)
    (gref,) = torch.autograd.grad(ref, x64, g.double().view(ref.shape))
    err = (gx.double() - gref).norm() / gref.norm().clamp(min=1e-30)
    assert err <= tol, f"normwise gradient error {err.item():.3e}"
    return gx


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("F,T", [(1, 1), (8, 4), (33, 1), (64, 1), (100, 4)])
@pytest.mark.parametrize("gather", [False, True], ids=["message", "gather"])
def test_backward_matches_fp64_autograd(cuda, dtype, F, T, gather):
    n_src, N, E = 600, 300, 4001
    src, dst = graph(cuda, n_src, N, E, hub_len=1200, seed=F + T)
    x = messages(cuda, dtype, n_src if gather else E, T, F, seed=13 + F)   # continuous: no ties
    _grad_check(x, src, dst, N, T, F, AGGS, SCALERS, gather, 1e-4 if dtype == torch.float32 else 2e-2, seed=F)


@pytest.mark.parametrize("agg", AGGS)
@pytest.mark.parametrize("scaler", SCALERS)
def test_backward_each_aggregator_and_scaler(cuda, agg, scaler):
    N, E, F = 200, 3000, 12
    src, dst = graph(cuda, 400, N, E, hub_len=800, seed=14, n_drop=9)
    for gather in (False, True):
        x = messages(cuda, torch.float32, 400 if gather else E, 1, F, seed=15)
        gx = _grad_check(x, src, dst, N, 1, F, (agg,), (scaler,), gather, 1e-4, seed=16)
        if not gather:  # dropped edges get no gradient
            dropped = dst >= N
            assert torch.equal(gx[dropped], torch.zeros_like(gx[dropped]))


@pytest.mark.parametrize("gather", [False, True], ids=["message", "gather"])
def test_backward_ties_route_to_the_lowest_edge(cuda, gather):
    n_src, N, E, F = 300, 150, 3000, 10
    src, dst = graph(cuda, n_src, N, E, hub_len=600, seed=17)
    g = torch.Generator(device=cuda).manual_seed(18)
    x = torch.randint(-2, 3, (n_src if gather else E, F), generator=g, device=cuda).float().requires_grad_(True)
    out = gno_b200.multi_aggregate(x, dst, N, ("min", "max"), ("identity",), src=src if gather else None)
    go = torch.randn(out.shape, generator=g, device=cuda)
    (gx,) = torch.autograd.grad(out, x, go)
    want = torch.zeros((E + 1, F), dtype=torch.float64, device=cuda)
    for i, red in enumerate(("min", "max")):
        _, arg = gno_b200.scatter(x.detach()[src] if gather else x.detach(), dst, 0, None, N, red, return_arg=True)
        want.scatter_add_(0, arg, go[:, i * F:(i + 1) * F].double())
    want = want[:E]
    if gather:
        want = torch.zeros((n_src, F), dtype=torch.float64, device=cuda).index_add_(0, src, want)
    assert torch.allclose(gx.double(), want, rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("gather", [False, True], ids=["message", "gather"])
def test_constant_rows_give_zero_std_gradient(cuda, gather):
    """Small-integer constant rows: var is exactly 0 and relu's gradient at 0 is 0."""
    n_src, N, E, F = 300, 120, 2500, 6
    src, dst = graph(cuda, n_src, N, E, hub_len=700, seed=19)
    g = torch.Generator(device=cuda).manual_seed(20)
    row_val = torch.randint(-5, 6, (N + 4, F), generator=g, device=cuda).float()
    if gather:  # every source feeds only rows of one value: make x constant over all nodes
        x = row_val[0].expand(n_src, F).contiguous()
    else:
        x = row_val[dst]
    x.requires_grad_(True)
    out = gno_b200.multi_aggregate(x, dst, N, ("std", "var"), ("identity", "linear"), AVG,
                                   src=src if gather else None)
    assert torch.allclose(out[:, :F], torch.full_like(out[:, :F], math.sqrt(1e-5)), rtol=1e-6, atol=0)
    (gx,) = torch.autograd.grad(out[:, :F].sum() + out[:, 2 * F:3 * F].sum(), x)
    assert torch.equal(gx, torch.zeros_like(gx))


def test_bit_reproducible_over_two_runs(cuda):
    """A size at which every CTA walks several groups of chunks."""
    N, E, F = 100_000, 8_000_000, 64
    g = torch.Generator(device=cuda).manual_seed(21)
    dst = (torch.rand(E, generator=g, device=cuda) ** 2 * N).long()
    x = torch.randn((E, F), generator=g, device=cuda).requires_grad_(True)
    go = torch.randn((N, 3 * 4 * F), generator=g, device=cuda)
    res = []
    for _ in range(2):
        out = gno_b200.multi_aggregate(x, dst, N, ("mean", "min", "max", "std"),
                                       ("identity", "amplification", "attenuation"), AVG)
        (gx,) = torch.autograd.grad(out, x, go)
        res.append((out, gx))
    assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1])


def test_plan_cache_training_step(cuda):
    gno_b200.clear_caches()
    n_src, N, E, F = 2000, 1500, 40_000, 64
    src, dst = graph(cuda, n_src, N, E, hub_len=3000, seed=22)
    x = messages(cuda, torch.float32, n_src, 1, F, seed=23).view(n_src, F).requires_grad_(True)
    misses = []
    for _ in range(3):
        m0 = gno_b200.plan_cache.misses
        out = gno_b200.multi_aggregate(x, dst, N, ("mean", "min", "max", "std"), ("identity", "amplification"),
                                       AVG, src=src)
        torch.autograd.grad(out.sum(), x)
        misses.append(gno_b200.plan_cache.misses - m0)
    assert misses[0] <= 2 and misses[1:] == [0, 0], misses


def test_no_edges_and_no_features(cuda):
    N = 5
    dst = torch.empty(0, dtype=torch.int64, device=cuda)
    x = torch.empty((0, 3), device=cuda, requires_grad=True)
    out = gno_b200.multi_aggregate(x, dst, N, AGGS, ("identity", "linear"), AVG)
    vals = torch.tensor([0, 0, 0, 0, 0, math.sqrt(1e-5)], device=cuda).repeat_interleave(3)
    lin = 1.0 / AVG["lin"]
    assert torch.allclose(out, torch.cat([vals, vals * lin]).expand(N, -1), rtol=1e-6, atol=0)
    (gx,) = torch.autograd.grad(out.sum(), x)
    assert gx.shape == (0, 3)
    xs = torch.randn((4, 3), device=cuda, requires_grad=True)
    out = gno_b200.multi_aggregate(xs, dst, N, src=dst)
    assert out.shape == (N, 12)
    assert torch.equal(torch.autograd.grad(out.sum(), xs)[0], torch.zeros_like(xs))
    idx = torch.tensor([0, 2, 2], device=cuda)
    x0 = torch.empty((3, 0), device=cuda, requires_grad=True)
    out = gno_b200.multi_aggregate(x0, idx, N)
    assert out.shape == (N, 0)
    assert torch.autograd.grad(out.sum(), x0)[0].shape == (3, 0)


def test_errors_on_device(cuda):
    dst = torch.tensor([0, 1, 1], device=cuda)
    with pytest.raises(IndexError):
        gno_b200.multi_aggregate(torch.randn(4, 3, device=cuda), dst, 2, src=torch.tensor([0, 4, 1], device=cuda))
    with pytest.warns(RuntimeWarning):
        gno_b200.multi_aggregate(torch.randn(3, 3, device=cuda), torch.tensor([0, 9, 1], device=cuda), 2)
    out = gno_b200.multi_aggregate(torch.ones(3, 2, device=cuda), dst)   # dim_size = index.max() + 1
    assert out.shape == (2, 8)


def test_full_size_products_bf16_message_form(cuda):
    import os
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench
    n, e, _, _, expo, off = bench.WORKLOADS["products"]
    F = 64
    src, dst = bench.make_graph(n, n, e, expo, off, cuda, 42)
    del src
    g = torch.Generator(device=cuda).manual_seed(24)
    x = torch.randn((e, F), generator=g, device=cuda, dtype=torch.bfloat16)
    out = gno_b200.multi_aggregate(x, dst, n, ("mean", "min", "max", "std"),
                                   ("identity", "amplification", "attenuation"), AVG)
    rows = torch.randperm(n, generator=g, device=cuda)[:4000]
    sel = torch.isin(dst, rows)
    remap = torch.full((n,), -1, dtype=torch.int64, device=cuda)
    remap[rows] = torch.arange(rows.numel(), device=cuda)
    check_forward(out[rows], x[sel].double(), remap[dst[sel]], rows.numel(), 1, F,
                  ("mean", "min", "max", "std"), ("identity", "amplification", "attenuation"), 1e-2)
