"""Graph attention on the fused path (gno_b200.softmax, gno_b200.attention_aggregate) against two
baselines on the same inputs, on the GATv2 shapes of the reference's models:

    (a) today's composition from this package: torch_scatter.composite.scatter_softmax, and H
        per-head weighted segment_reduce calls (forward) / materialised messages + scatter (backward)
    (b) native torch with PyG's formulas: scatter_reduce(amax) / index_select / index_add_

    python profiles/bench_attention.py [--iters 5] [--only products_f32,products_bf16,reddit_bf16]

Every op is timed the way a caller runs it (backward passes through torch.autograd.grad, for the
fused op and for the baselines alike).  One JSON line per measurement.  CUDA events on the current stream, 3 warm-ups, median of `iters`.
Every working set is far larger than the 126 MB L2 (products: 61.9 M edges; reddit: 115 M), so no
flush is needed.  Algorithmic bytes are computed from the shapes (see `bytes_*`); the softmax
counts the logits twice (the statistics pass reads them through perm, the apply pass again in
original order).  Also reports launches per call (gno_launch_count) and the output of the fused
op against baseline (b) at the timed size.

The GATv2 rows (gno_b200.gatv2_logits forward and backward, and a whole layer step: logits, softmax
and aggregate, forward, then torch.autograd.grad w.r.t. x_l, x_r and att) compare against native
torch only: PyG's `(leaky_relu(x_l[src] + x_r[dst]) * att).sum(-1)`.  They also report
torch.cuda.max_memory_allocated over the call.  A native run that does not fit in device memory is
recorded as "oom".
"""
import argparse
import gc
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "gnn-ops-benchmark_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import torch  # noqa: E402

import bench as B  # noqa: E402
import gno_b200  # noqa: E402
from gno_b200 import attention  # noqa: E402
from torch_scatter import composite  # noqa: E402

PEAK, PEAK_SRC = B.peaks()
# Denominator of frac_of_copy_peak: the device-to-device copy bandwidth measured on a B200
# (DESIGN.md §4 "Peak"); bench.peaks() is reported beside it, since it falls back to 6650 GB/s when
# MEASURED_PEAKS.json is absent.
COPY_PEAK = 6450.6
DEV = torch.device("cuda:0")
SHAPES = {"products_f32": ("products", 8, 16, torch.float32),
          "products_bf16": ("products", 8, 16, torch.bfloat16),
          "reddit_bf16": ("reddit", 4, 16, torch.bfloat16)}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as ex:
        q = repr(ex)
    return {"device": torch.cuda.get_device_name(DEV), "nvidia_smi": q}


def timeit(fn, iters):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return statistics.median(ts)


def launches(fn):
    torch.cuda.synchronize()
    n0 = gno_b200.launch_count()
    fn()
    torch.cuda.synchronize()
    return gno_b200.launch_count() - n0


def emit(**kw):
    print(json.dumps(kw), flush=True)


# ---- algorithmic bytes (s = element size) ----
def bytes_softmax_fwd(n, e, H, s):
    # pass 1: perm + erow + logits (via perm); pass 2: index (int64) + logits + y; stats [N, H] (m, d)
    return e * (4 + 4 + H * s) + e * (8 + 2 * H * s) + 2 * n * H * 8


def bytes_softmax_bwd(n, e, H, s):
    return e * (4 + 4 + 2 * H * s) + e * (8 + 3 * H * s) + 2 * n * H * 8


def bytes_aggregate(n_out, e, H, C, s):
    # per edge: gathered row + gather id + edge id + destination + the edge's H weights; per row: output
    return e * (H * C * s + 12 + H * s) + n_out * H * C * s


def bytes_edge_dot(n, e, H, C, s):
    # per edge: gathered x row + ids + dst + H outputs; grad_out rows once per row
    return e * (H * C * s + 12 + H * s) + n * H * C * s


def bytes_gatv2_fwd(n, e, H, C, s):
    # per edge: gathered x_l row + gidx, erow, eid + the edge's H logits; x_r rows once per row
    return e * (H * C * s + 12 + H * s) + n * H * C * s


def bytes_gatv2_bwd(n_src, n_dst, e, H, C, s):
    # two passes (dst plan: grad_x_r and grad_att; src plan: grad_x_l), each per edge: gathered
    # row + ids + the edge's H grad_logits; per row: own row read, gradient row written
    return 2 * e * (H * C * s + 12 + H * s) + 2 * (n_src + n_dst) * H * C * s


# ---- baselines ----
def native_softmax(a, dst, n):
    H = a.size(1)
    m = torch.full((n, H), torch.finfo(a.dtype).min, dtype=a.dtype, device=a.device)
    m = m.scatter_reduce(0, dst.view(-1, 1).expand(-1, H), a.detach(), "amax", include_self=True)
    m = m.masked_fill(m == torch.finfo(a.dtype).min, 0)
    ex = (a - m.index_select(0, dst)).exp()
    s = torch.zeros_like(m).index_add_(0, dst, ex)
    return ex / (s.index_select(0, dst) + 1e-16)


def native_aggregate(x, alpha, src, dst, n):
    return torch.zeros((n,) + tuple(x.shape[1:]), dtype=x.dtype, device=x.device).index_add_(
        0, dst, x.index_select(0, src) * alpha.unsqueeze(-1))


def composed_aggregate_fwd(plan, gidx, x, alpha, n):
    """Today's forward with this package: one weighted segment_reduce per head (strided C-column
    slices), the head's weights reordered by the plan."""
    N, H, C = x.shape
    x2 = x.view(N, H * C)
    out = torch.empty((n, H * C), dtype=x.dtype, device=x.device)
    perm = plan.perm.long()
    for h in range(H):
        w = alpha[:, h].index_select(0, perm)
        gno_b200.segment_reduce(plan, x2[:, h * C:(h + 1) * C], "sum", gidx=gidx, weights=w,
                                out=out[:, h * C:(h + 1) * C])
    return out


def composed_aggregate_diff(x, alpha, src, dst, n):
    """Today's differentiable form: materialised messages, then this package's scatter."""
    msg = x.index_select(0, src) * alpha.unsqueeze(-1)
    return gno_b200.autograd.scatter(msg, dst, 0, n, "sum")


def rel_err(got, want):
    """max |got - want| / max |want| (normwise: gradients cancel to near zero element-wise)"""
    got, want = got.detach().double(), want.detach().double()
    return float((got - want).abs().max() / want.abs().max().clamp(min=1e-30))


def run(key, iters):
    name, H, C, dtype = SHAPES[key]
    n, e = B.WORKLOADS[name][:2]
    ex, off = B.WORKLOADS[name][4:6]
    s = torch.finfo(dtype).bits // 8
    src, dst = B.make_graph(n, n, e, ex, off, DEV, 42)
    g = torch.Generator(device=DEV).manual_seed(7)
    logits = torch.randn((e, H), generator=g, device=DEV).to(dtype)
    x = torch.randn((n, H, C), generator=g, device=DEV).to(dtype)
    gy = torch.randn((e, H), generator=g, device=DEV).to(dtype)
    gout = torch.randn((n, H, C), generator=g, device=DEV).to(dtype)
    base = {"shape": key, "nodes": n, "edges": e, "heads": H, "channels": C, "dtype": str(dtype)[6:],
            "l2": "working set far larger than L2, no flush", "bench_peaks_GBps": PEAK,
            "bench_peaks_source": PEAK_SRC}

    def report(op, ms_fused, abytes, n_launch, baselines, **extra):
        gbs = abytes / (ms_fused * 1e-3) / 1e9
        emit(op=op, ms=round(ms_fused, 4), algorithmic_GB=round(abytes / 1e9, 3), achieved_GBps=round(gbs, 1),
             frac_of_copy_peak=round(gbs / COPY_PEAK, 4), copy_peak_GBps=COPY_PEAK,
             frac_of_bench_peaks=round(gbs / PEAK, 4), launches_per_call=n_launch,
             baseline_ms={k: round(v, 4) for k, v in baselines.items()},
             speedup={k: round(v / ms_fused, 2) for k, v in baselines.items()}, **base, **extra)

    # ---- softmax forward
    plan = gno_b200.plan_cache.get(dst, n)
    y = gno_b200.softmax(logits, dst, num_nodes=n)
    y_nat = native_softmax(logits.float(), dst, n)
    err = rel_err(y, y_nat)
    del y_nat
    ms = timeit(lambda: gno_b200.softmax(logits, dst, num_nodes=n), iters)
    ma = timeit(lambda: composite.scatter_softmax(logits, dst, dim=0, dim_size=n), iters)
    mb = timeit(lambda: native_softmax(logits, dst, n), iters)
    report("softmax forward", ms, bytes_softmax_fwd(n, e, H, s),
           launches(lambda: gno_b200.softmax(logits, dst, num_nodes=n)),
           {"(a) torch_scatter.composite.scatter_softmax": ma, "(b) native torch (PyG formula)": mb},
           logits_counted="twice", normwise_err_vs_native_fp32=err)

    # ---- softmax backward (all three through autograd.grad of their forward)
    la = logits.detach().requires_grad_()
    yf = gno_b200.softmax(la, dst, num_nodes=n)
    ms = timeit(lambda: torch.autograd.grad(yf, la, gy, retain_graph=True), iters)
    nl = launches(lambda: torch.autograd.grad(yf, la, gy, retain_graph=True))
    (g_fused,) = torch.autograd.grad(yf, la, gy, retain_graph=True)
    del yf
    ya = composite.scatter_softmax(la, dst, dim=0, dim_size=n)
    ma = timeit(lambda: torch.autograd.grad(ya, la, gy, retain_graph=True), iters)
    del ya
    yb = native_softmax(la, dst, n)
    mb = timeit(lambda: torch.autograd.grad(yb, la, gy, retain_graph=True), iters)
    (g_nat,) = torch.autograd.grad(native_softmax(la.float(), dst, n), la, gy.float())
    err = rel_err(g_fused, g_nat)
    del yb, g_nat, g_fused
    report("softmax backward", ms, bytes_softmax_bwd(n, e, H, s), nl,
           {"(a) autograd of scatter_softmax": ma, "(b) autograd of native torch": mb},
           logits_counted="y and g twice each", normwise_err_vs_native_fp32=err)

    # ---- aggregate forward
    alpha = y
    gidx = plan.sorted_ids(src)
    out = gno_b200.attention_aggregate(x, alpha, src, dst, n)
    ref = native_aggregate(x.float(), alpha.float(), src, dst, n)
    err = rel_err(out, ref)
    del ref
    ms = timeit(lambda: gno_b200.attention_aggregate(x, alpha, src, dst, n), iters)
    ma = timeit(lambda: composed_aggregate_fwd(plan, gidx, x, alpha, n), iters)
    mb = timeit(lambda: native_aggregate(x, alpha, src, dst, n), iters)
    report("attention_aggregate forward", ms, bytes_aggregate(n, e, H, C, s),
           launches(lambda: gno_b200.attention_aggregate(x, alpha, src, dst, n)),
           {"(a) H weighted segment_reduce calls": ma, "(b) native index_select * alpha + index_add_": mb},
           normwise_err_vs_native_fp32=err)

    # ---- aggregate backward (grad_x + grad_alpha)
    xg, ag = x.detach().requires_grad_(), alpha.detach().requires_grad_()
    of = gno_b200.attention_aggregate(xg, ag, src, dst, n)
    ms = timeit(lambda: torch.autograd.grad(of, (xg, ag), gout, retain_graph=True), iters)
    nl = launches(lambda: torch.autograd.grad(of, (xg, ag), gout, retain_graph=True))
    oa = composed_aggregate_diff(xg, ag, src, dst, n)
    ma = timeit(lambda: torch.autograd.grad(oa, (xg, ag), gout, retain_graph=True), iters)
    del oa
    ob = native_aggregate(xg, ag, src, dst, n)
    mb = timeit(lambda: torch.autograd.grad(ob, (xg, ag), gout, retain_graph=True), iters)
    del ob
    got = torch.autograd.grad(of, (xg, ag), gout)
    xf, af = x.float().requires_grad_(), alpha.float().requires_grad_()
    want = torch.autograd.grad(native_aggregate(xf, af, src, dst, n), (xf, af), gout.float())
    errs = {"grad_x": rel_err(got[0], want[0]), "grad_alpha": rel_err(got[1], want[1])}
    del got, want, xf, af
    report("attention_aggregate backward (grad_x + grad_alpha)", ms,
           bytes_aggregate(n, e, H, C, s) + bytes_edge_dot(n, e, H, C, s), nl,
           {"(a) autograd of materialised messages + scatter": ma, "(b) autograd of native torch": mb},
           normwise_err_vs_native_fp32=errs)
    del of

    # H = 1 against the existing weighted segment_reduce on the same graph (same work).  "repeated
    # alpha": the same alpha tensor every call (its sorted copy is memoised); "fresh alpha": the
    # sorted copy is rebuilt every call, as in training where each step brings a new alpha.
    x1 = x[:, :1].contiguous()
    a1 = alpha[:, :1].contiguous()
    w1 = a1[:, 0].index_select(0, plan.perm.long())
    m1 = timeit(lambda: gno_b200.attention_aggregate(x1, a1, src, dst, n), iters)

    def fresh():
        attention._sorted_alpha.clear()
        return gno_b200.attention_aggregate(x1, a1, src, dst, n)
    mf = timeit(fresh, iters)
    mw = timeit(lambda: gno_b200.segment_reduce(plan, x1.view(n, C), "sum", gidx=gidx, weights=w1), iters)
    perm = plan.perm.long()
    mp = timeit(lambda: gno_b200.segment_reduce(plan, x1.view(n, C), "sum", gidx=gidx,
                                                weights=a1[:, 0].index_select(0, perm)), iters)
    same = torch.equal(gno_b200.attention_aggregate(x1, a1, src, dst, n).view(n, C),
                       gno_b200.segment_reduce(plan, x1.view(n, C), "sum", gidx=gidx, weights=w1))
    emit(op="attention_aggregate H=1 vs weighted segment_reduce", ms=round(m1, 4),
         segment_reduce_weighted_ms=round(mw, 4), ratio=round(m1 / mw, 3),
         fresh_alpha_ms=round(mf, 4), permute_plus_segment_reduce_ms=round(mp, 4),
         ratio_fresh_vs_permute_plus_segment_reduce=round(mf / mp, 3),
         bit_identical=same, **base)
    del x1, a1, w1

    # ---- one full attention step: softmax -> aggregate -> backward of both
    def fused_step():
        lg, xs = logits.detach().requires_grad_(), x.detach().requires_grad_()
        o = gno_b200.attention_aggregate(xs, gno_b200.softmax(lg, dst, num_nodes=n), src, dst, n)
        return (o,) + torch.autograd.grad(o, (lg, xs), gout)

    def composed_step():
        lg, xs = logits.detach().requires_grad_(), x.detach().requires_grad_()
        o = composed_aggregate_diff(xs, composite.scatter_softmax(lg, dst, dim=0, dim_size=n), src, dst, n)
        torch.autograd.grad(o, (lg, xs), gout)

    def native_step(dt=dtype):
        lg, xs = logits.detach().to(dt).requires_grad_(), x.detach().to(dt).requires_grad_()
        o = native_aggregate(xs, native_softmax(lg, dst, n), src, dst, n)
        return (o,) + torch.autograd.grad(o, (lg, xs), gout.to(dt))

    ms = timeit(fused_step, iters)
    nl = launches(fused_step)
    ma = timeit(composed_step, iters)
    mb = timeit(native_step, iters)
    total = (bytes_softmax_fwd(n, e, H, s) + bytes_softmax_bwd(n, e, H, s) + 2 * bytes_aggregate(n, e, H, C, s)
             + bytes_edge_dot(n, e, H, C, s))
    got, want = fused_step(), native_step(torch.float32)
    errs = {k: rel_err(a, b) for k, a, b in zip(("out", "grad_logits", "grad_x"), got, want)}
    del got, want
    report("full attention step (softmax + aggregate, forward + backward)", ms, total, nl,
           {"(a) composed": ma, "(b) native torch": mb}, normwise_err_vs_native_fp32=errs)


def native_logits(x_l, x_r, att, src, dst):
    return (torch.nn.functional.leaky_relu(x_l[src] + x_r[dst], 0.2) * att).sum(-1)


def peak_gb(fn):
    """(torch.cuda.max_memory_allocated over one call, memory allocated before it), in GB."""
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    return round(torch.cuda.max_memory_allocated() / 1e9, 3), round(before / 1e9, 3)


def native_or_oom(fn, *args):
    """fn(*args), or "oom" when it does not fit in device memory."""
    try:
        return fn(*args)
    except torch.cuda.OutOfMemoryError:
        pass
    gc.collect()  # outside the handler: the traceback's frames no longer hold the partial results
    torch.cuda.empty_cache()
    return "oom"


def run_gatv2(key, iters):
    name, H, C, dtype = SHAPES[key]
    n, e = B.WORKLOADS[name][:2]
    ex, off = B.WORKLOADS[name][4:6]
    s = torch.finfo(dtype).bits // 8
    src, dst = B.make_graph(n, n, e, ex, off, DEV, 42)
    g = torch.Generator(device=DEV).manual_seed(11)
    x_l = torch.randn((n, H, C), generator=g, device=DEV).to(dtype)
    x_r = torch.randn((n, H, C), generator=g, device=DEV).to(dtype)
    att = torch.randn((H, C), generator=g, device=DEV).to(dtype)
    gl = torch.randn((e, H), generator=g, device=DEV).to(dtype)
    gout = torch.randn((n, H, C), generator=g, device=DEV).to(dtype)
    base = {"shape": key, "nodes": n, "edges": e, "heads": H, "channels": C, "dtype": str(dtype)[6:],
            "l2": "working set far larger than L2, no flush"}

    def report(op, ms, abytes, n_launch, native_ms, peak, native_peak, err):
        gbs = abytes / (ms * 1e-3) / 1e9
        emit(op=op, ms=round(ms, 4), algorithmic_GB=round(abytes / 1e9, 3), achieved_GBps=round(gbs, 1),
             frac_of_copy_peak=round(gbs / COPY_PEAK, 4), copy_peak_GBps=COPY_PEAK, launches_per_call=n_launch,
             native_ms=native_ms if native_ms == "oom" else round(native_ms, 4),
             speedup_vs_native=None if native_ms == "oom" else round(native_ms / ms, 2),
             max_memory_allocated_GB=peak[0], allocated_before_GB=peak[1],
             native_max_memory_allocated_GB=native_peak if native_peak == "oom" else native_peak[0],
             normwise_err_vs_native=err, **base)

    def native_err(got, names, want_fn):
        """Normwise error of `got` against native torch in fp32, or in the shape's dtype when the
        fp32 run does not fit in device memory."""
        for dt in dict.fromkeys((torch.float32, dtype)):
            want = native_or_oom(want_fn, dt)
            if want != "oom":
                return {"vs": f"native {str(dt)[6:]}", **{k: rel_err(a, b) for k, a, b in zip(names, got, want)}}
        return "native oom"

    # ---- logits forward
    fused_fwd = lambda: gno_b200.gatv2_logits(x_l, x_r, att, src, dst)  # noqa: E731
    nat_fwd = lambda: native_logits(x_l, x_r, att, src, dst)  # noqa: E731
    got = fused_fwd()
    err = native_err((got,), ("logits",),
                     lambda dt: (native_logits(x_l.to(dt), x_r.to(dt), att.to(dt), src, dst),))
    del got
    ms = timeit(fused_fwd, iters)
    peak = peak_gb(fused_fwd)
    nl = launches(fused_fwd)
    mb = native_or_oom(timeit, nat_fwd, iters)
    pb = native_or_oom(peak_gb, nat_fwd)
    report("gatv2_logits forward", ms, bytes_gatv2_fwd(n, e, H, C, s), nl, mb, peak, pb, err)

    # ---- logits backward (grad of x_l, x_r and att through autograd.grad)
    xs = [t.detach().requires_grad_() for t in (x_l, x_r, att)]
    lf = gno_b200.gatv2_logits(*xs, src, dst)
    bwd = lambda: torch.autograd.grad(lf, xs, gl, retain_graph=True)  # noqa: E731
    got = bwd()
    err = native_err(got, ("grad_x_l", "grad_x_r", "grad_att"), lambda dt: torch.autograd.grad(
        native_logits(*[t.to(dt) for t in xs], src, dst), xs, gl.to(dt)))
    del got
    ms = timeit(bwd, iters)
    peak = peak_gb(bwd)
    nl = launches(bwd)
    del lf

    def native_bwd_time():
        lb = native_logits(*xs, src, dst)
        nb = lambda: torch.autograd.grad(lb, xs, gl, retain_graph=True)  # noqa: E731
        return timeit(nb, iters), peak_gb(nb)
    r = native_or_oom(native_bwd_time)
    mb, pb = ("oom", "oom") if r == "oom" else r
    report("gatv2_logits backward (grad x_l, x_r, att)", ms, bytes_gatv2_bwd(n, n, e, H, C, s), nl, mb, peak, pb,
           err)

    # ---- a GATv2 layer step: logits -> softmax -> aggregate, forward + backward w.r.t. x_l, x_r, att
    def fused_layer():
        ts = [t.detach().requires_grad_() for t in (x_l, x_r, att)]
        lg = gno_b200.gatv2_logits(*ts, src, dst)
        o = gno_b200.attention_aggregate(ts[0], gno_b200.softmax(lg, dst, num_nodes=n), src, dst, n)
        return (o,) + torch.autograd.grad(o, ts, gout)

    def native_layer(dt=dtype):
        ts = [t.detach().to(dt).requires_grad_() for t in (x_l, x_r, att)]
        lg = native_logits(*ts, src, dst)
        o = native_aggregate(ts[0], native_softmax(lg, dst, n), src, dst, n)
        return (o,) + torch.autograd.grad(o, ts, gout.to(dt))

    got = fused_layer()
    err = native_err(got, ("out", "grad_x_l", "grad_x_r", "grad_att"), native_layer)
    del got
    ms = timeit(fused_layer, iters)
    peak = peak_gb(fused_layer)
    nl = launches(fused_layer)
    mb = native_or_oom(timeit, native_layer, iters)
    pb = native_or_oom(peak_gb, native_layer)
    total = (bytes_gatv2_fwd(n, e, H, C, s) + bytes_gatv2_bwd(n, n, e, H, C, s) + bytes_softmax_fwd(n, e, H, s)
             + bytes_softmax_bwd(n, e, H, s) + 2 * bytes_aggregate(n, e, H, C, s) + bytes_edge_dot(n, e, H, C, s))
    report("GATv2 layer step (logits + softmax + aggregate, forward + backward)", ms, total, nl, mb, peak, pb, err)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default=",".join(SHAPES))
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--ops", default="attention,gatv2", help="attention (softmax, aggregate), gatv2 (logits, layer)")
    args = ap.parse_args()
    emit(op="card", **card())
    runners = {"attention": run, "gatv2": run_gatv2}
    for k in args.only.split(","):
        for op in args.ops.split(","):
            gno_b200.clear_caches()
            gc.collect()
            torch.cuda.empty_cache()
            try:
                runners[op](k, args.iters)
            except Exception as ex:  # keep going: partial tables are still useful
                print(json.dumps({"shape": k, "ops": op, "error": repr(ex)[:500]}), flush=True)
