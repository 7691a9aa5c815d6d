"""Several aggregators in one pass (gno_b200.multi_aggregate, PNAConv.aggregate) against two
baselines on the same inputs, with the PNA set (aggregators mean, min, max, std; scalers identity,
amplification, attenuation):

    (a) today's composition on this package's torch_scatter shim with PNAConv's formulas: one
        scatter per statistic, std from scatter_mean of inputs * inputs, the degree from a
        scatter_add of ones, the scaler copies as node-level products
    (b) native torch: index_add / scatter_reduce(amin, amax) / bincount with the same formulas

and a sum-only segment_reduce over the same messages on the same plan (the bandwidth yardstick).

    python profiles/bench_multiagg.py [--iters 5] [--only products_msg_f32,...] [--out FILE]

Forward and backward (torch.autograd.grad w.r.t. the inputs, graph kept from one forward) are timed
with CUDA events on the current stream, 3 warm-ups, median of `iters`.  The products-shaped and
Reddit-shaped working sets are far larger than the 126 MB L2; the small shape (64 FakeDataset-sized
graphs) fits in L2 and is an overhead and launch measurement.  Algorithmic bytes come from the
shapes (`bytes_*`).  Each row also reports gno_b200 launches per call, the CUDA kernels per call
(torch.profiler), the peak of torch.cuda.max_memory_allocated over one call above what was
allocated before it, and the normwise error against an fp64 restatement on 4000 sampled
destination rows.  One JSON line per measurement.
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
import torch_scatter  # noqa: E402

COPY_PEAK = 6450.6  # GB/s, device-to-device copy measured on a B200 (DESIGN.md §4 "Peak")
DEV = torch.device("cuda:0")
AGGS = ("mean", "min", "max", "std")
SCALERS = ("identity", "amplification", "attenuation")
# name: (graph, form, F, dtype)
SHAPES = {"products_msg_f32": ("products", "message", 64, torch.float32),
          "products_msg_bf16": ("products", "message", 64, torch.bfloat16),
          "products_gather_f32": ("products", "gather", 100, torch.float32),
          "reddit_gather_bf16": ("reddit", "gather", 128, torch.bfloat16),
          "fake64_msg_f32": ("fake64", "message", 64, torch.float32)}


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


def counts(fn):
    """(gno_b200 launches, CUDA kernels, peak bytes above the allocation before the call) of one call."""
    torch.cuda.synchronize()
    n0 = gno_b200.launch_count()
    fn()
    torch.cuda.synchronize()
    gno = gno_b200.launch_count() - n0
    try:
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        kernels = sum(1 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                      and not e.name.startswith(("Memcpy", "Memset")))
    except Exception as ex:  # the profiler is a report, not a requirement
        kernels = repr(ex)[:80]
    gc.collect()
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated(DEV)
    torch.cuda.reset_peak_memory_stats(DEV)
    fn()
    torch.cuda.synchronize()
    return gno, kernels, torch.cuda.max_memory_allocated(DEV) - base


def emit(**kw):
    print(json.dumps(kw), flush=True)
    if ARGS.out:
        with open(ARGS.out, "a") as f:
            f.write(json.dumps(kw) + "\n")


# ---- algorithmic bytes (s = element size, W = feature columns, K = S*A output blocks) ----
def bytes_fwd(n, e, W, K, s):
    # per edge: message row + gather id + destination (+ edge id for the winners); per row: K blocks
    return e * (W * s + 12) + n * K * W * s


def bytes_yardstick(n, e, W, s):
    return e * (W * s + 8) + n * W * s


def bytes_bwd(form, n, n_src, e, W, K, s):
    state = n * W * 16  # mean, var (fp32), argmin, argmax (int32)
    if form == "message":
        # per edge: message row in, gradient row out, ids; per row: K gradient blocks, state
        return e * (2 * W * s + 12) + n * K * W * s + state
    # coefficients: K gradient blocks + state in, [P | Q], c_min, c_max out; transposed pass: per
    # edge a [P | Q] row and ids; per source: x in, gradient out; winner routing: c, winner, row id
    return (n * K * W * s + state + n * 4 * W * 4 + e * (2 * W * 4 + 8) + n_src * (W * s + 2 * W * 4 + W * s)
            + 2 * n * W * (4 + 8 + 4))


# ---- baselines ----
def pna_scale(out, deg, avg):
    d = deg.clamp(min=1).to(out.dtype).view(-1, 1)
    amp = torch.log(d + 1) / avg["log"]
    return torch.cat([out, out * amp, out * (1.0 / amp)], -1)


def composed(m, index, n, avg):
    """PNAConv.aggregate / degree scalers on the torch_scatter shim (PyG's formulas)."""
    outs = [torch_scatter.scatter(m, index, 0, None, n, reduce="mean"),
            torch_scatter.scatter(m, index, 0, None, n, reduce="min"),
            torch_scatter.scatter(m, index, 0, None, n, reduce="max")]
    mean = torch_scatter.scatter(m, index, 0, None, n, reduce="mean")
    mean_sq = torch_scatter.scatter(m * m, index, 0, None, n, reduce="mean")
    outs.append(torch.sqrt(torch.relu(mean_sq - mean * mean) + 1e-5))
    deg = torch_scatter.scatter(torch.ones_like(index), index, 0, None, n, reduce="sum")
    return pna_scale(torch.cat(outs, -1), deg, avg)


def native(m, index, n, avg):
    W = m.size(1)
    deg = torch.bincount(index, minlength=n)
    d = deg.clamp(min=1).to(m.dtype).view(-1, 1)
    z = torch.zeros((n, W), dtype=m.dtype, device=m.device)
    idx = index.view(-1, 1).expand_as(m)
    mean = z.index_add(0, index, m) / d
    mn = z.scatter_reduce(0, idx, m, "amin", include_self=False)
    mx = z.scatter_reduce(0, idx, m, "amax", include_self=False)
    var = z.index_add(0, index, m * m) / d - mean * mean
    out = torch.cat([mean, mn, mx, torch.sqrt(torch.relu(var) + 1e-5)], -1)
    return pna_scale(out, deg, avg)


def reference(m64, index, n, rows, avg):
    """fp64 restatement on the destination rows `rows` only: [len(rows), 12 W]."""
    remap = torch.full((n,), -1, dtype=torch.int64, device=index.device)
    remap[rows] = torch.arange(rows.numel(), device=index.device)
    r = remap[index]
    sel = r >= 0
    out = native(m64(sel), r[sel], rows.numel(), avg)
    return out


def make(name):
    graph, form, F, dtype = SHAPES[name]
    g = torch.Generator(device=DEV).manual_seed(42)
    if graph == "fake64":
        n_per, n_graphs, deg = 1000, 64, 10
        e_per = n_per * deg
        base = torch.arange(n_graphs, device=DEV).repeat_interleave(e_per) * n_per
        src = base + torch.randint(0, n_per, (n_graphs * e_per,), generator=g, device=DEV)
        dst = base + torch.randint(0, n_per, (n_graphs * e_per,), generator=g, device=DEV)
        n = n_per * n_graphs
    else:
        n, e, _, _, expo, off = B.WORKLOADS[graph]
        src, dst = B.make_graph(n, n, e, expo, off, DEV, 42)
    rows = src.numel() if form == "message" else n
    x = torch.randn((rows, F), generator=g, device=DEV, dtype=torch.float32).to(dtype)
    deg = torch.bincount(dst, minlength=n).double()
    avg = {"lin": float(deg.mean()), "log": float(torch.log(deg + 1).mean())}
    return form, n, src, dst, x, avg


def shape_rows(name, iters, info):
    form, n, src, dst, x, avg = make(name)
    E, W, s = dst.numel(), x.size(1), x.element_size()
    K = len(AGGS) * len(SCALERS)
    n_src = x.size(0)
    gs = src if form == "gather" else None
    msg = (lambda t: t.index_select(0, src)) if form == "gather" else (lambda t: t)
    g = torch.Generator(device=DEV).manual_seed(7)
    rows = torch.randperm(n, generator=g, device=DEV)[:4000]
    ref = reference(lambda sel: msg(x)[sel].double() if form == "message" else x.double()[src[sel]], dst, n, rows,
                    avg)
    base = dict(shape=name, form=form, nodes=n, edges=E, features=W, dtype=str(x.dtype).replace("torch.", ""),
                aggregators=AGGS, scalers=SCALERS, **info)
    go = torch.randn((n, K * W), generator=g, device=DEV, dtype=torch.float32).to(x.dtype)

    def err(out):
        o = out[rows].double()
        return float((o - ref).norm() / ref.norm())

    impls = {
        "fused": lambda t: gno_b200.multi_aggregate(t, dst, n, AGGS, SCALERS, avg, src=gs),
        "composed": lambda t: composed(msg(t), dst, n, avg),
        "native": lambda t: native(msg(t), dst, n, avg),
    }
    fb = bytes_fwd(n, E, W, K, s)
    bb = bytes_bwd(form, n, n_src, E, W, K, s)
    for impl, f in impls.items():
        try:
            xr = x.detach().requires_grad_(True)
            with torch.no_grad():
                e_out = err(f(x))
            t_f = timeit(lambda: f(x), iters)
            gno_f, k_f, mem_f = counts(lambda: f(x))
            emit(**base, impl=impl, direction="forward", ms=t_f, alg_bytes=fb,
                 frac_of_copy_peak=fb / (t_f * 1e-3) / (COPY_PEAK * 1e9), gno_launches=gno_f, cuda_kernels=k_f,
                 peak_mem_bytes=mem_f, normwise_err_fp64=e_out)
            out = f(xr)
            bwd = lambda: torch.autograd.grad(out, xr, go, retain_graph=True)  # noqa: E731
            t_b = timeit(bwd, iters)
            gno_b, k_b, mem_b = counts(bwd)
            emit(**base, impl=impl, direction="backward", ms=t_b, alg_bytes=bb,
                 frac_of_copy_peak=bb / (t_b * 1e-3) / (COPY_PEAK * 1e9), gno_launches=gno_b, cuda_kernels=k_b,
                 peak_mem_bytes=mem_b)
            del out, xr, bwd
        except torch.OutOfMemoryError:
            emit(**base, impl=impl, direction="forward+backward", ms="oom")
        gc.collect()
        torch.cuda.empty_cache()
    # bandwidth yardstick: sum-only segment reduce over the same messages on the same plan
    plan = gno_b200.plan_cache.get(dst, n)
    gidx = plan.perm if form == "message" else plan.sorted_ids(src)
    y = lambda: gno_b200.segment_reduce(plan, x, "sum", gidx=gidx)  # noqa: E731
    t_y = timeit(y, iters)
    gno_y, k_y, mem_y = counts(y)
    yb = bytes_yardstick(n, E, W, s)
    emit(**base, impl="segment_reduce_sum", direction="forward", ms=t_y, alg_bytes=yb,
         frac_of_copy_peak=yb / (t_y * 1e-3) / (COPY_PEAK * 1e9), gno_launches=gno_y, cuda_kernels=k_y,
         peak_mem_bytes=mem_y)


def main():
    global ARGS
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--only", default=",".join(SHAPES))
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    ARGS = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_multiagg.py needs a CUDA device")
    info = card()
    for name in ARGS.only.split(","):
        shape_rows(name, ARGS.iters, info)
        gno_b200.clear_caches()
        gc.collect()
        torch.cuda.empty_cache()


ARGS = None
if __name__ == "__main__":
    main()
