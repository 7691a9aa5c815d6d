"""bench.py — headline benchmark of the aggregation path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload rmat26] [--dump-outputs DIR]

Default workload = BASELINE.json configs[4], the configuration the metric's "at 1/2/4/8 B200"
is quoted on: dst-partitioned gather->scatter_add on a synthetic R-MAT scale-26 graph
(67,108,864 nodes, 1,073,741,824 edges, F=128 bf16), STRONG scaling: the graph is fixed; at N>1
every rank owns an edge-balanced destination range and the feature rows i with i % N == rank;
the one exchange step delivers exactly the source rows each rank's edges read (stored straight
into the peers' buffers over NVLink by the owners' gather kernel, pipelined over destination
sub-ranges so it overlaps the reduction); outputs stay partitioned.  It fits one GPU, so N=1 runs
the same graph.  A step = one pass of the hot path over the whole graph.

`value` = aggregated edges/s with plan and features resident in HBM; `e2e` = the same through
the host-buffer API (pinned host x and int64 edge_index -> device, plan build, aggregation,
result -> host); `roofline` = algorithmic bytes of the local segment-reduce launch / its
CUDA-event time against MEASURED_PEAKS.json; `parity` = this run's output checked against an
fp64 index_add_ of the same inputs on every rank; `per_config` (N=1) = kernel fractions of the
other BASELINE.json configs (C1, products, Reddit-shaped fp32/bf16, C4) from the same run.
`--workload products` keeps round 1's configs[1] bench (weak scaling at N>1).
One JSON line on stdout (rank 0).  `--dump-outputs DIR` also writes the output of the last timed
step (a fixed, seeded sample of its rows) as .npy files; nothing else is written.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "gnn-ops-benchmark_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOADS = {
    # name: (nodes, edges, features, dtype, zipf exponent, zipf offset)
    "products": (2_449_029, 61_859_140, 100, torch.float32, 0.75, 100.0),
    "c1": (100_000, 1_000_000, 64, torch.float32, 0.0, 1.0),
    "reddit": (232_965, 114_615_892, 602, torch.float32, 0.8, 300.0),
    "reddit_bf16": (232_965, 114_615_892, 602, torch.bfloat16, 0.8, 300.0),
}
RMAT_ABC = (0.57, 0.19, 0.19)  # a, b, c (d = 0.05)
RMAT_F = 128
TOL = {torch.float32: 1e-5, torch.bfloat16: 1e-2, torch.float16: 1e-2}


def is_rmat(name):
    return name.startswith("rmat")


def workload_shape(name):
    """(nodes, edges, features, dtype) of a workload."""
    if is_rmat(name):
        scale = int(name[4:])
        return 1 << scale, 1 << (scale + 4), RMAT_F, torch.bfloat16
    n, e, F, dtype, _, _ = WORKLOADS[name]
    return n, e, F, dtype


def dtype_name(dtype):
    return {torch.float32: "f32", torch.bfloat16: "bf16", torch.float16: "f16"}[dtype]


def config_of(name):
    """The workload description: IDENTICAL in the repo arm and the reference arm (the driver
    compares the two `config` objects).  Everything implementation-specific goes to `detail`."""
    n, e, F, dtype = workload_shape(name)
    if is_rmat(name):
        graph = ("R-MAT a,b,c,d=.57,.19,.19,.05, edge factor 16, seed 42 (src = column id, dst = row id), "
                 "unsorted int64 COO")
        scaling = "strong: the graph is fixed, destination rows are partitioned over the GPUs"
    else:
        graph = "power-law in-degrees (shifted Zipf over a random node permutation), uniform sources, seed 42"
        scaling = "weak: one graph of this size per GPU"
    return {"workload": name, "op": "fused index_select -> scatter_add (sum)", "nodes": n, "edges": e,
            "features": F, "feature_dtype": dtype_name(dtype), "graph": graph, "scaling_rule": scaling,
            "l2": "inputs far larger than the 126 MB L2; no flush needed",
            "tolerance": "|err| <= tol * sum|terms| per output element, tol 1e-5 fp32 / 1e-2 bf16 "
                         "(the error norm of a cancelling sum; DESIGN.md section 2)"}


def metric_of(name):
    if is_rmat(name):
        return "aggregation edges/s (dst-partitioned gather->scatter_add, RMAT graph)"
    return "aggregation edges/s (fused index_select->scatter_add, %s-shaped graph)" % name


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# --------------------------------------------------------------------------- graphs --
def make_graph(n_dst, n_src, n_edges, exponent, offset, device, seed):
    """Synthetic power-law graph: destination in-degrees follow a shifted Zipf law
    (weights (i+offset)^-exponent over a random node permutation), sources uniform."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    if exponent > 0:
        w = (torch.arange(n_dst, device=device, dtype=torch.float64) + offset) ** (-exponent)
        cdf = torch.cumsum(w, 0)
        cdf = (cdf / cdf[-1]).to(torch.float32)
        u = torch.rand(n_edges, device=device, generator=g)
        rank = torch.searchsorted(cdf, u).clamp_(max=n_dst - 1)
        relabel = torch.randperm(n_dst, device=device, generator=g)
        dst = relabel[rank]
        del w, cdf, u, rank, relabel
    else:
        dst = torch.randint(0, n_dst, (n_edges,), device=device, generator=g)
    src = torch.randint(0, n_src, (n_edges,), device=device, generator=g)
    return src, dst


def rmat_edges(scale, n_edges, device, seed, row_prefix=()):
    """R-MAT edge list: one quadrant choice per bit level.  Returns (src = column ids,
    dst = row ids), int64, identical on every rank for one seed.

    row_prefix fixes the top row bits: the result is then an exact sample of the sub-graph whose
    destination ids start with that prefix (the column bit of a fixed level is drawn from its
    conditional distribution), with dst returned relative to the slice."""
    a, b, c = RMAT_ABC
    d = 1.0 - a - b - c
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    rows = torch.zeros(n_edges, dtype=torch.int64, device=device)
    cols = torch.zeros(n_edges, dtype=torch.int64, device=device)
    for level in range(scale):
        u = torch.rand(n_edges, device=device, generator=g)
        if level < len(row_prefix):
            p1 = d / (c + d) if row_prefix[level] else b / (a + b)
            cols.mul_(2).add_((u < p1).to(torch.int64))
        else:
            rows.mul_(2).add_((u >= a + b).to(torch.int64))                           # quadrants c, d
            cols.mul_(2).add_((((u >= a) & (u < a + b)) | (u >= a + b + c)).to(torch.int64))  # b, d
        del u
    return cols, rows


def feature_block(owner, world, n_nodes, F, dtype, device):
    """Feature rows owned by `owner` under cyclic ownership (global row i = owner + world * j):
    every rank can regenerate any block, which is what the in-line parity check does."""
    rows = (n_nodes - owner + world - 1) // world
    g = torch.Generator(device=device)
    g.manual_seed(1000 + owner)
    out = torch.empty(rows, F, dtype=dtype, device=device)
    step = 1 << 22
    for r0 in range(0, rows, step):
        r1 = min(rows, r0 + step)
        out[r0:r1] = torch.randn(r1 - r0, F, device=device, generator=g, dtype=torch.float32).to(dtype)
    return out


# --------------------------------------------------------------------------- clocks --
class ClockSampler:
    """SM clock / throttle reasons sampled in a thread (NVML, 20 ms period; nvidia-smi -lms as the
    fallback) from start() to stop(); mark() brackets the exactly-timed region."""
    REASONS = (("hw_slowdown", "nvmlClocksEventReasonHwSlowdown"),
               ("hw_thermal_slowdown", "nvmlClocksEventReasonHwThermalSlowdown"),
               ("sw_thermal_slowdown", "nvmlClocksEventReasonSwThermalSlowdown"),
               ("sw_power_cap", "nvmlClocksEventReasonSwPowerCap"))

    def __init__(self, index):
        self.index, self.rows, self.marks = index, [], []
        self._stop = threading.Event()
        self.thread, self.proc, self.how = None, None, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            uuid = str(torch.cuda.get_device_properties(self.index).uuid)
            try:
                h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
            except Exception:
                h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            mx = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            masks = [(n, getattr(pynvml, attr)) for n, attr in self.REASONS]

            def loop():
                while not self._stop.is_set():
                    try:
                        sm = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                        bits = int(pynvml.nvmlDeviceGetCurrentClocksEventReasons(h))
                        pw = pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0
                        self.rows.append((time.perf_counter(), sm, mx, pw, [n for n, m in masks if bits & m]))
                    except Exception:
                        pass
                    self._stop.wait(0.02)
            self.thread = threading.Thread(target=loop, daemon=True)
            self.thread.start()
            self.how = "nvml, 20 ms period"
            return
        except Exception:
            pass
        try:
            q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                 "clocks_event_reasons.sw_power_cap")
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)

            def read():
                names = [n for n, _ in self.REASONS]
                for line in self.proc.stdout:
                    c = [v.strip() for v in line.split(",")]
                    try:
                        self.rows.append((time.perf_counter(), float(c[0]), float(c[1]), float(c[2]),
                                          [n for n, v in zip(names, c[3:7]) if v.lower().startswith("active")]))
                    except (ValueError, IndexError):
                        continue
            self.thread = threading.Thread(target=read, daemon=True)
            self.thread.start()
            self.how = "nvidia-smi -lms 50"
        except OSError:
            self.proc = None

    def mark(self):
        self.marks.append(time.perf_counter())

    def stop(self):
        self._stop.set()
        if self.proc is not None:
            time.sleep(0.1)
            self.proc.terminate()
        if self.thread is not None:
            self.thread.join(timeout=2)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no clock samples"], "samples": 0}
        t0 = self.marks[0] if self.marks else self.rows[0][0]
        t1 = self.marks[1] if len(self.marks) > 1 else self.rows[-1][0]
        t2 = self.marks[2] if len(self.marks) > 2 else t1
        timed = [r for r in self.rows if t0 <= r[0] <= t1]
        load = [r for r in self.rows if t0 <= r[0] <= t2]   # timed region + the kernel-only loop after it
        use = timed if len(timed) >= 3 else load
        reasons = sorted({n for r in use for n in r[4]})
        return {"sm_mhz": statistics.median(r[1] for r in use) if use else None,
                "sm_max_mhz": max(r[2] for r in self.rows), "reasons": reasons,
                "samples": len(use), "samples_in_timed_region": len(timed),
                "window": "timed region" if use is timed else "timed region + kernel-only loop (both under load)",
                "power_w_max": max(r[3] for r in use) if use else None, "how": self.how}


def algorithmic_bytes(n_rows, n_edges, F, es):
    """SURVEY.md §8(d): E*(F*s + 4) + N*(F*s_out + 4)."""
    return n_edges * (F * es + 4) + n_rows * (F * es + 4)


# ------------------------------------------------------------------- CPU reference --
def host_threads():
    """torchrun exports OMP_NUM_THREADS=1; the CPU arm uses every core this process may run on."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    torch.set_num_threads(max(1, n))
    return torch.get_num_threads()


def cpu_reference_step(x, src, dst, n_rows):
    """What the reference executes on CPU for this op: messages = x.index_select(0, src)
    (benchmark_fused_index_select_reduce.py:12-15 / PyG propagate), then
    torch_scatter.scatter_add == zeros.scatter_add_(0, expanded index, messages)
    (torch-scatter 2.0.9 scatter_sum; call site benchmark_scatter_add.py:18)."""
    msgs = x.index_select(0, src)
    out = torch.zeros(n_rows, x.size(1), dtype=x.dtype)
    out.scatter_add_(0, dst.view(-1, 1).expand(-1, x.size(1)), msgs)
    return out


# destination-id prefixes whose slices have about the graph's own density (edges per row):
# P(prefix) = .76^zeros * .24^ones ~ 2^-len.  (prefix, share of all edges)
RMAT_SLICES = [((0, 0, 1, 0, 0, 1, 0, 1, 0, 0, 1), 0.76 ** 7 * 0.24 ** 4),
               ((0, 0, 1, 0, 0, 1, 0, 1), 0.76 ** 5 * 0.24 ** 3),
               ((0, 0, 1, 0, 0, 1), 0.76 ** 4 * 0.24 ** 2),
               ((0, 0, 1), 0.76 ** 2 * 0.24)]


def time_cpu_rmat(name, budget_s, steps, warmup):
    """Reference CPU path on a bounded, exact sample of the R-MAT workload: ONE destination-row
    slice (all edges whose destination id starts with a bit prefix, sources over all nodes,
    output rows of the slice only), so edges, output rows and their zero-fill scale together.
    Returns (edges/s, description, cores, ms/step)."""
    cores = host_threads()
    n, e, F, dtype = workload_shape(name)
    scale = n.bit_length() - 1
    torch.manual_seed(42)
    # features: one random 2^20-row block tiled over all nodes (values do not change CPU time;
    # drawing 8.6e9 normals on the host would take minutes)
    blk = min(n, 1 << 20)
    x = torch.randn(blk, F, dtype=torch.float32).to(dtype).repeat(n // blk, 1)
    chosen = None
    per_edge = None
    for prefix, share in RMAT_SLICES:
        if len(prefix) >= scale:
            continue
        n_e = max(1, int(e * share))
        if per_edge is not None and per_edge * n_e * (steps + warmup) > budget_s:
            break
        src, dst = rmat_edges(scale, n_e, "cpu", 42, row_prefix=prefix)
        rows = n >> len(prefix)
        cpu_reference_step(x, src, dst, rows)
        t0 = time.perf_counter()
        cpu_reference_step(x, src, dst, rows)
        per_edge = (time.perf_counter() - t0) / n_e
        chosen = (prefix, src, dst, rows, n_e)
    prefix, src, dst, rows, n_e = chosen
    for _ in range(warmup):
        cpu_reference_step(x, src, dst, rows)
    t0 = time.perf_counter()
    for _ in range(steps):
        cpu_reference_step(x, src, dst, rows)
    dt = (time.perf_counter() - t0) / steps
    desc = (f"destination-row slice with id prefix {''.join(map(str, prefix))}: {n_e} of {e} edges into "
            f"{rows} of {n} rows, sources over all {n} nodes ({dtype_name(dtype)} features, a 2^20-row random "
            f"block tiled); torch CPU index_select + zeros + scatter_add_ (the calls torch_scatter 2.0.9 "
            f"scatter_sum makes), {steps} steps")
    return n_e / dt, desc, cores, dt * 1e3


def time_cpu_prefix(name, budget_s, steps, warmup):
    """Reference CPU path on a bounded sample of a power-law workload (same node set, first
    `sample` edges), all host threads. Returns (edges/s, description, cores, ms/step)."""
    cores = host_threads()
    n_nodes, n_edges, F, dtype, exponent, offset = WORKLOADS[name]
    torch.manual_seed(42)
    probe = min(n_edges, 1_000_000)
    src, dst = make_graph(n_nodes, n_nodes, probe, exponent, offset, "cpu", 42)
    x = torch.randn(n_nodes, F, dtype=torch.float32).to(dtype)
    cpu_reference_step(x, src, dst, n_nodes)
    t0 = time.perf_counter()
    cpu_reference_step(x, src, dst, n_nodes)
    per_edge = (time.perf_counter() - t0) / probe
    sample = int(min(n_edges, max(probe, budget_s / max(steps + warmup, 1) / per_edge)))
    if sample != probe:
        src, dst = make_graph(n_nodes, n_nodes, sample, exponent, offset, "cpu", 42)
    for _ in range(warmup):
        cpu_reference_step(x, src, dst, n_nodes)
    t0 = time.perf_counter()
    for _ in range(steps):
        cpu_reference_step(x, src, dst, n_nodes)
    dt = (time.perf_counter() - t0) / steps
    desc = (f"first {sample} of {n_edges} edges, same {n_nodes}-node feature matrix; torch CPU index_select + "
            f"zeros + scatter_add_ (the calls torch_scatter 2.0.9 scatter_sum makes), {steps} steps")
    return sample / dt, desc, cores, dt * 1e3


def time_cpu_baseline(name, budget_s, steps, warmup):
    return (time_cpu_rmat if is_rmat(name) else time_cpu_prefix)(name, budget_s, steps, warmup)


def run_reference(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    _, _, _, dtype = workload_shape(args.workload)
    v, desc, cores, ms = time_cpu_baseline(args.workload, 150.0, args.steps, args.warmup)
    emit_json({
        "impl": "reference", "metric": metric_of(args.workload), "value": v, "unit": "edges/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "strong" if is_rmat(args.workload) else "weak",
        "vs_baseline": None, "dtype": dtype_name(dtype), "data": "synthetic",
        "config": config_of(args.workload),
        "cpu_baseline": {"value": v, "unit": "edges/s", "cores": cores, "kind": "port", "sample": desc},
        "e2e": {"value": v, "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})


# ---------------------------------------------------------------------------- parity --
def parity_check(out, x_of, src, dst, row0, n_rows, tol, block_rows=1 << 21, edge_step=1 << 22):
    """max over the rank's output elements of |out - ref| / (tol * sum|terms|), ref = fp64
    index_add_ of the same inputs (native torch, original unsorted edge list — nothing of the
    plan is reused).  x_of(ids) returns the feature rows of global source ids."""
    dev = out.device
    worst = torch.zeros((), dtype=torch.float64, device=dev)
    F = out.size(1)
    for r0 in range(0, n_rows, block_rows):
        r1 = min(n_rows, r0 + block_rows)
        sel = torch.nonzero((dst >= row0 + r0) & (dst < row0 + r1)).flatten()
        ref = torch.zeros(r1 - r0, F, dtype=torch.float64, device=dev)
        mag = torch.zeros(r1 - r0, F, dtype=torch.float64, device=dev)
        for k0 in range(0, sel.numel(), edge_step):
            s = sel[k0:k0 + edge_step]
            v = x_of(src[s]).double()
            d = dst[s] - (row0 + r0)
            ref.index_add_(0, d, v)
            mag.index_add_(0, d, v.abs_())
            del v, d, s
        err = (out[r0:r1].double() - ref).abs_()
        worst = torch.maximum(worst, (err / (tol * mag + 1e-30)).max()) if err.numel() else worst
        del ref, mag, err, sel
    return worst


# ---------------------------------------------------------------------- --dump-outputs --
DUMP_BYTES = 32 << 20   # all ranks together; well under 64 MB with the row ids and .npy headers


def dump_outputs(dirname, out, row0, rank, world):
    """Writes this rank's output rows of the last timed step as float32 to DIR/out.npy, with
    their global row ids as float64 to DIR/out_rows.npy (suffix _rank<r> at N > 1).  Outputs
    larger than the budget are represented by a fixed, seeded sample of rows, so two builds run
    with the same arguments can be compared output for output."""
    n_rows, F = out.shape
    k = min(n_rows, DUMP_BYTES // world // (F * 4 + 8))
    if k == n_rows:
        rows = torch.arange(n_rows)
    else:
        rows = torch.randperm(n_rows, generator=torch.Generator().manual_seed(20240601))[:k].sort().values
    vals = out.index_select(0, rows.to(out.device)).float().cpu().numpy()
    suffix = "" if world == 1 else f"_rank{rank}"
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, f"out{suffix}.npy"), vals)
    np.save(os.path.join(dirname, f"out_rows{suffix}.npy"), (rows + row0).double().numpy())


# ------------------------------------------------------------------------ per_config --
def per_config(iters):
    """Kernel times / roofline fractions of the other BASELINE.json configs (profiles/bench_ops.py
    measures them; this just runs it in-process and keeps the numbers)."""
    sys.path.insert(0, os.path.join(ROOT, "profiles"))
    import bench_ops
    import gno_b200
    res = {}
    for key in ("c1", "c2", "c3", "c4"):
        gno_b200.clear_caches()
        torch.cuda.empty_cache()
        bench_ops.RESULTS.clear()
        try:
            bench_ops.RUNS[key](iters)
        except Exception as ex:
            res[key + " error"] = repr(ex)[:300]
        for line in bench_ops.RESULTS:
            res[line["op"]] = {"ms": line["ms"], "algorithmic_GB": line["algorithmic_GB"],
                               "frac_of_peak": line["frac_of_peak"]}
            if "frac_dram" in line:   # real DRAM traffic (ncu capture of the same launch) over the time measured here
                res[line["op"]]["frac_dram"] = line["frac_dram"]
    gno_b200.clear_caches()
    torch.cuda.empty_cache()
    return res


# ------------------------------------------------------------------------ RMAT bench --
def run_rmat(args):
    """BASELINE.json configs[4] (see the module docstring)."""
    import gno_b200
    from gno_b200 import plan as planmod
    from gno_b200.dist import DistAggregator, edge_balanced_ranges

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    N, E, F, dtype = workload_shape(args.workload)
    scale = N.bit_length() - 1
    es = 2
    sampler = ClockSampler(local_rank)
    sampler.start()

    src, dst = rmat_edges(scale, E, dev, 42)
    counts = torch.bincount(dst, minlength=N)
    # balance kernel time, not just edges: a row costs its output write plus a row switch in the
    # kernel; measured on 4 B200s a weight of 4 edges per row gives the shortest step
    bounds = edge_balanced_ranges(counts + args.row_weight, world).cpu()
    del counts
    lo, hi = int(bounds[rank]), int(bounds[rank + 1])
    if world > 1:
        m = (dst >= lo) & (dst < hi)
        src, dst = src[m], dst[m] - lo
        del m
    torch.cuda.empty_cache()
    e_local, n_out = src.numel(), hi - lo
    x_local = feature_block(rank, world, N, F, dtype, dev)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    agg = None
    stages = 1
    if world > 1:
        # Stage structure of the overlapped exchange, measured on 2 / 4 / 8 B200s
        # (profiles/scaling/r2h_*, r3d_* ... r3m_*; per-rank timelines in the same files).  Every N
        # splits by SOURCE and writes every output row at most TWICE: a 16-bit sum is rounded once
        # per stage that touches the row, and the stated tolerance (1e-2 of sum|terms|) holds two
        # bf16 roundings (2 * 2^-8), not three — three accumulating stages measured 1.06 of the bound.
        #   N=2: own-source edges, then the remote ones; the own half hides the whole exchange.
        #   N>=4: the own-source edges and the edges of the most-referenced remote rows in ONE
        #   two-buffer launch (merge_own: gathers from x_local and from the receive buffer) after a
        #   small first push, then the rest.  The first group is sized so that the merged launch ends
        #   when the exchange does: reduction work done beside the push is slow, work left for the
        #   last stage waits for the exchange.  N=4: the top 0.8 % of the remote rows (they carry 44 %
        #   of the remote edges), 8 KB push ring: 12.75 ms (0.4 / 1.5 / 3 / 6 / 10 %: 13.0 / 13.0 /
        #   13.3 / 14.2 / 15.0; three accumulating stages 12.7 but 3 roundings; unstaged 16.3).
        #   N=8: 10 %, 16 KB ring (the exchange is the critical path there; more bytes in flight under
        #   HBM contention): 7.44-7.68 ms (three stages 7.61; 8 KB ring 8.3; unstaged 10.1).
        # Also measured and not used: hybrid / destination splits, per-rank mixed structures (one
        # global barrier per stage makes every rank wait for the largest request list), larger push
        # grids (296 CTAs slow the reduction more than they speed the exchange), L2 evict-first
        # hints on the pushed rows (no effect).
        fracs = [float(v) for v in args.stage_fracs.split(",")] if args.stage_fracs else None
        if args.split == "auto":
            args.split = "source"
        if args.push_chunk < 0:
            args.push_chunk = 16384 if world >= 8 else 8192
        if args.merge_own < 0:
            args.merge_own = 1 if (world > 2 and args.split == "source") else 0
        if args.stages > 0:
            stages = args.stages
        elif args.split == "source":
            stages = 2 if world <= 2 else 3
            if fracs is None and stages == 3:
                if args.merge_own:
                    fracs = [0.1, 0.9] if world >= 8 else [0.008, 0.992]
                else:
                    fracs = [0.15, 0.85] if world >= 8 else [0.25, 0.75]
        elif args.split == "hybrid":
            stages = 2 if world <= 2 else 3
        else:
            stages = 4
        n_fr = stages - 1 if args.split in ("source", "hybrid") else stages
        if fracs is not None and len(fracs) != n_fr:
            raise SystemExit(f"--stage-fracs needs {n_fr} shares for {stages} {args.split} stages")
        own = args.ownership if args.ownership != "auto" else ("xorfold" if world & (world - 1) == 0 else "cyclic")
        kw = dict(rank=rank, world=world, cyclic_rows=N, stages=stages, stage_fracs=fracs,
                  row_weight=args.row_weight, split=args.split, ownership=own, push_blocks=args.push_blocks,
                  push_chunk=args.push_chunk, merge_own=bool(args.merge_own))
        try:
            agg = DistAggregator(bounds, src, dst, exchange=args.exchange, **kw)
            if args.exchange == "push":
                agg._push_buffer(F, dtype, dev)  # symmetric-memory rendezvous happens here
        except Exception as ex:  # no peer mapping on this box: same exchange through NCCL all-to-all
            if args.exchange != "push":
                raise
            print(f"push exchange unavailable ({ex!r}); using the NCCL needed-rows all-to-all", file=sys.stderr)
            args.exchange = "needed"
            agg = DistAggregator(bounds, src, dst, exchange="needed", **kw)
        plans = agg.xstage_plans()
        recv = torch.empty(agg.n_needed, F, device=dev, dtype=dtype) if args.exchange == "needed" else None
        n_needed, n_own = agg.n_needed, agg.recv_splits[rank]
    else:
        plan = planmod.build_plan(dst, n_out)
        gidx = plan.sorted_ids(src)
        plans = [(plan, gidx, plan.perm, 0, n_out, False)]
        n_needed = n_own = 0
    torch.cuda.synchronize()
    plan_ms = (time.perf_counter() - t0) * 1e3
    out = torch.empty(n_out, F, device=dev, dtype=dtype)

    def step():
        if world > 1:
            agg.aggregate(x_local, "sum", x_full=recv, out=out)
        else:
            gno_b200.segment_reduce(plan, x_local, "sum", gidx=gidx, out=out)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    warm = max(args.warmup, 3)
    for _ in range(warm):
        step()
    barrier()
    launches0 = gno_b200.launch_count()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.mark()
    a.record()
    for _ in range(args.steps):
        step()
    b.record()
    barrier()
    sampler.mark()
    launches = gno_b200.launch_count() - launches0
    total_ms = a.elapsed_time(b)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out, lo, rank, world)

    # ---- kernel-only: this rank's segment-reduce launches, no exchange (the roofline kernel) ----
    x_gather = x_local if world == 1 else (recv if recv is not None else agg._push_buffer(F, dtype, dev)[0][:n_needed])
    ka, kb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ka.record()
    for _ in range(args.steps):
        if world > 1:
            agg.reduce_stages(x_gather, "sum", out, x_local=x_local)
        else:
            gno_b200.segment_reduce(plan, x_gather, "sum", gidx=gidx, out=out)
    kb.record()
    torch.cuda.synchronize()
    sampler.mark()
    k_ms = ka.elapsed_time(kb) / args.steps
    # ---- exchange-only (N > 1): all stages back to back, nothing overlapped ----
    x_ms = 0.0
    if world > 1:
        barrier()
        xa, xb_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        xa.record()
        for _ in range(args.steps):
            if args.exchange == "push":
                agg.exchange_push(x_local)
            else:
                agg.exchange_needed(x_local, recv)
        xb_.record()
        barrier()
        x_ms = xa.elapsed_time(xb_) / args.steps
    clocks = sampler.stop()

    # ---- parity of the timed path's output, on every rank ----
    step()
    torch.cuda.synchronize()
    if world > 1:
        from gno_b200.dist import xorfold_global_ids
        x_glob = torch.empty(N, F, dtype=dtype, device=dev)
        for q in range(world):
            blk = x_local if q == rank else feature_block(q, world, N, F, dtype, dev)
            if own == "xorfold":
                x_glob[xorfold_global_ids(q, world, blk.size(0), dev)] = blk
            else:
                x_glob[q::world] = blk
            del blk
    else:
        x_glob = x_local
    t0 = time.perf_counter()
    worst = parity_check(out, lambda ids: x_glob[ids], src, dst, 0, n_out, TOL[dtype])
    nonzero_rows = (out != 0).any(1).sum().to(torch.float64)
    stats = torch.stack([torch.tensor(total_ms, dtype=torch.float64, device=dev),
                         torch.tensor(k_ms, dtype=torch.float64, device=dev),
                         torch.tensor(x_ms, dtype=torch.float64, device=dev), worst])
    sums = torch.stack([nonzero_rows, torch.tensor(float(e_local), dtype=torch.float64, device=dev)])
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
        dist.all_reduce(sums, op=dist.ReduceOp.SUM)
    total_ms, k_ms_max, x_ms_max, worst = (float(v) for v in stats.tolist())
    parity_s = time.perf_counter() - t0
    parity = {"checked": True, "max_err_over_bound": worst, "ok": bool(worst <= 1.0), "tol": TOL[dtype],
              "bound": "tol * sum|terms| per output element", "reference": "fp64 index_add_ over the original "
              "unsorted edge list (torch), all output rows of every rank", "ranks": world,
              "edges_checked": int(sums[1]), "nonzero_output_rows": int(sums[0]), "seconds": round(parity_s, 2)}
    del x_glob
    ms_per_step = total_ms / args.steps
    peak, peak_src = peaks()
    abytes = algorithmic_bytes(n_out, e_local, F, es)
    achieved = abytes / (k_ms * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath) and world == 1:
        with open(tpath) as f:
            traffic = json.load(f).get(args.workload)
    detail = {"edges_rank0": e_local, "rows_rank0": n_out, "plan_build_ms": plan_ms,
              "max_row_len": max(p.max_len for p, *_ in plans),
              "empty_rows_rank0": plans[0][0].n_empty if len(plans) == 1 else None,
              "chunk_len": plans[0][0].chunk_len,
              "exchange": args.exchange if world > 1 else None, "stages": stages if world > 1 else None,
              "stage_fracs": fracs if world > 1 else None,
              "split": args.split if world > 1 else None,
              "merge_own": bool(args.merge_own) if world > 1 else None,
              "push_chunk": args.push_chunk if world > 1 else None, "push_blocks": args.push_blocks if world > 1 else None,
              "stage_edges_rank0": [p.E for p, *_ in plans] if world > 1 else None,
              "stage_recv_rows_rank0": ([agg.stage_row0[s + 1] - agg.stage_row0[s] for s in range(stages)]
                                        if world > 1 else None),
              "exchange_bytes_in_rank0": (n_needed - n_own) * F * es,
              "local_reduce_ms_max_over_ranks": k_ms_max, "exchange_only_ms_max_over_ranks": x_ms_max,
              "parallelism": (f"edge-balanced dst ranges x{world} (row weight {args.row_weight}), {own} feature "
                              f"ownership, needed-rows {args.exchange} exchange in {stages} {args.split} stages "
                              "overlapped with the reduction") if world > 1 else "single GPU"}

    # ---- e2e: host buffers through the public API, every step ----
    del agg, plans, x_gather
    if world == 1:
        del plan, gidx
    try:
        need = x_local.numel() * es + src.numel() * 16 + out.numel() * es
        import psutil
        avail = psutil.virtual_memory().available
        if avail < 2 * need * max(1, world if world > 1 else 1) + (64 << 30):
            raise MemoryError(f"host has {avail >> 30} GiB available; pinning {need >> 30} GiB per rank "
                              "for the e2e leg was skipped")
        x_host = torch.empty(x_local.shape, dtype=dtype, pin_memory=True)
        x_host.copy_(x_local)
        ei_host = torch.empty((2, src.numel()), dtype=torch.int64, pin_memory=True)
        ei_host[0].copy_(src)
        ei_host[1].copy_(dst)
        out_host = torch.empty(out.shape, dtype=dtype, pin_memory=True)
        torch.cuda.synchronize()
        del src, dst, x_local, out
        gno_b200.clear_caches()
        torch.cuda.empty_cache()
        e2e = run_e2e_rmat(world, rank, dev, dist, bounds, x_host, ei_host, out_host, N, E,
                           own if world > 1 else "cyclic")
        del x_host, ei_host, out_host
    except Exception as ex:  # e.g. the box cannot pin 3 x 17 GB: keep the device-resident numbers
        e2e = {"value": None, "unit": "edges/s", "error": repr(ex)[:300]}
    torch.cuda.empty_cache()
    cpu = None
    pc = None
    if world == 1:
        v, desc, cores, _ = time_cpu_baseline(args.workload, 20.0, 3, 1)
        cpu = {"value": v, "unit": "edges/s", "cores": cores, "kind": "port", "sample": desc}
        if args.per_config:
            try:
                pc = per_config(5)
            except Exception as ex:
                pc = {"error": repr(ex)[:300]}
    if rank == 0:
        line = {"metric": metric_of(args.workload), "value": E / (ms_per_step * 1e-3), "unit": "edges/s",
                "n_gpus": world, "steps": args.steps, "warmup": warm, "ms_per_step": ms_per_step,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16",
                "data": "synthetic", "config": config_of(args.workload), "detail": detail, "clocks": clocks,
                "e2e": e2e, "gpu_launches": launches, "parity": parity,
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                             "frac": achieved / peak, "traffic": traffic,
                             "dram_frac": (traffic / (k_ms * 1e-3) / 1e9 / peak) if traffic else None,
                             "peak_source": peak_src,
                             "kernel": "segreduce_staged_kernel + segfinish_kernel (rank 0's shard)",
                             "kernel_ms": k_ms, "algorithmic_bytes": abytes}}
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if pc is not None:
            line["per_config"] = pc
        emit_json(line)
    if world > 1:
        dist.destroy_process_group()


def run_e2e_rmat(world, rank, dev, dist, bounds, x_host, ei_host, out_host, N, E, own):
    """Host-buffer path: every step copies that step's inputs (x shard and the int64 edge shard)
    from pinned host memory, builds the plan (N>1: the whole partitioned aggregator — request
    lists, NCCL needed-rows exchange), aggregates, and copies the result to pinned host memory."""
    import gno_b200
    es = x_host.element_size()
    n_out = out_host.size(0)
    steps = 3
    if world == 1:
        from gno_b200.host import gather_scatter_host

        def e2e_step():
            gno_b200.clear_caches()
            gather_scatter_host(x_host, ei_host, n_out, "sum", out_host)
        includes = ("H2D x + int64 edge_index (pinned), plan build (dst radix sort, overlapped with the x "
                    "copy), aggregation, D2H out; one call at a time, wall clock")
    else:
        from gno_b200.dist import DistAggregator

        def e2e_step():
            gno_b200.clear_caches()
            xd = x_host.to(dev, non_blocking=True)
            eid = ei_host.to(dev, non_blocking=True)
            a2 = DistAggregator(bounds, eid[0], eid[1], rank=rank, world=world, cyclic_rows=N,
                                exchange="needed", ownership=own)
            o = a2.aggregate(xd, "sum")
            out_host.copy_(o, non_blocking=True)
            torch.cuda.synchronize()
        includes = ("per rank: H2D x shard + int64 edge shard (pinned), partitioned-aggregator build (request "
                    "lists, dst radix sort), NCCL needed-rows all-to-all, aggregation, D2H out; wall clock, max over ranks")
    e2e_step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        e2e_step()
    torch.cuda.synchronize()
    e_ms = (time.perf_counter() - t0) * 1e3 / steps
    h2d = x_host.numel() * es + ei_host.numel() * 8
    d2h = out_host.numel() * es
    if world > 1:
        t = torch.tensor([e_ms, float(h2d), float(d2h)], device=dev, dtype=torch.float64)
        mx = t.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        e_ms, h2d, d2h = float(mx[0]), int(t[1]), int(t[2])
    return {"value": E / (e_ms * 1e-3), "unit": "edges/s", "h2d_bytes_per_step": h2d,
            "d2h_bytes_per_step": d2h, "ms_per_step": e_ms, "steps": steps, "includes": includes}


# ------------------------------------------------- power-law workloads (configs[1..3]) --
def run_weak(args):
    """Round 1's bench: products-shaped (or c1 / reddit) graph per GPU, all-gather of x at N>1."""
    import gno_b200
    from gno_b200 import plan as planmod

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        # High-priority NCCL stream: the chunk all-gathers of the staged exchange then get SMs as
        # aggregation CTAs retire instead of queueing behind the whole kernel (without it the
        # stages serialise: 10.0 -> 10.3 ms at N=4; with it 8.6 ms — profiles/scaling/stage_sweep_*).
        opts = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank), pg_options=opts)
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if args.stages <= 0:
        # measured (profiles/scaling/stage_sweep_{4,8}gpu_hipri.jsonl): 4 stages 8.63 vs 10.00 ms at
        # N=4, 13.30 vs 15.52 ms at N=8; at N=2 the peer-store all-gather (one stage) is used
        args.stages = 4 if world >= 4 else 1
    n_local, e_local, F, dtype, exponent, offset = WORKLOADS[args.workload]
    es = torch.empty((), dtype=dtype).element_size()
    n_global = n_local * world

    src, dst = make_graph(n_local, n_global, e_local, exponent, offset, dev, 42 + rank)
    gx = torch.Generator(device=dev)
    gx.manual_seed(1000 + rank)
    x_local = torch.randn(n_local, F, device=dev, generator=gx, dtype=torch.float32).to(dtype)
    x_full = torch.empty(n_global, F, device=dev, dtype=dtype) if world > 1 else x_local
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    agg = None
    xmode = None
    if world > 1:
        from gno_b200.dist import DistAggregator
        bounds = torch.arange(world + 1, dtype=torch.int64) * n_local
        # measured (profiles/scaling): the peer-store all-gather beats NCCL at N=2 (6.64 vs 7.18 ms),
        # ties at N=4 (10.16 vs 10.04) and loses at N=8 (17.4 vs 15.6)
        xmode = args.exchange if args.exchange in ("allgather", "allgather_push") else \
            ("allgather_push" if world <= 2 else "allgather")
        try:
            agg = DistAggregator(bounds, src, dst, rank=rank, world=world, stages=args.stages, exchange=xmode)
            if xmode == "allgather_push":
                x_full = agg.exchange_allgather_push(x_local)  # symmetric-memory rendezvous happens here
        except Exception as ex:  # no peer mapping on this box: NCCL all-gather
            if xmode != "allgather_push":
                raise
            print(f"allgather_push unavailable ({ex!r}); using the NCCL all-gather", file=sys.stderr)
            xmode = "allgather"
            agg = DistAggregator(bounds, src, dst, rank=rank, world=world, stages=args.stages)
        plan, gidx = agg.plan()
        if args.stages > 1:
            agg.stage_plans()
            stage_bufs = [torch.empty(world * r, F, device=dev, dtype=dtype) for r in agg.stage_rows]
    else:
        plan = planmod.build_plan(dst, n_local)
        gidx = plan.sorted_ids(src)
    torch.cuda.synchronize()
    plan_ms = (time.perf_counter() - t0) * 1e3
    out = torch.empty(n_local, F, device=dev, dtype=dtype)

    def step():
        if world > 1:  # all-gather of the feature shards, then the local gather-reduce
            agg.aggregate(x_local, "sum", x_full=x_full, out=out,
                          stage_bufs=stage_bufs if args.stages > 1 else None)
        else:
            gno_b200.segment_reduce(plan, x_full, "sum", gidx=gidx, out=out)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    sampler.start()
    warm = max(args.warmup, 3)
    for _ in range(warm):
        step()
    barrier()
    launches0 = gno_b200.launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    sampler.mark()
    ev[0].record()
    for i in range(args.steps):
        step()
    ev[1].record()
    barrier()
    sampler.mark()
    launches = gno_b200.launch_count() - launches0
    total_ms = ev[0].elapsed_time(ev[1])
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out, rank * n_local, rank, world)
    if world > 1:
        t = torch.tensor([total_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    value = e_local * world / (ms_per_step * 1e-3)

    # ---- kernel-only duration for the roofline (aggregation kernel alone, this rank) -------
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
           for _ in range(args.steps)]
    for a, b in kev:
        a.record()
        gno_b200.segment_reduce(plan, x_full, "sum", gidx=gidx, out=out)
        b.record()
    torch.cuda.synchronize()
    sampler.mark()
    clocks = sampler.stop()
    k_ms = statistics.mean(a.elapsed_time(b) for a, b in kev)
    peak, peak_src = peaks()
    abytes = algorithmic_bytes(n_local, e_local, F, es)
    achieved = abytes / (k_ms * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            traffic = json.load(f).get(args.workload)

    # ---- parity (the gather buffer of the last step still holds every rank's features) ----
    step()
    torch.cuda.synchronize()
    if world > 1:
        xg = agg.exchange(x_local)  # plain NCCL all-gather into the padded buffer, for the check only
        worst = parity_check(out, lambda ids: xg[ids], agg.src_padded, dst, 0, n_local, TOL[dtype])
        dist.all_reduce(worst, op=dist.ReduceOp.MAX)
        del xg
    else:
        worst = parity_check(out, lambda ids: x_full[ids], src, dst, 0, n_local, TOL[dtype])
    worst = float(worst)
    parity = {"checked": True, "max_err_over_bound": worst, "ok": bool(worst <= 1.0), "tol": TOL[dtype],
              "bound": "tol * sum|terms| per output element",
              "reference": "fp64 index_add_ over the original unsorted edge list (torch), all rows, every rank",
              "ranks": world}

    # ---- e2e: host buffers through the public API ------------------------------------------
    # Every step copies that step's inputs (x and the int64 edge_index) from pinned host memory,
    # builds the plan, aggregates and copies the result back to pinned host memory.  N=1 uses
    # gno_b200.host.HostPipeline (two steps in flight: the D2H of step i overlaps the H2D of
    # step i+1); N>1 runs the steps back to back through DistAggregator.
    cpu = None
    x_host = x_local.cpu().pin_memory()
    ei_host = torch.stack([src, dst]).cpu().pin_memory()
    out_hosts = [torch.empty(n_local, F, dtype=dtype).pin_memory() for _ in range(2)]
    e2e_steps = max(4, min(args.steps, 10))
    del src, dst
    torch.cuda.empty_cache()
    if world == 1:
        from gno_b200.host import HostPipeline, gather_scatter_host
        gno_b200.clear_caches()
        gather_scatter_host(x_host, ei_host, n_local, "sum", out_hosts[0])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        gather_scatter_host(x_host, ei_host, n_local, "sum", out_hosts[0])
        single_ms = (time.perf_counter() - t0) * 1e3
        pipe = HostPipeline(n_local, "sum")
        for i in range(2):  # warm-up
            pipe.submit(x_host, ei_host, out_hosts[i % 2])
            pipe.result()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        pipe.submit(x_host, ei_host, out_hosts[0])
        for i in range(1, e2e_steps):
            pipe.submit(x_host, ei_host, out_hosts[i % 2])
            pipe.result()
        pipe.result()
        torch.cuda.synchronize()
        e_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
        includes = ("H2D x + int64 edge_index (pinned), plan build (dst radix sort), aggregation, D2H out; "
                    "2 steps in flight (HostPipeline), wall clock over %d steps" % e2e_steps)
    else:
        from gno_b200.dist import DistAggregator
        single_ms = None

        def e2e_step():
            gno_b200.clear_caches()
            xd = x_host.to(dev, non_blocking=True)
            eid = ei_host.to(dev, non_blocking=True)
            a2 = DistAggregator(bounds, eid[0], eid[1], rank=rank, world=world)
            o = a2.aggregate(xd, "sum", x_full=x_full)
            out_hosts[0].copy_(o, non_blocking=True)

        e2e_step()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(e2e_steps):
            e2e_step()
        b.record()
        barrier()
        e_ms = a.elapsed_time(b) / e2e_steps
        t = torch.tensor([e_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e_ms = float(t.item())
        includes = "H2D x + int64 edge_index (pinned), plan build, NCCL all-gather, aggregation, D2H out"
    e2e = {"value": e_local * world / (e_ms * 1e-3), "unit": "edges/s",
           "h2d_bytes_per_step": (x_host.numel() * es + ei_host.numel() * 8) * world,
           "d2h_bytes_per_step": out_hosts[0].numel() * es * world,
           "ms_per_step": e_ms, "single_call_ms": single_ms, "includes": includes}
    del x_host, ei_host
    if rank == 0 and world == 1:
        v, desc, cores, _ = time_cpu_baseline(args.workload, 20.0, 3, 1)
        cpu = {"value": v, "unit": "edges/s", "cores": cores, "kind": "port", "sample": desc}

    if rank == 0:
        line = {
            "metric": metric_of(args.workload), "value": value, "unit": "edges/s", "n_gpus": world,
            "steps": args.steps, "warmup": warm, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": dtype_name(dtype), "data": "synthetic", "config": config_of(args.workload),
            "detail": {"nodes_per_gpu": n_local, "edges_per_gpu": e_local,
                       "index": "int64 edge_index -> cached dst-sorted CSR plan (int32)",
                       "plan_build_ms": plan_ms, "max_row_len": plan.max_len,
                       "chunk_len": plan.chunk_len, "rows_cut_by_chunks": plan.n_span,
                       "empty_rows": plan.n_empty,
                       "parallelism": (f"dst-partitioned x{world}, all-gather of x by "
                                       + ("peer-store kernel over NVLink (gno_push_rows)" if xmode == "allgather_push"
                                          else f"NCCL, {args.stages}-stage exchange")) if world > 1 else "single GPU"},
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "parity": parity,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic,
                         "dram_frac": (traffic / (k_ms * 1e-3) / 1e9 / peak) if traffic else None,
                         "peak_source": peak_src,
                         "kernel": "segreduce_staged_kernel (+ segfinish_kernel)", "kernel_ms": k_ms,
                         "algorithmic_bytes": abytes},
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
        emit_json(line)
    if world > 1:
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit_json(line):
    """The one JSON line goes to the real stdout; everything else (NCCL banners, warnings
    from libraries that print to fd 1) was redirected to stderr in main()."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, data)
    else:
        sys.stdout.write(data.decode())
        sys.stdout.flush()


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="rmat26",
                    choices=sorted(WORKLOADS) + ["rmat26", "rmat24", "rmat22", "rmat20", "rmat16"])
    ap.add_argument("--exchange", default="push", choices=["allgather", "allgather_push", "needed", "push"],
                    help="rmat workloads at N>1: the rows each rank's edges read, stored directly into the "
                         "peers' buffers by the owners' gather kernel over NVLink (push), or the same rows "
                         "through NCCL all-to-alls (needed); products workload: allgather | allgather_push")
    ap.add_argument("--row-weight", type=int, default=4,
                    help="rmat workloads: cost of one destination row in edge units when balancing ranges")
    ap.add_argument("--stages", type=int, default=0,
                    help="exchange pipeline depth at N>1 (rmat: destination sub-ranges, default 4; products: "
                         "row chunks of the all-gather, default 4 at N>=4)")
    ap.add_argument("--stage-fracs", default="",
                    help="rmat workloads: comma-separated shares of the stages (dest split: cost share of each "
                         "destination sub-range; source split: share of the remote rows in each remote stage)")
    ap.add_argument("--split", default="auto", choices=["auto", "source", "dest", "hybrid"],
                    help="rmat workloads at N>1: pipeline the exchange over groups of SOURCE rows (own rows, "
                         "then remote rows by decreasing reference count; stages accumulate), over DESTINATION "
                         "sub-ranges (every row written once), or hybrid (own-source edges, then the "
                         "remote-source edges by destination sub-range); auto = the measured best per N")
    ap.add_argument("--ownership", default="auto", choices=["auto", "cyclic", "xorfold"],
                    help="rmat workloads at N>1: feature row i lives on rank i %% N (cyclic) or on the XOR of "
                         "the log2(N)-bit groups of i (xorfold: balanced on R-MAT ids, whose bits are skewed); "
                         "auto = xorfold for power-of-two N")
    ap.add_argument("--merge-own", type=int, default=-1,
                    help="rmat workloads at N>1, source split: reduce the own-source edges and the first remote "
                         "group in one two-buffer launch (-1 = the measured best per N)")
    ap.add_argument("--push-chunk", type=int, default=-1,
                    help="rmat workloads at N>1: ring slot bytes of the TMA push (4096..16384; -1 = the measured "
                         "best per N: 8192 below 8 GPUs, 16384 at 8)")
    ap.add_argument("--push-blocks", type=int, default=148,
                    help="grid cap of the push kernel when it runs beside the reduction (0 = fill the chip)")
    ap.add_argument("--per-config", type=int, default=1,
                    help="N=1: also time the other BASELINE.json configs' kernels (per_config object)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the output of the last timed step to DIR/*.npy (float32, a fixed seeded "
                         "sample of rows when larger than 32 MB) for output-for-output comparison of builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    elif is_rmat(args.workload):
        run_rmat(args)
    else:
        run_weak(args)


if __name__ == "__main__":
    main()
