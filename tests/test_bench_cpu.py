"""CPU checks of bench.py's host logic: the reference arm's JSON line, the workload description
shared by both arms, and the R-MAT slice sampler the CPU baseline uses."""
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_line_and_shared_config():
    import bench as B
    env = dict(os.environ, OMP_NUM_THREADS="1")  # what torchrun exports: the arm must override it
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload",
                        "rmat16", "--steps", "2", "--warmup", "1", "--gpus", "2"], capture_output=True,
                       text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["unit"] == "edges/s" and line["value"] > 0
    assert line["config"] == B.config_of("rmat16")          # the repo arm emits the same object
    assert line["metric"] == B.metric_of("rmat16") and line["scaling"] == "strong"
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["value"] == line["value"]
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"]
    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:
        cores = os.cpu_count()
    assert line["cpu_baseline"]["cores"] == cores             # not torchrun's OMP_NUM_THREADS=1
    # non-zero ranks of a torchrun launch print nothing and exit 0
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload",
                        "rmat16"], capture_output=True, text=True, env=dict(env, RANK="1"), timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_rmat_slice_sampler_matches_the_full_graph():
    """rmat_edges(row_prefix=...) must be distributed like the edges of the full graph whose
    destination id starts with the prefix."""
    import bench as B
    scale, E = 8, 1 << 20
    src, dst = B.rmat_edges(scale, E, "cpu", 1)
    prefix = (0, 1)
    m = (dst >> (scale - 2)) == 0b01
    share = float(m.double().mean())
    assert abs(share - 0.76 * 0.24) < 0.005
    s_full, d_full = src[m], dst[m] & ((1 << (scale - 2)) - 1)
    s_sl, d_sl = B.rmat_edges(scale, int(m.sum()), "cpu", 2, row_prefix=prefix)
    assert int(d_sl.max()) < (1 << (scale - 2)) and int(s_sl.max()) < (1 << scale)
    for a, b in ((s_full, s_sl), (d_full, d_sl)):
        ha = torch.bincount(a, minlength=1 << scale).double() / a.numel()
        hb = torch.bincount(b, minlength=1 << scale).double() / b.numel()
        assert float((ha - hb).abs().sum()) < 0.06          # total-variation distance of the marginals
    # joint structure at the top level below the prefix: quadrant shares a, b, c, d
    top_r = (d_sl >> (scale - 3)) & 1
    top_c = (s_sl >> (scale - 3)) & 1
    q = [float(((top_r == r) & (top_c == c)).double().mean()) for r, c in ((0, 0), (0, 1), (1, 0), (1, 1))]
    for got, want in zip(q, (0.57, 0.19, 0.19, 0.05)):
        assert abs(got - want) < 0.01


def test_dump_outputs_sample_and_budget(tmp_path):
    """--dump-outputs: float32 rows with float64 global row ids, every row of a small output, the
    same seeded sample of a large one on every call, and the whole dump under 64 MB."""
    import numpy as np
    import bench as B
    small = torch.randn(100, 8, dtype=torch.bfloat16)
    B.dump_outputs(str(tmp_path / "s"), small, 0, 0, 1)
    v, r = np.load(tmp_path / "s" / "out.npy"), np.load(tmp_path / "s" / "out_rows.npy")
    assert v.dtype == np.float32 and r.dtype == np.float64
    assert np.array_equal(v, small.float().numpy()) and np.array_equal(r, np.arange(100.0))
    big = torch.arange(300_000, dtype=torch.float32)[:, None].expand(-1, 64).contiguous()
    for d in ("a", "b"):
        for rank in range(2):
            B.dump_outputs(str(tmp_path / d), big, 1000 + rank, rank, 2)
    for rank in range(2):
        va, ra = (np.load(tmp_path / "a" / f"{n}_rank{rank}.npy") for n in ("out", "out_rows"))
        vb, rb = (np.load(tmp_path / "b" / f"{n}_rank{rank}.npy") for n in ("out", "out_rows"))
        assert np.array_equal(va, vb) and np.array_equal(ra, rb)
        assert 0 < len(ra) < 300_000 and np.all(np.diff(ra) > 0)
        assert np.array_equal(va[:, 0], ra - 1000 - rank)         # each row is the output row its id names
    total = sum(os.path.getsize(p) for p in (tmp_path / "a").iterdir())
    assert total <= 64 << 20


def test_steps_must_be_positive():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload",
                        "rmat16", "--steps", "0"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and "--steps" in r.stderr and r.stdout.strip() == ""


def test_parity_check_detects_errors():
    import bench as B
    g = torch.Generator().manual_seed(0)
    n, E, F = 50, 2000, 8
    x = torch.randn(n, F, generator=g)
    src = torch.randint(0, n, (E,), generator=g)
    dst = torch.randint(0, n, (E,), generator=g)
    out = torch.zeros(n, F).index_add_(0, dst, x[src])
    assert float(B.parity_check(out, lambda ids: x[ids], src, dst, 0, n, 1e-5, block_rows=16, edge_step=300)) <= 1.0
    bad = out.clone()
    bad[7, 3] += 0.01
    assert float(B.parity_check(bad, lambda ids: x[ids], src, dst, 0, n, 1e-5, block_rows=16, edge_step=300)) > 1.0
