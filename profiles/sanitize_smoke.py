"""Small invocation of every kernel, for `compute-sanitizer --tool memcheck` (one tool per gpurun call):
    compute-sanitizer --tool memcheck --error-exitcode 1 python profiles/sanitize_smoke.py
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "gnn-ops-benchmark_b200"))
import torch  # noqa: E402

import gno_b200  # noqa: E402
from gno_b200 import plan as planmod  # noqa: E402

dev = torch.device("cuda:0")
g = torch.Generator(device=dev).manual_seed(0)
for dtype in (torch.float32, torch.bfloat16, torch.float16):
    for (E, N, F) in ((3000, 40, 100), (5000, 7, 602), (4097, 300, 7), (2000, 3000, 64), (999, 5, 1)):
        x = torch.randn(500, F, device=dev, generator=g).to(dtype)
        dst = (torch.rand(E, device=dev, generator=g) ** 3 * N).long().clamp_(0, N - 1)
        src = torch.randint(0, 500, (E,), device=dev, generator=g)
        for cl in (32, 256):
            plan = planmod.build_plan(dst, N, chunk_len=cl)
            gidx = plan.sorted_ids(src)
            for red in ("sum", "mean", "mul", "min", "max"):
                gno_b200.segment_reduce(plan, x, red, gidx=gidx, eid=plan.perm, want_arg=red in ("min", "max"))
        w = torch.rand(E, device=dev, generator=g).to(dtype)
        gno_b200.spmm(torch.stack([dst, src]), w, N, 500, x)
    s = torch.rand(97, 131, device=dev, generator=g).to(dtype)
    i2 = torch.randint(0, 50, (97, 131), device=dev, generator=g)
    for red in ("sum", "mean", "mul", "min", "max"):
        for dim in (0, 1):
            gno_b200.scatter(s, i2, dim, None, 50, red, return_arg=True)
            gno_b200.scatter(s, i2[0] if dim == 1 else i2[:, 0].contiguous(), dim, None, 50, red, return_arg=True)
    gno_b200.index_add(s, 1, torch.randint(0, 131, (131,), device=dev, generator=g), s.clone())
    gno_b200.index_select(s, 0, torch.randint(0, 97, (33,), device=dev, generator=g))
    gno_b200.index_select(s, 1, torch.randint(0, 131, (33,), device=dev, generator=g))
idx = torch.stack([torch.randint(0, 70, (9000,), device=dev, generator=g), torch.randint(0, 90, (9000,), device=dev, generator=g)])
val = torch.rand(9000, device=dev, generator=g)
ci, cv = gno_b200.coalesce(idx, val, 70, 90)
gno_b200.transpose(ci, cv, 70, 90)
gno_b200.transpose(idx, val, 70, 90)
for shape, dim in (((10007,), 0), ((50, 70), 0), ((50, 70), 1)):
    gno_b200.sort(torch.randn(*shape, device=dev, generator=g), dim)
k = torch.randint(0, 1 << 62, (70001,), device=dev, generator=g)
gno_b200.sort_pairs(k, torch.arange(70001, device=dev, dtype=torch.int32), 0, 64)
gno_b200.sort_pairs(k.to(torch.int32), None, 0, 32)
gno_b200.segment_csr(torch.randn(1000, 6, device=dev, generator=g), torch.tensor([0, 0, 10, 500, 1000], device=dev), None, "max", True)
# multi_aggregate: odd widths and towers, hub rows over several chunks, empty rows, dropped
# destinations; forward and both backward forms
avg = {"lin": 3.0, "log": 1.2}
for dtype in (torch.float32, torch.bfloat16, torch.float16):
    for (E, N, T, F) in ((3001, 40, 1, 7), (999, 300, 3, 5), (4097, 9, 2, 1), (2000, 64, 1, 100)):
        dst = (torch.rand(E, device=dev, generator=g) ** 3 * N).long()
        dst[::97] = N + 1
        src = torch.randint(0, 333, (E,), device=dev, generator=g)
        for form_src, rows in ((None, E), (src, 333)):
            x = torch.randn(rows, T, F, device=dev, generator=g).to(dtype).requires_grad_(True)
            out = gno_b200.multi_aggregate(x, dst, N, ("sum", "mean", "min", "max", "var", "std"),
                                           ("identity", "amplification", "attenuation", "linear", "inverse_linear"),
                                           avg, src=form_src)
            torch.autograd.grad(out.sum(), x)
# gatv2_attention: odd and wide heads, hub rows over several chunks, empty rows, N_src != N_dst;
# forward and backward
for dtype in (torch.float32, torch.bfloat16, torch.float16):
    for (E, n_src, n_dst, H, C) in ((3001, 50, 40, 3, 7), (999, 300, 200, 8, 33), (4097, 20, 9, 1, 1),
                                    (2000, 70, 64, 2, 130)):
        dst = (torch.rand(E, device=dev, generator=g) ** 3 * n_dst).long()
        dst[dst % 5 == 3] = 0
        src = torch.randint(0, n_src, (E,), device=dev, generator=g)
        ts = [torch.randn(r, H, C, device=dev, generator=g).to(dtype).requires_grad_(True)
              for r in (n_src, n_dst, 1)]
        out = gno_b200.gatv2_attention(ts[0], ts[1], ts[2], src, dst)
        torch.autograd.grad(out.sum(), ts)
torch.cuda.synchronize()
print("sanitize smoke ok")
