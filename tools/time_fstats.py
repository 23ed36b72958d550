"""Warm CUDA-event timing of the fused statistics entry points: python tools/time_fstats.py R C [culled]
`culled`: 20 % of the bins of both planes hold rounding-noise-level values (what round >= 2 of a pair tree sees: the
previous round's culled bins come back as ~1e-8 after the inverse + forward transform)."""
import sys, os
from pathlib import Path
import torch
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from shardmerge_b200 import engine as E
R, C = int(sys.argv[1]), int(sys.argv[2])
culled = len(sys.argv) > 3
dev = torch.device("cuda:0")
ws = E.get_workspace(R, C, dev)
g = torch.Generator(device=dev).manual_seed(1)
ws.re[0].copy_(torch.randn(ws.re[0].shape, generator=g, device=dev) * 0.7)
ws.re[1].copy_(0.5 * ws.re[0] + 0.6 * torch.randn(ws.re[0].shape, generator=g, device=dev))
if culled:
    for k in (0, 1):
        m = torch.rand(ws.re[k].shape, generator=g, device=dev) < 0.2
        ws.re[k][m] = (1e-8 * torch.randn(ws.re[k].shape, generator=g, device=dev))[m]
ws.re[0][:, ws.plan.Ch + 1:] = 0; ws.re[1][:, ws.plan.Ch + 1:] = 0
N = R * C
out = torch.empty_like(ws.re[0])
def run(fn, n=20):
    for _ in range(3): fn()
    torch.cuda.synchronize()
    a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n): fn()
    b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b) / n * 1000
ws.ctl.zero_()
cut = 0.08
cull = 0.10 if culled else 0.20
print(("culled " if culled else "plain  ") + f"{R}x{C}")
print("  cutoff  %.1f us" % run(lambda: E.fstats_cutoff(ws, ws.re[0], ws.re[1], int(2 * N * cut), 0.375)))
print("  blend   %.1f us" % run(lambda: E.fstats_blend_cull(ws, ws.re[0], ws.re[1], 1.0, out, int(N * cull))))
print("  sticky", ws.fs_status(), "thr_cut %.3e thr_cull %.3e" % (float(ws.flt[E.F_THR_CUT]), float(ws.flt[E.F_THR_CULL])))
