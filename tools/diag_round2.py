"""development: why is the fused cutoff pass slow on round-2 spectra of a pair tree?  python tools/diag_round2.py R C"""
import sys
from pathlib import Path
import torch
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from shardmerge_b200 import engine as E, _lib
from shardmerge_b200.config import MergeConfig
from shardmerge_b200.index import InMemoryIndex
from shardmerge_b200.merge.fast_fourier import FourierMerge
R, C = int(sys.argv[1]), int(sys.argv[2])
dev = torch.device("cuda:0")
g = torch.Generator(device=dev).manual_seed(1)
base = (0.02 * torch.randn((R, C), generator=g, device=dev)).to(torch.bfloat16)
sig, al = (0.002, 0.0026, 0.0023, 0.0029), (0.3, 0.5, 0.4, 0.2)
fts = [(base.float() + s * torch.randn((R, C), generator=g, device=dev)).to(torch.bfloat16) for s in sig]
fm = FourierMerge(MergeConfig(finetune_merge=[], output_base_model="b", output_dir="/tmp/unused"), index_manager=InMemoryIndex({}))
fm.keep_intermediates = True
fm.merge_sources([E.make_source(base, ft, weight=a, name=f"m{k}") for k, (ft, a) in enumerate(zip(fts, al))], base, dev, layer_name="x")
(_, _, ta), (_, _, tb) = fm.last_tree
ws = E.get_workspace(R, C, dev, lane="diag")
N = R * C
def spectra(x0, x1):
    ws.ctl.zero_()
    E.fwd_rows(ws, 0, E.Source(x32=x0), E.D_SUMSQ0); E.fwd_rows(ws, 1, E.Source(x32=x1), E.D_SUMSQ1)
    dbl, _, _, _ = ws.read_ctl()
    n0, n1 = float(dbl[0]) ** 0.5, float(dbl[1]) ** 0.5
    E.fwd_cols(ws, 0, scale=E.inv_norm_f32(E.f32(n0))); E.fwd_cols(ws, 1, scale=E.inv_norm_f32(E.f32(n1)))
def timeit(fn, n=10):
    for _ in range(2): fn()
    torch.cuda.synchronize()
    a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n): fn()
    b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b) / n * 1000
for tag, (x0, x1) in (("round 1 (deltas)", ((fts[0].float() - base.float()), (fts[1].float() - base.float()))), ("round 2 (intermediates)", (ta, tb))):
    spectra(x0.contiguous(), x1.contiguous())
    Ch = C // 2
    a, b = ws.re[0][:, :Ch + 1], ws.re[1][:, :Ch + 1]
    us = timeit(lambda: E.fstats_cutoff(ws, ws.re[0], ws.re[1], int(2 * N * 0.08), 0.5))
    h = ws.ctl.cpu()
    o = _lib.SM_CTL_FS
    st = h[o:o + _lib.SM_FS_STATE_BYTES]
    lo, hi = st[16:24].view(torch.int32).tolist()
    lo_f = torch.tensor([lo], dtype=torch.int32).view(torch.float32).item(); hi_f = torch.tensor([hi], dtype=torch.int32).view(torch.float32).item()
    inwin = (((a.abs() >= lo_f) & (a.abs() <= hi_f)).float().mean().item() + ((b.abs() >= lo_f) & (b.abs() <= hi_f)).float().mean().item()) / 2
    prod0 = ((a * b) == 0).float().mean().item()
    print(f"{tag}: cutoff {us:.1f} us  window [{lo_f:.3e}, {hi_f:.3e}] width 2^{(hi - lo).bit_length()}  keys in window {inwin:.4f}  "
          f"zero products {prod0:.4f}  exact zeros {((a == 0).float().mean().item()):.4f}/{((b == 0).float().mean().item()):.4f}  "
          f"|re| quantiles a {[float(q) for q in torch.quantile(a.abs().flatten()[:4000000], torch.tensor([0.05, 0.1, 0.2, 0.25, 0.5], device=dev))]}  sticky {ws.fs_status()}")
