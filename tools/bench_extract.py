"""Extracting a LoRA adapter from two checkpoints: the two kernels alone, and files in -> adapter out through extract_lora.
    python tools/bench_extract.py [--layers 8] [--root /dev/shm] [--rank 64] [--repeats 2] [--iters 50]

1. sm_lowrank_right / sm_lowrank_left (csrc/kernels_lowrank.cu, each a product kernel plus the fixed-order reduction of
   its split partials) at 14336x4096 and 4096x14336, bf16 W and M, k in {16, 72, 136, 264}: CUDA events around `--iters`
   back-to-back calls after a warm-up.  W + M are 235 MB, above the 126 MB L2, so every call reads them from HBM.  FMA/s
   counts k FMAs per element of Δ; TB/s counts the 4N bytes of W and M (the fp32 operand and result, k (R + C) x 4 bytes,
   are listed apart).  By these counts a kernel is HBM-bound below k ~ 20 and FMA-bound above (7.7 TB/s data-sheet HBM
   against the 36.7 TFMA/s FFMA2 rate of tools/ubench_f32x2.cu): an expectation, not a measurement.
2. A Llama-8B-shaped bf16 base and finetune (`--layers` transformer layers, bench.py's synthetic tensors) written as
   safetensors under ROOT, `extract_lora` at `--rank` into ROOT/out: Gparam/s over the wall clock, and the `timings` split
   into waiting for file reads, kernels, torch.linalg plumbing and writing (the first three overlap in time only where
   reads run ahead of the device; kernels and plumbing are CUDA-event sums).
The card's name and power limit are printed in the same run."""
import argparse, json, shutil, subprocess, sys, tempfile, time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import bench as B
from safetensors.torch import save_file
from shardmerge_b200 import extract

ap = argparse.ArgumentParser()
ap.add_argument("--layers", type=int, default=8)
ap.add_argument("--root", default="/dev/shm")
ap.add_argument("--rank", type=int, default=64)
ap.add_argument("--repeats", type=int, default=2)
ap.add_argument("--iters", type=int, default=50)
ap.add_argument("--skip-files", action="store_true")
args = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("bench_extract.py measures on a CUDA device; none is visible")
dev = torch.device("cuda:0")
card = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip()
print(f"card: {card}")

# ---- 1. kernels ------------------------------------------------------------------------------------------------------
rows = []
for R, C in [(14336, 4096), (4096, 14336)]:
    g = torch.Generator(device=dev).manual_seed(R + C)
    W = (0.02 * torch.randn((R, C), generator=g, device=dev)).to(torch.bfloat16)
    M = (W.float() + 0.002 * torch.randn((R, C), generator=g, device=dev)).to(torch.bfloat16)
    for k in (16, 72, 136, 264):
        X = torch.randn((C, k), generator=g, device=dev)
        Q = torch.randn((R, k), generator=g, device=dev)
        ws = extract._workspace(R, C, k, dev)
        for kind, call in (("right", lambda: extract.lowrank_right(W, M, X, ws=ws)),
                           ("left", lambda: extract.lowrank_left(W, M, Q, ws=ws))):
            for _ in range(5):
                call()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.iters):
                call()
            e1.record()
            torch.cuda.synchronize()
            t = e0.elapsed_time(e1) / 1e3 / args.iters
            n = R * C
            row = dict(kernel=kind, shape=f"{R}x{C}", k=k, us=round(t * 1e6, 1), TFMAps=round(k * n / t / 1e12, 2),
                       TBps=round(4 * n / t / 1e12, 2), operand_and_result_MB=round(4 * k * (R + C) / 1e6, 1))
            rows.append(row)
            print(f"{kind:>5} {row['shape']:>10} k={k:<3} {row['us']:8.1f} us  {row['TFMAps']:6.2f} TFMA/s  {row['TBps']:5.2f} TB/s")
    del W, M
print(json.dumps(dict(kernels="sm_lowrank_right / sm_lowrank_left, bf16 W and M", card=card, rows=rows)))
if args.skip_files:
    sys.exit(0)

# ---- 2. files in -> adapter out --------------------------------------------------------------------------------------
a = B.ARCH["llama8b"]
root = Path(tempfile.mkdtemp(prefix="shardmerge_extract_", dir=args.root))
try:
    per_layer = B.layer_tensors(a)
    for m in ("base", "model"):
        (root / m).mkdir()
    wm, idx, params = {}, 0, 0
    for layer in range(args.layers):
        shard = f"model-{layer + 1:05d}-of-{args.layers:05d}.safetensors"
        blobs = {"base": {}, "model": {}}
        for nm, shape in per_layer:
            name = f"model.layers.{layer}.{nm}"
            base, fts = B.synth_tensor(torch, shape, idx, 1, dev)
            blobs["base"][name] = base.cpu(); blobs["model"][name] = fts[0].cpu()
            wm[name] = shard; idx += 1; params += B.numel(shape)
        for m in ("base", "model"):
            save_file(blobs[m], str(root / m / shard), metadata={"format": "pt"})
    for m in ("base", "model"):
        (root / m / "model.safetensors.index.json").write_text(json.dumps({"metadata": {}, "weight_map": wm}))
    runs = []
    for rep in range(args.repeats):
        out = root / "out"
        timings = {}
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = extract.extract_lora(root / "base", root / "model", out, args.rank, timings=timings)
        dt = time.perf_counter() - t0
        size = sum(f.stat().st_size for f in out.iterdir())
        runs.append(dict(seconds=round(dt, 3), gparams_per_s=round(params / dt / 1e9, 3), adapter_MB=round(size / 1e6, 1),
                         pairs=len(res), **{k: round(v, 3) for k, v in timings.items()}))
        print(f"extract run {rep}: {dt:.3f} s  {params / dt / 1e9:.3f} Gparam/s  "
              + "  ".join(f"{k} {v:.3f} s" for k, v in sorted(timings.items())))
        shutil.rmtree(out)
    print(json.dumps(dict(workload=f"llama8b-shaped, {args.layers} layers, bf16 base + finetune on {args.root}, rank {args.rank}",
                          params=params, card=card, runs=runs)))
finally:
    shutil.rmtree(root, ignore_errors=True)
