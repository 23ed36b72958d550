"""LoRA adapters as finetunes: the materialize kernel alone, and files in -> files out through the public merge() API.
    python tools/bench_lora.py [--layers 8] [--root /dev/shm] [--repeats 2] [--skip-files]

1. sm_lora_materialize (csrc/kernels_lora.cu) at the Llama-8B projection shapes for r in {8, 16, 64, 256}, bf16 base and
   factors: CUDA events around `--iters` back-to-back launches after a warm-up.  GB/s counts the base read, the result
   write and the factors once; FMA/s counts r FMAs per element.  4096x4096 and 1024x4096 (base + result 64 MB / 16 MB) fit
   in the 126 MB L2, the two 14336-sized shapes (235 MB) do not.
2. Like tools/bench_files.py: a Llama-8B-shaped base, two full finetunes and LoRA adapters (r = 16) written as safetensors
   under ROOT, merged with FourierMerge + LocalSafetensorsIndex into ROOT/out, wall clock around merge().  Four runs: two
   full finetunes; one full finetune + one adapter on all seven projections; two such adapters; one full finetune + one
   adapter on q_proj and v_proj only.  In the last, the five untargeted tensors of each layer have a zero delta for the
   adapter, which the fused chain hands to the step-by-step path (the same as for a zero-delta full checkpoint).
The card's name and power limit are printed in the same run."""
import argparse, asyncio, json, shutil, subprocess, sys, tempfile, time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import bench as B
from safetensors.torch import save_file
from shardmerge_b200 import lora
from shardmerge_b200.config import MergeConfig, MergeModel
from shardmerge_b200.index import LocalSafetensorsIndex
from shardmerge_b200.merge.fast_fourier import FourierMerge
from shardmerge_b200.validate import verify_output

ap = argparse.ArgumentParser()
ap.add_argument("--layers", type=int, default=8)
ap.add_argument("--root", default="/dev/shm")
ap.add_argument("--repeats", type=int, default=2)
ap.add_argument("--iters", type=int, default=200)
ap.add_argument("--reader-threads", type=int, default=4)
ap.add_argument("--skip-files", action="store_true")
args = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("bench_lora.py measures on a CUDA device; none is visible")
dev = torch.device("cuda:0")
card = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip()
print(f"card: {card}")

# ---- 1. kernel -------------------------------------------------------------------------------------------------------
kernel_rows = []
for R, C in [(4096, 4096), (1024, 4096), (14336, 4096), (4096, 14336)]:
    for r in (8, 16, 64, 256):
        g = torch.Generator(device=dev).manual_seed(R + C + r)
        W = (0.02 * torch.randn((R, C), generator=g, device=dev)).to(torch.bfloat16)
        A = torch.randn((r, C), generator=g, device=dev).to(torch.bfloat16)
        Bf = (2.5e-4 * torch.randn((R, r), generator=g, device=dev)).to(torch.bfloat16)
        for _ in range(10):
            lora.materialize(W, A, Bf, 2.0)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.iters):
            lora.materialize(W, A, Bf, 2.0)
        e1.record()
        torch.cuda.synchronize()
        t = e0.elapsed_time(e1) / 1e3 / args.iters
        n = R * C
        nbytes = 2 * n + 2 * n + 2 * r * (R + C)
        row = dict(shape=f"{R}x{C}", r=r, us=round(t * 1e6, 2), GBps=round(nbytes / t / 1e9, 1),
                   TFMAps=round(r * n / t / 1e12, 2))
        kernel_rows.append(row)
        print(f"materialize {row['shape']:>10} r={r:<3}  {row['us']:8.2f} us  {row['GBps']:7.1f} GB/s  {row['TFMAps']:6.2f} TFMA/s")
        del W, A, Bf
print(json.dumps(dict(kernel="sm_lora_materialize bf16 base, bf16 factors", card=card, rows=kernel_rows)))
if args.skip_files:
    sys.exit(0)

# ---- 2. files in -> files out ----------------------------------------------------------------------------------------
a = B.ARCH["llama8b"]
root = Path(tempfile.mkdtemp(prefix="shardmerge_lora_", dir=args.root))
try:
    per_layer = B.layer_tensors(a)
    full_models = ["synth/base", "synth/ft0", "synth/ft1"]
    adapters = {"synth/ad0": B.layer_tensors(a), "synth/ad1": B.layer_tensors(a),
                "synth/adqv": [(n, s) for n, s in per_layer if n.startswith(("self_attn.q_proj", "self_attn.v_proj"))]}
    for m in full_models + list(adapters):
        (root / "storage" / m).mkdir(parents=True)
    wm, idx, params = {}, 0, 0
    ad_blobs = {m: {} for m in adapters}
    for layer in range(args.layers):
        shard = f"model-{layer + 1:05d}-of-{args.layers:05d}.safetensors"
        blobs = {m: {} for m in full_models}
        for nm, shape in per_layer:
            name = f"model.layers.{layer}.{nm}"
            base, fts = B.synth_tensor(torch, shape, idx, 2, dev)
            blobs["synth/base"][name] = base.cpu(); blobs["synth/ft0"][name] = fts[0].cpu(); blobs["synth/ft1"][name] = fts[1].cpu()
            wm[name] = shard; idx += 1; params += B.numel(shape)
            for k, (m, targets) in enumerate(adapters.items()):
                if len(shape) != 2 or nm not in dict(targets):
                    continue
                g = torch.Generator(device=dev).manual_seed(7919 * (k + 1) + idx)
                module = name[: -len(".weight")]
                ad_blobs[m][f"base_model.model.{module}.lora_A.weight"] = torch.randn((16, shape[1]), generator=g, device=dev).to(torch.bfloat16).cpu()
                ad_blobs[m][f"base_model.model.{module}.lora_B.weight"] = (2.5e-4 * torch.randn((shape[0], 16), generator=g, device=dev)).to(torch.bfloat16).cpu()
        for m in full_models:
            save_file(blobs[m], str(root / "storage" / m / shard), metadata={"format": "pt"})
    for m in full_models:
        (root / "storage" / m / "model.safetensors.index.json").write_text(json.dumps({"metadata": {}, "weight_map": wm}))
    for m, blob in ad_blobs.items():
        save_file(blob, str(root / "storage" / m / lora.WEIGHTS_FILE))
        (root / "storage" / m / lora.CONFIG_FILE).write_text(json.dumps({"peft_type": "LORA", "r": 16, "lora_alpha": 32}))
    bytes_of = lambda m: sum(f.stat().st_size for f in (root / "storage" / m).glob("*.safetensors"))

    runs = {"two full finetunes": ("synth/ft0", "synth/ft1"),
            "full + adapter (7 projections)": ("synth/ft0", "synth/ad0"),
            "two adapters (7 projections)": ("synth/ad0", "synth/ad1"),
            "full + adapter (q_proj, v_proj only)": ("synth/ft0", "synth/adqv")}
    results = []
    for label, (m0, m1) in runs.items():
        rates = []
        for rep in range(args.repeats):
            out = root / "out"
            cfg = MergeConfig(finetune_merge=[MergeModel(model=m0, base="synth/base", alpha=0.3, is_input=True),
                                              MergeModel(model=m1, base="synth/base", alpha=0.5, is_output=True)],
                              output_base_model="synth/base", output_dir=str(out), device=str(dev), storage_dir=str(root / "storage"))
            fm = FourierMerge(cfg, index_manager=LocalSafetensorsIndex(cfg.storage_path, reader_threads=args.reader_threads))
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            asyncio.run(fm.merge(str(dev)))
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            ok = verify_output(out, expected_dtype=torch.bfloat16).ok
            rates.append(params / dt)
            print(f"{label}, run {rep}: {dt:.3f} s  {params / dt / 1e9:.2f} Gparam/s  verified={ok}")
            shutil.rmtree(out)
        in_bytes = bytes_of("synth/base") + bytes_of(m0) + bytes_of(m1)
        results.append(dict(run=label, params_per_s=max(rates), input_bytes=in_bytes))
    print(json.dumps(dict(workload=f"llama8b-shaped, {args.layers} layers, 2 models on one base, safetensors on {args.root} in and out",
                          merged_params=params, card=card, runs=results, api="FourierMerge.merge() + LocalSafetensorsIndex + ModelWriter")))
finally:
    shutil.rmtree(root, ignore_errors=True)
