"""Times the TIES / DARE kernels (csrc/kernels_sparse.cu) and one files-in, files-out merge().

    python tools/bench_sparse.py [--iters 20] [--layers 2] [--out FILE]

Kernels: CUDA events around sm_sparse_select and sm_sparse_merge at the Llama-3.1-8B projection shapes, bf16, M = 2, 3, 8
finetunes, density 0.2 and 0.5.  Bytes are what the algorithm must move (bf16, N elements): the select reads 2(M+1)N in
each of its four passes (three radix digits and the tie count), the merge pass reads 2(M+1)N and writes 2N; DARE is the
merge pass alone.  The 4096x4096 working sets (3 to 9 tensors of 32 MB) fit partly in the 126 MB L2; the larger shapes
do not.  End to end: TiesMerge.merge() on a Llama-8B-shaped checkpoint (32000-token vocabulary) of --layers layers with 3 finetunes, written to and
read from a temporary directory.  The card's name and power limit are printed with the numbers."""
from __future__ import annotations

import argparse
import asyncio
import json
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from shardmerge_b200.merge import ties as T  # noqa: E402

SHAPES = [(4096, 4096), (1024, 4096), (14336, 4096), (4096, 14336)]


def card() -> str:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def timed(fn, iters: int) -> float:
    """milliseconds per call, CUDA events around `iters` calls after two warm-up calls"""
    fn(); fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def kernels(iters: int):
    dev = torch.device("cuda:0")
    rows = []
    for R, C in SHAPES:
        n = R * C
        base = (0.02 * torch.randn((R, C), device=dev)).to(torch.bfloat16)
        pool = [(base.float() + 0.002 * torch.randn((R, C), device=dev)).to(torch.bfloat16) for _ in range(8)]
        for M in (2, 3, 8):
            fts, w = pool[:M], [1.0 / M] * M
            for density in (0.2, 0.5):
                k = int(density * n)
                t_sel = timed(lambda: T.select_thresholds(base, fts, k), iters)
                t_ties = timed(lambda: T.sparse_merge(T.MODE_TIES, base, fts, w, density), iters)
                t_dare = timed(lambda: T.sparse_merge(T.MODE_DARE_TIES, base, fts, w, density, tensor_name="x"), iters)
                sel_bytes, merge_bytes = 4 * 2 * (M + 1) * n, 2 * (M + 1) * n + 2 * n
                row = dict(shape=f"{R}x{C}", M=M, density=density, select_ms=round(t_sel, 4),
                           select_GBps=round(sel_bytes / t_sel / 1e6, 1),
                           ties_total_ms=round(t_ties, 4), ties_merge_ms=round(t_ties - t_sel, 4),
                           ties_merge_GBps=round(merge_bytes / (t_ties - t_sel) / 1e6, 1),
                           dare_ms=round(t_dare, 4), dare_GBps=round(merge_bytes / t_dare / 1e6, 1))
                rows.append(row)
                print(json.dumps(row), flush=True)
        del pool
    return rows


def end_to_end(layers: int):
    from shardmerge_b200.config import MergeConfig, MergeModel
    from shardmerge_b200.index import LocalSafetensorsIndex
    from shardmerge_b200.merge import TiesMerge
    from tests.lora_util import llama_shapes, random_model, write_model
    shapes = llama_shapes(layers=layers, H=4096, KV=1024, I=14336, V=32000)     # Llama-2's vocabulary keeps the set-up short
    with tempfile.TemporaryDirectory() as tmp:
        root = Path(tmp)
        base = random_model(shapes, 0)
        write_model(root / "org" / "base", base)
        for s in (1, 2, 3):
            g = torch.Generator().manual_seed(s)
            write_model(root / "org" / f"ft{s}", {n: (t.float() + 0.002 * torch.randn(t.shape, generator=g)).to(t.dtype)
                                                  for n, t in base.items()})
        del base
        params = sum(int(torch.tensor(s).prod()) for s in shapes.values())
        best = None
        for rep in range(2):
            cfg = MergeConfig(finetune_merge=[MergeModel(model=f"org/ft{s}", base="org/base") for s in (1, 2, 3)],
                              output_base_model="org/base", output_dir=str(root / f"out{rep}"), storage_dir=str(root))
            strategy = TiesMerge(cfg, density=0.2, index_manager=LocalSafetensorsIndex(cfg.storage_path))
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            asyncio.run(strategy.merge("cuda:0"))
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
        row = dict(end_to_end="TiesMerge.merge", layers=layers, finetunes=3, params=params, best_s=round(best, 3),
                   Gparam_per_s=round(params / best / 1e9, 3))
        print(json.dumps(row), flush=True)
        return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--layers", type=int, default=2)
    ap.add_argument("--out", type=str, default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sparse.py needs a CUDA device")
    info = card()
    print(json.dumps(dict(card=info)), flush=True)
    result = dict(card=info, kernels=kernels(args.iters), end_to_end=end_to_end(args.layers))
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
