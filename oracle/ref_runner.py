"""ref_runner.py -- run the REFERENCE ITSELF (unmodified 54rt1n/shardmerge `shard` package) as checker / CPU arm.

TEST INFRASTRUCTURE.  Only tests/, __graft_entry__.smoke() and bench.py's CPU legs import this; nothing under
shardmerge_b200/ does.  The reference is found at oracle/_ref/shard: a git-ignored copy that
`make oracle_ref REFERENCE=<checkout of the reference>` makes (the repository holds no reference source).  Where it is
absent, the tests that run it skip.
`device="cuda"` on a B200 is the parity oracle for large tensors (same reference code, cuFFT + CUDA
reductions; the CPU reference's fp32 `.norm()` is biased at Llama sizes, SURVEY.md 0 / 7.3-0); `device="cpu"` is the
timed CPU baseline (`FourierMerge._merge_layer`, shard/merge/fast_fourier.py:103-276).
"""
from __future__ import annotations

import asyncio
import sys
import tempfile
from pathlib import Path

HERE = Path(__file__).resolve().parent
_CANDIDATES = [HERE / "_ref"]


def ref_root():
    for c in _CANDIDATES:
        if (c / "shard" / "tensor" / "functions.py").exists():
            return c
    return None


def available() -> bool:
    return ref_root() is not None


def load():
    """-> (shard.tensor.functions, FourierMerge, MergeConfig, MergeModel, ShardLayer) of the reference."""
    root = ref_root()
    if root is None:
        raise RuntimeError("reference not available: run `make oracle_ref REFERENCE=<checkout of the reference>`")
    if str(root) not in sys.path:
        sys.path.insert(0, str(root))
    import shard.tensor.functions as F
    from shard.config import MergeConfig, MergeModel
    from shard.merge.fast_fourier import FourierMerge
    from shard.writer import ShardLayer
    return F, FourierMerge, MergeConfig, MergeModel, ShardLayer


class _Promise:
    def __init__(self, t):
        self.t = t

    async def get(self):
        return self.t


class StubIndex:
    """Stands in for HFMultiModelIndex (shard/index.py:195-236) with in-memory tensors."""

    def __init__(self, tensors):
        self.tensors = tensors

    def get_tensor(self, model, layer_name, device="cpu"):
        return _Promise(self.tensors[(model, layer_name)].to(device))

    async def preload_tensor(self, model, layer_name):
        return None


def merge_layer(base, fts, alphas, device="cpu", layer="model.layers.3.mlp.up_proj.weight"):
    """The reference's FourierMerge._merge_layer on in-memory bf16 tensors -> merged tensor (on CPU)."""
    _, FourierMerge, MergeConfig, MergeModel, ShardLayer = load()
    tensors = {("org/base", layer): base}
    models = []
    for k, ft in enumerate(fts):
        tensors[(f"org/ft{k}", layer)] = ft
        models.append(MergeModel(model=f"org/ft{k}", base="org/base", alpha=alphas[k]))
    with tempfile.TemporaryDirectory() as td:
        cfg = MergeConfig(finetune_merge=models, output_base_model="org/base", output_dir=td + "/out",
                          cache_dir=td + "/cache", storage_dir=td + "/st")
        merger = FourierMerge(cfg, index_manager=StubIndex(tensors))
        out = asyncio.run(merger._merge_layer(ShardLayer(0, "s", layer, False), device))
    return out.cpu()
