"""TIES (Yadav et al. 2023) and DARE (Yu et al. 2023) task-vector merges: mergekit's `ties`, `dare_ties` and
`dare_linear`, restated with exact, device-independent definitions (DESIGN.md section 8).

For each tensor the deltas d_i = fp32(F_i) - fp32(W) of the participating finetunes against the output base W are
sparsified per model (TIES: the top `density` share by magnitude, ties to the lower flat index; DARE: a seeded Philox
drop mask, survivors rescaled by 1 / density), weighted by each model's alpha, combined by a sign-elected (TIES,
DARE-TIES) or plain (DARE-linear) disjoint mean, scaled and added back onto W.  Embed / final norm / lm_head tensors
pass through as in FourierMerge.  The hot path is csrc/kernels_sparse.cu through the C ABI; there is no CPU path."""
from __future__ import annotations

import ctypes
import hashlib
import logging
from typing import List

import torch

from .. import _lib
from .. import engine as E
from ..config import MergeConfig
from ..constants import INPUT_LAYER, OUTPUT_LAYER
from ..writer import ShardLayer
from .base import MergeTensorsBase

logger = logging.getLogger(__name__)

DTYPE_CODE = {torch.float32: 0, torch.bfloat16: 1, torch.float16: 2}
MAX_MODELS = 64
MODE_TIES, MODE_DARE_TIES, MODE_DARE_LINEAR = 0, 1, 2


def dare_key(seed: int, model_index: int, tensor_name: str):
    """Philox key (k0, k1) of model `model_index`'s DARE mask on `tensor_name`: the first 8 bytes of
    sha256(f"{seed}/{model_index}/{tensor_name}"), little-endian, k0 the low word.  The mask depends on nothing else, so
    it is the same on every GPU, in every tensor order and on every run."""
    v = int.from_bytes(hashlib.sha256(f"{seed}/{model_index}/{tensor_name}".encode()).digest()[:8], "little")
    return v & 0xFFFFFFFF, v >> 32


def _inputs(base: torch.Tensor, fts: List[torch.Tensor], what: str):
    """Contiguous, 16-byte aligned device tensors and their dtype codes; ValueError on a dtype or shape the kernels
    do not take."""
    if not 1 <= len(fts) <= MAX_MODELS:
        raise ValueError(f"{what}: 1..{MAX_MODELS} models per tensor, got {len(fts)}")
    for t in [base] + list(fts):
        if t.dtype not in DTYPE_CODE:
            raise ValueError(f"{what}: tensors must be float32, bfloat16 or float16, got {t.dtype}")
        if tuple(t.shape) != tuple(base.shape):
            raise ValueError(f"{what}: finetune / base shape mismatch: {tuple(t.shape)} vs {tuple(base.shape)}")

    def fix(t):
        t = t.contiguous()
        return t if t.data_ptr() % 16 == 0 else t.clone()
    base, fts = fix(base), [fix(t) for t in fts]
    codes = (ctypes.c_int * len(fts))(*[DTYPE_CODE[t.dtype] for t in fts])
    ptrs = (ctypes.c_void_p * len(fts))(*[t.data_ptr() for t in fts])
    return base, fts, codes, ptrs


def select_thresholds(base: torch.Tensor, fts: List[torch.Tensor], k: int) -> torch.Tensor:
    """Enqueue the per-model magnitude selects (sm_sparse_select) of the k largest |delta| of each finetune; returns the
    workspace, whose first 16 * len(fts) bytes hold one sm_sparse_thr {u32 key, u32 status, i64 last} per model."""
    base, fts, codes, ptrs = _inputs(base, fts, "sparse select")
    lib = _lib.load()
    n = base.numel()
    ws = torch.empty(lib.sm_sparse_ws_bytes(n, len(fts)), dtype=torch.uint8, device=base.device)
    _lib.check(lib.sm_sparse_select(n, int(k), DTYPE_CODE[base.dtype], base.data_ptr(), codes, ptrs, len(fts), ws.data_ptr(),
                                    ws.numel(), E._stream(base.device)), "sm_sparse_select")
    return ws


def read_thresholds(ws: torch.Tensor, n_models: int):
    """[(key, status, last)] per model from a select_thresholds workspace (synchronises)."""
    raw = ws[: 16 * n_models].cpu()
    words, last = raw.view(torch.int32).view(-1, 4), raw.view(torch.int64).view(-1, 2)[:, 1]
    return [(int(w[0]) & 0xFFFFFFFF, int(w[1]) & 0xFFFFFFFF, int(j)) for w, j in zip(words, last)]


def sparse_merge(mode: int, base: torch.Tensor, fts: List[torch.Tensor], weights: List[float], density: float,
                 scale: float = 1.0, seed: int = 0, tensor_name: str = "", model_indices=None):
    """Enqueue one tensor's merge on the current stream -> (out in base's dtype, per-model count of non-finite deltas as
    an int32 device tensor).  model_indices: each model's position in finetune_merge, which keys its DARE mask."""
    base, fts, codes, ptrs = _inputs(base, fts, f"sparse merge of {tensor_name or 'tensor'}")
    lib = _lib.load()
    M, n = len(fts), base.numel()
    idx = list(range(M)) if model_indices is None else list(model_indices)
    ws = select_thresholds(base, fts, int(density * n)) if mode == MODE_TIES else None
    keys = None
    if mode != MODE_TIES:
        keys = (ctypes.c_uint32 * (2 * M))(*[w for i in idx for w in dare_key(seed, i, tensor_name)])
    out = torch.empty_like(base)
    nonfinite = torch.empty(M, dtype=torch.int32, device=base.device)
    _lib.check(lib.sm_sparse_merge(mode, n, DTYPE_CODE[base.dtype], base.data_ptr(), codes, ptrs, M,
                                   (ctypes.c_float * M)(*weights), keys, float(density), int(density * 2 ** 24),
                                   float(scale), None if ws is None else ws.data_ptr(), nonfinite.data_ptr(),
                                   out.data_ptr(), E._stream(base.device)), "sm_sparse_merge")
    return out, nonfinite


class _Pending:
    """A merged tensor whose non-finite counts are still on the device."""

    def __init__(self, out, nonfinite, layer_name, models):
        self.out, self.nonfinite, self.layer_name, self.models = out, nonfinite, layer_name, models

    def check(self):
        for model, count in zip(self.models, self.nonfinite.tolist()):
            if count:
                raise ValueError(f"non-finite delta in {self.layer_name} of model {model}: {count} elements are NaN or Inf "
                                 f"in fp32(finetune) - fp32(base)")


class _TaskVectorMerge(MergeTensorsBase):
    mode = MODE_TIES
    method = ""
    pipeline_depth = 1           # merge(): one tensor stays in flight while the previous one's status is read

    def __init__(self, config: MergeConfig, density: float, scale: float = 1.0, seed: int = 0, index_manager=None):
        super().__init__(config, index_manager)
        self.density, self.scale, self.seed = density, scale, seed
        self.pending: List[_Pending] = []
        self.defer_checks = False        # True inside merge(): _merge_layer returns before the status is read

    def get_readme(self) -> str:
        return f"""# Merged Model

Base Model: {self.config.output_base_model}
Finetuned Models:
{chr(10).join(f'- {m.model} (weight {m.alpha})' for m in self.config.finetune_merge)}

This model was created with {self.method} (density {self.density}, scale {self.scale}{self._seed_note()}): each finetuned
model's delta from the base model was sparsified, weighted, combined by a disjoint mean and added back onto the base.
"""

    def _seed_note(self) -> str:
        return ""

    async def initialize(self):
        """Every refusal before any tensor data is read or output written: density, bases, adapters (base class),
        models per tensor and dtypes."""
        if not 0.0 < float(self.density) <= 1.0:
            raise ValueError(f"{type(self).__name__}: density must be in (0, 1], got {self.density}")
        base = self.config.output_base_model
        for m in self.config.finetune_merge:
            if m.base != base:
                raise ValueError(f"{type(self).__name__}: finetune {m.model} has base {m.base}; TIES and DARE take every delta "
                                 f"against the one output base {base}")
        await super().initialize()
        dtypes_of = getattr(self.index_manager, "tensor_dtypes", None)
        dtypes = {uri: dtypes_of(uri) for uri in [base] + [m.model for m in self.config.finetune_merge]} if dtypes_of else None
        for name in self.index_manager.get_layer_order(base):
            try:
                number = ShardLayer(0, "", name, False).layer_number
            except ValueError:
                continue                                       # unknown names are reported by the writer
            if number in (INPUT_LAYER, OUTPUT_LAYER):
                continue
            models = [m.model for m in self.config.finetune_merge if m.use_layer_index(number)]
            if len(models) > MAX_MODELS:
                raise ValueError(f"{type(self).__name__}: {len(models)} models take part in {name}; at most {MAX_MODELS}")
            if dtypes is not None and models:
                bad = [(uri, dtypes[uri][name]) for uri in [base] + models if dtypes[uri][name] not in DTYPE_CODE]
                if bad:
                    raise ValueError(f"{type(self).__name__}: {name} of {bad[0][0]} is {bad[0][1]}; the kernels take "
                                     f"float32, bfloat16 and float16")

    def _participants(self, number: int):
        return [(i, m) for i, m in enumerate(self.config.finetune_merge) if m.use_layer_index(number)]

    def prefetch_layer(self, shard_layer: ShardLayer, device: str):
        prefetch = getattr(self.index_manager, "prefetch", None)
        if prefetch is None or not str(device).startswith("cuda"):
            return
        if shard_layer.layer_number in (INPUT_LAYER, OUTPUT_LAYER):
            self._prefetch_passthrough(shard_layer, device, prefetch)
            return
        for uri in dict.fromkeys([self.config.output_base_model] + [m.model for _, m in self._participants(shard_layer.layer_number)]):
            prefetch(uri, shard_layer.layer_name, device)

    async def _merge_layer(self, shard_layer: ShardLayer, device: str) -> torch.Tensor:
        number, name = shard_layer.layer_number, shard_layer.layer_name
        if number in (INPUT_LAYER, OUTPUT_LAYER):
            return await self._passthrough(shard_layer, device)
        E._require_cuda(device)
        logger.info(f"Processing layer: {name}")
        base = await self.index_manager.get_tensor(self.config.output_base_model, name, device=device).get()
        parts = self._participants(number)
        if not parts:
            return base
        fts = [await self.index_manager.get_tensor(m.model, name, device=device).get() for _, m in parts]
        out, nonfinite = sparse_merge(self.mode, base, fts, [m.alpha for _, m in parts], self.density, self.scale, self.seed,
                                      name, [i for i, _ in parts])
        pend = _Pending(out, nonfinite, name, [m.model for _, m in parts])
        if self.defer_checks:
            self.pending.append(pend)
        else:
            pend.check()
        return out

    def _finalize(self, tensor: torch.Tensor):
        """Read the non-finite counts of `tensor` (and of every older pending tensor) and raise on any."""
        for i, pend in enumerate(self.pending):
            if pend.out is tensor:
                head, self.pending = self.pending[: i + 1], self.pending[i + 1:]
                for p in head:
                    p.check()
                return


class TiesMerge(_TaskVectorMerge):
    """TIES: per model the top `density` share of the delta by magnitude, sign election, disjoint mean"""
    mode = MODE_TIES
    method = "TIES merging"

    def __init__(self, config: MergeConfig, density: float, scale: float = 1.0, index_manager=None):
        super().__init__(config, density, scale, 0, index_manager)


class DareTiesMerge(_TaskVectorMerge):
    """DARE-TIES: seeded random drop at rate 1 - density with 1 / density rescaling, sign election, disjoint mean"""
    mode = MODE_DARE_TIES
    method = "DARE-TIES merging"

    def _seed_note(self) -> str:
        return f", seed {self.seed}"


class DareLinearMerge(_TaskVectorMerge):
    """DARE-linear: seeded random drop at rate 1 - density with 1 / density rescaling, weighted mean"""
    mode = MODE_DARE_LINEAR
    method = "DARE-linear merging"

    def _seed_note(self) -> str:
        return f", seed {self.seed}"
