"""FourierMerge -- the SLERP-FFT merge strategy with the interface of
shard/merge/fast_fourier.py (FourierMerge :79-276), device-resident.

`_merge_layer(shard_layer, device)` keeps the reference's contract: embed / final norm /
lm_head tensors are passed through from the is_input / is_output model (:104-130); every
other tensor is the pairwise-tree spectral merge of the applicable finetunes' deltas
(:132-257), added onto the output base, NaN -> 0, Inf -> ValueError, cast to bf16 (:269-276).

What differs is where the bytes live: deltas are never materialised (the row-pass kernel
subtracts bf16 base from bf16 finetune on load), spectra and tree intermediates stay in HBM,
and the reference's TensorDiskCache round trips (:46-77, torch.save/torch.load of every delta
and intermediate) have no equivalent.  `name_hash` is kept because the intermediate names show
up in log lines.
"""
from __future__ import annotations

import asyncio
import hashlib
import logging
import os
from typing import List, NamedTuple, Optional

import torch

from .. import engine as E
from ..config import MergeConfig
from ..constants import INPUT_LAYER, OUTPUT_LAYER
from ..tensor.functions import correlated_pairs, retry_on_select_miss
from .base import MergeTensorsBase

logger = logging.getLogger(__name__)


def name_hash(name: str) -> str:
    """First four characters of every '_'-separated part, '::', first 8 hex digits of sha256(name)
    (shard/merge/fast_fourier.py:36-41)."""
    short = "_".join(part[:4] for part in name.split("_"))
    return f"{short}::{hashlib.sha256(name.encode()).hexdigest()[:8]}"


def task_arithmetic(t0: torch.Tensor, t1: torch.Tensor) -> torch.Tensor:
    """t0 + t1 where the signs agree, else t0 (shard/merge/fast_fourier.py:30-34; unused by the merge)."""
    return torch.where(torch.sign(t0) == torch.sign(t1), t0 + t1, t0)


def clamp(value: float, min_value: float, max_value: float) -> float:
    return max(min_value, min(value, max_value))


class TreeStep(NamedTuple):
    """One entry of a round of the pair tree, in the order correlated_pairs yields it (the order of the next round's
    stack).  y = -1: the model at x is carried to the next round unmerged (a_w is its weight, b_w is 0)."""
    x: int
    y: int
    a_w: float
    b_w: float
    cull_pct: float
    last: bool           # the pair of the last round: it gives the merged tensor


def tree_plan(sumsq: List[float], weights: List[float], cull_start_pct: float, target_norm_offset: float):
    """The schedule of the pairwise tree of fast_fourier.py:165-254 -> (fp32 norms, target_norm, rounds of TreeSteps).
    The reference pairs every round by the products of the ORIGINAL norms list (stale after round 1, :180-184), so the
    whole schedule follows from the models' sums of squares of delta and their weights."""
    norms = [E.f32(v ** 0.5) for v in sumsq]
    target_norm = torch.tensor(norms, dtype=torch.float32).mean().item() + target_norm_offset      # fp32 mean, :165
    nt = torch.tensor(norms, dtype=torch.float32)
    rounds, w, cull_pct = [], list(weights), cull_start_pct
    while len(w) > 1:
        n = len(w)
        corr = torch.triu(nt[:n, None] * nt[None, :n], diagonal=1)                                 # fp32 products
        steps = [TreeStep(x, y, w[x], w[y] if y >= 0 else 0.0, cull_pct, n == 2)
                 for x, y, _ in correlated_pairs(corr, way="least")]
        rounds.append(steps)
        w = [s.a_w if s.y < 0 else (s.a_w + s.b_w) / 2.0 for s in steps]
        cull_pct = cull_pct / 2.0                                                                  # :254
    return norms, target_norm, rounds


class _PendingTree:
    """Deferred check of a pair tree: the per-pair handles of engine.pair_merge_async behind the interface of one."""

    def __init__(self, out, parts, layer_name, norms, target_norm):
        self.out, self.parts, self.layer_name = out, parts, layer_name
        self.norms, self.target_norm = norms, target_norm
        self.redo = None
        self.phase_b = None            # enqueues the pair merges once the norms are on the host (FourierMerge._merge_sources_tree)

    def run_phase_b(self):
        fn, self.phase_b = self.phase_b, None
        if fn is not None:
            fn()

    def resolve(self) -> dict:
        self.run_phase_b()
        infos = [p.resolve() for p in self.parts]
        sticky = 0
        flags = [0, 0, 0, 0]
        for i in infos:
            sticky |= i["select_sticky"]
            flags = [f + g for f, g in zip(flags, i["flags"])]
        branch = next((i["branch"] for i in infos if i["branch"] != "slerp"), "slerp")
        return dict(norms=list(self.norms), target_norm=self.target_norm, swap=[i["swap"] for i in infos], branch=branch,
                    branches=[i["branch"] for i in infos], select_sticky=sticky, flags=flags)


class FourierMerge(MergeTensorsBase):
    merges_adapters = True       # a LoRA adapter's finetuned tensor is formed on the device from its factors (lora.py)
    pipeline_depth = 1           # merge(): one tensor stays in flight while the previous one is settled / written
    # Consecutive tensors alternate between `lanes` CUDA streams (each with its own workspace): every kernel of the
    # chain has a latency-bound prologue / epilogue (single-CTA statistics epilogues, launch gaps, tail waves) that
    # a second tensor's kernels fill.  The reference merges strictly one tensor at a time (shard/merge/base.py:215-220).
    lanes = max(1, int(os.environ.get("SHARDMERGE_LANES", "3")))

    def __init__(self, config: MergeConfig, task_add_models: Optional[List[str]] = None,
                 target_norm_offset: float = 1e-10, cull_start_pct: float = 0.20, index_manager=None, **kwargs):
        super().__init__(config, index_manager)
        self.task_add_models = task_add_models or []
        self.target_norm_offset = target_norm_offset
        self.cull_start_pct = cull_start_pct
        self.last_info: dict = {}
        self.pending: list = []          # deferred checks of fused pair merges (resolve_all)
        self.defer_checks = False        # True inside merge(): _merge_layer returns before the check
        self._lane_streams: dict = {}    # device index -> [streams]
        self._lane_next = 0
        self._tree_waiting: list = []    # pair trees whose row passes are enqueued but whose norms have not been read yet
        self.keep_intermediates = False  # tests: keep the tree's fp32 round results in self.last_tree (the step path also keeps
                                         # the last round's when the output base is not bf16: the merged delta before the base)
        self.last_tree: list = []

    def get_readme(self) -> str:
        models = "\n".join(f"- {m.model} (vs {m.base})" for m in self.config.finetune_merge)
        return f"# SLERP-FFT Merged Model\nBase: {self.config.output_base_model}\nModels merged:\n{models}\n"

    async def initialize(self):
        """Index set-up of the base class, then every merged tensor's shape is checked against the FFT plans BEFORE any
        work is done or output written (the reference's torch.fft takes any shape; here an odd last dimension or a prime
        factor above 1021 has no plan, and that should not surface in the middle of a 70B merge)."""
        await super().initialize()
        shapes_of = getattr(self.index_manager, "tensor_shapes", None)
        if shapes_of is None:
            return
        from .. import _lib
        from ..writer import ShardLayer
        lib = _lib.load()
        bad = []
        for name, shape in shapes_of(self.config.output_base_model).items():
            try:
                if ShardLayer(0, "", name, False).layer_number < 0:
                    continue                                   # pass-through tensors are never transformed
            except ValueError:
                continue                                       # unknown names are reported by the writer, as in the reference
            if len(shape) == 0:
                bad.append((name, shape, "a 0-d tensor has nothing to transform"))
                continue
            R, C = (1, shape[0]) if len(shape) == 1 else (shape[-2], shape[-1])
            if len(shape) == 2 and C % 2 == 1 and R % 2 == 0:
                R, C = C, R                                    # merged as its transpose (merge_sources)
            stack = 1
            for d in shape[:-2]:
                stack *= d
            # the slices' column sweeps need a plan for [R][C]; rows and statistics one for all stack * R rows
            for rows in {int(R), int(R) * int(stack)}:
                plan = lib.sm_plan_create(rows, int(C))
                if not plan:
                    bad.append((name, shape, lib.sm_last_error().decode()))
                    break
                lib.sm_plan_destroy(plan)
        if bad:
            lines = "\n".join(f"  {n} {tuple(s)}: {why}" for n, s, why in bad[:20])
            raise E.UnsupportedShape(f"{len(bad)} tensors of {self.config.output_base_model} cannot be merged on the sm_100a "
                                     f"FFT path:\n{lines}")

    # -------------------------------------------------------------------------------------
    def prefetch_layer(self, shard_layer, device: str):
        prefetch = getattr(self.index_manager, "prefetch", None)
        if prefetch is None or not str(device).startswith("cuda"):
            return
        number, name = shard_layer.layer_number, shard_layer.layer_name
        if number in (INPUT_LAYER, OUTPUT_LAYER):
            self._prefetch_passthrough(shard_layer, device, prefetch)
            return
        wanted = [self.config.output_base_model]
        for m in self.config.finetune_merge:
            if m.use_layer_index(number):
                wanted += [m.base, m.model]
        for uri in dict.fromkeys(wanted):
            prefetch(uri, name, device)

    async def _merge_layer(self, shard_layer, device: str) -> torch.Tensor:
        number = shard_layer.layer_number
        if number in (INPUT_LAYER, OUTPUT_LAYER):
            return await self._passthrough(shard_layer, device)

        dev = E._require_cuda(device)
        name = shard_layer.layer_name
        models = [m for m in self.config.finetune_merge if m.use_layer_index(number)]
        preload = getattr(self.index_manager, "preload_tensor", None)
        if preload is not None:
            await asyncio.gather(*[preload(m.model, name) for m in models])

        async def fetch(model_name):
            return await self.index_manager.get_tensor(model_name, name, device=device).get()

        base_cache: dict = {}
        sources: List[E.Source] = []
        for m in models:
            if m.base not in base_cache:
                base_cache[m.base] = await fetch(m.base)
            part = self._adapter_part(m.model, name)
            ft = await fetch(m.model) if part is None else await self._adapter_tensor(m.model, part, base_cache[m.base], device)
            sources.append(E.make_source(base_cache[m.base], ft, weight=m.alpha, name=m.model))
        base_out = base_cache.get(self.config.output_base_model)
        if base_out is None:
            base_out = await fetch(self.config.output_base_model)
        return self.merge_sources(sources, base_out, dev, layer_name=name, defer=self.defer_checks)

    def _finalize(self, tensor: torch.Tensor):
        """Resolve the deferred check of `tensor` (and of every older deferred tensor): wait for its scalar block,
        redo it step by step if the device chose another branch, raise on Inf.  Pass-through and step-path tensors
        never enter `self.pending` and are final already.  The handle is found by identity, not by position:
        `_process_layers` interleaves fused, pass-through and step-path tensors."""
        for i, pend in enumerate(self.pending):
            if pend.out is tensor:
                head, self.pending = self.pending[: i + 1], self.pending[i + 1:]
                for p in head:
                    if p in self._tree_waiting:
                        self._tree_waiting.remove(p)
                    self._resolve(p)
                return

    # -------------------------------------------------------------------------------------
    def merge_sources(self, sources: List[E.Source], base_out: torch.Tensor, dev, layer_name: str = "",
                      safe_select: bool = False, defer: bool = False) -> torch.Tensor:
        """The regular-layer part of _merge_layer (fast_fourier.py:147-276) on device tensors.

        Two bf16 finetunes on a bf16 base take the fused chain (csrc/pipeline.cu): everything is
        enqueued from one C call and no host synchronisation happens until the scalar block is
        checked -- right away (defer=False) or later through resolve_all() (defer=True: the returned
        tensor is valid once resolve_all() has returned)."""
        for src in sources:
            shp = tuple(src.x32.shape) if src.x32 is not None else tuple(src.base.shape)
            if src.x32 is None and tuple(src.ft.shape) != shp:
                raise ValueError(f"finetune / base shape mismatch for {layer_name}: {tuple(src.ft.shape)} vs {shp}")
            if int(torch.tensor(shp).prod()) != base_out.numel():
                raise ValueError(f"tensor shape mismatch for {layer_name}: {shp} vs output base {tuple(base_out.shape)}")
        if base_out.ndim == 2 and base_out.shape[1] % 2 == 1 and base_out.shape[0] % 2 == 0:
            # The packed real row transform needs an even row length.  fft2(X^T) = fft2(X)^T, and everything between the two
            # transforms is element-wise or a statistic over all bins, so an [R][odd C] tensor is merged as its [C][R]
            # transpose (contiguous copies: a rare shape, no LLM weight has it) and the result transposed back.
            tr = lambda x: None if x is None else x.t().contiguous()
            t_sources = [E.Source(base=tr(sr.base), ft=tr(sr.ft), x32=tr(sr.x32), weight=sr.weight, name=sr.name) for sr in sources]
            merged_t = self.merge_sources(t_sources, tr(base_out), dev, layer_name, safe_select, defer=False)
            for sr, ts in zip(sources, t_sources):
                sr.norm = ts.norm
            return merged_t.t().contiguous()
        all_bf16 = (not safe_select and base_out.dtype == torch.bfloat16 and base_out.ndim in (1, 2)
                    and all(src.is_bf16 for src in sources))
        is_tree = all_bf16 and 3 <= len(sources) <= 120
        if self._tree_waiting and not is_tree:
            # a pair tree whose norms have not been read yet keeps its row spectra in its lane's workspace: enqueue its
            # pair merges before anything else may be given that lane
            waiting, self._tree_waiting = self._tree_waiting, []
            for pend in waiting:
                pend.run_phase_b()
        if is_tree:
            return self._merge_sources_tree(sources, base_out, dev, layer_name, defer)
        fused_ok = len(sources) == 2 and all_bf16
        if not fused_ok:
            return self._merge_sources_steps(sources, base_out, dev, layer_name, safe_select)
        R, C = E.shape_rc(base_out)
        out = torch.empty(base_out.shape, dtype=torch.bfloat16, device=dev)
        a_w, b_w = sources[0].weight, sources[1].weight
        base_c = base_out.contiguous()
        # on a lane the caller's stream is not made to wait for the chain -- whoever consumes `out` does so after
        # resolve (a host-side wait for the lane's last event)
        ws, lane = self._lane_workspace(dev, defer, R, C, 2, [out, base_c] + [t for src in sources for t in (src.base, src.ft)])
        with torch.cuda.stream(lane):
            pend = E.pair_merge_async(ws, sources[0], sources[1], base_c, out, t=a_w / (a_w + b_w), t_sum=1.0,
                                      cutoff_pct=0.08, cull_pct=self.cull_start_pct,
                                      target_norm_offset=self.target_norm_offset, layer_name=layer_name)
        pend.redo = lambda: self._merge_sources_steps(sources, base_out, dev, layer_name, False)
        if defer:
            self.pending.append(pend)
            return out
        self._resolve(pend)
        return out

    def _lane_workspace(self, dev, defer: bool, R: int, C: int, n_spectra: int, tensors):
        """(workspace, stream) for one tensor's fused chains.  Deferred with several lanes, consecutive tensors take turns
        on the lane streams: the lane waits for the caller's stream (the inputs and a new workspace are ready there) and
        `tensors` are recorded on it, so their memory is not reused before the lane is done.  Otherwise: lane 0 on the
        caller's stream."""
        caller = torch.cuda.current_stream(dev)
        lane_i, lane = 0, caller
        if self.lanes > 1 and defer:
            streams = self._lane_streams.get(dev.index)
            if streams is None:
                streams = self._lane_streams[dev.index] = [torch.cuda.Stream(device=dev) for _ in range(self.lanes)]
            lane_i = self._lane_next % self.lanes
            self._lane_next += 1
            lane = streams[lane_i]
        ws = E.get_workspace(R, C, dev, n_spectra=n_spectra, lane=lane_i)
        if lane is not caller:
            lane.wait_event(caller.record_event())
            for t in tensors:
                t.record_stream(lane)
        return ws, lane

    # -------------------------------------------------------------------------------------
    def _merge_sources_tree(self, sources: List[E.Source], base_out: torch.Tensor, dev, layer_name: str = "",
                            defer: bool = False) -> torch.Tensor:
        """Three or more bf16 finetunes: the pairwise tree of fast_fourier.py:171-254 with every pair merge on the fused
        chain.  One host read per tensor -- the models' norms, which pair them up (correlated_pairs over norm products,
        :180-186; later rounds keep using the ORIGINAL norms list, the reference's stale-norms quirk) and give
        target_norm (:165).  Round 1 merges row spectra that are already in the workspace into fp32 intermediates,
        later rounds read fp32 tensors, the last pair writes base + merged as bf16; role / branch decisions of every
        pair are made on the device and checked afterwards (a non-SLERP branch anywhere redoes the tensor step by step)."""
        R, C = E.shape_rc(base_out)
        M = len(sources)
        out = torch.empty(base_out.shape, dtype=torch.bfloat16, device=dev)
        base_c = base_out.contiguous()
        ws, lane = self._lane_workspace(dev, defer, R, C, M, [out, base_c] + [t for src in sources for t in (src.base, src.ft)])
        # ---- phase A (enqueue only): every model's row pass, the sums of squares on their way to pinned host memory
        with torch.cuda.stream(lane):
            sums = torch.zeros(M, dtype=torch.float64, device=dev)
            for i, src in enumerate(sources):
                E.fwd_rows_ptr(ws, i, src, sums.data_ptr() + 8 * i)
            slot = E.take_pinned_slot()                       # pinned landing zone from the pool (no cudaHostAlloc per tensor)
            sums_host = slot[: 8 * M].view(torch.float64)
            sums_host.copy_(sums, non_blocking=True)
            sums_ready = torch.cuda.Event()
            sums_ready.record(lane)
        pend = _PendingTree(out, [], layer_name, None, None)

        # ---- phase B: the one host wait (norms), pairing on the host, every pair merge as a fused chain on the lane
        def phase_b():
            sums_ready.synchronize()
            sumsq = sums_host.tolist()
            E.give_pinned_slot(slot)
            norms, target_norm, rounds = tree_plan(sumsq, [src.weight for src in sources], self.cull_start_pct,
                                                   self.target_norm_offset)
            pend.norms, pend.target_norm = norms, target_norm
            with torch.cuda.stream(lane):
                # stack entry: (source, slot holding its row spectrum or None, sum of squares or None)
                stack = [(src, i, sumsq[i]) for i, src in enumerate(sources)]
                kept = []
                for steps in rounds:
                    nxt = []
                    for st in steps:
                        if st.y < 0:
                            nxt.append((stack[st.x][0], None, None))    # carried over; its rows are redone when it is paired
                            continue
                        (sa, slot_a, ss_a), (sb, slot_b, ss_b) = stack[st.x], stack[st.y]
                        rows_done = slot_a is not None and slot_b is not None
                        res = out if st.last else torch.empty((R, C), dtype=torch.float32, device=dev)
                        pend.parts.append(E.pair_merge_async(
                            ws, sa, sb, base_c, res, t=st.a_w / (st.a_w + st.b_w), t_sum=1.0, cutoff_pct=0.08,
                            cull_pct=st.cull_pct, target_norm_offset=self.target_norm_offset, layer_name=layer_name,
                            slots=(slot_a, slot_b) if rows_done else (0, 1), rows_done=rows_done,
                            sumsq=(ss_a, ss_b) if rows_done else None, target_norm=target_norm))
                        if not st.last:
                            inter = E.Source(x32=res, weight=(st.a_w + st.b_w) / 2.0, name=name_hash(f"{sa.name}_{sb.name}"))
                            nxt.append((inter, None, None))
                            if self.keep_intermediates:
                                kept.append((sa.name, sb.name, res))
                    stack = nxt
            if self.keep_intermediates:
                self.last_tree = kept

        pend.phase_b = phase_b
        pend.redo = lambda: self._merge_sources_steps(sources, base_out, dev, layer_name, False)
        if defer:
            # The host wait for this tensor's norms is put off until the NEXT tree tensor's row passes are enqueued (on
            # another lane), so the GPU has work while the host waits; at most one tensor waits (its row spectra occupy its
            # lane's workspace until its chains are enqueued, and the lanes take turns).
            self._tree_waiting.append(pend)
            while len(self._tree_waiting) > (1 if self.lanes > 1 else 0):
                self._tree_waiting.pop(0).run_phase_b()
            self.pending.append(pend)
            return out
        pend.run_phase_b()
        self._resolve(pend)
        return out

    def _resolve(self, pend):
        info = pend.resolve()
        if info["branch"] != "slerp" or info["select_sticky"] != 0:
            # the device found another branch (or a select window missed): the step-by-step path decides
            if info["select_sticky"] != 0:
                logger.warning(f"select window miss on {pend.layer_name}; re-running step by step")
            pend.out.copy_(pend.redo().reshape(pend.out.shape))
            return
        self.last_info = dict(branches=info.get("branches", ["slerp"]), layer=pend.layer_name, norms=info["norms"],
                              target_norm=info["target_norm"], flags=info["flags"], swap=info["swap"])
        if info["flags"][1] > 0:
            raise ValueError("Inf in ifft output")                          # functions.py:215-217
        if info["flags"][3] > 0:
            raise ValueError(f"Inf in merged tensor for {pend.layer_name}")  # fast_fourier.py:273-274

    def resolve_all(self):
        """Check every deferred fused merge (one wait per tensor, all already in flight)."""
        pending, self.pending = self.pending, []
        waiting, self._tree_waiting = self._tree_waiting, []
        for pend in waiting:                      # enqueue what is still held back, oldest first, before any wait
            pend.run_phase_b()
        for pend in pending:
            self._resolve(pend)

    def _merge_sources_steps(self, sources: List[E.Source], base_out: torch.Tensor, dev, layer_name: str = "",
                             safe_select: bool = False) -> torch.Tensor:
        """Step-by-step path: any number of models, any branch, host decisions between the stages."""
        if len(sources) == 0:
            raise IndexError("list index out of range")      # what the reference does with no applicable model
        return retry_on_select_miss(lambda safe: self._steps_pass(sources, base_out, dev, layer_name, safe),
                                    f"on {layer_name}", safe_select)

    def _steps_pass(self, sources: List[E.Source], base_out: torch.Tensor, dev, layer_name: str, safe_select: bool):
        """One run of the step path -> (merged tensor or None, sticky status of its order statistics)."""
        R, C = E.shape_rc(base_out)              # a tensor with leading dimensions is a stack of slices: all its rows
        base_bf16 = base_out if base_out.dtype == torch.bfloat16 else None
        # its own workspace (lane "steps"): a redo or a 1 / 3+ model tensor runs on the caller's stream while fused
        # chains of the same shape may still be in flight on the lane streams with the lane workspaces
        ws = E.ws_for(base_out, dev, n_spectra=max(2, len(sources)), safe_select=safe_select, lane="steps")
        ws.ctl.zero_()
        info = dict(branches=[], layer=layer_name)
        self.last_info = info

        # row passes of every model: delta, row FFT, sum of squares -> norms in one read-back
        extra = torch.zeros(max(len(sources), 2), dtype=torch.float64, device=dev)
        for i, s in enumerate(sources):
            E.fwd_rows_ptr(ws, i, s, extra.data_ptr() + 8 * i)
        norms, target_norm, rounds = tree_plan(extra.to("cpu").tolist()[: len(sources)], [s.weight for s in sources],
                                               self.cull_start_pct, self.target_norm_offset)
        for s, n in zip(sources, norms):
            s.norm = n
        info["norms"] = list(norms)
        info["target_norm"] = target_norm

        if len(sources) == 1:
            # loop skipped: result = raw delta, alpha ignored (fast_fourier.py:171,256-257)
            return _finish_elementwise(sources[0], None, 1.0, 0.0, 1.0, base_out, ws), 0

        # stack entries: (source, slot of its row spectrum or None)
        stack = [(s, i) for i, s in enumerate(sources)]
        out_final: Optional[torch.Tensor] = None
        kept = []
        for steps in rounds:
            nxt = []
            for st in steps:
                if st.y < 0:
                    nxt.append(stack[st.x])
                    continue
                (sa, slot_a), (sb, slot_b) = stack[st.x], stack[st.y]
                a_w, b_w = st.a_w, st.b_w
                # intermediates of an earlier round have no row spectrum yet: run their row pass into a
                # slot nobody in the current stack still needs (norm_a/norm_b of :209-210 come with it)
                busy = {sl for _, sl in stack if sl is not None} | {sl for _, sl in nxt if sl is not None}
                if slot_a is None:
                    slot_a = next(i for i in range(ws.n_spectra) if i not in busy)
                    busy.add(slot_a)
                    sa.norm = _rows_and_norm(ws, slot_a, sa)
                if slot_b is None:
                    slot_b = next(i for i in range(ws.n_spectra) if i not in busy)
                    busy.add(slot_b)
                    sb.norm = _rows_and_norm(ws, slot_b, sb)
                na, nb = sa.norm, sb.norm
                if abs(na) < abs(nb):                          # larger norm becomes `a`; weights stay put (:212-215)
                    sa, sb, slot_a, slot_b, na, nb = sb, sa, slot_b, slot_a, nb, na
                cnorm_a, cnorm_b = abs(na / target_norm), abs(nb / target_norm)
                n_ratio = cnorm_b / (cnorm_a + 1e-10)
                final = st.last
                out = (torch.empty((R, C) if base_out.ndim >= 2 else (C,), dtype=torch.bfloat16, device=dev)
                       if (final and base_bf16 is not None)
                       else torch.empty((R, C) if base_out.ndim >= 2 else (C,), dtype=torch.float32, device=dev))
                if cnorm_a < 1e-6:                             # :223-225  merged = a + b
                    info["branches"].append("add")
                    merged = _pair_elementwise(sa, sb, 1.0, 1.0, 1.0, final, base_out, ws, out)
                elif cnorm_b < 1e-6 or n_ratio < 0.1:          # :226-232  arithmetic-FFT
                    info["branches"].append("arith")
                    norm_scale = target_norm / na
                    weight_scale = b_w / (a_w + 1e-10)
                    # FFT is linear: a*s and (b*w)*s scale the spectra instead of the inputs
                    E.spectral_pair(ws, slot_a, slot_b, scale0=E.f32(norm_scale),
                                    scale1=E.f32(E.f32(weight_scale) * E.f32(norm_scale)), mode="arith", t=1.0,
                                    agreement=True, out_scale=1.0, base=base_bf16 if final else None, out=out,
                                    check_ifft=False)
                    merged = out
                    logger.info(f"Arithmetic-FFT Merged {sb.name} x {weight_scale} on to {sa.name} x {norm_scale}")
                else:                                          # :233-244  SLERP-FFT
                    a_prop = a_w / (a_w + b_w)
                    branch = _slerp_pair(ws, slot_a, slot_b, sa, sb, na, nb, a_prop, st.cull_pct, target_norm,
                                         base_bf16 if final else None, out, final, base_out)
                    info["branches"].append(branch)
                    merged = out
                    logger.info(f"SLERP-FFT Merged {sa.name} and {sb.name} with weight {a_prop}")
                if final and merged.dtype == torch.bfloat16:
                    out_final = merged
                    nxt.append((None, None))
                else:
                    inter = E.Source(x32=merged.reshape(R, C) if merged.ndim == 1 else merged,
                                     weight=(a_w + b_w) / 2.0, name=name_hash(f"{sa.name}_{sb.name}"))
                    nxt.append((inter, None))
                    kept.append((sa.name, sb.name, inter.x32))
            stack = nxt
        if self.keep_intermediates:
            self.last_tree = kept

        _, _, flags, _ = ws.read_ctl()
        info["flags"] = [int(v) for v in flags]
        if ws.select_sticky() != 0:
            return None, ws.select_sticky()
        if int(flags[1]) > 0:
            raise ValueError("Inf in ifft output")             # functions.py:215-217
        if out_final is None:
            # non-bf16 base or an FFT-free last pair: finish with torch ops exactly as :269-276
            res = stack[0][0].x32.reshape(base_out.shape)
            res = base_out.to(torch.float32) + res
            res = torch.where(torch.isnan(res), torch.zeros_like(res), res)
            if torch.any(torch.isinf(res)):
                raise ValueError(f"Inf in merged tensor for {layer_name}")
            return res.to(torch.bfloat16), 0
        if int(flags[3]) > 0:
            raise ValueError(f"Inf in merged tensor for {layer_name}")   # fast_fourier.py:273-274
        return out_final.reshape(base_out.shape), 0


# ------------------------------------------------------------------------------------------
def _rows_and_norm(ws: E.Workspace, slot: int, src: E.Source) -> float:
    acc = torch.zeros(1, dtype=torch.float64, device=ws.plan.device)
    E.fwd_rows_ptr(ws, slot, src, acc.data_ptr())
    return E.f32(acc.item() ** 0.5)


def _slerp_pair(ws, slot_a, slot_b, sa, sb, na, nb, t, cull_pct, target_norm, base_bf16, out, final, base_out) -> str:
    """merge_tensors_fft2_slerp as called at fast_fourier.py:235-243 (t_sum=1, cutoff 0.08), x target_norm."""
    if nb < 1e-4 or na < 1e-4:
        # functions.py:184-190: returns the normalised v0 unchanged
        src = sa
        scale = E.inv_norm_f32(na)
        x = src.delta_f32() * scale if na != 0 else src.delta_f32()
        res = x * E.f32(target_norm)
        _store(res, final, base_out, out)
        return "slerp-early"
    ratio = nb / (na + 1e-10)
    if ratio < 0.1:
        # functions.py:199-202 (unreachable from _merge_layer, which required n_ratio >= 0.1)
        x = sa.delta_f32() * E.inv_norm_f32(na) + (sb.delta_f32() * E.inv_norm_f32(nb)) * E.f32(t)
        _store(x * E.f32(target_norm), final, base_out, out)
        return "slerp-linear"
    E.spectral_pair(ws, slot_a, slot_b, scale0=E.inv_norm_f32(na), scale1=E.inv_norm_f32(nb), mode="slerp", t=t,
                    t_sum=1.0, cutoff_pct=0.08, cull_pct=cull_pct, out_scale=E.f32(target_norm),
                    base=base_bf16, out=out, check_ifft=True)
    return "slerp"


def _store(res32: torch.Tensor, final: bool, base_out: torch.Tensor, out: torch.Tensor):
    res32 = res32.reshape(out.shape)
    if out.dtype == torch.bfloat16:
        y = base_out.to(torch.float32).reshape(out.shape) + res32
        y = torch.where(torch.isnan(y), torch.zeros_like(y), y)
        if torch.any(torch.isinf(y)):
            raise ValueError("Inf in merged tensor")
        out.copy_(y.to(torch.bfloat16))
    else:
        out.copy_(res32)


def _pair_elementwise(sa, sb, ca, cb, scale, final, base_out, ws, out):
    """merged = ca*a + cb*b (FFT-free branches)."""
    if final and out.dtype == torch.bfloat16 and sa.is_bf16 and sb.is_bf16:
        E.delta_axpby_bf16(base_out, sa, ca, sb, cb, scale, out, ws.flags)
        return out
    # a stacked source's delta keeps its leading dimensions, a tree intermediate is one [R][C] matrix
    res = (sa.delta_f32().reshape(out.shape) * ca + sb.delta_f32().reshape(out.shape) * cb) * scale
    _store(res, final, base_out, out)
    return out


def _finish_elementwise(sa, sb, ca, cb, scale, base_out, ws):
    out = torch.empty_like(base_out, dtype=torch.bfloat16)
    if sa.is_bf16 and base_out.dtype == torch.bfloat16:
        E.delta_axpby_bf16(base_out, sa, ca, None, 0.0, scale, out, ws.flags)
        _, _, flags, _ = ws.read_ctl()
        if int(flags[3]) > 0:
            raise ValueError("Inf in merged tensor")
        return out
    _store(sa.delta_f32() * ca, True, base_out, out)
    return out
