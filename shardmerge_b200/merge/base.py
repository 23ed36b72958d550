"""MergeTensorsBase -- orchestration with the interface of shard/merge/base.py:96-223.

A strategy implements `_merge_layer(shard_layer, device) -> Tensor`; `merge(device)` walks the
output shards in file-name order, the tensors of a shard in canonical layer order, skips what
an earlier run already wrote (resume, shard/writer.py:93-113) and hands every result to the
writer.  The index manager is duck-typed (shard/index.py:HFMultiModelIndex or
shardmerge_b200.index.*): it needs add_model, model_indexes, get_model_keys, get_layer_order,
get_tensor(model, name, device) -> promise with `await .get()`.
"""
from __future__ import annotations

import logging
from abc import ABC, abstractmethod
from typing import List

import torch

from ..config import MergeConfig, MergeModel
from ..lora import UnsupportedAdapter
from ..writer import ModelWriter, ShardLayer

logger = logging.getLogger(__name__)


class MergeTensorsBase(ABC):
    merges_adapters = False      # True: _merge_layer forms a LoRA adapter's finetuned tensors (index managers with is_adapter)

    def __init__(self, config: MergeConfig, index_manager=None):
        if index_manager is None:
            raise ValueError("shardmerge_b200 strategies need an index_manager (see shardmerge_b200.index)")
        self.config = config
        self.index_manager = index_manager

    @abstractmethod
    def get_readme(self) -> str:
        return "No readme defined"

    @abstractmethod
    async def _merge_layer(self, shard_layer: ShardLayer, device: str) -> torch.Tensor:
        raise NotImplementedError

    async def get_base_output_tensor(self, shard_layer: ShardLayer, device: str) -> torch.Tensor:
        """fp32 copy of the output-base tensor (shard/merge/base.py:117-119)."""
        t = await self.index_manager.get_tensor(self.config.output_base_model, shard_layer.layer_name, device=device).get()
        return t.to(torch.float32)

    async def get_delta_for_models(self, models: List[MergeModel], shard_layer: ShardLayer, device: str,
                                   apply_alpha: bool = True) -> list:
        """fp32(finetune) - fp32(base) per model, optionally x alpha (shard/merge/base.py:121-137).
        The fused path never calls this (the row kernel forms the delta on load); it is kept for
        strategies and callers that want the explicit tensors."""
        out, bases = [], {}
        for m in models:
            if m.base not in bases:
                bases[m.base] = (await self.index_manager.get_tensor(m.base, shard_layer.layer_name, device=device).get()).to(torch.float32)
            ft = (await self.index_manager.get_tensor(m.model, shard_layer.layer_name, device=device).get()).to(torch.float32)
            out.append((ft - bases[m.base]).detach() * (m.alpha if apply_alpha else 1))
        return out

    async def initialize(self):
        im = self.index_manager
        await im.add_model(self.config.output_base_model)
        self.index_doc = im.model_indexes[self.config.output_base_model]
        for m in self.config.finetune_merge:
            await im.add_model(m.base)
            await im.add_model(m.model)
        is_adapter = getattr(im, "is_adapter", None)
        if is_adapter is not None:
            if is_adapter(self.config.output_base_model):
                raise UnsupportedAdapter(f"adapter {self.config.output_base_model}: output_base_model must be a full model")
            for m in self.config.finetune_merge:
                if not is_adapter(m.model):
                    continue
                if not self.merges_adapters:
                    raise UnsupportedAdapter(f"adapter {m.model}: {type(self).__name__} does not merge LoRA adapters; "
                                             f"FourierMerge (merge/fast_fourier.py) does, or merge the materialised checkpoint")
                im.bind_adapter(m.model, m.base)      # the adapter is applied to this entry's base; refusals raise here
        want = im.get_model_keys(self.config.output_base_model)
        for m in self.config.finetune_merge:
            have = im.get_model_keys(m.model)
            if want - have or have - want:
                raise ValueError(f"Model {m.model} architecture mismatch with base model {self.config.output_base_model}\n"
                                 f"Missing keys: {want - have}\nExtra keys: {have - want}")

    def get_writer(self, layer_order: list, **kwargs) -> ModelWriter:
        return ModelWriter(base_index=self.index_doc, output_path=self.config.output_path, layer_order=layer_order,
                           output_astype=self.config.output_astype, **kwargs)

    async def merge(self, device: str):
        await self.initialize()
        layer_order = self.index_manager.get_layer_order(self.config.output_base_model)
        writer = self.get_writer(layer_order)
        if self.pipeline_depth > 0:
            self.defer_checks = True
        try:
            for group in writer.shard_layers():
                await self._process_layers(writer, [sl for sl in group if not sl.written], device)
        except BaseException:
            writer.flush_partial()       # keep what was merged: the next run resumes behind it (shard/writer.py:93-113)
            raise
        finally:
            self.defer_checks = False
        writer.finalize()
        readme = self.get_readme() or "No README defined"
        with open(self.config.output_path / "README.md", "w") as fh:
            fh.write(readme)
        logger.info(f"Merge complete. Output saved to {self.config.output_path}")

    # Strategies whose _merge_layer only ENQUEUES device work (FourierMerge's fused chain) set
    # pipeline_depth > 0: the loop then keeps that many tensors in flight before it settles the
    # oldest one (waits for its device-side status) and hands it to the writer, so the GPU never
    # drains between tensors.  depth 0 = the reference's strictly sequential behaviour.
    pipeline_depth = 0

    def _finalize(self, tensor: torch.Tensor):
        """Make `tensor` (a value `_merge_layer` returned) final before it is handed to the writer.  Strategies
        whose `_merge_layer` only enqueues device work override this: they wait for that tensor's device-side
        status, redo it on another path if the device asked for that, and raise what the reference would raise."""

    def prefetch_layer(self, shard_layer: ShardLayer, device: str):
        """Start the host-to-device copies of the tensors `_merge_layer(shard_layer)` will ask for (override per
        strategy; needs an index manager with `prefetch`, see shardmerge_b200/index.py)."""

    prefetch_depth = 3           # tensors whose uploads may be in flight ahead of the one being merged

    async def _process_layers(self, writer: ModelWriter, shard_layers: List[ShardLayer], device: str):
        current = None
        in_flight = []
        ahead = 0                # shard_layers[:ahead] have had their uploads started
        try:
            for i, current in enumerate(shard_layers):
                while ahead < len(shard_layers) and ahead <= i + self.prefetch_depth:
                    self.prefetch_layer(shard_layers[ahead], device)       # uploads overlap the kernels of tensors i..
                    ahead += 1
                in_flight.append((current, await self._merge_layer(current, device)))
                while len(in_flight) > self.pipeline_depth:
                    done, tensor = in_flight.pop(0)
                    self._finalize(tensor)
                    writer.add_tensor(done.layer_name, tensor)
            while in_flight:
                done, tensor = in_flight.pop(0)
                self._finalize(tensor)
                writer.add_tensor(done.layer_name, tensor)
        except Exception as exc:
            logger.error(f"Error processing {getattr(current, 'layer_name', '?')}: {exc}")
            raise
