"""PEFT LoRA adapters as finetunes: the one module that knows the adapter format.

A PEFT LoRA adapter directory holds `adapter_config.json` and `adapter_model.safetensors`.  Its tensors are keyed by the
module path under `base_model.model.`:

  <prefix><module>.lora_A.weight   [r][in]    low-rank factors of a linear module whose base weight is <module>.weight
  <prefix><module>.lora_B.weight   [out][r]
  <prefix><name>                   a full tensor (`modules_to_save`, trained biases): the finetune's <name> as it is

For every base tensor W of the base the adapter is bound to, the finetune's tensor is
  - with a LoRA pair:      round_to_dtype(W)( fp32(W) + s * (fp32(B) @ fp32(A)) ), formed on the device by `materialize`
                           (csrc/kernels_lora.cu), s = alpha / r or alpha / sqrt(r) with `use_rslora`;
  - with a full tensor:    that tensor;
  - otherwise:             W itself.
`Adapter.bind` checks every key and shape against the base and raises `UnsupportedAdapter` for what it cannot represent.
"""
from __future__ import annotations

import json
import math
import re
from dataclasses import dataclass
from pathlib import Path
from typing import Dict, Optional, Tuple

import torch

CONFIG_FILE = "adapter_config.json"
WEIGHTS_FILE = "adapter_model.safetensors"
KEY_PREFIX = "base_model.model."
_PAIR = re.compile(r"^(?P<module>.+)\.lora_(?P<which>[AB])\.weight$")
_DTYPE_CODE = {torch.float32: 0, torch.bfloat16: 1, torch.float16: 2}


class UnsupportedAdapter(ValueError):
    """An adapter this project cannot apply exactly; the message names the adapter and the reason."""


def is_adapter_dir(path) -> bool:
    """A directory with an adapter config and weights and no full-model index."""
    path = Path(path)
    return ((path / CONFIG_FILE).is_file() and (path / WEIGHTS_FILE).is_file()
            and not (path / "model.safetensors.index.json").exists())


@dataclass(frozen=True)
class Part:
    """How one base tensor's finetuned value is obtained from an adapter.
    kind "lora": from the factors under keys (lora_A key, lora_B key) and `scaling`;
    kind "full": the adapter's tensor under keys[0];  kind "base": the base tensor itself (keys is empty)."""
    kind: str
    keys: Tuple[str, ...] = ()
    scaling: float = 0.0


BASE_PART = Part("base")


def _f32(x: float) -> float:
    return float(torch.tensor(x, dtype=torch.float32))


def scaling_for(config: dict, module: str, r: int) -> float:
    """fp32(alpha / r), or fp32(alpha / sqrt(r)) with use_rslora; alpha is the value of the first `alpha_pattern` key that
    matches `module` as `(.*\\.)?{key}$`, else `lora_alpha`."""
    alpha = config.get("lora_alpha", 8)
    for key, value in (config.get("alpha_pattern") or {}).items():
        if re.match(rf"(.*\.)?{key}$", module):
            alpha = value
            break
    return _f32(alpha / math.sqrt(r) if config.get("use_rslora", False) else alpha / r)


def read_config(directory) -> dict:
    with open(Path(directory) / CONFIG_FILE) as fh:
        return json.load(fh)


class Adapter:
    """One adapter: its config and the (dtype, shape) of every tensor in its weights file, as read from the header."""

    def __init__(self, name: str, config: dict, tensors: Dict[str, Tuple[torch.dtype, tuple]]):
        self.name, self.config, self.tensors = name, config, tensors
        self.base: Optional[str] = None
        self.parts: Dict[str, Part] = {}
        peft_type = str(config.get("peft_type", "")).upper()
        if peft_type != "LORA":
            self._refuse(f"peft_type is {config.get('peft_type')!r}, only LORA adapters are supported")
        if config.get("use_dora", False) or any("lora_magnitude_vector" in k for k in tensors):
            self._refuse("DoRA (use_dora, lora_magnitude_vector) is not supported")
        if config.get("fan_in_fan_out", False):
            self._refuse("fan_in_fan_out (transposed Conv1D factors) is not supported")
        emb = [k for k in tensors if "lora_embedding_A" in k or "lora_embedding_B" in k]
        if emb:
            self._refuse(f"embedding LoRA (lora_embedding_A / lora_embedding_B) is not supported: {emb[0]}")

    def _refuse(self, why: str):
        raise UnsupportedAdapter(f"adapter {self.name}: {why}")

    def bind(self, base: str, base_shapes: Dict[str, tuple]) -> None:
        """Map every adapter key to a base tensor of `base` (a {name: shape} dict) and check the shapes.  Binding again to
        the same base is a no-op; to another base, a refusal."""
        if self.base is not None:
            if self.base != base:
                self._refuse(f"used with two different bases, {self.base} and {base}")
            return
        pairs: Dict[str, Dict[str, str]] = {}
        parts: Dict[str, Part] = {}
        for key in sorted(self.tensors):
            if not key.startswith(KEY_PREFIX):
                self._refuse(f"key {key} does not start with {KEY_PREFIX!r}")
            name = key[len(KEY_PREFIX):]
            m = _PAIR.match(name)
            if m:
                pairs.setdefault(m.group("module"), {})[m.group("which")] = key
                continue
            if name not in base_shapes:
                self._refuse(f"key {key} does not map to a tensor of {base}")
            if tuple(self.tensors[key][1]) != tuple(base_shapes[name]):
                self._refuse(f"{key} has shape {tuple(self.tensors[key][1])}, {base}'s {name} {tuple(base_shapes[name])}")
            parts[name] = Part("full", (key,))
        for module, keys in pairs.items():
            target = module + ".weight"
            if set(keys) != {"A", "B"}:
                self._refuse(f"{module} has lora_{''.join(sorted(keys))} without its other factor")
            if target not in base_shapes:
                self._refuse(f"key {keys['A']} does not map to a tensor of {base} ({target})")
            if target in parts:
                self._refuse(f"{target} has both a LoRA pair and a full tensor")
            shape = tuple(base_shapes[target])
            a_shape, b_shape = tuple(self.tensors[keys["A"]][1]), tuple(self.tensors[keys["B"]][1])
            if (len(shape) != 2 or len(a_shape) != 2 or len(b_shape) != 2 or a_shape[0] < 1 or a_shape[0] != b_shape[1]
                    or a_shape[1] != shape[1] or b_shape[0] != shape[0]):
                self._refuse(f"lora_A {a_shape} / lora_B {b_shape} of {module} do not match {base}'s {target} {shape} "
                             f"(want lora_A [r][{shape[-1]}], lora_B [{shape[0]}][r])")
            parts[target] = Part("lora", (keys["A"], keys["B"]), scaling_for(self.config, module, a_shape[0]))
        self.base, self.parts = base, parts

    def part(self, tensor_name: str) -> Part:
        return self.parts.get(tensor_name, BASE_PART)


def materialize(base: torch.Tensor, lora_A: torch.Tensor, lora_B: torch.Tensor, scaling: float) -> torch.Tensor:
    """The finetuned tensor round_to_dtype(base)(fp32(base) + scaling * fp32(lora_B) @ fp32(lora_A)) on base's CUDA device,
    enqueued on the current stream (csrc/kernels_lora.cu).  base [R][C] in fp32 / bf16 / fp16; lora_A [r][C] and lora_B [R][r]
    in one of those dtypes."""
    from . import _lib
    from . import engine as E

    if base.device.type != "cuda" or lora_A.device != base.device or lora_B.device != base.device:
        raise RuntimeError(f"lora.materialize needs the three tensors on one CUDA device (got {base.device}, "
                           f"{lora_A.device}, {lora_B.device}); there is no CPU path")
    if base.dtype not in _DTYPE_CODE or lora_A.dtype not in _DTYPE_CODE or lora_B.dtype != lora_A.dtype:
        raise NotImplementedError(f"lora.materialize: base and factors in fp32 / bf16 / fp16, factors of one dtype "
                                  f"(got {base.dtype}, {lora_A.dtype}, {lora_B.dtype})")
    if base.ndim != 2 or lora_A.ndim != 2 or lora_B.ndim != 2:
        raise ValueError("lora.materialize: 2-D base and factors")
    R, C = base.shape
    r = lora_A.shape[0]
    if r < 1 or tuple(lora_A.shape) != (r, C) or tuple(lora_B.shape) != (R, r):
        raise ValueError(f"lora.materialize: lora_A {tuple(lora_A.shape)} / lora_B {tuple(lora_B.shape)} do not fit base {(R, C)}")
    base, lora_A, lora_B = base.contiguous(), lora_A.contiguous(), lora_B.contiguous()
    out = torch.empty_like(base)
    if out.numel() == 0:
        return out
    rc = _lib.load().sm_lora_materialize(int(R), int(C), int(r), _DTYPE_CODE[base.dtype], base.data_ptr(),
                                         _DTYPE_CODE[lora_A.dtype], lora_A.data_ptr(), lora_B.data_ptr(), float(scaling),
                                         out.data_ptr(), E._stream(base.device))
    _lib.check(rc, "sm_lora_materialize")
    return out
