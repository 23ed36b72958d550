"""Synthetic Llama-shaped models and PEFT LoRA adapters on disk, for the adapter tests."""
from __future__ import annotations

import json
import re
from pathlib import Path

import torch
from safetensors.torch import save_file

PROJ = ("self_attn.q_proj", "self_attn.k_proj", "self_attn.v_proj", "self_attn.o_proj",
        "mlp.gate_proj", "mlp.up_proj", "mlp.down_proj")


def llama_shapes(layers: int = 2, H: int = 128, KV: int = 64, I: int = 256, V: int = 256) -> dict:
    out = {"model.embed_tokens.weight": (V, H)}
    proj = {"self_attn.q_proj": (H, H), "self_attn.k_proj": (KV, H), "self_attn.v_proj": (KV, H), "self_attn.o_proj": (H, H),
            "mlp.gate_proj": (I, H), "mlp.up_proj": (I, H), "mlp.down_proj": (H, I)}
    for li in range(layers):
        for p in PROJ:
            out[f"model.layers.{li}.{p}.weight"] = proj[p]
        out[f"model.layers.{li}.input_layernorm.weight"] = (H,)
        out[f"model.layers.{li}.post_attention_layernorm.weight"] = (H,)
    out["model.norm.weight"] = (H,)
    out["lm_head.weight"] = (V, H)
    return out


def random_model(shapes: dict, seed: int, dtype=torch.bfloat16, scale: float = 0.02) -> dict:
    g = torch.Generator().manual_seed(seed)
    return {n: (scale * torch.randn(s, generator=g)).to(dtype) for n, s in shapes.items()}


def write_model(directory: Path, tensors: dict):
    """One shard per transformer layer plus one for the rest, and model.safetensors.index.json."""
    directory.mkdir(parents=True, exist_ok=True)
    shards: dict = {}
    for name, t in tensors.items():
        m = re.match(r"model\.layers\.(\d+)\.", name)
        shards.setdefault(f"model-layer{int(m.group(1)):05d}.safetensors" if m else "model-misc.safetensors", {})[name] = t
    wm = {}
    for shard, blob in shards.items():
        save_file({k: v.contiguous() for k, v in blob.items()}, str(directory / shard), metadata={"format": "pt"})
        wm.update({k: shard for k in blob})
    (directory / "model.safetensors.index.json").write_text(json.dumps({"metadata": {}, "weight_map": wm}))


def adapter_tensors(shapes: dict, targets, r: int, seed: int, dtype=torch.bfloat16, full=(), base=None) -> dict:
    """PEFT-keyed factors for every 2-D tensor whose module name ends with one of `targets`, drawn so that
    scaling * B @ A is a few percent of a 0.02-scale base; `full` names get a whole tensor (modules_to_save)."""
    g = torch.Generator().manual_seed(seed)
    out = {}
    for name, shape in shapes.items():
        module = name[: -len(".weight")]
        if len(shape) == 2 and any(module.endswith(t) for t in targets):
            R, C = shape
            out[f"base_model.model.{module}.lora_A.weight"] = (torch.randn((r, C), generator=g) / C ** 0.5).to(dtype)
            out[f"base_model.model.{module}.lora_B.weight"] = (1e-3 * torch.randn((R, r), generator=g)).to(dtype)
    for name in full:
        src = base[name].float() if base is not None else torch.zeros(shapes[name])
        out[f"base_model.model.{name}"] = (src + 0.01 * torch.randn(shapes[name], generator=g)).to(dtype)
    return out


def write_adapter(directory: Path, tensors: dict, r: int = 16, alpha: float = 32.0, **config):
    directory.mkdir(parents=True, exist_ok=True)
    cfg = {"peft_type": "LORA", "r": r, "lora_alpha": alpha, "base_model_name_or_path": "some-hub/quantised-variant",
           "target_modules": sorted({k.split(".lora_")[0].rsplit(".", 1)[-1] for k in tensors if ".lora_" in k}),
           "use_rslora": False, "use_dora": False, "fan_in_fan_out": False}
    cfg.update(config)
    (directory / "adapter_config.json").write_text(json.dumps(cfg))
    save_file({k: v.contiguous() for k, v in tensors.items()}, str(directory / "adapter_model.safetensors"))
