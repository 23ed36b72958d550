"""PEFT LoRA adapters as finetunes, host side: key mapping, scaling, the refusals of initialize(), and the directory
rules of LocalSafetensorsIndex.  No GPU: every refusal happens before any tensor data is read or output written."""
import asyncio
import json
import math

import pytest
import torch

from shardmerge_b200 import lora
from shardmerge_b200.config import MergeConfig, MergeModel
from shardmerge_b200.index import LocalSafetensorsIndex
from shardmerge_b200.lora import UnsupportedAdapter
from shardmerge_b200.merge.addition import AdditionMerge
from shardmerge_b200.merge.fast_fourier import FourierMerge
from shardmerge_b200.merge.fourier import FourierMerge as InRamFourierMerge
from shardmerge_b200.merge.taskaddition import TaskAdditionMerge
from tests.lora_util import adapter_tensors, llama_shapes, random_model, write_adapter, write_model

SHAPES = llama_shapes(layers=2)


@pytest.fixture
def storage(tmp_path):
    write_model(tmp_path / "org" / "base", random_model(SHAPES, 0))
    write_model(tmp_path / "org" / "base2", random_model(SHAPES, 1))
    return tmp_path


def _adapter(storage, name, r=8, targets=("q_proj", "v_proj"), full=(), tensors=None, extra=None, **config):
    t = adapter_tensors(SHAPES, targets, r, seed=7, full=full) if tensors is None else tensors
    t.update(extra or {})
    write_adapter(storage / "org" / name, t, r=r, **config)
    return f"org/{name}"


def _fm(storage, models, cls=FourierMerge, out="out"):
    cfg = MergeConfig(finetune_merge=[MergeModel(model=m, base=b) for m, b in models], output_base_model="org/base",
                      output_dir=str(storage / out), storage_dir=str(storage))
    return cls(cfg, index_manager=LocalSafetensorsIndex(cfg.storage_path))


def _bind(storage, uri, base="org/base"):
    im = LocalSafetensorsIndex(storage)
    asyncio.run(im.add_model(base))
    asyncio.run(im.add_model(uri))
    im.bind_adapter(uri, base)
    return im


# ---- key mapping ---------------------------------------------------------------------------------------------------
def test_key_mapping_pairs_full_tensors_and_biases(storage):
    bias = {"base_model.model.model.layers.0.self_attn.q_proj.bias": torch.zeros(128)}
    base = random_model(SHAPES, 0)
    for li in range(2):                                # every layer has the same components (canonical_layer_order)
        base[f"model.layers.{li}.self_attn.q_proj.bias"] = torch.zeros(128, dtype=torch.bfloat16)
    write_model(storage / "org" / "base", base)
    uri = _adapter(storage, "a", full=("lm_head.weight",), extra=bias)
    im = _bind(storage, uri)
    q = im.adapter_part(uri, "model.layers.1.self_attn.q_proj.weight")
    assert q.kind == "lora" and q.keys == ("base_model.model.model.layers.1.self_attn.q_proj.lora_A.weight",
                                          "base_model.model.model.layers.1.self_attn.q_proj.lora_B.weight")
    assert im.adapter_part(uri, "lm_head.weight") == lora.Part("full", ("base_model.model.lm_head.weight",))
    assert im.adapter_part(uri, "model.layers.0.self_attn.q_proj.bias") == \
        lora.Part("full", ("base_model.model.model.layers.0.self_attn.q_proj.bias",))
    assert im.adapter_part(uri, "model.layers.0.self_attn.k_proj.weight") is lora.BASE_PART
    assert im.adapter_part("org/base", "lm_head.weight") is None
    # the adapter reports its base's keys, order and shapes
    assert im.get_model_keys(uri) == im.get_model_keys("org/base")
    assert im.get_layer_order(uri) == im.get_layer_order("org/base")
    assert im.tensor_shapes(uri) == im.tensor_shapes("org/base")


# ---- scaling -------------------------------------------------------------------------------------------------------
def _f32(x):
    return float(torch.tensor(x, dtype=torch.float32))


def test_scaling_lora_alpha_and_rslora():
    assert lora.scaling_for({"lora_alpha": 16}, "model.layers.0.self_attn.q_proj", 8) == 2.0
    assert lora.scaling_for({"lora_alpha": 7}, "m.q_proj", 3) == _f32(7 / 3)
    assert lora.scaling_for({"lora_alpha": 16, "use_rslora": True}, "m.q_proj", 8) == _f32(16 / math.sqrt(8))
    assert lora.scaling_for({"lora_alpha": 5, "use_rslora": True}, "m.q_proj", 320) == _f32(5 / math.sqrt(320))


def test_scaling_alpha_pattern_exact_and_suffix():
    cfg = {"lora_alpha": 16, "alpha_pattern": {"model.layers.1.self_attn.q_proj": 4, "v_proj": 64, "proj": 1}}
    assert lora.scaling_for(cfg, "model.layers.1.self_attn.q_proj", 8) == 0.5        # exact
    assert lora.scaling_for(cfg, "model.layers.0.self_attn.v_proj", 8) == 8.0        # suffix after a dot
    assert lora.scaling_for(cfg, "model.layers.0.self_attn.q_proj", 8) == 2.0        # "proj" is not a dotted suffix of q_proj
    assert lora.scaling_for(cfg, "model.layers.0.mlp.proj", 8) == _f32(1 / 8)
    # the first matching key wins
    assert lora.scaling_for({"lora_alpha": 1, "alpha_pattern": {"q_proj": 2, "self_attn.q_proj": 3}}, "a.self_attn.q_proj", 1) == 2.0


def test_bound_scaling_uses_the_factor_rank(storage):
    uri = _adapter(storage, "a", r=8, lora_alpha=24, alpha_pattern={"layers.1.self_attn.v_proj": 4})
    im = _bind(storage, uri)
    cfg = json.loads((storage / "org" / "a" / "adapter_config.json").read_text())
    cfg["r"] = 99                                      # the config's r is not what scales: lora_A's row count is
    (storage / "org" / "a" / "adapter_config.json").write_text(json.dumps(cfg))
    im2 = _bind(storage, uri)
    for i in (im, im2):
        assert i.adapter_part(uri, "model.layers.0.self_attn.q_proj.weight").scaling == 3.0
        assert i.adapter_part(uri, "model.layers.1.self_attn.v_proj.weight").scaling == 0.5


# ---- refusals from initialize(), before any output ----------------------------------------------------------------
def _refused(storage, models, match, cls=FourierMerge):
    fm = _fm(storage, models, cls)
    with pytest.raises(UnsupportedAdapter, match=match):
        asyncio.run(fm.merge("cuda"))
    assert not (storage / "out").exists()


def test_refuses_non_lora_peft_type(storage):
    _refused(storage, [(_adapter(storage, "ia3", peft_type="IA3"), "org/base")], "org/ia3.*peft_type")


def test_refuses_dora(storage):
    _refused(storage, [(_adapter(storage, "dora", use_dora=True), "org/base")], "org/dora.*DoRA")
    mag = {"base_model.model.model.layers.0.self_attn.q_proj.lora_magnitude_vector": torch.ones(128)}
    _refused(storage, [(_adapter(storage, "dora2", extra=mag), "org/base")], "org/dora2.*DoRA")


def test_refuses_fan_in_fan_out(storage):
    _refused(storage, [(_adapter(storage, "fifo", fan_in_fan_out=True), "org/base")], "org/fifo.*fan_in_fan_out")


def test_refuses_embedding_lora(storage):
    emb = {"base_model.model.model.embed_tokens.lora_embedding_A": torch.zeros(8, 256),
           "base_model.model.model.embed_tokens.lora_embedding_B": torch.zeros(128, 8)}
    _refused(storage, [(_adapter(storage, "emb", extra=emb), "org/base")], "org/emb.*lora_embedding")


@pytest.mark.parametrize("which,shape", [("A", (8, 127)), ("B", (129, 8)), ("B", (128, 7)), ("A", (0, 128))])
def test_refuses_pair_shape_mismatch(storage, which, shape):
    t = adapter_tensors(SHAPES, ("q_proj",), 8, seed=1)
    t[f"base_model.model.model.layers.0.self_attn.q_proj.lora_{which}.weight"] = torch.zeros(shape, dtype=torch.bfloat16)
    _refused(storage, [(_adapter(storage, "bad", tensors=t), "org/base")], "org/bad.*q_proj")


def test_refuses_unmapped_keys(storage):
    for i, extra in enumerate([{"base_model.model.model.layers.0.self_attn.rotary.lora_A.weight": torch.zeros(8, 128),
                                "base_model.model.model.layers.0.self_attn.rotary.lora_B.weight": torch.zeros(128, 8)},
                               {"base_model.model.model.layers.9.input_layernorm.weight": torch.zeros(128)},
                               {"model.layers.0.input_layernorm.weight": torch.zeros(128)},
                               {"base_model.model.model.layers.0.mlp.up_proj.lora_A.weight": torch.zeros(8, 128)}]):
        _refused(storage, [(_adapter(storage, f"u{i}", extra=extra), "org/base")], f"org/u{i}")


def test_refuses_full_tensor_shape_mismatch(storage):
    extra = {"base_model.model.lm_head.weight": torch.zeros(300, 128)}
    _refused(storage, [(_adapter(storage, "head", extra=extra), "org/base")], "org/head.*lm_head")


def test_refuses_one_adapter_with_two_bases(storage):
    uri = _adapter(storage, "a")
    _refused(storage, [(uri, "org/base"), (uri, "org/base2")], "org/a.*two different bases")


def test_refuses_adapter_as_base(storage):
    uri = _adapter(storage, "a")
    _refused(storage, [(uri, "org/base"), (_adapter(storage, "b"), uri)], "org/b.*not a full model")


@pytest.mark.parametrize("cls", [AdditionMerge, TaskAdditionMerge, InRamFourierMerge])
def test_other_strategies_refuse_adapters(storage, cls):
    _refused(storage, [(_adapter(storage, "a"), "org/base")], f"org/a.*{cls.__name__} does not merge LoRA adapters", cls=cls)


def test_valid_adapter_passes_the_architecture_check(storage):
    uri = _adapter(storage, "a", full=("lm_head.weight",))
    fm = _fm(storage, [(uri, "org/base")], AdditionMerge)
    fm.merges_adapters = True                          # the base-class part of initialize(), without FFT plans
    asyncio.run(fm.initialize())
    assert fm.index_manager.is_adapter(uri) and not fm.index_manager.is_adapter("org/base")


# ---- directory rules ----------------------------------------------------------------------------------------------
def test_directory_with_index_stays_a_full_model(storage):
    d = storage / "org" / "both"
    write_model(d, random_model(SHAPES, 3))
    write_adapter(d, adapter_tensors(SHAPES, ("q_proj",), 8, seed=1))
    im = LocalSafetensorsIndex(storage)
    asyncio.run(im.add_model("org/both"))
    assert not im.is_adapter("org/both")
    assert im.get_model_keys("org/both") == set(SHAPES)
    assert im.adapter_part("org/both", "lm_head.weight") is None


def test_directory_without_index_or_adapter_is_not_found(storage):
    (storage / "org" / "empty").mkdir()
    (storage / "org" / "empty" / "adapter_config.json").write_text("{}")      # config without weights: not an adapter
    with pytest.raises(FileNotFoundError):
        asyncio.run(LocalSafetensorsIndex(storage).add_model("org/empty"))
