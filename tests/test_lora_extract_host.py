"""Extracting a LoRA adapter from two checkpoints, without a GPU: the refusals, the adapter files `lora.save_adapter`
writes, and the fp64 prototype of the randomized SVD that the GPU results are compared against."""
import asyncio
import json

import pytest
import torch
from safetensors import safe_open

from shardmerge_b200 import extract, lora
from shardmerge_b200.index import LocalSafetensorsIndex
from tests.lora_util import llama_shapes, random_model, write_adapter, write_model


# ---- the reference: the algorithm of extract._factorize in fp64 on the CPU -------------------------------------------
def prototype(delta: torch.Tensor, om: torch.Tensor, r: int, power_iters: int = 2):
    """lora_A [r'][C], lora_B [R][r'] and the singular values of Bm, in fp64, for Δ `delta` and test matrix `om`."""
    delta, om = delta.double(), om.double()
    R, C = delta.shape
    rr = min(r, R, C)

    def orth(Y):
        return torch.linalg.qr(Y).Q

    Y = delta @ om
    for _ in range(power_iters):
        Q = orth(Y)
        Y = delta @ orth((Q.T @ delta).T)
    Q = orth(Y)
    Qb, Rb = torch.linalg.qr((Q.T @ delta).T)
    Us, S, Vh = torch.linalg.svd(Rb.T)
    root = S[:rr].sqrt()
    return root[:, None] * (Vh[:rr] @ Qb.T), (Q @ Us[:, :rr]) * root, S


def spectrum_matrix(R: int, C: int, kind: str, seed: int) -> torch.Tensor:
    """fp64 [R][C] with singular values 1/i ("inv"), 0.9^i ("geo") or those of a Gaussian matrix ("gauss")."""
    g = torch.Generator().manual_seed(seed)
    if kind == "gauss":
        return torch.randn((R, C), generator=g, dtype=torch.float64)
    n = min(R, C)
    i = torch.arange(1, n + 1, dtype=torch.float64)
    s = 1.0 / i if kind == "inv" else 0.9 ** i
    U = torch.linalg.qr(torch.randn((R, n), generator=g, dtype=torch.float64)).Q
    V = torch.linalg.qr(torch.randn((C, n), generator=g, dtype=torch.float64)).Q
    return (U * s) @ V.T


# residual of the prototype over the optimal sqrt(Σ_{i>r} σ_i²), measured on the shapes below at r = 16 and 64 with the
# default oversample 8 and 2 power iterations: at most 1.0075 (1/i), 1.00002 (0.9^i), 1.017 (Gaussian)
NEAR_OPTIMAL = {"inv": 1.02, "geo": 1.001, "gauss": 1.03}


@pytest.mark.parametrize("r", [16, 64])
@pytest.mark.parametrize("kind", sorted(NEAR_OPTIMAL))
@pytest.mark.parametrize("shape", [(512, 2048), (4096, 4096)], ids=lambda s: f"{s[0]}x{s[1]}")
def test_prototype_near_optimal(shape, kind, r):
    R, C = shape
    delta = spectrum_matrix(R, C, kind, seed=R + r)
    A, B, S = prototype(delta, extract.omega(f"spectrum.{kind}", C, min(r + 8, R, C)), r)
    tail = float(torch.linalg.svdvals(delta)[r:].square().sum().sqrt())
    got = float((delta - B @ A).norm())
    assert tail <= got * (1 + 1e-12) and got <= NEAR_OPTIMAL[kind] * tail, (got, tail)
    # the residual formula from the singular values agrees with the direct one
    assert abs(extract._residual(float(delta.square().sum()), S, r) - got / float(delta.norm())) < 1e-6


def test_prototype_recovers_exact_rank():
    g = torch.Generator().manual_seed(3)
    L = torch.randn((300, 8), generator=g, dtype=torch.float64) @ torch.randn((8, 500), generator=g, dtype=torch.float64)
    A, B, _ = prototype(L, extract.omega("x", 500, 16), 8)
    assert float((L - B @ A).norm() / L.norm()) < 1e-12


def test_omega_depends_on_name_and_seed_only():
    a = extract.omega("model.layers.0.mlp.up_proj.weight", 64, 9)
    assert a.dtype == torch.float32 and a.shape == (64, 9)
    assert torch.equal(a, extract.omega("model.layers.0.mlp.up_proj.weight", 64, 9))
    assert not torch.equal(a, extract.omega("model.layers.1.mlp.up_proj.weight", 64, 9))
    assert not torch.equal(a, extract.omega("model.layers.0.mlp.up_proj.weight", 64, 9, seed=1))
    assert abs(float(a.std()) - 1.0) < 0.15


# ---- refusals: before any device work, nothing created at output_dir ------------------------------------------------
SHAPES = llama_shapes(layers=1, H=32, KV=16, I=64, V=64)


@pytest.fixture
def pair(tmp_path):
    base = random_model(SHAPES, 0)
    write_model(tmp_path / "base", base)
    write_model(tmp_path / "model", {n: (t.float() + 0.01).to(t.dtype) for n, t in base.items()})
    return tmp_path


def _refused(root, exc, match, base="base", model="model", out="out", **kw):
    kw.setdefault("rank", 4)
    with pytest.raises(exc, match=match):
        extract.extract_lora(root / base, root / model, root / out, **kw)
    assert not (root / out).exists() or not any((root / out).iterdir())
    assert [p.name for p in root.iterdir() if p.name.startswith(".")] == []


@pytest.mark.parametrize("kw,match", [(dict(rank=0), "rank must be >= 1"), (dict(oversample=-1), "oversample"),
                                      (dict(power_iters=-1), "power_iters"), (dict(dtype=torch.float64), "fp32, bf16 or fp16")])
def test_refuses_bad_parameters(pair, kw, match):
    _refused(pair, ValueError, match, **kw)


def test_refuses_directories_without_index(pair):
    _refused(pair, FileNotFoundError, "base .*nowhere has no model.safetensors.index.json", base="nowhere")
    write_adapter(pair / "adapter", {"base_model.model.model.norm.weight": torch.ones(32)})
    _refused(pair, FileNotFoundError, "LoRA adapter, not a full checkpoint", model="adapter")


def test_refuses_different_names(pair):
    base = random_model(SHAPES, 0)
    base.pop("model.norm.weight")
    base["extra.weight"] = torch.zeros(3)
    write_model(pair / "other", base)
    _refused(pair, ValueError, r"only in the base: \[model.norm.weight\]; only in the model: \[extra.weight\]", model="other")


def test_refuses_different_shapes(pair):
    base = random_model(SHAPES, 0)
    base["model.norm.weight"] = torch.zeros(31)
    write_model(pair / "other", base)
    _refused(pair, ValueError, r"model.norm.weight has shape \(32,\) in the base, \(31,\) in the model", model="other")


def test_refuses_non_empty_output(pair):
    (pair / "out").mkdir()
    (pair / "out" / "keep.txt").write_text("x")
    with pytest.raises(FileExistsError, match="not an empty directory"):
        extract.extract_lora(pair / "base", pair / "model", pair / "out", 4)
    assert [p.name for p in (pair / "out").iterdir()] == ["keep.txt"]


def test_cli_refusal_needs_no_device(pair):
    with pytest.raises(ValueError, match="rank must be >= 1"):
        extract.main([str(pair / "base"), str(pair / "model"), str(pair / "out"), "--rank", "0"])
    assert not (pair / "out").exists()


# ---- save_adapter -----------------------------------------------------------------------------------------------------
def test_save_adapter_keys_config_and_bind(tmp_path):
    base = random_model(SHAPES, 0)
    write_model(tmp_path / "base", base)
    q, down = "model.layers.0.self_attn.q_proj.weight", "model.layers.0.mlp.down_proj.weight"
    tensors = {q: (torch.randn(8, 32), torch.randn(32, 8)),
               down: (torch.randn(3, 64).to(torch.bfloat16), torch.randn(32, 3).to(torch.bfloat16)),
               "lm_head.weight": (torch.randn(8, 32), torch.randn(64, 8)),
               "model.norm.weight": torch.randn(32),
               "model.embed_tokens.weight": torch.randn(64, 32).to(torch.bfloat16)}
    (tmp_path / "ad").mkdir()                                             # an empty directory may exist
    lora.save_adapter(tmp_path / "ad", tensors, {"r": 8, "base_model_name_or_path": str(tmp_path / "base")})
    assert sorted(p.name for p in tmp_path.iterdir()) == ["ad", "base"]
    assert sorted(p.name for p in (tmp_path / "ad").iterdir()) == [lora.CONFIG_FILE, lora.WEIGHTS_FILE]
    cfg = json.loads((tmp_path / "ad" / lora.CONFIG_FILE).read_text())
    assert cfg["peft_type"] == "LORA" and cfg["r"] == 8 and cfg["lora_alpha"] == 8
    assert cfg["alpha_pattern"] == {"model.layers.0.mlp.down_proj": 3}
    assert cfg["target_modules"] == ["down_proj", "lm_head", "q_proj"]
    assert cfg["modules_to_save"] == ["model.embed_tokens", "model.norm"]
    assert cfg["base_model_name_or_path"] == str(tmp_path / "base")
    assert cfg["use_dora"] is False and cfg["fan_in_fan_out"] is False and cfg["use_rslora"] is False
    with safe_open(str(tmp_path / "ad" / lora.WEIGHTS_FILE), "pt") as f:
        assert f.metadata() == {"format": "pt"}
        keys = set(f.keys())
        for name, value in tensors.items():
            if isinstance(value, tuple):
                module = name[: -len(".weight")]
                assert torch.equal(f.get_tensor(f"base_model.model.{module}.lora_A.weight"), value[0])
                assert torch.equal(f.get_tensor(f"base_model.model.{module}.lora_B.weight"), value[1])
            else:
                assert torch.equal(f.get_tensor(f"base_model.model.{name}"), value)
    assert len(keys) == 2 * 3 + 2
    # read back through the project's own reader (headers only): every pair has scaling exactly 1
    im = LocalSafetensorsIndex(tmp_path)
    asyncio.run(im.add_model("base"))
    asyncio.run(im.add_model("ad"))
    im.bind_adapter("ad", "base")
    for name in (q, down, "lm_head.weight"):
        part = im.adapter_part("ad", name)
        assert part.kind == "lora" and part.scaling == 1.0, name
    assert im.adapter_part("ad", "model.norm.weight").kind == "full"
    assert im.adapter_part("ad", "model.layers.0.mlp.up_proj.weight").kind == "base"


def test_save_adapter_refuses_non_empty_directory_and_bad_pairs(tmp_path):
    (tmp_path / "ad").mkdir()
    (tmp_path / "ad" / "x").write_text("")
    with pytest.raises(FileExistsError):
        lora.save_adapter(tmp_path / "ad", {}, {"r": 4})
    with pytest.raises(ValueError, match="1 <= r' <= 4"):
        lora.save_adapter(tmp_path / "ad2", {"a.weight": (torch.zeros(5, 3), torch.zeros(2, 5))}, {"r": 4})
    assert sorted(p.name for p in tmp_path.iterdir()) == ["ad"]
