"""PEFT LoRA adapters on the device: sm_lora_materialize against the definition, merges with adapters bit-identical to
merges of the checkpoints the adapters materialise to, and what an adapter model reads from disk."""
import asyncio
import copy

import numpy as np
import pytest
import torch
from safetensors.torch import load_file

from shardmerge_b200 import lora
from shardmerge_b200.config import MergeConfig, MergeModel
from shardmerge_b200.index import LocalSafetensorsIndex
from shardmerge_b200.merge.fast_fourier import FourierMerge
from tests.lora_util import adapter_tensors, llama_shapes, random_model, write_adapter, write_model

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}


def _scaling(r):
    return float(np.float32(2.0 / r))


def _draw(R, C, r, base_dt, ab_dt, seed):
    """Base ~ 0.02 N(0,1); factors such that _scaling(r) * B @ A is about 5 % of the base's magnitude, as in trained adapters."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    W = (0.02 * torch.randn((R, C), generator=g, device=DEV)).to(base_dt)
    A = torch.randn((r, C), generator=g, device=DEV).to(ab_dt)
    B = (torch.randn((R, r), generator=g, device=DEV) * (1e-3 / (_scaling(r) * r ** 0.5))).to(ab_dt)
    return W, A, B


def _ordered(bits16: torch.Tensor) -> torch.Tensor:
    u = bits16.view(torch.int16).to(torch.int32) & 0xFFFF
    return torch.where(u >= 0x8000, 0x8000 - (u & 0x7FFF), u + 0x8000)


def _ref64(W, A, B, s):
    return W.double() + float(s) * (B.double() @ A.double())


@pytest.mark.parametrize("base_name", ["bf16", "fp16", "fp32"])
@pytest.mark.parametrize("ab_name", ["fp32", "bf16", "fp16"])
@pytest.mark.parametrize("r", [1, 8, 16, 64, 320])
@pytest.mark.parametrize("shape", [(77, 300), (1024, 4096), (14336, 4096), (4096, 14336)], ids=lambda s: f"{s[0]}x{s[1]}")
def test_materialize_vs_definition(shape, r, ab_name, base_name):
    R, C = shape
    base_dt, ab_dt = DTYPES[base_name], DTYPES[ab_name]
    W, A, B = _draw(R, C, r, base_dt, ab_dt, seed=R * 7 + C + r)
    s = _scaling(r)
    out = lora.materialize(W, A, B, s)
    torch.cuda.synchronize()
    assert out.dtype == base_dt and out.shape == W.shape
    ref = _ref64(W, A, B, s)
    delta = (ref - W.double()).abs() / W.double().abs().clamp_min(1e-30)
    assert 0.001 < float(delta.median()) < 0.2                     # the drawn delta is a few percent of the base
    # error bound of the fp32 evaluation the definition prescribes: r FMAs, the product with s and the add
    bound = (r + 2) * 2.0 ** -24 * (W.double().abs() + abs(s) * (B.double().abs() @ A.double().abs()))
    err = (out.double() - ref).abs()
    if base_dt != torch.float32:
        ulp = (_ordered(out) - _ordered(ref.to(base_dt))).abs()
        assert float((ulp == 0).double().mean()) >= 0.999
        # within 1 ulp, except where W + s * acc nearly cancels: there |W + s * acc| << |W|, the fp32 evaluation's
        # absolute error (about 2^-24 |W|) is many bf16 ulps of the result, and that evaluation is the definition
        half_ulp = out.double().abs() * 2.0 ** -(8 if base_dt == torch.bfloat16 else 11)
        assert bool(((ulp <= 1) | (err <= bound + half_ulp)).all())
    else:
        assert bool((err <= bound).all())
    if r == 1:                                                      # bit-exact against the same steps in numpy float32
        w, a, b = (t.float().cpu().numpy() for t in (W, A, B))
        acc = b[:, :1] * a[:1, :]                                   # fma(b, a, 0) == b * a rounded once
        y = torch.from_numpy(w + np.float32(s) * acc).to(base_dt)
        assert torch.equal(out.cpu().view(torch.uint8), y.view(torch.uint8))


@pytest.mark.parametrize("base_name", ["bf16", "fp32"])
def test_materialize_non_finite_factors(base_name):
    R, C, r = 77, 300, 5
    base_dt = DTYPES[base_name]
    W, A, B = _draw(R, C, r, base_dt, torch.float32, seed=11)
    A[2, 7] = float("nan")
    A[4, 100] = float("inf")
    B[30, 4] = float("-inf")
    B[31, 0] = 0.0
    A[0, 200] = float("inf")                                        # 0 * Inf = NaN at (31, 200)
    out = lora.materialize(W, A, B, 0.25).double()
    ref = _ref64(W, A, B, 0.25)
    assert torch.equal(torch.isnan(out), torch.isnan(ref))
    assert torch.equal(torch.isposinf(out), torch.isposinf(ref)) and torch.equal(torch.isneginf(out), torch.isneginf(ref))
    assert bool(torch.isnan(out[:, 7]).all()) and bool(torch.isnan(out[31, 200]))
    fin = torch.isfinite(ref)
    assert torch.allclose(out[fin], ref[fin], rtol=1e-2, atol=0)


def test_materialize_unaligned_and_strided_inputs():
    # odd column counts take the element-wise epilogue; a transposed view is made contiguous
    for (R, C) in [(65, 129), (3, 7), (128, 1)]:
        W, A, B = _draw(R, C, 3, torch.bfloat16, torch.bfloat16, seed=R + C)
        out = lora.materialize(W, A, B, 0.5)
        ulp = (_ordered(out) - _ordered(_ref64(W, A, B, 0.5).to(torch.bfloat16))).abs()
        assert int(ulp.max()) <= 1
    W, A, B = _draw(256, 128, 8, torch.bfloat16, torch.bfloat16, seed=5)
    Wt = W.t().contiguous().t()
    assert torch.equal(lora.materialize(Wt, A, B, 0.5), lora.materialize(W, A, B, 0.5))


# ---- merges: an adapter is an ordinary finetune once materialised ---------------------------------------------------
SHAPES = llama_shapes(layers=3)


def _storage(root):
    base = random_model(SHAPES, 0)
    write_model(root / "org" / "base", base)
    write_model(root / "org" / "full", {n: (t.float() + 0.002 * torch.randn(t.shape, generator=torch.Generator().manual_seed(9))).to(t.dtype)
                                        for n, t in base.items()})
    every = ("q_proj", "k_proj", "v_proj", "o_proj", "gate_proj", "up_proj", "down_proj")
    write_adapter(root / "org" / "ad1", adapter_tensors(SHAPES, every, 16, seed=1, full=("lm_head.weight",), base=base), r=16,
                  lora_alpha=32)
    write_adapter(root / "org" / "ad2", adapter_tensors(SHAPES, every, 8, seed=2, dtype=torch.float32), r=8, lora_alpha=16,
                  use_rslora=True, alpha_pattern={"down_proj": 4})
    write_adapter(root / "org" / "qv", adapter_tensors(SHAPES, ("q_proj", "v_proj"), 16, seed=3, full=("lm_head.weight",),
                                                       base=base), r=16, lora_alpha=16)
    return base


def _materialised_checkpoint(root, adapter, base):
    """The full checkpoint an adapter stands for, formed with lora.materialize and saved as a normal model."""
    im = LocalSafetensorsIndex(root)
    asyncio.run(im.add_model("org/base"))
    asyncio.run(im.add_model(adapter))
    im.bind_adapter(adapter, "org/base")
    out = {}
    for name, t in base.items():
        part = im.adapter_part(adapter, name)
        got = [im.get_tensor(adapter, k, device=str(DEV)) for k in part.keys]
        got = [asyncio.run(p.get()) for p in got]
        if part.kind == "lora":
            out[name] = lora.materialize(t.to(DEV), got[0], got[1], part.scaling).cpu()
        elif part.kind == "full":
            out[name] = got[0].cpu()
        else:
            out[name] = t
    write_model(root / (adapter + "_ckpt"), out)


def _merge(root, entries, out, lanes=3):
    cfg = MergeConfig(finetune_merge=[MergeModel(**e) for e in entries], output_base_model="org/base",
                      output_dir=str(root / out), device="cuda", storage_dir=str(root))
    fm = FourierMerge(cfg, index_manager=LocalSafetensorsIndex(cfg.storage_path))
    fm.lanes = lanes
    asyncio.run(fm.merge("cuda:0"))
    tensors = {}
    for f in sorted((root / out).glob("*.safetensors")):
        tensors.update(load_file(str(f)))
    return fm, tensors


CASES = {
    "two_adapters": [dict(model="org/ad1", base="org/base", alpha=0.3, is_input=True),
                     dict(model="org/ad2", base="org/base", alpha=0.5, is_output=True)],
    "adapter_and_full": [dict(model="org/full", base="org/base", alpha=0.4, is_input=True),
                         dict(model="org/ad1", base="org/base", alpha=0.6, is_output=True)],
    "tree_of_three": [dict(model="org/ad1", base="org/base", alpha=0.3),
                      dict(model="org/full", base="org/base", alpha=0.5, is_output=True),
                      dict(model="org/ad2", base="org/base", alpha=0.7, is_input=True)],
    "layer_range": [dict(model="org/ad1", base="org/base", alpha=0.3, is_output=True),
                    dict(model="org/ad2", base="org/base", alpha=0.5, start_layer=1, end_layer=1),
                    dict(model="org/full", base="org/base", alpha=0.5)],
    # k / o / gate / up / down have a zero delta for the q / v adapter: the fused chain hands them to the step-by-step path
    "untargeted_tensors": [dict(model="org/qv", base="org/base", alpha=0.5, is_output=True),
                           dict(model="org/full", base="org/base", alpha=0.5)],
}


@pytest.fixture(scope="module")
def lora_storage(tmp_path_factory):
    root = tmp_path_factory.mktemp("lora_merge")
    base = _storage(root)
    for a in ("org/ad1", "org/ad2", "org/qv"):
        _materialised_checkpoint(root, a, base)
    return root


@pytest.mark.parametrize("lanes", [1, 3])
@pytest.mark.parametrize("case", sorted(CASES))
def test_merge_bit_identical_to_materialised_checkpoints(lora_storage, case, lanes):
    entries = CASES[case]
    _, got = _merge(lora_storage, entries, f"out_{case}_{lanes}_adapter", lanes)
    ckpt = copy.deepcopy(entries)
    for e in ckpt:
        if e["model"] != "org/full":
            e["model"] += "_ckpt"
    _, want = _merge(lora_storage, ckpt, f"out_{case}_{lanes}_ckpt", lanes)
    assert sorted(got) == sorted(want) == sorted(SHAPES)
    for name in want:
        assert torch.equal(got[name].view(torch.uint8), want[name].view(torch.uint8)), name


def test_adapter_reads_only_factors_and_replacements(lora_storage, monkeypatch):
    read = []
    orig = LocalSafetensorsIndex._read_into

    def counting(self, model_uri, tensor_name, buf):
        t = orig(self, model_uri, tensor_name, buf)
        read.append((model_uri, tensor_name, t.numel() * t.element_size()))
        return t

    monkeypatch.setattr(LocalSafetensorsIndex, "_read_into", counting)
    entries = [dict(model="org/full", base="org/base", alpha=0.4, is_input=True),
               dict(model="org/ad1", base="org/base", alpha=0.6, is_output=True)]
    _merge(lora_storage, entries, "out_bytes")
    ad = [(k, n) for u, k, n in read if u == "org/ad1"]
    header = LocalSafetensorsIndex(lora_storage)._meta(lora_storage / "org" / "ad1" / lora.WEIGHTS_FILE)[1]
    adapter_bytes = {k: b1 - b0 for k, (_, _, b0, b1) in header.items()}
    assert sorted(k for k, _ in ad) == sorted(adapter_bytes)               # every factor / replacement exactly once
    assert sum(n for _, n in ad) == sum(adapter_bytes.values())
    base_reads = [k for u, k, _ in read if u == "org/base"]
    assert len(base_reads) == len(set(base_reads))                          # no base tensor read twice
    assert "lm_head.weight" not in base_reads                               # the adapter's replacement is the output
