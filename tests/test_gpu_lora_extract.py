"""Extracting a LoRA adapter on the device: sm_lowrank_right / sm_lowrank_left against fp64, exact-rank recovery,
near-optimality against the fp64 prototype, and the round trip through this project's adapter reader and merge."""
import asyncio
import copy
import math

import pytest
import torch
from safetensors.torch import load_file

from shardmerge_b200 import _lib, extract, lora
from shardmerge_b200.config import MergeConfig, MergeModel
from shardmerge_b200.index import LocalSafetensorsIndex
from shardmerge_b200.merge.fast_fourier import FourierMerge
from tests.lora_util import llama_shapes, random_model, write_model
from tests.test_lora_extract_host import NEAR_OPTIMAL, prototype, spectrum_matrix

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}
U32 = 2.0 ** -24


def _gamma(n):
    return n * U32 / (1 - n * U32)


def _pair(R, C, w_dt, m_dt, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    W = (0.02 * torch.randn((R, C), generator=g, device=DEV)).to(w_dt)
    M = (W.float() + 0.002 * torch.randn((R, C), generator=g, device=DEV)).to(m_dt)
    return W, M, g


def _ordered(bits16):
    u = bits16.view(torch.int16).to(torch.int32) & 0xFFFF
    return torch.where(u >= 0x8000, 0x8000 - (u & 0x7FFF), u + 0x8000)


# ---- the kernels against fp64 -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("dts", ["bf16/bf16", "fp16/fp16", "fp32/fp32", "bf16/fp16"])
@pytest.mark.parametrize("k", [1, 8, 72, 264])
@pytest.mark.parametrize("shape", [(1, 4096), (77, 300), (1024, 4096), (14336, 4096), (4096, 14336)],
                         ids=lambda s: f"{s[0]}x{s[1]}")
def test_kernels_vs_fp64(shape, k, dts):
    R, C = shape
    w_dt, m_dt = (DTYPES[n] for n in dts.split("/"))
    W, M, g = _pair(R, C, w_dt, m_dt, seed=R * 31 + C + k)
    X = torch.randn((C, k), generator=g, device=DEV)
    Q = torch.randn((R, k), generator=g, device=DEV)
    d64 = (M.float() - W.float()).double()                 # Δ: one rounded fp32 subtraction per element
    Y, ss = extract.lowrank_right(W, M, X, sumsq=True)
    Z = extract.lowrank_left(W, M, Q)
    for got, ref, bound in ((Y, d64 @ X.double(), _gamma(C) * (d64.abs() @ X.double().abs())),
                            (Z, Q.double().T @ d64, _gamma(R) * (Q.double().abs().T @ d64.abs()))):
        err = (got.double() - ref).abs()
        assert bool((err <= bound).all()), float((err - bound).max())
        assert float(err.norm() / ref.norm()) <= 1e-5
    ss_ref = float(d64.square().sum())
    assert abs(float(ss) - ss_ref) <= 1e-6 * ss_ref
    # deterministic: a second launch, and one on another stream, give the same bits
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        Y2, ss2 = extract.lowrank_right(W, M, X, sumsq=True)
        Z2 = extract.lowrank_left(W, M, Q)
    side.synchronize()
    Y3, _ = extract.lowrank_right(W, M, X)
    assert torch.equal(Y, Y2) and torch.equal(Y, Y3) and torch.equal(Z, Z2) and float(ss) == float(ss2)


def test_kernels_unaligned_and_argument_errors():
    W, M, g = _pair(65, 131, torch.bfloat16, torch.float32, seed=4)     # odd C: the scalar-tail loads
    X = torch.randn((131, 5), generator=g, device=DEV)
    Y, _ = extract.lowrank_right(W[:, 1:], M[:, 1:], X[1:].contiguous())  # contiguous copies of offset views
    d64 = (M[:, 1:].float() - W[:, 1:].float()).double()
    assert float((Y.double() - d64 @ X[1:].double()).norm() / (d64 @ X[1:].double()).norm()) <= 1e-6
    lib = _lib.load()
    ws = torch.empty(16, dtype=torch.uint8, device=DEV)
    rc = lib.sm_lowrank_right(1024, 4096, 8, 1, W.data_ptr(), 1, M.data_ptr(), X.data_ptr(), Y.data_ptr(), None,
                              ws.data_ptr(), 16, torch.cuda.current_stream().cuda_stream)
    assert rc == -2 and b"workspace" in lib.sm_last_error()
    assert lib.sm_lowrank_left(0, 4, 1, 1, None, 1, None, None, None, None, 0, None) == -2
    assert lib.sm_lowrank_left(4, 4, 1, 3, None, 1, None, None, None, None, 0, None) == -2
    assert lib.sm_lowrank_right(9_000_000, 4, 1, 1, None, 1, None, None, None, None, None, 0, None) == -2
    assert b"grid" in lib.sm_last_error()


# ---- exact-rank recovery ----------------------------------------------------------------------------------------------
def _low_rank(R, C, r0, seed, scale):
    g = torch.Generator().manual_seed(seed)
    L = torch.randn((R, r0), generator=g, dtype=torch.float64) @ torch.randn((r0, C), generator=g, dtype=torch.float64)
    return L * (scale / float(L.std()))


def _read_pair(directory, name):
    t = load_file(str(directory / lora.WEIGHTS_FILE))
    module = name[: -len(".weight")]
    return t[f"base_model.model.{module}.lora_A.weight"], t[f"base_model.model.{module}.lora_B.weight"]


def _check_bf16_round_trip(got, Wb, Mb, A, B, L):
    """`got` = materialize(Wb, A, B, 1.0) for a bf16 model Mb = bf16(Wb + L) with L of rank r0 = A.shape[0].

    Δ = fp32(Mb) − fp32(Wb) = L + e carries Mb's own bf16 rounding e, which is full rank: no rank-r0 adapter holds it, so
    "within 1 bf16 ulp of Mb everywhere" cannot hold where Wb + L nearly cancels (|Mb| far below |Wb|; there e, and the
    part of it the factors leave out, is many ulps of the small result).  What does hold:
      - the factors are as close to Δ as the true low-rank part is: ‖BA − Δ‖ ≤ ‖e‖ up to fp32 rounding;
      - wherever BA is within half a bf16 ulp of Δ (less the fp32 error of the evaluation), got is within 1 ulp of Mb;
      - everywhere, got is the bf16 rounding of a value within that element's factor error of Mb."""
    d64 = (Mb.float() - Wb.float()).double()
    BA = B.double() @ A.double()
    e = d64 - L
    assert float((BA - d64).norm()) <= (1 + 1e-3) * float(e.norm())
    fe = (BA - d64).abs()                                                   # the factors' error per element
    f32 = (A.shape[0] + 2) * 2.0 ** -24 * (Wb.double().abs() + B.double().abs() @ A.double().abs())
    t = fe + f32                                                            # |value materialize rounds − Mb|
    ulp = (_ordered(got) - _ordered(Mb)).abs()
    assert bool(((t > Mb.double().abs() * 2.0 ** -9) | (ulp <= 1)).all())  # 2^-9 |x| <= half a bf16 ulp of x
    assert bool(((got.double() - Mb.double()).abs() <= t + 2.0 ** -8 * (Mb.double().abs() + t)).all())


@pytest.mark.parametrize("r0", [1, 8, 64])
@pytest.mark.parametrize("shape", [(77, 300), (1024, 4096), (4096, 14336)], ids=lambda s: f"{s[0]}x{s[1]}")
def test_exact_rank_recovery(tmp_path, shape, r0):
    R, C = shape
    name = "model.layers.0.mlp.up_proj.weight"
    W = 0.02 * torch.randn((R, C), generator=torch.Generator().manual_seed(r0))
    M = (W.double() + _low_rank(R, C, r0, seed=R + r0, scale=0.002)).float()
    write_model(tmp_path / "base", {name: W})
    write_model(tmp_path / "model", {name: M})
    res = extract.extract_lora(tmp_path / "base", tmp_path / "model", tmp_path / "out", r0)
    A, B = _read_pair(tmp_path / "out", name)
    assert A.dtype == torch.float32 and A.shape == (r0, C) and B.shape == (R, r0)
    d64 = (M - W).double()
    # Δ = L + the fp32 rounding of M: about 2^-24 |W| = 6e-7 |L| here (|W| = 10 |L|); the factors' own error is a few fp32
    # roundings of sums over R or C
    rel = float((d64 - B.double() @ A.double()).norm() / d64.norm())
    assert rel <= 1e-5, rel
    assert abs(res[name] - rel) <= 1e-3

    # bf16 base and model, fp32 factors: materialising the adapter gives M back up to what a rank-r0 adapter can hold
    Wb = W.to(torch.bfloat16)
    L = _low_rank(R, C, r0, seed=R + r0, scale=0.002)
    Mb = (Wb.double() + L).to(torch.bfloat16)
    write_model(tmp_path / "base_b", {name: Wb})
    write_model(tmp_path / "model_b", {name: Mb})
    extract.extract_lora(tmp_path / "base_b", tmp_path / "model_b", tmp_path / "out_b", r0)
    A, B = _read_pair(tmp_path / "out_b", name)
    got = lora.materialize(Wb.to(DEV), A.to(DEV), B.to(DEV), 1.0).cpu()
    _check_bf16_round_trip(got, Wb, Mb, A, B, L)


# ---- near-optimality --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("r", [16, 64])
@pytest.mark.parametrize("kind", sorted(NEAR_OPTIMAL))
@pytest.mark.parametrize("shape", [(512, 2048), (4096, 4096)], ids=lambda s: f"{s[0]}x{s[1]}")
def test_near_optimal_vs_prototype(shape, kind, r):
    R, C = shape
    M = spectrum_matrix(R, C, kind, seed=R + r).float()
    d64 = M.double()                                             # W = 0: Δ is M exactly
    om = extract.omega(f"spectrum.{kind}", C, min(r + 8, R, C))
    Md = M.to(DEV)
    A, B, S, norm2 = extract._factorize(torch.zeros_like(Md), Md, r, 8, 2, om.to(DEV))
    gpu = float((d64 - B.double().cpu() @ A.double().cpu()).norm())
    pa, pb, _ = prototype(d64, om, r)
    proto = float((d64 - pb @ pa).norm())
    assert abs(gpu - proto) <= 1e-3 * proto, (gpu, proto)
    tail = float(torch.linalg.svdvals(d64.to(DEV)).cpu()[r:].square().sum().sqrt())
    assert proto <= NEAR_OPTIMAL[kind] * tail
    assert abs(extract._residual(float(norm2), S, r) - gpu / float(d64.norm())) <= 1e-3


# ---- round trip through this project ----------------------------------------------------------------------------------
SHAPES = llama_shapes(layers=2)
EXACT = ("model.layers.0.self_attn.q_proj.weight", "model.layers.0.self_attn.v_proj.weight",
         "model.layers.1.mlp.down_proj.weight")
FULL_RANK = "model.layers.1.mlp.up_proj.weight"
NORM = "model.layers.0.input_layernorm.weight"


def _changed_model(base):
    model = dict(base)
    g = torch.Generator().manual_seed(7)
    for i, name in enumerate(EXACT):
        R, C = SHAPES[name]
        model[name] = (base[name].double() + _low_rank(R, C, 8, seed=100 + i, scale=0.002)).to(torch.bfloat16)
    model[FULL_RANK] = (base[FULL_RANK].float() + 0.002 * torch.randn(SHAPES[FULL_RANK], generator=g)).to(torch.bfloat16)
    model[NORM] = (base[NORM].float() + 0.01 * torch.randn(SHAPES[NORM], generator=g)).to(torch.bfloat16)
    # lm_head saved in fp32 with the base's values: a zero Δ whose bytes differ, stored whole
    model["lm_head.weight"] = base["lm_head.weight"].float()
    return model


@pytest.fixture(scope="module")
def round_trip(tmp_path_factory):
    root = tmp_path_factory.mktemp("extract")
    base = random_model(SHAPES, 0)
    model = _changed_model(base)
    write_model(root / "org" / "base", base)
    write_model(root / "org" / "model", model)
    return root, base, model


def _materialise(root, adapter, base):
    im = LocalSafetensorsIndex(root)
    asyncio.run(im.add_model("org/base"))
    asyncio.run(im.add_model(adapter))
    im.bind_adapter(adapter, "org/base")
    out = {}
    for name, t in base.items():
        part = im.adapter_part(adapter, name)
        got = [asyncio.run(im.get_tensor(adapter, k, device=str(DEV)).get()) for k in part.keys]
        if part.kind == "lora":
            assert part.scaling == 1.0
            out[name] = lora.materialize(t.to(DEV), got[0], got[1], part.scaling).cpu()
        elif part.kind == "full":
            out[name] = got[0].cpu()
        else:
            out[name] = t
    return out


def _merge(root, entries, out):
    cfg = MergeConfig(finetune_merge=[MergeModel(**e) for e in entries], output_base_model="org/base",
                      output_dir=str(root / out), device="cuda", storage_dir=str(root))
    asyncio.run(FourierMerge(cfg, index_manager=LocalSafetensorsIndex(cfg.storage_path)).merge("cuda:0"))
    tensors = {}
    for f in sorted((root / out).glob("*.safetensors")):
        tensors.update(load_file(str(f)))
    return tensors


@pytest.mark.parametrize("factor", ["fp32", "bf16", "fp16"])
def test_round_trip(round_trip, factor):
    root, base, model = round_trip
    ad = f"org/ad_{factor}"
    res = extract.extract_lora(root / "org" / "base", root / "org" / "model", root / ad, 8, dtype=DTYPES[factor])
    keys = set(load_file(str(root / ad / lora.WEIGHTS_FILE)))
    pairs = {k[len("base_model.model."): -len(".lora_A.weight")] + ".weight" for k in keys if k.endswith(".lora_A.weight")}
    full = {k[len("base_model.model."):] for k in keys if ".lora_" not in k}
    assert pairs == set(EXACT) | {FULL_RANK} and sorted(res) == sorted(pairs)
    assert full == {NORM, "lm_head.weight"} and len(keys) == 2 * len(pairs) + len(full)

    got = _materialise(root, ad, base)
    for name in full:
        assert got[name].dtype == model[name].dtype and torch.equal(got[name].view(torch.uint8), model[name].view(torch.uint8))
    tensors = load_file(str(root / ad / lora.WEIGHTS_FILE))
    for name in pairs:
        d64 = (model[name].float() - base[name].float()).double()
        module = name[: -len(".weight")]
        A = tensors[f"base_model.model.{module}.lora_A.weight"].double()
        B = tensors[f"base_model.model.{module}.lora_B.weight"].double()
        assert A.shape[0] == 8 and abs(res[name] - float((d64 - B @ A).norm() / d64.norm())) <= 1e-3, name
        if name in EXACT and factor == "fp32":
            L = _low_rank(*SHAPES[name], 8, seed=100 + EXACT.index(name), scale=0.002)
            _check_bf16_round_trip(got[name], base[name], model[name], A.float(), B.float(), L)
    assert res[FULL_RANK] > 0.5 and max(res[n] for n in EXACT) < 0.05

    # a merge with the adapter as a finetune is bit-identical to the merge of the checkpoint it materialises to
    write_model(root / f"{ad}_ckpt", got)
    entries = [dict(model=ad, base="org/base", alpha=0.5, is_output=True),
               dict(model="org/model", base="org/base", alpha=0.4, is_input=True)]
    merged = _merge(root, entries, f"merge_{factor}")
    ckpt = copy.deepcopy(entries)
    ckpt[0]["model"] += "_ckpt"
    want = _merge(root, ckpt, f"merge_{factor}_ckpt")
    assert sorted(merged) == sorted(want) == sorted(SHAPES)
    for name in want:
        assert torch.equal(merged[name].view(torch.uint8), want[name].view(torch.uint8)), name

    # extracting again gives the same bytes
    extract.extract_lora(root / "org" / "base", root / "org" / "model", root / f"{ad}_again", 8, dtype=DTYPES[factor])
    for f in (lora.CONFIG_FILE, lora.WEIGHTS_FILE):
        assert (root / ad / f).read_bytes() == (root / f"{ad}_again" / f).read_bytes(), f


def test_cli_prints_worst_residuals(round_trip, capsys):
    root, _, _ = round_trip
    assert extract.main([str(root / "org" / "base"), str(root / "org" / "model"), str(root / "cli_out"), "--rank", "4",
                         "--dtype", "bf16"]) == 0
    out = capsys.readouterr().out
    assert "4 LoRA pairs at rank 4" in out and FULL_RANK in out
    assert (root / "cli_out" / lora.WEIGHTS_FILE).is_file()


@pytest.mark.parametrize("where", ["model.layers.1.mlp.gate_proj.weight", NORM])
def test_nan_in_delta_raises_and_writes_nothing(tmp_path, where):
    base = random_model(SHAPES, 0)
    model = dict(base)
    bad = base[where].clone()
    bad.view(-1)[3] = float("nan")
    model[where] = bad
    write_model(tmp_path / "base", base)
    write_model(tmp_path / "model", model)
    with pytest.raises(ValueError, match=f"difference of {where.replace('.', '[.]')} holds NaN or Inf"):
        extract.extract_lora(tmp_path / "base", tmp_path / "model", tmp_path / "out", 8)
    assert sorted(p.name for p in tmp_path.iterdir()) == ["base", "model"]


def test_timings_cover_the_phases(round_trip):
    root, _, _ = round_trip
    t = {}
    extract.extract_lora(root / "org" / "base", root / "org" / "model", root / "timed", 8, timings=t)
    assert set(t) == {"kernels", "linalg", "read_wait", "write", "total"}
    assert all(math.isfinite(v) and v >= 0 for v in t.values()) and t["kernels"] > 0 and t["linalg"] > 0
