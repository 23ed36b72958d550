"""FourierMerge's step-by-step path (merge/fast_fourier.py: _merge_sources_steps / _steps_pass) against the numpy oracle.

Every input other than bf16 finetunes on a bf16 base takes this path: fp16 and fp32 checkpoints and mixes of dtypes
(engine.make_source turns such a pair into an fp32 delta that sm_fwd_rows_f32 transforms), stacked tensors, and every
branch that is not SLERP.  Each case runs FourierMerge.merge_sources on device tensors and oracle_np.merge_layer on the
same stored values, and compares the branches, target_norm and the bf16 output, with the bounds the suite already holds
for this algorithm:

  FFT branches       test_pair_merge_vs_oracle_mid_size: within 1 ulp on >= 99.99 % when the fp32 merged delta's raw
                     rel-L2 is <= 1e-5, else on >= 98.5 % with the flip-accounted residual (k = 16) <= 1e-5; never more
                     than one bf16 ulp of the largest value apart.  The merged delta is compared with the oracle's without
                     the nested imaginary path (interp_imag=False), which returns Im X0 only up to rounding noise.
  FFT-free branches  within 1 ulp everywhere: the GPU multiplies by an fp32 reciprocal where the oracle divides.
  trees              test_fused_tree_rounds_vs_oracle and test_tree_of_four_finetunes_vs_oracle: round 1 flip-accounted
                     <= 1e-5; later rounds blend spectra whose culled bins are rounding noise in the reference too, so the
                     final delta is pinned by its rel-L2 (< 0.5) and its norm (within 5 %).
Run with `pytest -m gpu tests/test_gpu_step_path.py -s` to see where each case sits against its bound."""
import asyncio

import numpy as np
import pytest
import torch

from oracle import oracle_np as O
from tests.parity_util import bf16_ulp_distance, flip_accounted, rel_l2

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
LAYER = "model.layers.0.x"
DT = {"bf16": torch.bfloat16, "fp16": torch.float16, "fp32": torch.float32}
ALPHAS = (0.3, 0.5, 0.4, 0.2)
SIG = (0.002, 0.0026, 0.0023, 0.0029)


@pytest.fixture(scope="module")
def E():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from shardmerge_b200 import engine
    return engine


def _merger(models=None, tensors=None):
    from shardmerge_b200.config import MergeConfig
    from shardmerge_b200.index import InMemoryIndex
    from shardmerge_b200.merge.fast_fourier import FourierMerge
    cfg = MergeConfig(finetune_merge=models or [], output_base_model="org/base", output_dir="/tmp/unused")
    fm = FourierMerge(cfg, index_manager=InMemoryIndex(tensors or {}))
    fm.keep_intermediates = True
    return fm


def stored(t):
    """A tensor as the oracle takes it: bf16 as uint16 bit patterns, fp16 / fp32 as they are."""
    t = t.detach().contiguous().cpu()
    return t.view(torch.int16).numpy().view(np.uint16) if t.dtype == torch.bfloat16 else t.numpy()


def bits(t):
    return t.detach().contiguous().view(torch.int16).cpu().numpy().view(np.uint16)


def draw(shape, seed, base_dt, ft_dts, sig=SIG, mean=0.0, bs=0.02):
    """test_pair_merge_vs_oracle_mid_size's inputs: base ~ mean + bs N(0, 1), finetune k = base + sig[k] N(0, 1), each
    stored in its own dtype."""
    g = torch.Generator(device=DEV).manual_seed(1234 + seed)
    base = (mean + bs * torch.randn(shape, generator=g, device=DEV)).to(DT[base_dt])
    fts = []
    for k, dt in enumerate(ft_dts):
        gk = torch.Generator(device=DEV).manual_seed(100000 * (k + 1) + seed)
        fts.append((base.float() + sig[k] * torch.randn(shape, generator=gk, device=DEV)).to(DT[dt]))
    return base, fts


def run(E, fm, base, fts, base_out=None, alphas=ALPHAS):
    base_out = base if base_out is None else base_out
    srcs = [E.make_source(base, ft, weight=a, name=f"m{k}") for k, (ft, a) in enumerate(zip(fts, alphas))]
    return fm.merge_sources(srcs, base_out, torch.device(DEV), layer_name=LAYER)


def oracle(base, fts, base_out=None, alphas=ALPHAS, interp_imag=True):
    info = {}
    models = [dict(base=stored(base), ft=stored(ft), alpha=a, name=f"m{k}") for k, (ft, a) in enumerate(zip(fts, alphas))]
    out = O.merge_layer(stored(base if base_out is None else base_out), models, info=info, interp_imag=interp_imag)
    return out, info


def check_decisions(fm, info):
    """The branches (the oracle records slerp-early as slerp) and target_norm."""
    got = ["slerp" if b == "slerp-early" else b for b in fm.last_info["branches"]]
    assert got == info["branches"], (fm.last_info["branches"], info["branches"])
    assert abs(fm.last_info["target_norm"] / info["target_norm"] - 1) < 1e-6, (fm.last_info["target_norm"], info["target_norm"])


def check_fft(tag, out, oo, m32, ref32):
    """The mid-size bounds.  m32: our fp32 merged delta (before the base is added), ref32: the oracle's."""
    raw, resid, share = flip_accounted(np.asarray(m32).reshape(oo.shape), np.asarray(ref32).reshape(oo.shape), k=16)
    u = bf16_ulp_distance(bits(out).reshape(oo.shape), oo)
    frac1 = float((u <= 1).mean())
    want = O.bf16_to_f32(oo)
    absd = np.abs(O.bf16_to_f32(bits(out).reshape(oo.shape)) - want)
    print(f"\n[{tag}] fp32 merged delta: raw rel-L2 {raw:.3e}, flip-accounted {resid:.3e} (top-16 bins carry {share:.4f}); "
          f"bf16 exact {float((u == 0).mean()):.6f} within-1ulp {frac1:.6f} max-abs-diff {absd.max():.3e}")
    assert resid <= 1e-5, (tag, raw, resid, share)
    assert frac1 >= (0.9999 if raw <= 1e-5 else 0.985), (tag, frac1, raw)
    assert absd.max() <= 2.0 ** -7 * np.abs(want).max() + 1e-4, (tag, absd.max())


def check_within_1ulp(tag, out, oo):
    u = bf16_ulp_distance(bits(out).reshape(oo.shape), oo)
    print(f"\n[{tag}] bf16 exact {float((u == 0).mean()):.6f} max ulp {int(u.max())}")
    assert int(u.max()) <= 1, (tag, int(u.max()))


def fp32_result(fm):
    """The step path's fp32 merged delta: its last round's result when the output base is not bf16."""
    return fm.last_tree[-1][2].cpu().numpy()


def merged_vs_oracle(E, tag, base, fts, base_out=None, alphas=ALPHAS):
    """One FFT-branch case end to end: decisions, fp32 merged delta and bf16 output against the oracle."""
    fm = _merger()
    out = run(E, fm, base, fts, base_out, alphas)
    oo, info = oracle(base, fts, base_out, alphas)
    check_decisions(fm, info)
    _, info_ni = oracle(base, fts, base_out, alphas, interp_imag=False)
    check_fft(tag, out, oo, fp32_result(fm), info_ni["merged_f32"])
    return fm, out


# ---------------------------------------------------------------------------------------------------- SLERP, every dtype
@pytest.mark.parametrize("dt,shape,seed", [("fp16", (1024, 4096), 31), ("fp16", (512, 2048), 32), ("fp32", (1024, 4096), 33)])
def test_slerp_on_fp16_and_fp32_checkpoints(E, dt, shape, seed):
    """sm_fwd_rows_f32 on the fp32 deltas, sm_inv_rows_f32, and the torch ops that add the fp16 / fp32 base."""
    base, fts = draw(shape, seed, dt, (dt, dt))
    fm, out = merged_vs_oracle(E, f"slerp {dt} {shape}", base, fts)
    assert fm.last_info["branches"] == ["slerp"] and out.dtype == torch.bfloat16 and tuple(out.shape) == shape


@pytest.mark.parametrize("case", ["bf16 base, fp32 finetune", "fp16 base, bf16 finetunes"])
def test_mixed_dtypes(E, case):
    """A bf16 pair next to an fp32 delta into the bf16 epilogue (sm_inv_rows_bf16); fp32 deltas of bf16 finetunes on an fp16
    base into the torch finish."""
    shape = (1024, 4096)
    if case.startswith("bf16"):
        base, fts = draw(shape, 41, "bf16", ("bf16", "fp32"))
        fm = _merger()
        out = run(E, fm, base, fts)
        oo, info = oracle(base, fts)
        check_decisions(fm, info)
        assert fm.last_info["branches"] == ["slerp"]
        # the merged delta of the same kernels, taken before the bf16 epilogue: the same sources on an fp32 output base
        fm32 = _merger()
        run(E, fm32, base, fts, base_out=base.float())
        _, info_ni = oracle(base, fts, interp_imag=False)
        check_fft(case, out, oo, fp32_result(fm32), info_ni["merged_f32"])
    else:
        base, fts = draw(shape, 42, "fp16", ("bf16", "bf16"))
        fm, _ = merged_vs_oracle(E, case, base, fts)
        assert fm.last_info["branches"] == ["slerp"]


# ---------------------------------------------------------------------------------------------------- other branches
def test_arith_with_fp32_output(E):
    """A norm ratio below 0.1: the arithmetic-FFT branch with an fp32 result (fp32 base)."""
    base, fts = draw((512, 2048), 51, "fp32", ("fp32", "fp32"), sig=(0.0026, 0.0001))
    fm, _ = merged_vs_oracle(E, "arith fp32", base, fts)
    assert fm.last_info["branches"] == ["arith"]


def test_add_on_fp32_deltas(E):
    """Two finetunes equal to the base: their pair takes the add branch on fp32 deltas (exactly zero), and the
    arithmetic-FFT branch merges that with the third model."""
    base, (ft,) = draw((512, 2048), 52, "fp32", ("fp32",))
    fts = [base.clone(), base.clone(), ft]
    fm, _ = merged_vs_oracle(E, "add fp32", base, fts, alphas=(0.3, 0.5, 0.4))
    assert fm.last_info["branches"] == ["add", "arith"]
    assert not fm.last_tree[0][2].any()


def _nudged(base, idx, v):
    ft = base.clone()
    ft.view(-1)[idx] = (base.view(-1)[idx].float() + v).to(base.dtype)
    return ft


def test_slerp_early_on_fp16(E):
    """Delta norms below 1e-4 (a few elements moved by ~3e-5): merge_tensors_fft2_slerp returns the normalised larger
    delta (functions.py:184-190) without a transform -- _slerp_pair's early return on fp32 deltas."""
    shape = (512, 2048)
    base, _ = draw(shape, 53, "fp16", ())
    idx0, idx1 = torch.tensor([12345, 99, 777777], device=DEV), torch.tensor([777, 4242], device=DEV)
    base.view(-1)[torch.cat([idx0, idx1])] = 0.01          # fp16 spacing 2^-17 there: the deltas are 4 ulps
    fts = [_nudged(base, idx0, 3e-5), _nudged(base, idx1, 3e-5)]
    fm = _merger()
    out = run(E, fm, base, fts)
    oo, info = oracle(base, fts)
    assert fm.last_info["branches"] == ["slerp-early"]
    assert all(n < 1e-4 for n in fm.last_info["norms"])
    check_decisions(fm, info)
    check_within_1ulp("slerp-early fp16", out, oo)


def test_one_model_on_fp16(E):
    """A layer range leaves one model: its raw delta is added to the base, alpha ignored (fast_fourier.py:171,256-257),
    in fp32 -- the same two roundings as the oracle's, so the same bits."""
    from shardmerge_b200.config import MergeModel
    from shardmerge_b200.writer import ShardLayer
    name = "model.layers.3.mlp.up_proj.weight"
    base, fts = draw((512, 2048), 54, "fp16", ("fp16", "fp16"))
    models = [MergeModel(model="org/ft0", base="org/base", alpha=0.3),
              MergeModel(model="org/ft1", base="org/base", alpha=0.5, start_layer=5)]
    tensors = {"org/base": {name: base}, "org/ft0": {name: fts[0]}, "org/ft1": {name: fts[1]}}
    fm = _merger(models, tensors)
    out = asyncio.run(fm._merge_layer(ShardLayer(0, "s", name, False), DEV))
    oo, info = oracle(base, fts[:1], alphas=(0.3,))
    check_decisions(fm, info)
    assert fm.last_info["branches"] == [] and out.dtype == torch.bfloat16
    assert np.array_equal(bits(out), oo)


# ---------------------------------------------------------------------------------------------------- trees and shapes
def check_tree(tag, fm, out, base_out, oo, info_ni, n_models, shape):
    """round 1 against the oracle's intermediates (info_ni: without the nested imaginary path), the final delta loosely
    (see the module docstring)"""
    names = {f"m{k}" for k in range(n_models)}
    round1 = [(a, b, t) for a, b, t in fm.last_tree if a in names and b in names]
    assert len(round1) == n_models // 2
    inter = info_ni["intermediates"]
    for a, b, t in round1:
        key = next(k for k in inter if set(k.split("_")) == {a, b})
        raw, resid, share = flip_accounted(t.cpu().numpy().reshape(shape), inter[key].reshape(shape), k=16)
        print(f"\n[{tag} round 1 {key}] raw {raw:.3e} flip-accounted {resid:.3e}")
        assert resid <= 1e-5, (tag, key, raw, resid, share)
    basef = O.widen(stored(base_out)).reshape(shape)
    do, dr = O.bf16_to_f32(bits(out)).reshape(shape) - basef, O.bf16_to_f32(oo).reshape(shape) - basef
    ratio = np.linalg.norm(do) / np.linalg.norm(dr)
    print(f"[{tag}] final delta rel-L2 vs oracle {rel_l2(do, dr):.3f}, norm ratio {ratio:.4f}")
    assert np.isfinite(do).all()
    assert rel_l2(do, dr) < 0.5 and abs(ratio - 1) < 0.05, (tag, rel_l2(do, dr), ratio)


def tree_vs_oracle(E, tag, base, fts):
    fm = _merger()
    out = run(E, fm, base, fts)
    oo, info = oracle(base, fts)
    check_decisions(fm, info)
    assert fm.last_info["branches"] == ["slerp"] * (len(fts) - 1)
    _, info_ni = oracle(base, fts, interp_imag=False)
    check_tree(tag, fm, out, base, oo, info_ni, len(fts), tuple(base.shape))
    return fm, out


@pytest.mark.parametrize("n_models", [3, 4])
def test_tree_on_fp32(E, n_models):
    """Rounds >= 2 on the step path: fp32 intermediates get their row pass into a free slot, carried models keep theirs.
    Every pair after the first runs on the workspace the earlier pairs used."""
    base, fts = draw((512, 2048), 60 + n_models, "fp32", ("fp32",) * n_models)
    fm, out = tree_vs_oracle(E, f"tree{n_models} fp32", base, fts)
    if n_models != 4:
        return
    # The last round pinned exactly, as test_fused_tree_matches_merge_sources_steps does for the fused tree: its two fp32
    # inputs (the tree's own round-1 results) through the tensor function, with the same t and cull, give the same tensor.
    from shardmerge_b200.tensor import functions as F
    (a0, a1, ta), (b0, b1, tb), _ = fm.last_tree
    w = {f"m{k}": a for k, a in enumerate(ALPHAS)}
    wa, wb = (w[a0] + w[a1]) / 2, (w[b0] + w[b1]) / 2
    x, y = (ta, tb) if float(ta.norm()) >= float(tb.norm()) else (tb, ta)     # larger norm takes role v0; t is not swapped
    m, _, _ = F.merge_tensors_fft2_slerp(x, y, t=wa / (wa + wb), device=DEV, t_sum=1.0, cutoff_pct=0.08, cull_pct=0.10)
    final = (base.float() + m.to(DEV) * E.f32(fm.last_info["target_norm"])).to(torch.bfloat16)
    u = bf16_ulp_distance(bits(out), bits(final))
    print(f"[tree4 fp32 last round vs the tensor function] bf16 exact {float((u == 0).mean()):.6f} max ulp {int(u.max())}")
    assert float((u == 0).mean()) >= 0.9999 and int(u.max()) <= 1, (float((u == 0).mean()), int(u.max()))


@pytest.mark.parametrize("n_models", [2, 3])
def test_stack_on_fp16(E, n_models):
    """A tensor with a leading dimension: column sweeps per slice, inv_rows' 1 / N over one slice, norms and order
    statistics over the whole tensor; fp16, with two models and with a tree of three."""
    shape = (3, 352, 512)
    base, fts = draw(shape, 70 + n_models, "fp16", ("fp16",) * n_models)
    if n_models == 2:
        fm, out = merged_vs_oracle(E, "stack fp16 x2", base, fts)
        assert tuple(out.shape) == shape
    else:
        tree_vs_oracle(E, "stack fp16 x3", base, fts)


@pytest.mark.parametrize("dt", ["fp16", "bf16"])
def test_stack_of_unchanged_tensors_adds_zero(E, dt):
    """Three finetunes that left a stacked tensor (e.g. frozen experts) as it was: both rounds take the add branch, the
    second one on a [R][C] intermediate and a model whose delta keeps the tensor's leading dimension."""
    shape = (3, 352, 512)
    base, _ = draw(shape, 75, dt, ())
    fts = [base.clone() for _ in range(3)]
    fm = _merger()
    out = run(E, fm, base, fts)
    oo, info = oracle(base, fts)
    check_decisions(fm, info)
    assert fm.last_info["branches"] == ["add", "add"] and tuple(out.shape) == shape
    assert np.array_equal(bits(out), oo)
    assert torch.equal(out.float(), base.to(torch.bfloat16).float())       # values: base + 0 turns a -0.0 into +0.0


def test_one_dimensional_fp32(E):
    """A layer-norm-like vector (mean 1.0): the R = 1 plans."""
    base, fts = draw((4096,), 81, "fp32", ("fp32", "fp32"), sig=(0.01, 0.013), mean=1.0, bs=0.1)
    fm, out = merged_vs_oracle(E, "1-D fp32", base, fts)
    assert fm.last_info["branches"] == ["slerp"] and tuple(out.shape) == (4096,)


def test_odd_row_length_fp32(E):
    """[256][333] has no packed real row transform: merge_sources merges the fp32 transposes and transposes back."""
    shape = (256, 333)
    base, fts = draw(shape, 82, "fp32", ("fp32", "fp32"))
    fm = _merger()
    out = run(E, fm, base, fts)
    oo, info = oracle(base, fts)
    check_decisions(fm, info)
    assert fm.last_info["branches"] == ["slerp"] and tuple(out.shape) == shape
    _, info_ni = oracle(base, fts, interp_imag=False)
    check_fft("odd C fp32", out, oo, fp32_result(fm).T, info_ni["merged_f32"])


# ---------------------------------------------------------------------------------------------------- range and non-finite
def test_fp16_deltas_beyond_the_fp16_range(E):
    """Elements moved from -60000 to +60000 (fp16 holds at most 65504): the fp32 delta carries them, nothing overflows.
    A handful of such elements dominate both spectra, so bins are decided by rounding there; the output is checked for
    the decisions, the norms and finiteness, and where it sits against the oracle is printed."""
    shape = (256, 1024)
    base, fts = draw(shape, 91, "fp16", ("fp16", "fp16"))
    for (r, c), (b, f0, f1) in (((5, 7), (-60000, 60000, 50000)), ((100, 200), (60000, -60000, -55000))):
        base[r, c], fts[0][r, c], fts[1][r, c] = b, f0, f1
    fm = _merger()
    out = run(E, fm, base, fts)
    oo, info = oracle(base, fts)
    check_decisions(fm, info)
    assert min(fm.last_info["norms"]) > 1.5e5
    assert torch.isfinite(out.float()).all()
    u = bf16_ulp_distance(bits(out), oo)
    print(f"\n[fp16 range] branches {fm.last_info['branches']}, bf16 within-1ulp of the oracle {float((u <= 1).mean()):.6f}, "
          f"at the moved elements {[int(u[5, 7]), int(u[100, 200])]} ulp")


def outcome(fn):
    try:
        return "bits", fn()
    except Exception as exc:               # noqa: BLE001 -- the exception type is the outcome
        return "raises", type(exc)


@pytest.mark.parametrize("n_models", [1, 2, 3])
def test_inf_in_an_fp16_finetune(E, n_models):
    """An Inf in one finetune: the same outcome as the oracle -- the same exception type, or the same bits.  One model:
    base + Inf is Inf (ValueError).  Two or three: that model's norm products are infinite, and pairing, which runs over
    finite products only, has nothing left to pair it with (ValueError) -- rather than a tensor of zeros (NaN -> 0)."""
    base, fts = draw((256, 1024), 92, "fp16", ("fp16",) * n_models)
    fts[0][17, 3] = float("inf")
    fm = _merger()
    got = outcome(lambda: bits(run(E, fm, base, fts)))
    with np.errstate(invalid="ignore", over="ignore"):
        want = outcome(lambda: oracle(base, fts)[0])
    print(f"\n[inf x{n_models}] ours {got[0]} {got[1] if got[0] == 'raises' else ''}, oracle {want[0]} "
          f"{want[1] if want[0] == 'raises' else ''}")
    assert got[0] == want[0]
    if got[0] == "raises":
        assert got[1] is want[1]
    else:
        assert np.array_equal(got[1], want[1])


# ---------------------------------------------------------------------------------------------------- without the oracle
def test_bf16_and_fp32_storage_agree(E):
    """The same values, all exactly bf16, stored as bf16 (the fused chain) and as fp32 (the step path): the same decisions,
    and the two results within the mid-size bounds of each other, the fused chain's fp32 merged delta taken from the same
    chain with an fp32 output."""
    R, C = 1024, 4096
    base, fts = draw((R, C), 21, "bf16", ("bf16", "bf16"))
    fm = _merger()
    fused = run(E, fm, base, fts)
    info_f = dict(fm.last_info)
    assert "swap" in info_f                                  # the fused chain ran: it records its device role decision
    base32, fts32 = base.float(), [ft.float() for ft in fts]
    steps = run(E, fm, base32, fts32)
    assert info_f["branches"] == fm.last_info["branches"] == ["slerp"]
    assert abs(info_f["target_norm"] / fm.last_info["target_norm"] - 1) < 1e-7
    m_steps = fp32_result(fm)
    ws = E.get_workspace(R, C, DEV, lane="dtype-invariance")
    m_fused = torch.empty((R, C), dtype=torch.float32, device=DEV)
    srcs = [E.make_source(base, ft, weight=a, name=f"m{k}") for k, (ft, a) in enumerate(zip(fts, ALPHAS))]
    pinfo = E.pair_merge_async(ws, srcs[0], srcs[1], None, m_fused, t=0.3 / 0.8, cutoff_pct=0.08, cull_pct=0.20,
                               layer_name=LAYER).resolve()
    assert pinfo["branch"] == "slerp" and pinfo["select_sticky"] == 0
    check_fft("bf16 vs fp32 storage", steps, bits(fused), m_steps, m_fused.cpu().numpy())


# ---------------------------------------------------------------------------------------------------- from files to files
@pytest.mark.parametrize("dt", ["fp16", "fp32"])
def test_merge_checkpoint_files(E, tmp_path, dt):
    """FourierMerge.merge() on a Llama-shaped fp16 / fp32 checkpoint from files to files: the output verifies, every tensor
    is written in the configured output dtype (bf16 -- the writer casts pass-through tensors too, shard/writer.py:133),
    pass-through tensors are the is_input / is_output model's values, every merged tensor meets the FFT bounds."""
    from safetensors.torch import load_file
    from shardmerge_b200 import validate
    from shardmerge_b200.config import MergeConfig, MergeModel
    from shardmerge_b200.index import LocalSafetensorsIndex
    from shardmerge_b200.merge.fast_fourier import FourierMerge
    from tests.lora_util import llama_shapes, random_model, write_model
    shapes = llama_shapes(layers=2)
    base = random_model(shapes, 0, dtype=DT[dt])
    fts = []
    for k, s in enumerate(SIG[:2]):
        g = torch.Generator().manual_seed(10 + k)
        fts.append({n: (t.float() + s * torch.randn(t.shape, generator=g)).to(DT[dt]) for n, t in base.items()})
    write_model(tmp_path / "org" / "base", base)
    for k, ft in enumerate(fts):
        write_model(tmp_path / "org" / f"ft{k}", ft)
    cfg = MergeConfig(finetune_merge=[MergeModel(model="org/ft0", base="org/base", alpha=ALPHAS[0], is_input=True),
                                      MergeModel(model="org/ft1", base="org/base", alpha=ALPHAS[1], is_output=True)],
                      output_base_model="org/base", output_dir=str(tmp_path / "out"), device="cuda", storage_dir=str(tmp_path))
    asyncio.run(FourierMerge(cfg, index_manager=LocalSafetensorsIndex(cfg.storage_path)).merge(DEV))
    rep = validate.verify_output(tmp_path / "out", expected_dtype=cfg.output_astype, expected_shapes=shapes)
    assert rep.ok and rep.tensors == len(shapes), rep.summary()
    got = {}
    for f in sorted((tmp_path / "out").glob("*.safetensors")):
        got.update(load_file(str(f)))
    passthrough = {"model.embed_tokens.weight": fts[0], "model.norm.weight": fts[1], "lm_head.weight": fts[1]}
    for name, src in passthrough.items():
        assert torch.equal(got[name].view(torch.int16), src[name].to(torch.bfloat16).view(torch.int16)), name
    merged = [n for n in shapes if n not in passthrough]
    assert len(merged) == 18
    for name in merged:
        b, f = base[name].to(DEV), [ft[name].to(DEV) for ft in fts]
        fm = _merger()
        again = run(E, fm, b, f)                      # the same tensor through merge_sources: its fp32 merged delta
        assert torch.equal(again.cpu().view(torch.int16), got[name].view(torch.int16)), name
        oo, info = oracle(b, f)
        check_decisions(fm, info)
        _, info_ni = oracle(b, f, interp_imag=False)
        check_fft(f"{dt} {name}", got[name], oo, fp32_result(fm), info_ni["merged_f32"])
