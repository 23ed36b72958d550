"""GPU parity at the BASELINE.json shapes themselves (VERDICT r1, "next round" item 1).  Run with `pytest -m gpu`.

  (a) forward spectrum and inverse transform of every 2-D Llama-3.1-8B / 70B / TinyLlama shape against an independent
      fp64 FFT (torch.fft on the device -- TEST-ONLY checker, cuFFT never runs on the product path), through
      Plan.row_freq(): one case per packed kernel instantiation the bench times, plus the one-row kernels
      (k_row_fwd_tma / k_row_inv_tma, k_row_fwd_ct / k_row_inv_ct) at the shapes and input types that select them;
  (b) FourierMerge.merge_sources against oracle/oracle_np.merge_layer at 1024x4096, 4096x4096, 14336x4096, 4096x14336
      and 8192x8192 with north_star's bounds: fp32 merged delta rel-L2 <= 1e-5 once the flipped bins are set aside
      (and outright when nothing flips), bf16 within 1 ulp on >= 99.99 % when nothing flips; flips are listed;
  (c) the goldens' stage taps (the reference's own spectra fft0 / fft1) through the CUDA interpolate_fft_components:
      zero / cull masks identical to the reference's res_real_noimag;
  (d) every record is printed and, when SM_PARITY_REPORT names a file, collected there as JSON (profiles/r02_parity.json
      is one such report): per shape raw rel-L2, flip-accounted rel-L2, flipped bins, within-1-ulp, exact, max-abs-diff;
  (e) when oracle/_ref is present (make oracle_ref), the REFERENCE ITSELF with device="cuda" as the oracle.
"""
import glob
import json
import os
import time
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import oracle_np as O
from tests.parity_util import bf16_ulp_distance, flip_accounted, flipped_bins, rel_l2

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
ROOT = Path(__file__).resolve().parent.parent
REPORT = Path(os.environ["SM_PARITY_REPORT"]) if os.environ.get("SM_PARITY_REPORT") else None

LLAMA8B = [(4096, 4096), (1024, 4096), (14336, 4096), (4096, 14336)]
LLAMA70B = [(8192, 8192), (1024, 8192), (28672, 8192), (8192, 28672)]
TINYLLAMA = [(2048, 2048), (256, 2048), (5632, 2048), (2048, 5632)]


def record(section, key, **values):
    """Print one record and append it to the parity report, if one is asked for (a JSON file that survives `pytest -q`)."""
    if REPORT is not None:
        try:
            REPORT.parent.mkdir(parents=True, exist_ok=True)
            doc = json.loads(REPORT.read_text()) if REPORT.exists() else {}
            doc.setdefault(section, {})[key] = values
            REPORT.write_text(json.dumps(doc, indent=1, sort_keys=True))
        except OSError:
            pass
    print(f"\n[{section}] {key}: " + ", ".join(f"{k}={v}" for k, v in values.items()))


@pytest.fixture(scope="module")
def E():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from shardmerge_b200 import engine
    return engine


def bits(t):
    return t.contiguous().view(torch.int16).cpu().numpy().view(np.uint16)


def synth(shape, seed):
    g = torch.Generator(device=DEV).manual_seed(1234 + seed)
    base = (0.02 * torch.randn(shape, generator=g, device=DEV)).to(torch.bfloat16)
    fts = []
    for k, sig in enumerate((0.002, 0.0026)):
        gk = torch.Generator(device=DEV).manual_seed(100000 * (k + 1) + seed)
        fts.append((base.float() + sig * torch.randn(shape, generator=gk, device=DEV)).to(torch.bfloat16))
    return base, fts


def _rel(a, b):
    return float(((a - b).abs() ** 2).sum().sqrt() / (b.abs() ** 2).sum().sqrt())


def forward_inverse_check(E, shape, seed=0, f32=False):
    """-> (forward rel-L2 vs fp64 rfft2, inverse rel-L2 vs the input given the fp64 spectrum).
    f32: the forward pass reads the delta as an fp32 source instead of forming it from the bf16 pair."""
    R, C = shape
    base, fts = synth(shape, seed)
    delta = fts[0].float() - base.float()
    ws = E.get_workspace(R, C, DEV)
    pl = ws.plan
    ws.ctl.zero_()
    src = E.Source(x32=delta) if f32 else E.Source(base=base, ft=fts[0])
    E.fwd_rows(ws, 0, src, E.D_SUMSQ0)
    E.fwd_cols(ws, 0, scale=1.0)
    freq = pl.row_freq().to(DEV)
    ref = torch.fft.rfft2(delta.double())                     # [R][Ch+1] complex128, natural row order
    ref_stored = ref[freq]                                     # stored row i holds frequency freq[i]
    got = torch.complex(ws.re[0][:, : pl.Ch + 1].double(), ws.im[0][:, : pl.Ch + 1].double())
    fwd = _rel(got, ref_stored)
    pad_ok = bool((ws.re[0][:, pl.Ch + 1:] == 0).all()) and bool((ws.im[0][:, pl.Ch + 1:] == 0).all())
    del got
    # inverse, fed with the checker's spectrum (rounded to fp32): the inverse kernels are checked on their own,
    # not only as the inverse of our forward transform
    ws.re[0][:, : pl.Ch + 1] = ref_stored.real.float()
    ws.im[0][:, : pl.Ch + 1] = ref_stored.imag.float()
    del ref, ref_stored
    out = torch.empty((R, C), dtype=torch.float32, device=DEV)
    E.inv_cols(ws, ws.re[0], ws.im[0], cull=False)
    E.inv_rows(ws, ws.re[0], ws.im[0], False, 1.0, None, out, check_ifft=True)
    inv = _rel(out.double(), delta.double())
    return fwd, inv, pad_ok, pl.describe()


@pytest.mark.parametrize("shape", LLAMA8B + LLAMA70B + TINYLLAMA)
def test_forward_and_inverse_vs_fp64_fft(E, shape):
    fwd, inv, pad_ok, desc = forward_inverse_check(E, shape)
    record("fft_vs_fp64", f"{shape[0]}x{shape[1]}", forward_rel_l2=fwd, inverse_rel_l2=inv, plan=desc)
    assert fwd <= 1e-6 and inv <= 1e-6 and pad_ok, (fwd, inv, pad_ok)
    E.clear_caches()
    torch.cuda.empty_cache()


# The paired-row kernels take bf16 pairs of rows only.  An fp32 source, an odd row count or a single row selects the one-row
# kernels instead: k_row_fwd_tma / k_row_inv_tma where the row and its staging fit in shared memory (fp32 at the Llama-8B
# shapes; 4095x4096, 2047x2048), else k_row_fwd_ct / k_row_inv_ct (a single row; fp32 at 8192x28672).
ONE_ROW = [(s, True) for s in LLAMA8B] + [((4095, 4096), False), ((2047, 2048), False), ((1, 4096), False),
                                         ((1, 8192), False), ((8192, 28672), True)]


@pytest.mark.parametrize("shape,f32", ONE_ROW, ids=lambda v: f"{v[0]}x{v[1]}" if isinstance(v, tuple) else ("f32" if v else "bf16"))
def test_one_row_kernels_vs_fp64_fft(E, shape, f32):
    fwd, inv, pad_ok, desc = forward_inverse_check(E, shape, f32=f32)
    record("fft_vs_fp64_one_row", f"{shape[0]}x{shape[1]}" + (" f32" if f32 else ""), forward_rel_l2=fwd, inverse_rel_l2=inv, plan=desc)
    assert fwd <= 1e-6 and inv <= 1e-6 and pad_ok, (fwd, inv, pad_ok)
    E.clear_caches()
    torch.cuda.empty_cache()


def _merger():
    from shardmerge_b200.config import MergeConfig
    from shardmerge_b200.index import InMemoryIndex
    from shardmerge_b200.merge.fast_fourier import FourierMerge
    cfg = MergeConfig(finetune_merge=[], output_base_model="org/base", output_dir="/tmp/unused")
    return FourierMerge(cfg, index_manager=InMemoryIndex({}))


def parity_metrics(out_bits, ref_bits, base_bits, shape):
    """north_star's end-to-end figures for one tensor: bf16 ulp statistics and max-abs-diff of the outputs, rel-L2 of the
    merged deltas (output - base, what the bf16 outputs can resolve) raw and with the flipped bins set aside."""
    u = bf16_ulp_distance(out_bits, ref_bits)
    of, rf, bf = O.bf16_to_f32(out_bits), O.bf16_to_f32(ref_bits), O.bf16_to_f32(base_bits)
    return dict(within_1ulp=float((u <= 1).mean()), exact=float((u == 0).mean()), max_ulp=int(u.max()),
                max_abs_diff=float(np.abs(of - rf).max()), max_abs_ref=float(np.abs(rf).max()))


@pytest.mark.parametrize("shape,seed", [((1024, 4096), 31), ((4096, 4096), 32), ((14336, 4096), 33), ((4096, 14336), 34),
                                        ((8192, 8192), 35)])
def test_merge_vs_oracle_full_size(E, shape, seed):
    """FourierMerge.merge_sources (the fused chain: what bench.py times) vs the numpy oracle on the same bits."""
    from shardmerge_b200.tensor import functions as F
    base, fts = synth(shape, seed)
    fm = _merger()
    srcs = [E.make_source(base, fts[k], weight=a, name=f"m{k}") for k, a in enumerate((0.3, 0.5))]
    out = fm.merge_sources(srcs, base, torch.device(DEV), layer_name="model.layers.0.x")
    assert fm.last_info["branches"] == ["slerp"]
    # fp32 intermediates: the merged delta through the tensor-function API (fp32 in / out) on identical fp32 deltas
    d0 = fts[0].float() - base.float(); d1 = fts[1].float() - base.float()
    a_, b_ = (d0, d1) if float(d0.norm()) >= float(d1.norm()) else (d1, d0)
    m, _, _ = F.merge_tensors_fft2_slerp(a_, b_, t=0.3 / 0.8, device=DEV, t_sum=1.0, cutoff_pct=0.08, cull_pct=0.20)
    m = m.numpy()
    bb, f0, f1 = bits(base), bits(fts[0]), bits(fts[1])
    out_bits = bits(out)
    del d0, d1, a_, b_, out, srcs, base, fts
    E.clear_caches(); torch.cuda.empty_cache()
    t0 = time.time()
    info = {}
    oo = O.merge_layer(bb, [dict(base=bb, ft=f0, alpha=0.3, name="m0"), dict(base=bb, ft=f1, alpha=0.5, name="m1")], info=info)
    oracle_s = time.time() - t0
    assert info["branches"] == ["slerp"]
    assert abs(fm.last_info["target_norm"] / info["target_norm"] - 1) < 1e-6
    mo = info["merged_f32"].reshape(shape)                                 # oracle: merged delta x target_norm, fp32
    m = m * np.float32(info["target_norm"])
    # flips are expected at ~1e-6 per element (SURVEY 7.3-1: ~2.5e-7 per element and decision type, two mirror bins
    # each), so the number of bins set aside scales with the tensor: at most 4e-6 of the spectrum
    kmax = max(16, int(4e-6 * m.size))
    raw, resid, share = flip_accounted(m, mo, k=kmax)
    flips = flipped_bins(m, mo, tol=1e-5, kmax=kmax)
    flips["bins"] = flips["bins"][:24]
    met = parity_metrics(out_bits, oo, bb, shape)
    record("merge_vs_oracle", f"{shape[0]}x{shape[1]}", fp32_rel_l2_raw=raw, fp32_rel_l2_flip_accounted=resid,
           flipped_bins=flips["bins"], n_flipped=flips["n"], bins_allowed=kmax, oracle_seconds=round(oracle_s, 1), **met)
    assert resid <= 1e-5, (raw, resid, share)                             # north_star: fp32 intermediates
    if flips["n"] == 0:
        assert raw <= 1e-5 and met["within_1ulp"] >= 0.9999, (raw, met)   # north_star: bf16 within 1 ulp on >= 99.99 %
    else:
        # every flipped Hermitian bin pair is one sinusoid over the whole tensor; its amplitude is far below a typical
        # bf16 ulp, so it moves a small fraction of roundings (those with near-zero base values)
        assert met["within_1ulp"] >= 0.99, met
    assert met["max_abs_diff"] <= 2.0 ** -7 * met["max_abs_ref"] + 1e-4


def test_golden_taps_through_cuda_blend(E, golden_dir):
    """The reference's own spectra (stage taps fft0 / fft1 of the fixtures) through the CUDA blend: the result's zero set
    (culled bins) must be the reference's, values within fp32 reduction error (same bar as the oracle's test,
    tests/test_oracle_golden.py:44-55)."""
    from shardmerge_b200.tensor import functions as F
    for f in sorted(glob.glob(str(golden_dir / "tensor_*.npz"))):
        d = np.load(f)
        r = F.interpolate_fft_components(torch.from_numpy(d["fft0"]), torch.from_numpy(d["fft1"]), 0.375, DEV, t_sum=1.0,
                                         cutoff_pct=0.08, cull_pct=0.20, interp_imag=False).cpu().numpy()
        ref = d["res_real_noimag"]
        # the CUDA path keeps the Hermitian half spectrum (columns 0..C/2) and mirrors it on the way out
        C = ref.shape[-1]
        half = (slice(None),) * (ref.ndim - 1) + (slice(0, C // 2 + 1),)
        mism = int(np.count_nonzero((r.real[half] == 0) != (ref[half] == 0)))
        err = rel_l2(r.real[half], ref[half])
        record("golden_taps_cuda_blend", Path(f).stem, mask_mismatches=mism, rel_l2=err)
        assert mism == 0, (f, mism)
        assert err < 1e-6, (f, err)
        assert np.array_equal(r.imag[half], d["fft0"].imag[half])         # interp_imag=False: Im X0 (functions.py:160)
        # the other tensor-function entry points on the same taps
        inv = F.ifft_transform(torch.from_numpy(d["res"]), DEV).numpy()
        assert rel_l2(inv, d["merged"]) < 2e-6, f
        ar = F.arithmetic_fft_components(torch.from_numpy(d["fft0"]), torch.from_numpy(d["fft1"]), 1.0, True, DEV,
                                         do_imag=False).numpy()
        oa = O.arithmetic_fft_components(d["fft0"], d["fft1"], 1.0, True, do_imag=False)
        # (the C ABI packs a full spectrum into the Hermitian half with the projection (X[k] + conj X[-k]) / 2, so the
        # reference's not-quite-Hermitian MKL spectra come out within rounding, not bit for bit)
        assert rel_l2(ar.real[half], np.asarray(oa).real[half]) < 1e-6, f
        ta = F.task_arithmetic_fft2(torch.from_numpy(d["v0"]), torch.from_numpy(d["v1"]), 1.0, DEV, agreement=True).numpy()
        to = O.task_arithmetic_fft2(d["v0"], d["v1"], 1.0, agreement=True)
        assert flip_accounted(ta, np.asarray(to), k=8)[1] < 1e-5, f


# ------------------------------------------------------------------------------------------ the reference itself
def _ref():
    from oracle import ref_runner as RR
    if not RR.available():
        pytest.skip("needs a copy of the reference in oracle/_ref (make oracle_ref REFERENCE=<checkout of the reference>)")
    return RR


@pytest.mark.parametrize("shape,seed", [((256, 2048), 41), ((1024, 4096), 42), ((4096, 4096), 43), ((14336, 4096), 44)])
def test_merge_vs_reference_on_cuda(E, shape, seed):
    """SURVEY 8c: the unmodified reference (`FourierMerge._merge_layer`, shard/merge/fast_fourier.py:103-276) run with
    device="cuda" on this box is the parity oracle for large tensors (cuFFT + CUDA reductions; its CPU path's fp32
    norms are biased at these sizes).  The reference's cuFFT calls are the CHECKER here, never the product path."""
    RR = _ref()
    base, fts = synth(shape, seed)
    fm = _merger()
    srcs = [E.make_source(base, fts[k], weight=a, name=f"m{k}") for k, a in enumerate((0.3, 0.5))]
    out = fm.merge_sources(srcs, base, torch.device(DEV), layer_name="model.layers.0.x")
    out_bits, bb = bits(out), bits(base)
    t0 = time.time()
    ref = RR.merge_layer(base, fts, [0.3, 0.5], device=DEV)
    torch.cuda.synchronize()
    ref_s = time.time() - t0
    ref_bits = bits(ref)
    degenerate = float((ref_bits == bb).mean())
    met = parity_metrics(out_bits, ref_bits, bb, shape)
    basef = O.bf16_to_f32(bb)
    raw, resid, share = flip_accounted(O.bf16_to_f32(out_bits) - basef, O.bf16_to_f32(ref_bits) - basef, k=16)
    floor = {}
    if shape[0] * shape[1] <= 1024 * 4096:
        # the floor any implementation faces: the SAME reference code, CPU (MKL) against CUDA (cuFFT), same metric
        # (SURVEY 7.3-1c; at larger sizes the CPU reference's biased fp32 norms make the comparison meaningless)
        ref_cpu = bits(RR.merge_layer(base.cpu(), [f.cpu() for f in fts], [0.3, 0.5], device="cpu"))
        fm_ = parity_metrics(ref_cpu, ref_bits, bb, shape)
        floor = dict(reference_cpu_vs_cuda_within_1ulp=fm_["within_1ulp"], reference_cpu_vs_cuda_exact=fm_["exact"])
    record("merge_vs_reference_cuda", f"{shape[0]}x{shape[1]}", reference_seconds=round(ref_s, 2),
           reference_equals_base_fraction=degenerate, bf16_delta_rel_l2_raw=raw, bf16_delta_rel_l2_flip_accounted=resid,
           **floor, **met)
    if degenerate > 0.5:
        pytest.skip("the reference degenerates on CUDA for this input (NaN imaginary path, SURVEY 7.3-2): recorded only")
    # the bf16 outputs quantise the delta (|delta| ~ 0.1 ulp of |base|), so the delta comparison resolves ~1e-2 only;
    # the ulp statistics are the tight end-to-end check here.  One flipped bin weighs 1 / sqrt(N): small tensors show it more
    # (measured 0.9940 at 256x2048, 0.9978 - 0.9986 at the Llama shapes; the reference's own CPU path reaches 0.92 at 1024x4096)
    assert met["within_1ulp"] >= (0.985 if shape[0] * shape[1] < (1 << 21) else 0.99), met
    assert met["max_abs_diff"] <= 2.0 ** -7 * met["max_abs_ref"] + 1e-4


@pytest.mark.parametrize("shape,seed", [((1024, 4096), 51), ((4096, 4096), 52)])
def test_tensor_function_vs_reference_on_cuda(E, shape, seed):
    """merge_tensors_fft2_slerp, fp32 in / fp32 out, ours vs the reference's on device="cuda": north_star's fp32 bound."""
    RR = _ref()
    from shardmerge_b200.tensor import functions as F
    RF = RR.load()[0]
    base, fts = synth(shape, seed)
    d0 = fts[1].float() - base.float(); d1 = fts[0].float() - base.float()     # larger norm first, as _merge_layer orders them
    kw = dict(t=0.375, t_sum=1.0, cutoff_pct=0.08, cull_pct=0.20)
    m, n0, n1 = F.merge_tensors_fft2_slerp(d0, d1, device=DEV, **kw)
    r, rn0, rn1 = RF.merge_tensors_fft2_slerp(d0.clone(), d1.clone(), device=DEV, **kw)
    m, r = m.numpy(), r.cpu().numpy()
    kmax = max(16, int(4e-6 * m.size))
    raw, resid, share = flip_accounted(m, r, k=kmax)
    flips = flipped_bins(m, r, tol=1e-5, kmax=kmax)
    flips["bins"] = flips["bins"][:24]
    record("tensor_function_vs_reference_cuda", f"{shape[0]}x{shape[1]}", fp32_rel_l2_raw=raw, fp32_rel_l2_flip_accounted=resid,
           n_flipped=flips["n"], flipped_bins=flips["bins"], norm_rel_err=[abs(n0 / rn0 - 1), abs(n1 / rn1 - 1)],
           reference_zero_fraction=float((r == 0).mean()))
    assert abs(n0 / rn0 - 1) < 1e-6 and abs(n1 / rn1 - 1) < 1e-6
    if float((r == 0).mean()) > 0.5:
        pytest.skip("the reference degenerates on CUDA for this input: recorded only")
    assert resid <= 1e-5, (raw, resid, share)


# ------------------------------------------------------------------------------------------ lengths that do not factor
AWKWARD = [(74, 296), (1002, 668), (18944, 3584), (3584, 18944), (16032, 8192), (1, 18944), (167, 4096)]


@pytest.mark.parametrize("shape", AWKWARD)
def test_generic_radix_lengths_vs_fp64_fft(E, shape):
    """VERDICT r1 missing #1: the reference's torch.fft takes any length (functions.py:55-58).  Prime factors above 13
    (37 in Qwen2.5's 18944, 167 in Llama-3's 128256-row embeddings; 16032 = 2^5 * 3 * 167 is the CI-sized stand-in for
    those) run as generic radix stages: forward and inverse against the fp64 FFT like every other shape."""
    if shape[0] == 1:
        R, C = shape
        g = torch.Generator(device=DEV).manual_seed(C)
        x = torch.randn((1, C), generator=g, device=DEV, dtype=torch.float32)
        ws = E.get_workspace(1, C, DEV)
        ws.ctl.zero_()
        E.fwd_rows(ws, 0, E.Source(x32=x), E.D_SUMSQ0)
        E.fwd_cols(ws, 0, scale=1.0)
        ref = torch.fft.rfft(x.double(), dim=1)
        got = torch.complex(ws.re[0][:, : C // 2 + 1].double(), ws.im[0][:, : C // 2 + 1].double())
        fwd = _rel(got, ref)
        out = torch.empty((1, C), dtype=torch.float32, device=DEV)
        E.inv_rows(ws, ws.re[0], ws.im[0], False, 1.0, None, out, check_ifft=True)
        inv = _rel(out.double(), x.double())
        desc = ws.plan.describe()
    else:
        fwd, inv, pad_ok, desc = forward_inverse_check(E, shape, seed=3)
        assert pad_ok
    record("fft_vs_fp64_generic_radix", f"{shape[0]}x{shape[1]}", forward_rel_l2=fwd, inverse_rel_l2=inv, plan=desc)
    assert fwd <= 1e-6 and inv <= 1e-6, (fwd, inv)
    E.clear_caches()
    torch.cuda.empty_cache()


def test_config5_embedding_shape_merge(E):
    """BASELINE config 5: the 128256 x 8192 embedding / lm_head shape (1.05 G elements) through the tensor-level merge on
    ONE B200 (it fits: 17 GB of planes).  CI-sized stand-in 16032 x 8192 (same awkward factors 3 * 167) is checked
    against the reference itself on device="cuda" when oracle/_ref is present; the full shape is merged, timed, and
    checked through size-independent properties (finite, norm of the merged delta, output = base where both deltas
    are zero is covered elsewhere)."""
    from oracle import ref_runner as RR
    fm = _merger()
    # --- CI size vs the reference on CUDA
    shape = (16032, 8192)
    base, fts = synth(shape, 61)
    srcs = [E.make_source(base, fts[k], weight=a, name=f"m{k}") for k, a in enumerate((0.3, 0.5))]
    out = fm.merge_sources(srcs, base, torch.device(DEV), layer_name="model.layers.0.x")
    assert fm.last_info["branches"] == ["slerp"]
    if RR.available():
        ref = RR.merge_layer(base, fts, [0.3, 0.5], device=DEV)
        met = parity_metrics(bits(out), bits(ref), bits(base), shape)
        record("config5", "16032x8192_vs_reference_cuda", **met)
        assert met["within_1ulp"] >= 0.99, met
        del ref
    del base, fts, srcs, out
    E.clear_caches(); torch.cuda.empty_cache()
    # --- full size
    shape = (128256, 8192)
    base, fts = synth(shape, 62)
    srcs = [E.make_source(base, fts[k], weight=a, name=f"m{k}") for k, a in enumerate((0.3, 0.5))]
    out = fm.merge_sources(srcs, base, torch.device(DEV), layer_name="model.layers.0.x")      # warm-up: plans, tables
    torch.cuda.synchronize()
    t0 = time.time()
    out = fm.merge_sources(srcs, base, torch.device(DEV), layer_name="model.layers.0.x")
    torch.cuda.synchronize()
    dt = time.time() - t0
    assert fm.last_info["branches"] == ["slerp"]
    d = out.float() - base.float()
    d0 = fts[0].float() - base.float()
    ratio = float(d.norm() / d0.norm())
    finite = bool(torch.isfinite(out.float()).all())
    record("config5", "128256x8192_one_gpu", seconds=round(dt, 3), params_per_s=shape[0] * shape[1] / dt,
           merged_delta_norm_over_delta0_norm=ratio, finite=finite, plan=E.get_plan(*shape, DEV).describe())
    assert finite and 0.3 < ratio < 1.5
    E.clear_caches(); torch.cuda.empty_cache()


@pytest.mark.parametrize("case", ["arith_1024x4096", "tree4_512x2048", "norm_1d_8192", "norm_1d_4096"])
def test_other_branches_vs_reference_on_cuda(E, case):
    """The branches the BASELINE inputs do not take, against the unmodified reference on device="cuda": the arithmetic-FFT
    branch (norm ratio < 0.1, fast_fourier.py:226-232), a 4-finetune pair tree (:171-254; pinned loosely, see DESIGN 4) and 1-D
    tensors (layer norms; SURVEY 7.3-2 asked whether the reference's nested imaginary path degenerates there on CUDA)."""
    RR = _ref()
    g = torch.Generator(device=DEV).manual_seed(len(case) * 17)
    if case.startswith("norm_1d"):
        n = int(case.split("_")[-1])
        base = (1.0 + 0.1 * torch.randn((n,), generator=g, device=DEV)).to(torch.bfloat16)
        sig, alphas = (0.01, 0.013), (0.3, 0.5)
        shape = (n,)
    elif case.startswith("arith"):
        shape, sig, alphas = (1024, 4096), (0.0026, 0.0001), (0.3, 0.5)
        base = (0.02 * torch.randn(shape, generator=g, device=DEV)).to(torch.bfloat16)
    else:
        shape, sig, alphas = (512, 2048), (0.002, 0.0026, 0.0023, 0.0029), (0.3, 0.5, 0.4, 0.2)
        base = (0.02 * torch.randn(shape, generator=g, device=DEV)).to(torch.bfloat16)
    fts = [(base.float() + s * torch.randn(shape, generator=g, device=DEV)).to(torch.bfloat16) for s in sig]
    fm = _merger()
    srcs = [E.make_source(base, f, weight=a, name=f"m{k}") for k, (f, a) in enumerate(zip(fts, alphas))]
    layer = "model.layers.0.input_layernorm.weight" if len(shape) == 1 else "model.layers.0.mlp.up_proj.weight"
    out = fm.merge_sources(srcs, base, torch.device(DEV), layer_name=layer)
    ref = RR.merge_layer(base, fts, list(alphas), device=DEV, layer=layer)
    ob, rb, bb = bits(out), bits(ref), bits(base)
    met = parity_metrics(ob, rb, bb, shape)
    degenerate = float((rb == bb).mean())
    basef = O.bf16_to_f32(bb)
    do, dr = O.bf16_to_f32(ob) - basef, O.bf16_to_f32(rb) - basef
    rel = float(np.linalg.norm(do - dr) / max(np.linalg.norm(dr), 1e-30))
    record("other_branches_vs_reference_cuda", case, branches=fm.last_info["branches"], reference_equals_base_fraction=degenerate,
           bf16_delta_rel_l2=rel, **met)
    if degenerate > 0.5:
        pytest.skip("the reference degenerates on CUDA for this input (merged delta = 0): recorded only")
    if case.startswith("arith"):
        assert fm.last_info["branches"] == ["arith"] and met["within_1ulp"] >= 0.999, met
    elif case.startswith("tree4"):
        assert fm.last_info["branches"] == ["slerp"] * 3
        assert rel < 0.6 and abs(np.linalg.norm(do) / np.linalg.norm(dr) - 1) < 0.1, rel
    else:
        assert fm.last_info["branches"] == ["slerp"] and met["within_1ulp"] >= 0.97, met
