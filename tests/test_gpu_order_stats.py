"""Order statistics on adversarial spectra.

The SLERP blend reproduces the reference only if both of its thresholds are the exact key at the reference's rank
(torch.sort of the full, mirrored |Re|).  Two engines find those keys from a sampled window -- the fused statistics
(csrc/kernels_fstats.cu, every SLERP pair above 2^20 elements) and the sampled mode of sm_select_kth_abs
(csrc/kernels_stats.cu, above 4 Mi keys) -- and either one must give the exact key with status 0 or raise its status
with a NaN threshold, never a finite wrong key.  Here they run on distributions that stress the window: exact zeros,
tied keys (the warp-combined "dense" path), ties confined to the multiplicity-1 edge columns, products that underflow,
a gap at the rank, NaN / Inf keys, ranks at either end, and ties packed into one pass CTA (side-list overflow).  The
exhaustive select is the control.  The public functions must redo a flagged tensor with the exhaustive select.
"""
import logging
import zlib

import numpy as np
import pytest
import torch

from oracle import oracle_np as O
from tests.parity_util import bf16_ulp_distance, flip_accounted, rel_l2
from tests.test_gpu_parity import _np_blend, half_weights, planes_to_numpy

DEV = "cuda:0"
gpu = pytest.mark.gpu
T = 0.375


@pytest.fixture(scope="module")
def E():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from shardmerge_b200 import engine
    return engine


# ------------------------------------------------------------------------------------------
# exact reference
# ------------------------------------------------------------------------------------------
def exact_keys(planes, w, ranks):
    """The keys torch.sort of the full (mirrored) |Re| of half-planar `planes` puts at `ranks`: every stored bin repeated
    by its Hermitian multiplicity `w`, NaN sorted last and +Inf just below it, a rank past the end -> the last key."""
    keys = np.concatenate([np.repeat(np.abs(np.asarray(p, dtype=np.float32)).ravel(), w.ravel()) for p in planes])
    ks = [min(int(k), keys.size - 1) for k in ranks]
    part = np.partition(keys, sorted(set(ks)))
    return [np.float32(part[k]) for k in ks]


def same_key(got, want):
    got, want = np.float32(got), np.float32(want)
    return bool(np.isnan(got) and np.isnan(want)) or got.view(np.uint32) == want.view(np.uint32)


def hermitian_full(half, C):
    """half-planar [R][C//2+1] real part -> the full [R][C] real part of a Hermitian spectrum (exact mirror)."""
    R, Ch = half.shape[0], C // 2
    mr = (-np.arange(R)) % R
    h = half.copy()
    for e in (0, Ch):                                       # edge columns are their own mirror: Re[r] == Re[-r]
        h[:, e] = np.where(np.arange(R) <= mr, h[:, e], h[mr, e])
    full = np.empty((R, C), dtype=h.dtype)
    full[:, : Ch + 1] = h
    full[:, Ch + 1:] = h[mr][:, 1:Ch][:, ::-1]
    return h, full


def test_exact_keys_match_full_sort():
    """The weighted-repeat reference against oracle_np.kth_abs (the reference's torch.sort) on full np.fft.fft2 spectra,
    with ties, zeros, NaN and +-Inf, one and two planes, every kind of rank."""
    rng = np.random.default_rng(11)
    R, C = 24, 32
    halves, fulls = [], []
    for s in range(2):
        F = np.fft.fft2(rng.standard_normal((R, C)))
        F = 0.5 * (F + np.conj(F[(-np.arange(R)) % R][:, (-np.arange(C)) % C]))     # exactly Hermitian
        re = F.real.astype(np.float32)
        re[np.abs(re) < 0.5] = 0.0
        re[re > 4.0] = np.float32(4.0)
        full = re.copy()
        for (r, c), v in zip([(1, 3), (2, 0), (5, C // 2), (7, 9)], [np.nan, np.inf, -np.inf, np.nan if s else -np.inf]):
            full[r, c] = full[(-r) % R, (-c) % C] = v
        h, full2 = hermitian_full(full[:, : C // 2 + 1], C)
        assert np.array_equal(full2.view(np.uint32), full.view(np.uint32))
        halves.append(h); fulls.append(full)
    w = half_weights(R, C)
    for planes, fl in (([halves[0]], fulls[0]), (halves, np.concatenate([f.ravel() for f in fulls]))):
        n = np.abs(fl).size
        ranks = [0, 1, n // 3, n // 2, n - 9, n - 5, n - 2, n - 1, n, n + 7]
        got = exact_keys(planes, w, ranks)
        for k, g in zip(ranks, got):
            assert same_key(g, O.kth_abs(np.abs(fl), k)), (k, g, O.kth_abs(np.abs(fl), k))


# ------------------------------------------------------------------------------------------
# plane generators: half-planar [R][Ch+1] fp32 real parts of two spectra, and the ranks to test
# ------------------------------------------------------------------------------------------
def _gauss(rng, R, Ch):
    p0 = (rng.standard_normal((R, Ch + 1)) * 0.7).astype(np.float32)
    p1 = (0.5 * p0 + 0.6 * rng.standard_normal((R, Ch + 1))).astype(np.float32)
    return p0, p1


def _tie_values(n, exp):
    """n distinct keys whose low 18 bits are zero: each sits on the lower edge of a sample-histogram bin."""
    return np.array([(1.0 + j / 32.0) * 2.0 ** exp for j in range(n)], dtype=np.float32)


def _below(planes, w, v):
    return int(sum((w * (np.abs(p) < v)).sum() for p in planes))


def case_planes(name, R, C, seed=0):
    """-> dict(p0, p1, cut=[2-plane ranks], one=[1-plane ranks on p0], cull=[cull fractions], strict, sampled_strict):
    strict -- the fused statistics must be exact; sampled_strict -- the sampled select as well"""
    Ch, N = C // 2, R * C
    rng = np.random.default_rng(zlib.crc32(f"{name} {R}x{C} {seed}".encode()))
    w = half_weights(R, C)
    p0, p1 = _gauss(rng, R, Ch)
    fr = lambda fs, tot: [int(tot * f) for f in fs]
    cut, one, cull, strict = fr((0.08, 0.5, 0.02), 2 * N), fr((0.2, 0.1), N), (0.2, 0.1, 0.05), True
    sampled_strict = True
    if name == "D2":                                         # exact zeros, independent positions
        for p in (p0, p1):
            p[rng.random(p.shape) < 0.3] = 0.0
        # the blend output holds ~9 % zeros (both operands zero): its cull ranks stay clear of that block
        cut, one, cull = fr((0.1, 0.25, 0.35), 2 * N), fr((0.15, 0.29), N), (0.2, 0.3, 0.4)
        # a window that starts at key 0 takes in the whole zero block (30 % of the keys), more than the sampled select's
        # candidate buffer (1/16 of them) holds: it has to flag the ranks inside the block (status bit 1)
        sampled_strict = False
    elif name == "D3":                                       # tied tiny +- keys, ranks inside the tie block
        vals = _tie_values(10, -30)
        for p in (p0, p1):
            m = rng.random(p.shape) < 0.12
            p[m] = vals[rng.integers(0, 10, m.sum())] * rng.choice(np.float32([-1, 1]), m.sum())
        cut, one = fr((0.03, 0.06, 0.1), 2 * N), fr((0.05, 0.09), N)
    elif name == "D4":                                       # a tie only in the multiplicity-1 columns 0 and Ch
        v = np.float32(0.5)
        for p in (p0, p1):
            p[np.abs(p) == v] *= np.float32(0.5)            # the tie is the edge columns' alone
            p[:, 0] = v; p[:, Ch] = -v
        b2, b1 = _below([p0, p1], w, v), _below([p0], w, v)
        cut, one = [b2 - 1, b2 + 4 * R - 1, b2 + 4 * R], [b1 + 2 * R - 1, b1 + 2 * R]
    elif name == "D5":                                       # +-0.0 and tiny pairs whose product underflows to 0
        m = rng.random(p0.shape)
        tiny = (rng.random(p0.shape) + 0.5).astype(np.float32) * np.float32(1e-23)
        sg = rng.choice(np.float32([-1, 1]), p0.shape)
        p0[m < 0.3] = (sg * tiny)[m < 0.3]
        p1[m < 0.3] = (np.where(m < 0.15, sg, -sg) * tiny[::-1, ::-1])[m < 0.3]
        z = (m >= 0.3) & (m < 0.36)
        p0[z] = np.where(sg > 0, np.float32(0.0), np.float32(-0.0))[z]
        p1[(m >= 0.33) & (m < 0.39)] = -0.0
        cut, one = fr((0.1, 0.2, 0.3), 2 * N), fr((0.1, 0.2), N)
    elif name == "D6":                                       # a gap at the rank
        for p in (p0, p1):
            small = rng.random(p.shape) < 0.08
            mag = np.where(small, 1e-4, 1e-1) * (1 + 0.05 * rng.standard_normal(p.shape))
            p[:] = (mag * np.sign(p + (p == 0))).astype(np.float32)
        b2, b1 = _below([p0, p1], w, np.float32(1e-3)), _below([p0], w, np.float32(1e-3))
        cut, one, strict = [int(2 * N * 0.08), b2 - 1, b2], [int(N * 0.08), b1 - 1, b1], False
    elif name == "D7":                                       # NaN / +-Inf keys, never in a same-sign pair
        idx = rng.choice(p0.size, 600, replace=False)
        r, c = np.unravel_index(idx, p0.shape)
        p0[r[:200], c[:200]] = np.inf; p1[r[:200], c[:200]] = -np.abs(p1[r[:200], c[:200]]) - 0.1
        p1[r[200:400], c[200:400]] = -np.inf; p0[r[200:400], c[200:400]] = np.abs(p0[r[200:400], c[200:400]]) + 0.1
        p0[r[400:500], c[400:500]] = np.nan; p1[r[400:500], c[400:500]] += np.float32(0.1) * np.sign(p1[r[400:500], c[400:500]] + 1e-3)
        p1[r[500:], c[500:]] = np.nan; p0[r[500:], c[500:]] += np.float32(0.1) * np.sign(p0[r[500:], c[500:]] + 1e-3)
        n_nan2 = int(sum((w * np.isnan(p)).sum() for p in (p0, p1)))
        n_inf2 = int(sum((w * np.isinf(p)).sum() for p in (p0, p1)))
        n_nan1, n_inf1 = int((w * np.isnan(p0)).sum()), int((w * np.isinf(p0)).sum())
        cut = [int(2 * N * 0.5), 2 * N - n_nan2 - n_inf2 - 1, 2 * N - n_nan2 - n_inf2 // 2, 2 * N - n_nan2 - 1]
        one = [int(N * 0.2), N - n_nan1 - n_inf1 - 1, N - n_nan1 - 1]
        strict = False
    elif name == "D8":                                       # ranks at either end
        cut = [0, 1, 2 * N - 1, int(2 * N * 1e-4), int(2 * N * 0.9999)]
        one = [0, 1, N - 1, int(N * 1e-4), int(N * 0.9999)]
        cull, strict = (1e-4, 0.9999, 0.2, 1e-4, 0.9999), False
    elif name == "D9":                                       # equal-sign ties packed into the first rows (one pass CTA)
        v = exact_keys([p0, p1], w, [int(2 * N * 0.08)])[0]
        p0[:8, 1:Ch] = v; p1[:8, 1:Ch] = v
        cut, one, strict = fr((0.08,), 2 * N), fr((0.08,), N), False
    else:
        assert name == "D1"
    return dict(p0=p0, p1=p1, cut=cut, one=one, cull=cull, strict=strict, sampled_strict=strict and sampled_strict)


def _fill(E, ws, p0, p1):
    """the two planes into ws.re[0], ws.re[1] row for row (the statistics and the blend do not depend on which frequency a
    stored row holds, and D9's ties stay in the first stored rows); the padding columns stay zero"""
    Ch = ws.plan.Ch
    for slot, p in ((0, p0), (1, p1)):
        ws.re[slot].zero_()
        ws.re[slot][:, : Ch + 1] = torch.from_numpy(np.ascontiguousarray(p)).to(DEV)


def _sel_status(sel, which):
    return int(sel.view(torch.int32)[16 * which + 9].item())


def _check(tag, status, thr, want, strict):
    """exact: status 0 and the key's bits; flagged: status != 0 and a NaN threshold; anything else fails."""
    if status == 0:
        assert same_key(thr, want), (tag, "wrong key with status 0", float(thr), float(want))
    else:
        assert not strict, (tag, "flagged", status, float(thr), float(want))
        assert np.isnan(thr), (tag, "flag without a NaN threshold", status, float(thr))
    return status == 0


def _tsign(x):
    s = np.sign(x)
    s[np.isnan(s)] = 0                                       # torch.sign(NaN) == 0
    return s


def _run_fused(E, ws, d, R, C):
    w = half_weights(R, C)
    p0, p1 = d["p0"], d["p1"]
    N = R * C
    wf = w.astype(np.float64)
    cuts = exact_keys([p0, p1], w, d["cut"])
    for i, (k2, want) in enumerate(zip(d["cut"], cuts)):
        cullp = d["cull"][i % len(d["cull"])]
        k1 = int(N * cullp)
        ws.ctl.zero_()
        E.fstats_cutoff(ws, ws.re[0], ws.re[1], k2, T)
        out = torch.empty_like(ws.re[0])
        E.fstats_blend_cull(ws, ws.re[0], ws.re[1], 1.0, out, k1)
        dbl, flt, _, _ = ws.read_ctl()
        st0, st1 = ws.fs_status()
        thr = np.float32(flt[E.F_THR_CUT].item())
        if not _check(("fused cutoff", k2), st0, thr, want, d["strict"]):
            continue
        sl = (_tsign(p0) == _tsign(p1)) & ~(np.abs(p1) < thr)
        a, b = p0.astype(np.float64), p1.astype(np.float64)
        s00, s11, s01 = (wf * a * a)[sl].sum(), (wf * b * b)[sl].sum(), (wf * a * b)[sl].sum()
        # (a threshold above every finite key leaves the sums empty: both zero)
        assert abs(float(dbl[E.D_S00]) - s00) <= 2e-7 * s00 and abs(float(dbl[E.D_S11]) - s11) <= 2e-7 * s11, (k2, float(dbl[E.D_S00]), s00)
        assert abs(float(dbl[E.D_S01]) - s01) <= 2e-7 * np.sqrt(s00 * s11), (k2, float(dbl[E.D_S01]), s01)
        dot, ct, sn, rn = (flt[E.F_DOT + j].item() for j in range(4))
        expect, _ = _np_blend(p0, p1, thr, dot, ct, sn, rn, 1.0)
        got = out[:, : C // 2 + 1].cpu().numpy()
        eq = (got.view(np.uint32) == expect.view(np.uint32)) | (np.isnan(got) & np.isnan(expect))
        assert eq.all(), (k2, int((~eq).sum()))
        _check(("fused cull", k1), st1, np.float32(flt[E.F_THR_CULL].item()), exact_keys([expect], w, [k1])[0], d["strict"])


def _run_select(E, ws, d, R, C, strict):
    w = half_weights(R, C)
    for k2, want in zip(d["cut"], exact_keys([d["p0"], d["p1"]], w, d["cut"])):
        ws.ctl.zero_()
        E.select_kth(ws, ws.re[0], ws.re[1], k2, E.F_THR_CUT, which=0)
        _, flt, _, sel = ws.read_ctl()
        _check(("select2", ws.safe_select, k2), _sel_status(sel, 0), np.float32(flt[E.F_THR_CUT].item()), want, strict)
    for k1, want in zip(d["one"], exact_keys([d["p0"]], w, d["one"])):
        ws.ctl.zero_()
        E.select_kth(ws, ws.re[0], None, k1, E.F_THR_CULL, which=1)
        _, flt, _, sel = ws.read_ctl()
        _check(("select1", ws.safe_select, k1), _sel_status(sel, 1), np.float32(flt[E.F_THR_CULL].item()), want, strict)


CASES = ["D1", "D2", "D3", "D4", "D5", "D6", "D7", "D8", "D9"]
SHAPES = [(1024, 2048), (2048, 4096), (2049, 1024), (1024, 5632)]


@gpu
@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("case", CASES)
def test_order_statistics_adversarial(E, case, shape):
    """Fused statistics, sampled select and exhaustive select on one adversarial distribution: exact or flagged as the
    case allows; where the fused cutoff is exact, the SLERP sums, the blend output and the cull threshold as well."""
    R, C = shape
    d = case_planes(case, R, C)
    ws = E.get_workspace(R, C, DEV)
    _fill(E, ws, d["p0"], d["p1"])
    _run_fused(E, ws, d, R, C)
    if R * C * 2 > (4 << 20):                               # 1024 x 2048: 4 Mi keys, the select is exhaustive there
        _fill(E, ws, d["p0"], d["p1"])
        _run_select(E, ws, d, R, C, d["sampled_strict"])
    safe = E.get_workspace(R, C, DEV, safe_select=True)
    _fill(E, safe, d["p0"], d["p1"])
    _run_select(E, safe, d, R, C, True)


@gpu
def test_order_statistics_on_tree_round_spectra(E):
    """D3r: the Re planes of the two round-1 fp32 intermediates of a four-finetune tree, transformed by the kernels'
    forward pass -- the culled bins are rounding noise with a handful of distinct keys (the fused pass's dense path)."""
    R, C = 1024, 2048
    g = torch.Generator(device=DEV).manual_seed(4321)
    base = (0.02 * torch.randn((R, C), generator=g, device=DEV)).to(torch.bfloat16)
    sig, alphas = (0.002, 0.0026, 0.0023, 0.0029), (0.3, 0.5, 0.4, 0.2)
    fts = [(base.float() + s * torch.randn((R, C), generator=g, device=DEV)).to(torch.bfloat16) for s in sig]
    from tests.test_gpu_parity import _merger
    fm = _merger()
    fm.keep_intermediates = True
    fm.merge_sources([E.make_source(base, ft, weight=a, name=f"m{k}") for k, (ft, a) in enumerate(zip(fts, alphas))],
                     base, torch.device(DEV), layer_name="model.layers.0.x")
    (_, _, ta), (_, _, tb) = fm.last_tree
    ws = E.get_workspace(R, C, DEV)
    ws.ctl.zero_()
    for slot, x in ((0, ta), (1, tb)):
        E.fwd_rows(ws, slot, E.Source(x32=x.contiguous()), E.D_SUMSQ0 + slot)
        E.fwd_cols(ws, slot, scale=E.inv_norm_f32(float(x.norm())))
    p0, p1 = (planes_to_numpy(ws, s).real.astype(np.float32) for s in (0, 1))
    w = half_weights(R, C)
    N = R * C
    low = np.abs(p0)[np.abs(p0) < np.quantile(np.abs(p0), 0.08)]
    print(f"\n[tree round 2 spectra] {np.unique(low).size} distinct keys among the {low.size} smallest")
    d = dict(p0=p0, p1=p1, cut=[int(2 * N * f) for f in (0.08, 0.02, 0.15)], one=[int(N * f) for f in (0.1, 0.05)],
             cull=(0.1, 0.05, 0.2), strict=True)
    _fill(E, ws, p0, p1)
    _run_fused(E, ws, d, R, C)
    safe = E.get_workspace(R, C, DEV, safe_select=True)
    _fill(E, safe, p0, p1)
    _run_select(E, safe, d, R, C, True)


# ------------------------------------------------------------------------------------------
# public functions: a flagged select is redone with the exhaustive one
# ------------------------------------------------------------------------------------------
def _pair(shape, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    v0 = 0.002 * torch.randn(shape, generator=g)
    v1 = 0.6 * v0 + 0.0018 * torch.randn(shape, generator=g)
    return v0, v1


def _d6_time_domain(R, C, seed):
    d = case_planes("D6", R, C, seed)
    return [torch.from_numpy(np.fft.irfft2(p.astype(np.float64), s=(R, C)).astype(np.float32)) for p in (d["p0"], d["p1"])]


PCTS = [(1e-4, 0.2), (0.08, 1e-4), (0.08, 0.9999)]


@gpu
@pytest.mark.parametrize("shape", [(1024, 2048), (2048, 4096)])
@pytest.mark.parametrize("pcts", PCTS + ["d6"])
def test_merge_tensors_fft2_slerp_extreme_percentages(E, shape, pcts):
    """Cutoff / cull percentages whose sampled window falls off either end (and a spectrum with a gap at the rank) are
    legal in the reference; the tensor function must redo a flagged tensor and match the oracle."""
    from shardmerge_b200.tensor import functions as F
    R, C = shape
    if pcts == "d6":
        v0, v1 = _d6_time_domain(R, C, 1)
        cutoff, cull = 0.08, 0.2
    else:
        v0, v1 = _pair(shape, R + C)
        cutoff, cull = pcts
    m, n0, n1 = F.merge_tensors_fft2_slerp(v0, v1, t=T, device=DEV, t_sum=1.0, cutoff_pct=cutoff, cull_pct=cull)
    mo, no0, no1 = O.merge_tensors_fft2_slerp(v0.numpy(), v1.numpy(), T, t_sum=1.0, cutoff_pct=cutoff, cull_pct=cull,
                                              interp_imag=False)
    assert abs(n0 / no0 - 1) < 1e-6 and abs(n1 / no1 - 1) < 1e-6
    m, mo = m.numpy(), np.asarray(mo)
    assert np.abs(m).max() > 0
    raw, resid, share = flip_accounted(m, mo, k=16)
    print(f"\n[{shape} {pcts}] raw rel-L2 {raw:.3e}, flip-accounted {resid:.3e}")
    assert resid <= 1e-5, (raw, resid, share)
    if cull > 0.99:
        # ~0.01 % of the real parts survive the cull, Im X0 dominates the tensor: count the surviving bins directly
        So, Sr = np.fft.rfft2(m.astype(np.float64)).real, np.fft.rfft2(mo.astype(np.float64)).real
        tau = 1e-3 * np.abs(Sr).max()
        ns_o, ns_r = int((np.abs(So) > tau).sum()), int((np.abs(Sr) > tau).sum())
        assert abs(ns_o - ns_r) <= 2 and ns_r > 0, (ns_o, ns_r)
        sv = (np.abs(So) > tau) & (np.abs(Sr) > tau)
        assert rel_l2(So[sv], Sr[sv]) < 1e-5


def _full_spectrum(case, R, C):
    d = case_planes(case, R, C, seed=3)
    fulls = [hermitian_full(p, C)[1] for p in (d["p0"], d["p1"])]
    return [torch.complex(torch.from_numpy(f), torch.zeros(f.shape)) for f in fulls]


@gpu
@pytest.mark.parametrize("case,cutoff,cull", [("D3", 0.06, 0.2), ("D6", 0.08, 0.2), ("D8", 1e-4, 0.9999),
                                              ("D8", 0.9999, 1e-4)])
def test_interpolate_fft_components_adversarial(E, case, cutoff, cull):
    """The step-by-step blend (sampled select at this size) on full Hermitian spectra with tied keys, a gap and
    extreme ranks: the same zero mask as the oracle and rel-L2 < 1e-6."""
    from shardmerge_b200.tensor import functions as F
    R, C = 2048, 4096
    z0, z1 = _full_spectrum(case, R, C)
    got = F.interpolate_fft_components(z0, z1, T, DEV, t_sum=1.0, cutoff_pct=cutoff, cull_pct=cull,
                                       interp_imag=False).cpu().numpy()
    want = O.interpolate_fft_components(z0.numpy(), z1.numpy(), T, t_sum=1.0, cutoff_pct=cutoff, cull_pct=cull,
                                        interp_imag=False)
    assert np.array_equal(got.real == 0, want.real == 0), int(((got.real == 0) != (want.real == 0)).sum())
    assert rel_l2(got.real, want.real) < 1e-6


def _bf16_pair(R, C, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    base = (0.02 * torch.randn((R, C), generator=g, device=DEV)).to(torch.bfloat16)
    fts = [(base.float() + s * torch.randn((R, C), generator=g, device=DEV)).to(torch.bfloat16) for s in (0.002, 0.0026)]
    return base, fts


def _bits(t):
    return t.contiguous().view(torch.int16).cpu().numpy().view(np.uint16)


@gpu
@pytest.mark.parametrize("defer", [False, True])
def test_fourier_merge_redoes_flagged_tensor(E, caplog, defer):
    """FourierMerge(cull_start_pct=1e-4): the fused chain's cull window falls off the low end, the flag must send the
    tensor through the step path to the exhaustive select (PendingPair -> _merge_sources_steps -> safe_select) and the
    result match the oracle.  The next, unflagged tensor on the same merger must not see the flag."""
    from shardmerge_b200.config import MergeConfig
    from shardmerge_b200.index import InMemoryIndex
    from shardmerge_b200.merge.fast_fourier import FourierMerge
    R, C = 1024, 2048
    fm = FourierMerge(MergeConfig(finetune_merge=[], output_base_model="org/base", output_dir="/tmp/unused"),
                      index_manager=InMemoryIndex({}), cull_start_pct=1e-4)
    alphas = (0.3, 0.5)
    for cull, seed, flagged in ((1e-4, 71, True), (0.2, 72, False)):
        fm.cull_start_pct = cull
        base, fts = _bf16_pair(R, C, seed)
        srcs = [E.make_source(base, ft, weight=a, name=f"m{k}") for k, (ft, a) in enumerate(zip(fts, alphas))]
        caplog.clear()
        with caplog.at_level(logging.WARNING):
            out = fm.merge_sources(srcs, base, torch.device(DEV), layer_name="model.layers.0.x", defer=defer)
            if defer:
                fm.resolve_all()
            torch.cuda.synchronize()
        missed = any("select window miss" in r.getMessage() for r in caplog.records)
        assert missed == flagged, (cull, [r.getMessage() for r in caplog.records])
        models = [dict(base=_bits(base), ft=_bits(ft), alpha=a, name=f"m{k}") for k, (ft, a) in enumerate(zip(fts, alphas))]
        info = {}
        oo = O.merge_layer(_bits(base), models, cull_start_pct=cull, info=info)
        assert fm.last_info["branches"] == ["slerp"] == info["branches"]
        basef = O.bf16_to_f32(_bits(base))
        raw, resid, share = flip_accounted(O.bf16_to_f32(_bits(out)) - basef, O.bf16_to_f32(oo) - basef, k=16)
        u = bf16_ulp_distance(_bits(out), oo)
        print(f"\n[cull {cull} defer {defer}] delta raw {raw:.3e} flip-accounted {resid:.3e} within 1 ulp {float((u <= 1).mean()):.6f}")
        assert float((u <= 1).mean()) >= 0.99, float((u <= 1).mean())
        assert resid < 0.05, (raw, resid, share)
