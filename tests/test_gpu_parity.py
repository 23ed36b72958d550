"""GPU parity tests: the sm_100a kernels, called through the C ABI (ctypes), against the numpy
oracle and the golden fixtures generated from the reference.  Run with `pytest -m gpu`.

Tolerances (north_star): fp32 intermediates rel L2 <= 1e-5 per tensor, checked stage by stage
with identical stage inputs; end to end additionally flip-accounted (tests/parity_util.py)
because the reference's masks / order statistics are discontinuous; final bf16 within 1 ulp on
>= 99.99 % of elements for the stages where that is well defined (epilogue given the same
spectrum), with the end-to-end fraction reported and bounded more loosely.
"""
import glob

import numpy as np
import pytest
import torch

from oracle import oracle_np as O
from tests.parity_util import bf16_ulp_distance, flip_accounted, rel_l2

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


@pytest.fixture(scope="module")
def E():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from shardmerge_b200 import engine
    return engine


def planes_to_numpy(ws, slot):
    """half-planar stored order -> complex128 [R][Ch+1] in natural frequency order"""
    pl = ws.plan
    re = ws.re[slot][:, : pl.Ch + 1].double().cpu().numpy()
    im = ws.im[slot][:, : pl.Ch + 1].double().cpu().numpy()
    z = re + 1j * im
    out = np.empty_like(z)
    out[pl.row_freq().numpy()] = z
    return out


def numpy_to_planes(ws, slot, z):
    """complex [R][Ch+1] natural order -> planes (stored order)"""
    pl = ws.plan
    zs = z[pl.row_freq().numpy()]
    ws.re[slot].zero_(); ws.im[slot].zero_()
    ws.re[slot][:, : pl.Ch + 1] = torch.from_numpy(np.ascontiguousarray(zs.real, dtype=np.float32)).to(DEV)
    ws.im[slot][:, : pl.Ch + 1] = torch.from_numpy(np.ascontiguousarray(zs.imag, dtype=np.float32)).to(DEV)


def half_weights(R, C):
    w = np.full((R, C // 2 + 1), 2, dtype=np.int64)
    w[:, 0] = 1; w[:, C // 2] = 1
    return w


def bits(t):
    return t.contiguous().view(torch.int16).cpu().numpy().view(np.uint16)


def from_bits(u16):
    return torch.from_numpy(u16.view(np.int16).copy()).view(torch.bfloat16).to(DEV)


SHAPES = [(1, 2), (1, 16), (1, 2048), (1, 8192), (2, 4), (8, 8), (32, 64), (96, 40), (352, 96), (143, 26),
          (256, 2048), (1024, 512), (512, 5632), (2048, 2048), (1792, 1024)]


@pytest.mark.parametrize("shape", SHAPES)
def test_forward_fft_matches_numpy(E, shape):
    R, C = shape
    g = torch.Generator(device=DEV).manual_seed(R * 7919 + C)
    x = torch.randn((R, C), generator=g, device=DEV, dtype=torch.float32)
    ws = E.get_workspace(R, C, DEV)
    ws.ctl.zero_()
    E.fwd_rows(ws, 0, E.Source(x32=x), E.D_SUMSQ0)
    E.fwd_cols(ws, 0, scale=1.0)
    got = planes_to_numpy(ws, 0)
    xs = x.double().cpu().numpy()
    ref = np.fft.rfft2(xs) if R > 1 else np.fft.rfft(xs, axis=1)
    assert rel_l2(got, ref) < 1e-6
    dbl, _, _, _ = ws.read_ctl()
    assert abs(float(dbl[E.D_SUMSQ0]) / float((xs ** 2).sum()) - 1) < 5e-7     # fp32 per-thread partials, fp64 across
    # inverse: back to the input (x 1/N inside the epilogue)
    out = torch.empty((R, C), dtype=torch.float32, device=DEV)
    E.inv_cols(ws, ws.re[0], ws.im[0], cull=False)
    E.inv_rows(ws, ws.re[0], ws.im[0], False, 1.0, None, out, check_ifft=True)
    assert rel_l2(out.cpu().numpy(), x.cpu().numpy()) < 1e-6


def test_forward_bf16_delta(E):
    R, C = 256, 2048
    g = torch.Generator(device=DEV).manual_seed(5)
    base = (0.02 * torch.randn((R, C), generator=g, device=DEV)).to(torch.bfloat16)
    ft = (base.float() + 0.002 * torch.randn((R, C), generator=g, device=DEV)).to(torch.bfloat16)
    ws = E.get_workspace(R, C, DEV)
    ws.ctl.zero_()
    E.fwd_rows(ws, 0, E.Source(base=base, ft=ft), E.D_SUMSQ0)
    E.fwd_cols(ws, 0, scale=1.0)
    delta = (ft.float() - base.float()).double().cpu().numpy()
    assert rel_l2(planes_to_numpy(ws, 0), np.fft.rfft2(delta)) < 1e-6
    dbl, _, _, _ = ws.read_ctl()
    assert abs(float(dbl[E.D_SUMSQ0]) / float((delta ** 2).sum()) - 1) < 5e-7


@pytest.mark.parametrize("shape", [(2, 4096), (6, 4096), (5, 4096), (2, 8192), (6, 8192), (7, 8192), (2, 14336), (3, 14336),
                                   (2, 28672), (5, 28672), (130, 4096), (150, 14336), (2, 2048), (260, 2048), (3, 5632), (6, 5632), (200, 5632)])
def test_paired_row_kernels_edge_row_counts(E, shape):
    """Every family of the packed-f32x2 row kernels (row pairs at C = 4096 / 8192, even / odd halves at C = 14336 /
    28672) at the smallest and at odd row counts (odd R falls back to the one-row kernels where pairs are needed):
    bf16 delta -> spectrum vs numpy, sum of squares, and back through the bf16 epilogue (x scale, + base, RNE)."""
    R, C = shape
    g = torch.Generator(device=DEV).manual_seed(R * 31 + C)
    base = (0.02 * torch.randn((R, C), generator=g, device=DEV)).to(torch.bfloat16)
    ft = (base.float() + 0.002 * torch.randn((R, C), generator=g, device=DEV)).to(torch.bfloat16)
    ws = E.get_workspace(R, C, DEV)
    ws.ctl.zero_()
    E.fwd_rows(ws, 0, E.Source(base=base, ft=ft), E.D_SUMSQ0)
    E.fwd_cols(ws, 0, scale=1.0)
    delta = (ft.float() - base.float()).double().cpu().numpy()
    assert rel_l2(planes_to_numpy(ws, 0), np.fft.rfft2(delta)) < 1e-6
    dbl, _, _, _ = ws.read_ctl()
    assert abs(float(dbl[E.D_SUMSQ0]) / float((delta ** 2).sum()) - 1) < 5e-7
    E.inv_cols(ws, ws.re[0], ws.im[0], cull=False)
    out = torch.empty((R, C), dtype=torch.bfloat16, device=DEV)
    E.inv_rows(ws, ws.re[0], ws.im[0], False, 0.37, base, out, check_ifft=True)     # 0.5 would put half the results on exact bf16 ties
    want = (base.float() + 0.37 * (ft.float() - base.float())).to(torch.bfloat16)
    u = bf16_ulp_distance(bits(out), bits(want))
    # (an ulp distance > 1 only happens next to zero, where base + 0.37 delta cancels and the ulp is tiny)
    assert float((u <= 1).mean()) >= 0.9999 and float((u == 0).mean()) >= 0.995, (float((u <= 1).mean()), float((u == 0).mean()))
    assert float((out.float() - want.float()).abs().max()) <= 2.0 ** -8 * float(want.float().abs().max())
    _, _, flags, _ = ws.read_ctl()
    assert [int(v) for v in flags[:4]] == [0, 0, 0, 0]


def _expanded_sorted(planes, R, C):
    w = half_weights(R, C)
    keys = np.concatenate([np.repeat(np.abs(p).ravel(), w.ravel()) for p in planes])
    keys.sort(kind="stable")
    return keys


@pytest.mark.parametrize("shape,safe", [((64, 128), False), ((1, 4096), False), ((1024, 4096), False),
                                        ((1024, 4096), True), ((2048, 2048), False)])
def test_select_kth_exact(E, shape, safe):
    """order statistics == sorted(cat(|re0|,|re1|))[k] with Hermitian multiplicities, bit exact."""
    R, C = shape
    ws = E.get_workspace(R, C, DEV, safe_select=safe)
    g = torch.Generator(device=DEV).manual_seed(R + C)
    for slot in (0, 1):
        ws.re[slot].copy_(torch.randn(ws.re[slot].shape, generator=g, device=DEV) * (0.7 + 0.3 * slot))
    Ch = C // 2
    p0 = ws.re[0][:, : Ch + 1].cpu().numpy(); p1 = ws.re[1][:, : Ch + 1].cpu().numpy()
    N = R * C
    both = _expanded_sorted([p0, p1], R, C)
    one = _expanded_sorted([p0], R, C)
    for pct in (0.08, 0.2, 0.5, 0.0001, 0.999999):
        ws.ctl.zero_()
        k2 = int((2 * N) * pct); k1 = int(N * pct)
        E.select_kth(ws, ws.re[0], ws.re[1], k2, E.F_THR_CUT, which=0)
        E.select_kth(ws, ws.re[0], None, k1, E.F_THR_CULL, which=1)
        _, flt, _, sel = ws.read_ctl()
        status = sel.view(torch.int32)[9].item(), sel.view(torch.int32)[16 + 9].item()
        assert status == (0, 0), (pct, status)
        assert np.float32(flt[E.F_THR_CUT].item()) == both[k2], (pct, flt[E.F_THR_CUT].item(), both[k2])
        assert np.float32(flt[E.F_THR_CULL].item()) == one[k1], (pct, flt[E.F_THR_CULL].item(), one[k1])


def test_select_window_miss_is_reported(E):
    """A degenerate distribution (most keys identical) must either give the exact answer or raise
    the status flag -- never a silently wrong threshold."""
    R, C = 2048, 4096
    ws = E.get_workspace(R, C, DEV)
    ws.re[0].fill_(1.0); ws.re[1].fill_(1.0)
    ws.re[0][:, :64] = torch.randn((R, 64), device=DEV)
    ws.ctl.zero_()
    k = int(2 * R * C * 0.08)
    E.select_kth(ws, ws.re[0], ws.re[1], k, E.F_THR_CUT, which=0)
    _, flt, _, sel = ws.read_ctl()
    status = sel.view(torch.int32)[9].item()
    if status == 0:
        assert flt[E.F_THR_CUT].item() == 1.0
    else:
        assert np.isnan(flt[E.F_THR_CUT].item())
    ws2 = E.get_workspace(R, C, DEV, safe_select=True)
    ws2.re[0].copy_(ws.re[0]); ws2.re[1].copy_(ws.re[1]); ws2.ctl.zero_()
    E.select_kth(ws2, ws2.re[0], ws2.re[1], k, E.F_THR_CUT, which=0)
    _, flt2, _, sel2 = ws2.read_ctl()
    assert sel2.view(torch.int32)[9].item() == 0 and flt2[E.F_THR_CUT].item() == 1.0


def _np_blend(re0, re1, thr, dot, ct, sn, rn, t_sum):
    f = np.float32
    same = np.sign(re0) == np.sign(re1)
    small = np.abs(re1) < f(thr)
    out = np.where(np.abs(re0) > np.abs(re1), re0, re1).astype(f)
    sl = same & ~small
    rel = (re1 - (re0 * f(dot)).astype(f)).astype(f)
    val = ((re0 * f(ct)).astype(f) + ((rel / f(rn)).astype(f) * f(sn)).astype(f)).astype(f)
    out[sl] = val[sl]
    sm = same & small
    out[sm] = (re0 + (f(t_sum) * re1).astype(f)).astype(f)[sm]
    return out, sl


@pytest.mark.parametrize("shape", [(1, 2048), (96, 40), (512, 1024)])
def test_reduce_scalars_blend_bit_exact(E, shape):
    R, C = shape
    Ch = C // 2
    ws = E.get_workspace(R, C, DEV)
    g = torch.Generator(device=DEV).manual_seed(77)
    ws.re[0].copy_(torch.randn(ws.re[0].shape, generator=g, device=DEV))
    ws.re[1].copy_(0.6 * ws.re[0] + 0.8 * torch.randn(ws.re[0].shape, generator=g, device=DEV))
    ws.re[0][0, 0] = 0.0; ws.re[1][0, 0] = 0.0            # sign(0) == sign(0) participates
    ws.re[0][0, 1] = 0.0
    re0 = ws.re[0][:, : Ch + 1].cpu().numpy(); re1 = ws.re[1][:, : Ch + 1].cpu().numpy()
    ws.ctl.zero_()
    thr = 0.1
    ws.flt[E.F_THR_CUT] = thr
    E.slerp_reduce(ws, ws.re[0], ws.re[1])
    E.slerp_scalars(ws, 0.375)
    out = torch.empty_like(ws.re[0])
    E.blend(ws, 0, True, ws.re[0], ws.re[1], 1.0, out)
    dbl, flt, _, _ = ws.read_ctl()
    w = half_weights(R, C).astype(np.float64)
    sl = (np.sign(re0) == np.sign(re1)) & ~(np.abs(re1) < np.float32(thr))
    a, b = re0.astype(np.float64), re1.astype(np.float64)
    s00, s11, s01 = (w * a * a)[sl].sum(), (w * b * b)[sl].sum(), (w * a * b)[sl].sum()
    assert abs(float(dbl[E.D_S00]) / s00 - 1) < 1e-12 and abs(float(dbl[E.D_S11]) / s11 - 1) < 1e-12
    assert abs(float(dbl[E.D_S01]) / s01 - 1) < 1e-11
    dot, ct, sn, rn = (flt[i].item() for i in (E.F_DOT, E.F_COS, E.F_SIN, E.F_RELNORM))
    dref = s01 / np.sqrt(s00 * s11)
    assert abs(dot - dref) < 2e-7
    assert abs(ct - np.cos(np.arccos(dref) * 0.375)) < 2e-7 and abs(sn - np.sin(np.arccos(dref) * 0.375)) < 2e-7
    assert abs(rn / np.sqrt(s11 - 2 * dot * s01 + dot * dot * s00) - 1) < 1e-6
    expect, _ = _np_blend(re0, re1, thr, dot, ct, sn, rn, 1.0)
    got = out[:, : Ch + 1].cpu().numpy()
    assert np.array_equal(got.view(np.uint32), expect.view(np.uint32))
    # arithmetic functor (functions.py:273-284)
    E.blend(ws, 1, True, ws.re[0], ws.re[1], 0.5, out)
    exp2 = np.where(np.sign(re0) == np.sign(re1), (re0 + (np.float32(0.5) * re1).astype(np.float32)).astype(np.float32), re1)
    assert np.array_equal(out[:, : Ch + 1].cpu().numpy().view(np.uint32), exp2.astype(np.float32).view(np.uint32))


@pytest.mark.parametrize("shape", [(1024, 4096), (2048, 2048), (512, 5632), (4096, 4096)])
def test_fused_stats_match_separate_kernels(E, shape, safe=False):
    """kernels_fstats.cu (one pass: cutoff statistic + SLERP sums + scalars; one pass: blend + cull statistic)
    against the exact sort and against the step-by-step kernels: thresholds bit-exact, sums to 1e-12,
    blend output bit-exact."""
    R, C = shape
    Ch = C // 2
    ws = E.get_workspace(R, C, DEV, safe_select=safe)
    g = torch.Generator(device=DEV).manual_seed(R * 3 + C)
    ws.re[0].copy_(torch.randn(ws.re[0].shape, generator=g, device=DEV) * 0.7)
    ws.re[1].copy_(0.5 * ws.re[0] + 0.6 * torch.randn(ws.re[0].shape, generator=g, device=DEV))
    ws.re[0][0, 0] = 0.0; ws.re[1][0, 0] = 0.0
    N = R * C
    re0 = ws.re[0][:, : Ch + 1].cpu().numpy(); re1 = ws.re[1][:, : Ch + 1].cpu().numpy()
    for cutoff, cullp in ((0.08, 0.20), (0.5, 0.10), (0.02, 0.05)):
        ws.ctl.zero_()
        k2 = int((2 * N) * cutoff); k1 = int(N * cullp)
        E.fstats_cutoff(ws, ws.re[0], ws.re[1], k2, 0.375)
        out = torch.empty_like(ws.re[0])
        E.fstats_blend_cull(ws, ws.re[0], ws.re[1], 1.0, out, k1)
        dbl, flt, _, _ = ws.read_ctl()
        assert ws.fs_status() == (0, 0), (cutoff, ws.fs_status())
        thr = np.float32(flt[E.F_THR_CUT].item())
        both = _expanded_sorted([re0, re1], R, C)
        assert thr == both[k2], (cutoff, thr, both[k2])
        w = half_weights(R, C).astype(np.float64)
        sl = (np.sign(re0) == np.sign(re1)) & ~(np.abs(re1) < thr)
        a, b = re0.astype(np.float64), re1.astype(np.float64)
        s00, s11, s01 = (w * a * a)[sl].sum(), (w * b * b)[sl].sum(), (w * a * b)[sl].sum()
        # fp32 products / 4-element fp32 partials inside the streaming pass, fp64 across
        assert abs(float(dbl[E.D_S00]) / s00 - 1) < 2e-7 and abs(float(dbl[E.D_S11]) / s11 - 1) < 2e-7
        assert abs(float(dbl[E.D_S01]) - s01) < 2e-7 * np.sqrt(s00 * s11)
        scal = [float(flt[E.F_DOT + i].item()) for i in range(4)]
        # the same scalars from the step-by-step kernel given the fused sums
        ws2 = E.Workspace(E.get_plan(R, C, DEV), 2, False)
        ws2.ctl.zero_()
        ws2.dbl[E.D_S00:E.D_S00 + 3] = torch.tensor([float(dbl[E.D_S00]), float(dbl[E.D_S11]), float(dbl[E.D_S01])],
                                                    dtype=torch.float64, device=DEV)
        ws2.flt[E.F_THR_CUT] = float(thr)
        E.slerp_scalars(ws2, 0.375)
        out2 = torch.empty_like(ws.re[0])
        E.blend(ws2, 0, True, ws.re[0], ws.re[1], 1.0, out2)
        _, flt2, _, _ = ws2.read_ctl()
        assert scal == [float(flt2[E.F_DOT + i].item()) for i in range(4)]
        o1 = out[:, : Ch + 1].cpu().numpy(); o2 = out2[:, : Ch + 1].cpu().numpy()
        assert np.array_equal(o1.view(np.uint32), o2.view(np.uint32))
        one = _expanded_sorted([o2], R, C)
        assert np.float32(flt[E.F_THR_CULL].item()) == one[k1], (cullp, flt[E.F_THR_CULL].item(), one[k1])


def test_fused_stats_window_miss_is_reported(E):
    """Degenerate distribution: either the exact answer or a raised status, never a silently wrong threshold."""
    R, C = 2048, 4096
    ws = E.get_workspace(R, C, DEV)
    ws.re[0].fill_(1.0); ws.re[1].fill_(1.0)
    ws.re[0][:, :64] = torch.randn((R, 64), device=DEV)
    ws.ctl.zero_()
    E.fstats_cutoff(ws, ws.re[0], ws.re[1], int(2 * R * C * 0.08), 0.375)
    _, flt, _, _ = ws.read_ctl()
    st = ws.fs_status()[0]
    if st == 0:
        assert flt[E.F_THR_CUT].item() == 1.0
    else:
        assert np.isnan(flt[E.F_THR_CUT].item())


@pytest.mark.parametrize("shape", [(1, 4096), (256, 512), (352, 96), (1024, 2048)])
def test_inverse_epilogue_bf16_within_1ulp(E, shape):
    """Given the same spectrum, iFFT + x scale + base + bf16 RNE matches the oracle's epilogue on
    >= 99.99 % of elements within 1 ulp (and the cull on load zeroes exactly |re| < thr)."""
    R, C = shape
    rng = np.random.default_rng(3)
    m = (rng.standard_normal((R, C)) * 0.003).astype(np.float32)
    base = O.f32_to_bf16((rng.standard_normal((R, C)) * 0.02).astype(np.float32))
    Z = np.fft.rfft2(m.astype(np.float64)) if R > 1 else np.fft.rfft(m.astype(np.float64), axis=1)
    thr = np.float32(np.quantile(np.abs(Z.real), 0.2))
    Zc = np.where(np.abs(Z.real.astype(np.float32)) < thr, 0.0, Z.real.astype(np.float32)) + 1j * Z.imag.astype(np.float32)
    # oracle: full-spectrum inverse of the culled Hermitian spectrum
    mc = (np.fft.irfft2(Zc, s=(R, C)) if R > 1 else np.fft.irfft(Zc, n=C, axis=1)).astype(np.float32)
    scale = np.float32(7.25)
    expect = O.f32_to_bf16((O.bf16_to_f32(base) + (mc * scale).astype(np.float32)).astype(np.float32))
    ws = E.get_workspace(R, C, DEV)
    ws.ctl.zero_()
    numpy_to_planes(ws, 0, Z)
    ws.flt[E.F_THR_CULL] = float(thr)
    out = torch.empty((R, C), dtype=torch.bfloat16, device=DEV)
    E.inv_cols(ws, ws.re[0], ws.im[0], cull=True)
    E.inv_rows(ws, ws.re[0], ws.im[0], True, float(scale), from_bits(base.reshape(R, C)), out, check_ifft=True)
    u = bf16_ulp_distance(bits(out).reshape(R, C), expect)
    assert float((u <= 1).mean()) >= 0.9999, float((u <= 1).mean())
    assert float((u == 0).mean()) >= 0.995
    _, _, flags, _ = ws.read_ctl()
    assert [int(v) for v in flags] == [0, 0, 0, 0]


@pytest.mark.parametrize("shape", [(8, 64), (4, 4096), (4, 8192), (4, 14336), (3, 28672), (4, 2048), (3, 5632)])
def test_epilogue_nan_inf_policy(E, shape):
    """NaN -> 0 (counted), Inf kept (counted) after the base add (fast_fourier.py:270-274), in every epilogue variant
    (one-row, row pairs, even / odd halves)."""
    R, C = shape
    ws = E.get_workspace(R, C, DEV)
    ws.ctl.zero_()
    Z = np.zeros((R, C // 2 + 1), dtype=np.complex128)
    numpy_to_planes(ws, 0, Z)
    base = torch.zeros((R, C), dtype=torch.bfloat16, device=DEV)
    base[0, 0] = float("inf"); base[0, 1] = float("nan")
    base[R - 1, C - 1] = float("nan"); base[R - 1, C - 2] = float("-inf"); base[1, 7] = float("nan")
    out = torch.empty((R, C), dtype=torch.bfloat16, device=DEV)
    E.inv_cols(ws, ws.re[0], ws.im[0], cull=False)
    E.inv_rows(ws, ws.re[0], ws.im[0], False, 1.0, base, out, check_ifft=True)
    _, _, flags, _ = ws.read_ctl()
    assert int(flags[2]) == 3 and int(flags[3]) == 2 and int(flags[0]) == 0 and int(flags[1]) == 0
    assert out[0, 1].item() == 0.0 and torch.isinf(out[0, 0])
    assert out[R - 1, C - 1].item() == 0.0 and out[R - 1, C - 2].item() == float("-inf") and out[1, 7].item() == 0.0
    assert int(torch.count_nonzero(out.float() != 0)) == 2


# ------------------------------------------------------------------------------------------
# golden fixtures (reference outputs) and oracle, end to end
# ------------------------------------------------------------------------------------------
def _merger():
    from shardmerge_b200.config import MergeConfig, MergeModel
    from shardmerge_b200.index import InMemoryIndex
    from shardmerge_b200.merge.fast_fourier import FourierMerge
    cfg = MergeConfig(finetune_merge=[], output_base_model="org/base", output_dir="/tmp/unused")
    return FourierMerge(cfg, index_manager=InMemoryIndex({}))


def _run_layer_case(E, d, n_models=None):
    fm = _merger()
    alphas = d["alphas"][:n_models] if n_models else d["alphas"]
    base = from_bits(d["base"])
    srcs = [E.make_source(base, from_bits(d[f"ft{k}"]), weight=float(a), name=f"org/ft{k}") for k, a in enumerate(alphas)]
    out = fm.merge_sources(srcs, base, torch.device(DEV), layer_name=str(d["layer"]))
    return bits(out).reshape(d["base"].shape), fm.last_info


@pytest.mark.parametrize("name,branches,min_within1", [
    ("slerp_256x512", ["slerp"], 0.999), ("slerp_swapped_128x256", ["slerp"], 0.98),
    ("slerp_a7b2_128x256", ["slerp"], 0.98), ("slerp_1d_2048", ["slerp"], 0.98), ("slerp_352x96", ["slerp"], 0.98),
    ("arith_128x256", ["arith"], 0.9999), ("onezero_64x128", ["arith"], 0.9999),
    ("single_64x128", [], 1.0), ("add_zero_64x128", ["add"], 1.0),
])
def test_golden_layer_cases(E, golden_dir, name, branches, min_within1):
    """FourierMerge on the reference's own inputs vs the reference's bf16 outputs.  Small tensors
    make a single flipped spectrum bin visible in a few % of the bf16 roundings, hence the
    per-case floors; the flip-accounted residual of the fp32 delta is the tight check."""
    d = np.load(golden_dir / f"layer_{name}.npz")
    got, info = _run_layer_case(E, d)
    assert info["branches"] == branches
    u = bf16_ulp_distance(got, d["out"])
    frac1 = float((u <= 1).mean())
    assert frac1 >= min_within1, (name, frac1, int(u.max()))
    if min_within1 == 1.0:
        assert np.array_equal(got, d["out"])
    if "slerp" in branches or "arith" in branches:
        # same inputs through the oracle: ours and the oracle should bracket the reference alike
        models = [dict(base=d["base"], ft=d[f"ft{k}"], alpha=float(a), name=f"org/ft{k}") for k, a in enumerate(d["alphas"])]
        oo = O.merge_layer(d["base"], models)
        basef = O.bf16_to_f32(d["base"])
        raw, resid, share = flip_accounted(O.bf16_to_f32(got) - basef, O.bf16_to_f32(oo) - basef, k=8)
        # bf16 quantisation of (base + delta) limits what the delta comparison can resolve
        assert resid < 0.05, (name, raw, resid, share)


@pytest.mark.parametrize("shape,seed", [((256, 333), 61), ((1024, 1001), 62)])
def test_pair_merge_odd_row_length_vs_oracle(E, shape, seed):
    """[R][odd C] tensors have no packed real row transform; they are merged as their transpose (fft2(X^T) = fft2(X)^T and
    the blend is element-wise / global).  Against the oracle, which transforms the tensor as it is."""
    R, C = shape
    g = torch.Generator(device=DEV).manual_seed(1234 + seed)
    base = (0.02 * torch.randn(shape, generator=g, device=DEV)).to(torch.bfloat16)
    fts = [(base.float() + sg * torch.randn(shape, generator=g, device=DEV)).to(torch.bfloat16) for sg in (0.002, 0.0026)]
    fm = _merger()
    srcs = [E.make_source(base, fts[k], weight=a, name=f"m{k}") for k, a in enumerate((0.3, 0.5))]
    out = fm.merge_sources(srcs, base, torch.device(DEV), layer_name="model.layers.0.x")
    assert tuple(out.shape) == shape and out.dtype == torch.bfloat16 and fm.last_info["branches"] == ["slerp"]
    models = [dict(base=bits(base), ft=bits(fts[k]), alpha=a, name=f"m{k}") for k, a in enumerate((0.3, 0.5))]
    info = {}
    oo = O.merge_layer(bits(base), models, info=info)
    assert abs(fm.last_info["target_norm"] / info["target_norm"] - 1) < 1e-6
    basef = O.bf16_to_f32(bits(base))
    raw, resid, share = flip_accounted(O.bf16_to_f32(bits(out)) - basef, O.bf16_to_f32(oo) - basef, k=16)
    u = bf16_ulp_distance(bits(out), oo)
    frac1 = float((u <= 1).mean())
    print(f"\n[{shape}] odd row length: raw {raw:.3e} flip-accounted {resid:.3e} within 1 ulp {frac1:.6f}")
    assert resid < 0.05 and frac1 >= 0.98, (raw, resid, share, frac1)


def test_golden_layer_range(E, golden_dir):
    d = np.load(golden_dir / "layer_layer_range_64x128.npz")
    got, info = _run_layer_case(E, d, n_models=2)
    u = bf16_ulp_distance(got, d["out"])
    assert float((u <= 1).mean()) >= 0.98


def test_golden_tensor_cases(E, golden_dir):
    """merge_tensors_fft2_slerp (fp32 in, fp32 out) vs the reference's result: flip-accounted <= 1e-5."""
    from shardmerge_b200.tensor import functions as F
    for f in sorted(glob.glob(str(golden_dir / "tensor_*.npz"))):
        d = np.load(f)
        m, n0, n1 = F.merge_tensors_fft2_slerp(torch.from_numpy(d["v0"]), torch.from_numpy(d["v1"]), t=0.375, device=DEV,
                                               t_sum=1.0, cutoff_pct=0.08, cull_pct=0.20)
        assert abs(n0 / float(d["n0"]) - 1) < 1e-6 and abs(n1 / float(d["n1"]) - 1) < 1e-6
        raw, resid, share = flip_accounted(m.numpy(), d["merged"], k=8)
        assert resid < 1e-5, (f, raw, resid, share)
        # forward transform vs the reference's (MKL) spectrum
        X = F.fft_transform(torch.from_numpy(d["v0"]) / np.float32(d["n0"]), DEV).numpy()
        assert rel_l2(X, d["fft0"]) < 2e-6


@pytest.mark.parametrize("shape,seed", [((1024, 4096), 21), ((2048, 1024), 22), ((1, 8192), 23), ((512, 8192), 24),
                                        ((256, 14336), 25), ((128, 28672), 26)])
def test_pair_merge_vs_oracle_mid_size(E, shape, seed):
    """Synthetic Llama-like tensors (SURVEY 8d) at sizes the oracle finishes in seconds."""
    R, C = shape
    g = torch.Generator(device=DEV).manual_seed(1234 + seed)
    sh = (R, C) if R > 1 else (C,)
    mean, bs, sig = (1.0, 0.1, (0.01, 0.013)) if R == 1 else (0.0, 0.02, (0.002, 0.0026))
    base = (mean + bs * torch.randn(sh, generator=g, device=DEV)).to(torch.bfloat16)
    fts = []
    for k in range(2):
        gk = torch.Generator(device=DEV).manual_seed(100000 * (k + 1) + seed)
        fts.append((base.float() + sig[k] * torch.randn(sh, generator=gk, device=DEV)).to(torch.bfloat16))
    fm = _merger()
    srcs = [E.make_source(base, fts[k], weight=a, name=f"m{k}") for k, a in enumerate((0.3, 0.5))]
    out = fm.merge_sources(srcs, base, torch.device(DEV), layer_name="model.layers.0.x")
    assert fm.last_info["branches"] == ["slerp"]
    models = [dict(base=bits(base), ft=bits(fts[k]), alpha=a, name=f"m{k}") for k, a in enumerate((0.3, 0.5))]
    info = {}
    oo = O.merge_layer(bits(base), models, info=info)
    assert abs(fm.last_info["target_norm"] / info["target_norm"] - 1) < 1e-6
    # (a) fp32 intermediates: the merged delta of the tensor function vs the oracle on identical fp32 deltas.
    #     north_star tolerance: rel L2 <= 1e-5 -- met outright when no decision flips, and by the residual
    #     once the <= 8 flipped Hermitian bin pairs are set aside (SURVEY 7.3: discontinuous algorithm).
    from shardmerge_b200.tensor import functions as F
    d0 = fts[0].float() - base.float(); d1 = fts[1].float() - base.float()
    n0, n1 = float(d0.norm()), float(d1.norm())
    a_, b_ = (d0, d1) if n0 >= n1 else (d1, d0)
    m, _, _ = F.merge_tensors_fft2_slerp(a_, b_, t=0.3 / 0.8, device=DEV, t_sum=1.0, cutoff_pct=0.08, cull_pct=0.20)
    mo, _, _ = O.merge_tensors_fft2_slerp(a_.cpu().numpy(), b_.cpu().numpy(), 0.3 / 0.8, t_sum=1.0, cutoff_pct=0.08,
                                          cull_pct=0.20, interp_imag=False)
    raw, resid, share = flip_accounted(m.cpu().numpy().reshape(sh), np.asarray(mo).reshape(sh), k=16)
    print(f"\n[{shape}] fp32 merged delta: raw rel-L2 {raw:.3e}, flip-accounted {resid:.3e} (top-16 bins carry {share:.4f})")
    assert resid <= 1e-5, (raw, resid, share)
    # (b) final bf16: within 1 ulp on >= 99.99 % when nothing flipped; one flipped bin pair is a sinusoid of
    #     ~3 % of a typical bf16 ulp over the whole tensor, which moves ~0.5 % of the near-zero elements by > 1 ulp.
    u = bf16_ulp_distance(bits(out), oo)
    frac1 = float((u <= 1).mean())
    absd = np.abs(O.bf16_to_f32(bits(out)) - O.bf16_to_f32(oo))
    print(f"[{shape}] bf16 exact {float((u == 0).mean()):.6f} within-1ulp {frac1:.6f} max-abs-diff {absd.max():.3e}")
    assert frac1 >= (0.9999 if raw <= 1e-5 else 0.985), (frac1, raw)
    assert absd.max() <= 2.0 ** -7 * np.abs(O.bf16_to_f32(oo)).max() + 1e-4   # never more than one bf16 ulp of the largest value


@pytest.mark.parametrize("shape", [(4096, 4096), (14336, 4096), (4096, 14336), (1024, 4096),
                                   (8192, 8192), (1024, 8192), (28672, 8192), (8192, 28672)])
def test_full_size_properties(E, shape):
    """Llama-3.1-8B and 70B shapes, size-independent properties: FFT round trip, Parseval, linearity, exact
    rank of the order statistic (by counting), bf16 output finite."""
    R, C = shape
    g = torch.Generator(device=DEV).manual_seed(R + 3 * C)
    base = (0.02 * torch.randn((R, C), generator=g, device=DEV)).to(torch.bfloat16)
    ft = (base.float() + 0.002 * torch.randn((R, C), generator=g, device=DEV)).to(torch.bfloat16)
    delta = ft.float() - base.float()
    ws = E.get_workspace(R, C, DEV)
    ws.ctl.zero_()
    E.fwd_rows(ws, 0, E.Source(base=base, ft=ft), E.D_SUMSQ0)
    E.fwd_cols(ws, 0, scale=1.0)
    Ch = C // 2
    w = torch.full((Ch + 1,), 2.0, device=DEV, dtype=torch.float64); w[0] = 1; w[Ch] = 1
    energy = ((ws.re[0][:, : Ch + 1].double() ** 2 + ws.im[0][:, : Ch + 1].double() ** 2) * w).sum().item()
    ss = (delta.double() ** 2).sum().item()
    dbl, _, _, _ = ws.read_ctl()
    assert abs(float(dbl[E.D_SUMSQ0]) / ss - 1) < 1e-7
    assert abs(energy / (ss * R * C) - 1) < 1e-5                      # Parseval
    # exact rank by counting
    N = R * C
    k = int(N * 0.2)
    E.select_kth(ws, ws.re[0], None, k, E.F_THR_CULL, which=1)
    _, flt, _, sel = ws.read_ctl()
    assert sel.view(torch.int32)[16 + 9].item() == 0
    thr = flt[E.F_THR_CULL].item()
    a = ws.re[0][:, : Ch + 1].abs()
    below = ((a < thr).double() * w).sum().item(); upto = ((a <= thr).double() * w).sum().item()
    assert below <= k < upto, (below, k, upto)
    # round trip
    out = torch.empty((R, C), dtype=torch.float32, device=DEV)
    E.inv_cols(ws, ws.re[0], ws.im[0], cull=False)
    E.inv_rows(ws, ws.re[0], ws.im[0], False, 1.0, None, out, check_ifft=True)
    err = ((out.double() - delta.double()) ** 2).sum().sqrt().item() / ss ** 0.5
    assert err < 1e-6, err


@pytest.mark.parametrize("shape", [(1, 4096), (256, 512), (1024, 4096), (2048, 5632)])
def test_fused_chain_matches_step_path(E, shape):
    """The host-sync-free fused chain (csrc/pipeline.cu: device-side role / branch / target_norm
    decisions) gives the same tensor as the step-by-step path with host decisions, both ways round
    (model 0 larger and model 1 larger)."""
    R, C = shape
    sh = (R, C) if R > 1 else (C,)
    for sig in ((0.002, 0.0026), (0.0026, 0.002)):
        g = torch.Generator(device=DEV).manual_seed(R + C)
        base = (0.02 * torch.randn(sh, generator=g, device=DEV)).to(torch.bfloat16)
        fts = [(base.float() + s * torch.randn(sh, generator=g, device=DEV)).to(torch.bfloat16) for s in sig]
        fm = _merger()
        mk = lambda: [E.make_source(base, ft, weight=a, name=f"m{k}") for k, (ft, a) in enumerate(zip(fts, (0.3, 0.5)))]
        fused = fm.merge_sources(mk(), base, torch.device(DEV), layer_name="model.layers.0.x")
        info_f = dict(fm.last_info)
        steps = fm._merge_sources_steps(mk(), base, torch.device(DEV), layer_name="model.layers.0.x")
        assert info_f["branches"] == ["slerp"] and fm.last_info["branches"] == ["slerp"]
        assert info_f["swap"] == (1 if sig[1] > sig[0] else 0)
        assert abs(info_f["target_norm"] / fm.last_info["target_norm"] - 1) < 1e-7
        u = bf16_ulp_distance(bits(fused), bits(steps))
        assert float((u == 0).mean()) >= 0.9999 and int(u.max()) <= 1, (float((u == 0).mean()), int(u.max()))


def test_fused_stats_survive_a_select_on_the_same_workspace(E):
    """sm_select_kth_abs (step path, tree rounds >= 2) uses the front of the statistics workspace, the fused
    statistics keep their (persistently zeroed) histograms at its end: a select in between must not cost the next
    fused call its sample window."""
    R, C = 1024, 2048
    ws = E.get_workspace(R, C, DEV)
    g = torch.Generator(device=DEV).manual_seed(77)
    ws.re[0].copy_(torch.randn(ws.re[0].shape, generator=g, device=DEV))
    ws.re[1].copy_(torch.randn(ws.re[0].shape, generator=g, device=DEV))
    N = R * C
    for _ in range(2):
        ws.ctl.zero_()
        E.select_kth(ws, ws.re[0], ws.re[1], int(2 * N * 0.08), E.F_THR_CUT)
        _, flt, _, _ = ws.read_ctl()
        want = flt[E.F_THR_CUT].item()
        ws.ctl.zero_()
        E.fstats_cutoff(ws, ws.re[0], ws.re[1], int(2 * N * 0.08), 0.375)
        _, flt, _, _ = ws.read_ctl()
        assert ws.fs_status()[0] == 0
        assert flt[E.F_THR_CUT].item() == want


def test_tree_of_four_finetunes_vs_oracle(E):
    """BASELINE config 4 (four finetunes): round 1 = two pair merges on the fused chain, round 2 = one pair merge of the
    fp32 intermediates on the step path (fast_fourier.py:171-254); against the numpy oracle at a size it finishes
    in seconds."""
    R, C = 1024, 2048
    g = torch.Generator(device=DEV).manual_seed(4321)
    base = (0.02 * torch.randn((R, C), generator=g, device=DEV)).to(torch.bfloat16)
    sig, alphas = (0.002, 0.0026, 0.0023, 0.0029), (0.3, 0.5, 0.4, 0.2)
    fts = [(base.float() + s * torch.randn((R, C), generator=g, device=DEV)).to(torch.bfloat16) for s in sig]
    fm = _merger()
    srcs = [E.make_source(base, ft, weight=a, name=f"m{k}") for k, (ft, a) in enumerate(zip(fts, alphas))]
    out = fm.merge_sources(srcs, base, torch.device(DEV), layer_name="model.layers.0.x")
    assert fm.last_info["branches"] == ["slerp", "slerp", "slerp"]
    models = [dict(base=bits(base), ft=bits(ft), alpha=a, name=f"m{k}") for k, (ft, a) in enumerate(zip(fts, alphas))]
    info = {}
    oo = O.merge_layer(bits(base), models, info=info)
    assert abs(fm.last_info["target_norm"] / info["target_norm"] - 1) < 1e-6
    # Round >= 2 blends spectra in which the previous cull left 20 % of the real parts at rounding-noise level: the
    # sign mask there -- and ~10 % of the output bins -- is decided by FFT rounding noise in the reference itself
    # (tests/test_oracle_golden.py::test_tree_merges_structure: the oracle against the reference's own fixture shows the
    # same spread), so only the branch structure, the norms and the overall delta can be pinned for a tree.
    basef = O.bf16_to_f32(bits(base))
    do, dr = O.bf16_to_f32(bits(out)) - basef, O.bf16_to_f32(oo) - basef
    print(f"\n[tree4 {R}x{C}] delta rel-L2 vs oracle {rel_l2(do, dr):.3f}, norm ratio {np.linalg.norm(do) / np.linalg.norm(dr):.4f}")
    assert rel_l2(do, dr) < 0.5
    assert abs(np.linalg.norm(do) / np.linalg.norm(dr) - 1) < 0.05
    assert np.isfinite(do).all()


def test_fused_chain_falls_back_on_other_branches(E):
    """Device-side branch detection: a near-zero second delta (arithmetic branch) and identical
    models (add branch) are re-run on the step path and match the reference fixtures."""
    import numpy as np
    from pathlib import Path
    gd = Path(__file__).resolve().parent / "golden"
    for name, branch in (("arith_128x256", "arith"), ("add_zero_64x128", "add"), ("onezero_64x128", "arith")):
        d = np.load(gd / f"layer_{name}.npz")
        got, info = _run_layer_case(E, d)
        assert info["branches"] == [branch]
        u = bf16_ulp_distance(got, d["out"])
        assert float((u <= 1).mean()) >= 0.9999


def test_deferred_checks_pipeline(E):
    """defer=True: several tensors enqueued back to back, settled afterwards."""
    fm = _merger()
    outs, refs = [], []
    for i, (R, C) in enumerate([(256, 512), (128, 256), (256, 512), (1, 2048)]):
        sh = (R, C) if R > 1 else (C,)
        g = torch.Generator(device=DEV).manual_seed(50 + i)
        base = (0.02 * torch.randn(sh, generator=g, device=DEV)).to(torch.bfloat16)
        fts = [(base.float() + s * torch.randn(sh, generator=g, device=DEV)).to(torch.bfloat16) for s in (0.002, 0.0026)]
        mk = lambda base=base, fts=fts: [E.make_source(base, ft, weight=a, name=f"m{k}")
                                         for k, (ft, a) in enumerate(zip(fts, (0.3, 0.5)))]
        outs.append(fm.merge_sources(mk(), base, torch.device(DEV), layer_name=f"model.layers.{i}.x", defer=True))
        refs.append((mk, base))
    assert len(fm.pending) == 4
    fm.resolve_all()
    assert not fm.pending
    for out, (mk, base) in zip(outs, refs):
        steps = fm._merge_sources_steps(mk(), base, torch.device(DEV), layer_name="x")
        u = bf16_ulp_distance(bits(out), bits(steps))
        assert int(u.max()) <= 1 and float((u == 0).mean()) >= 0.9999


def test_lanes_do_not_change_results(E):
    """Consecutive tensors spread over several streams (FourierMerge.lanes) give bit-identical outputs to the
    single-stream schedule: same kernels, same order per tensor, separate workspaces."""
    shapes = [(1024, 2048), (512, 1024), (1024, 2048), (1, 4096), (2048, 1024), (1024, 2048)]
    results = {}
    for lanes in (1, 3):
        fm = _merger()
        fm.lanes = lanes
        outs = []
        for i, (R, C) in enumerate(shapes):
            sh = (R, C) if R > 1 else (C,)
            g = torch.Generator(device=DEV).manual_seed(900 + i)
            base = (0.02 * torch.randn(sh, generator=g, device=DEV)).to(torch.bfloat16)
            fts = [(base.float() + s * torch.randn(sh, generator=g, device=DEV)).to(torch.bfloat16) for s in (0.002, 0.0026)]
            srcs = [E.make_source(base, ft, weight=a, name=f"m{k}") for k, (ft, a) in enumerate(zip(fts, (0.3, 0.5)))]
            outs.append(fm.merge_sources(srcs, base, torch.device(DEV), layer_name=f"model.layers.{i}.x", defer=True))
        fm.resolve_all()
        torch.cuda.synchronize()
        results[lanes] = [bits(o) for o in outs]
    for a, b in zip(results[1], results[3]):
        assert np.array_equal(a, b)


def test_shape_mismatch_is_refused(E):
    fm = _merger()
    base = torch.zeros((64, 128), dtype=torch.bfloat16, device=DEV)
    other = torch.zeros((2048,), dtype=torch.bfloat16, device=DEV)
    srcs = [E.make_source(other, other, weight=0.3), E.make_source(other, other, weight=0.5)]
    with pytest.raises(ValueError):
        fm.merge_sources(srcs, base, torch.device(DEV), layer_name="model.layers.0.x")


# ----------------------------------------------------------------------------- element-wise strategies (SURVEY 8f N3)
def _nan_equal_bits(a, b):
    fa, fb = O.bf16_to_f32(a), O.bf16_to_f32(b)
    return (a == b) | ((fa != fa) & (fb != fb))


from tests.parity_util import ELEM_CASES, elem_case as _elem_case, elem_same as _elem_same

_ELEM_TORCH = {"bf16": torch.bfloat16, "f16": torch.float16, "f32": torch.float32}


def _elem_to_torch(dt, a):
    return torch.from_numpy(a.view(np.int16).copy()).view(torch.bfloat16) if dt == "bf16" else torch.from_numpy(a.copy())


def _elem_to_numpy(dt, t):
    return bits(t) if dt == "bf16" else t.detach().cpu().numpy()


@pytest.mark.parametrize("name", ELEM_CASES)
def test_elementwise_strategies_golden(E, golden_dir, name):
    """AdditionMerge / TaskAdditionMerge through the reference's class interface (`_merge_layer`) on the reference's own
    inputs: bit-identical to the reference's output (NaN payloads aside) for bf16, fp16 and fp32 models, 2..35 finetunes."""
    import asyncio
    from shardmerge_b200.config import MergeConfig, MergeModel
    from shardmerge_b200.index import InMemoryIndex
    from shardmerge_b200.merge import AdditionMerge, TaskAdditionMerge
    from shardmerge_b200.writer import ShardLayer
    dt, base, fts, want = _elem_case(golden_dir, name)
    n = len(fts)
    layer = "model.layers.3.mlp.up_proj.weight"
    models = {"org/base": {layer: _elem_to_torch(dt, base)}}
    for k in range(n):
        models[f"org/ft{k}"] = {layer: _elem_to_torch(dt, fts[k])}
    cfg = MergeConfig(finetune_merge=[MergeModel(model=f"org/ft{k}", base="org/base", alpha=1.0) for k in range(n)],
                      output_base_model="org/base", output_dir="/tmp/unused")
    cls = TaskAdditionMerge if "taskaddition" in name else AdditionMerge
    out = asyncio.run(cls(cfg, index_manager=InMemoryIndex(models))._merge_layer(ShardLayer(0, "s", layer, False), DEV))
    assert out.dtype == _ELEM_TORCH[dt] and out.is_cuda
    assert _elem_same(dt, _elem_to_numpy(dt, out), want).all()


@pytest.mark.parametrize("mode,n_models,numel,dt", [(0, 3, 1 << 20, "f32"), (1, 17, (1 << 20) + 3, "f32"), (1, 5, (1 << 21) + 1, "f16"),
                                                     (1, 9, (1 << 20) + 7, "bf16"), (0, 12, 1000003, "bf16"), (1, 33, 300001, "f16")])
def test_elementwise_general_kernel_vs_oracle(E, mode, n_models, numel, dt):
    """The run-time-model-count kernel (any dtype, > 8 models) at ragged sizes against the numpy oracle, bit for bit."""
    from shardmerge_b200.merge._elementwise import elem_merge
    td = _ELEM_TORCH[dt]
    g = torch.Generator(device=DEV).manual_seed(950 + mode * 100 + n_models)
    base = (0.02 * torch.randn(numel, generator=g, device=DEV)).to(td)
    fts = [(base.float() + 0.003 * torch.randn(numel, generator=g, device=DEV)).to(td) for _ in range(n_models)]
    fts[0][:64] = base[:64]                                           # zero deltas
    fts[1][100] = float("nan"); fts[0][101] = float("inf")
    out = elem_merge(mode, base, fts, torch.device(DEV))
    want = (O.taskaddition_merge if mode == 1 else O.addition_merge)(_elem_to_numpy(dt, base), [_elem_to_numpy(dt, t) for t in fts], dt)
    assert _elem_same(dt, _elem_to_numpy(dt, out), want).all()


def test_elementwise_rejects_mixed_dtypes(E):
    from shardmerge_b200.merge._elementwise import elem_merge
    base = torch.zeros(64, dtype=torch.bfloat16, device=DEV)
    with pytest.raises(NotImplementedError):
        elem_merge(0, base, [base.float()], torch.device(DEV))
    with pytest.raises(NotImplementedError):
        elem_merge(0, base.double(), [base.double()], torch.device(DEV))


@pytest.mark.parametrize("mode,n_models,numel", [(0, 2, 4096 * 4096), (1, 3, 4096 * 4096), (1, 4, 1024 * 4096 + 5), (0, 8, 1000003)])
def test_elementwise_kernels_vs_oracle(E, mode, n_models, numel):
    """Large and ragged sizes (vector body + scalar tail) against the numpy oracle, bit for bit."""
    from shardmerge_b200.merge._elementwise import elem_merge
    g = torch.Generator(device=DEV).manual_seed(900 + mode * 10 + n_models)
    base = (0.02 * torch.randn(numel, generator=g, device=DEV)).to(torch.bfloat16)
    fts = [(base.float() + 0.003 * torch.randn(numel, generator=g, device=DEV)).to(torch.bfloat16) for _ in range(n_models)]
    fts[0][:64] = base[:64]                                           # zero deltas
    out = elem_merge(mode, base, fts, torch.device(DEV))
    want = (O.taskaddition_merge if mode == 1 else O.addition_merge)(bits(base), [bits(t) for t in fts])
    assert _nan_equal_bits(bits(out), want).all()


def test_elementwise_kernel_bandwidth(E):
    """The element-wise strategies are pure streams: (M + 2) x 2 bytes per element.  Prints the achieved HBM
    bandwidth (warm, CUDA events) -- a measurement, with a loose floor as the assertion."""
    from shardmerge_b200.merge._elementwise import elem_merge
    numel = 14336 * 4096
    g = torch.Generator(device=DEV).manual_seed(7)
    base = (0.02 * torch.randn(numel, generator=g, device=DEV)).to(torch.bfloat16)
    fts = [(base.float() + 0.003 * torch.randn(numel, generator=g, device=DEV)).to(torch.bfloat16) for _ in range(2)]
    for mode in (0, 1):
        for _ in range(3):
            elem_merge(mode, base, fts, torch.device(DEV))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            elem_merge(mode, base, fts, torch.device(DEV))
        e1.record(); torch.cuda.synchronize()
        gbs = 10 * numel * 2 * 4 / (e0.elapsed_time(e1) / 1e3) / 1e9
        print(f"\n[elem mode {mode}] {numel} elements x 2 finetunes: {gbs:.0f} GB/s of algorithmic traffic")
        assert gbs > 1500


@pytest.mark.parametrize("n_models,shape", [(4, (512, 2048)), (3, (1024, 2048)), (4, (1, 8192)), (5, (256, 4096))])
def test_fused_tree_matches_merge_sources_steps(E, n_models, shape):
    """BASELINE config 4: the pair tree with every pair merge on the fused chain (FourierMerge._merge_sources_tree: fp32
    intermediates, external target norm, device-side role / branch decisions) against the host-driven step path on the
    same kernels -- same spectra, same exact thresholds, so the same tensor."""
    R, C = shape
    sh = (R, C) if R > 1 else (C,)
    g = torch.Generator(device=DEV).manual_seed(77 + n_models + R)
    mean, bs = (1.0, 0.1) if R == 1 else (0.0, 0.02)
    base = (mean + bs * torch.randn(sh, generator=g, device=DEV)).to(torch.bfloat16)
    sig = (0.002, 0.0026, 0.0023, 0.0029, 0.0021)[:n_models]
    if R == 1:
        sig = tuple(5 * s for s in sig)
    alphas = (0.3, 0.5, 0.4, 0.2, 0.6)[:n_models]
    fts = [(base.float() + s * torch.randn(sh, generator=g, device=DEV)).to(torch.bfloat16) for s in sig]
    srcs = lambda: [E.make_source(base, ft, weight=a, name=f"m{k}") for k, (ft, a) in enumerate(zip(fts, alphas))]
    fm = _merger()
    got = fm.merge_sources(srcs(), base, torch.device(DEV), layer_name="model.layers.0.x")
    info = dict(fm.last_info)
    assert info["branches"] == ["slerp"] * (n_models - 1)
    assert len(info["swap"]) == n_models - 1                 # the fused tree ran: one device role decision per pair
    # deferred on the lanes as merge() does it
    fm.defer_checks = True
    got2 = fm.merge_sources(srcs(), base, torch.device(DEV), layer_name="model.layers.0.x", defer=True)
    fm.resolve_all()
    torch.cuda.synchronize()
    assert np.array_equal(bits(got), bits(got2))
    fm_steps = _merger()
    want = fm_steps._merge_sources_steps(srcs(), base, torch.device(DEV), layer_name="model.layers.0.x")
    assert fm_steps.last_info["branches"] == ["slerp"] * (n_models - 1)
    assert abs(info["target_norm"] / fm_steps.last_info["target_norm"] - 1) < 1e-7
    # Rounds >= 2 blend spectra whose culled bins hold rounding noise: the last bit of a round-1 scalar decides ~10 % of
    # the later rounds' bins (in the reference as well, see test_tree_of_four_finetunes_vs_oracle), so two correct
    # evaluations agree on the final tensor only loosely ...
    basef = base.float().cpu().numpy()
    dg, dw = got.float().cpu().numpy() - basef, want.float().cpu().numpy() - basef
    assert rel_l2(dg, dw) < 0.5 and abs(np.linalg.norm(dg) / np.linalg.norm(dw) - 1) < 0.05
    if n_models != 4 or R == 1:
        return
    # ... but the LAST round of the fused tree can be pinned exactly: feed its two fp32 inputs (the tree's own round-1
    # results) to the step-by-step tensor function with the same t and cull: same kernels' arithmetic on identical
    # inputs -> the same bf16 tensor.
    from shardmerge_b200.tensor import functions as F
    fm.keep_intermediates = True
    got3 = fm.merge_sources(srcs(), base, torch.device(DEV), layer_name="model.layers.0.x")
    assert np.array_equal(bits(got3), bits(got))
    (a0, a1, ta), (b0, b1, tb) = fm.last_tree                 # round-1 results in the order round 2 stacks them
    w = {f"m{k}": a for k, a in enumerate(alphas)}
    wa, wb = (w[a0] + w[a1]) / 2, (w[b0] + w[b1]) / 2
    x, y = (ta, tb) if float(ta.norm()) >= float(tb.norm()) else (tb, ta)     # larger norm takes role v0; t is not swapped
    m, _, _ = F.merge_tensors_fft2_slerp(x, y, t=wa / (wa + wb), device=DEV, t_sum=1.0, cutoff_pct=0.08, cull_pct=0.10)
    final = (base.float() + m.to(DEV) * E.f32(info["target_norm"])).to(torch.bfloat16)
    u = bf16_ulp_distance(bits(got), bits(final))
    assert float((u == 0).mean()) >= 0.9999 and int(u.max()) <= 1, (float((u == 0).mean()), int(u.max()))


def test_fused_tree_rounds_vs_oracle(E):
    """VERDICT r1 weak #4: pin what is deterministic in a tree.  Round 1 (pairs of deltas, cull 0.20): the fp32
    intermediates against the oracle's, flip-accounted <= 1e-5.  Round 2 (cull 0.10) blends spectra whose culled bins
    hold rounding noise, so ~10 % of its output bins are decided by noise in the reference itself: given IDENTICAL fp32
    inputs (the oracle's round-1 results) our pair merge must agree with the oracle's on every bin whose two inputs are
    above the noise floor."""
    from shardmerge_b200.tensor import functions as F
    R, C = 512, 2048
    g = torch.Generator(device=DEV).manual_seed(991)
    base = (0.02 * torch.randn((R, C), generator=g, device=DEV)).to(torch.bfloat16)
    sig, alphas = (0.002, 0.0026, 0.0023, 0.0029), (0.3, 0.5, 0.4, 0.2)
    fts = [(base.float() + s * torch.randn((R, C), generator=g, device=DEV)).to(torch.bfloat16) for s in sig]
    fm = _merger()
    fm.keep_intermediates = True
    srcs = [E.make_source(base, ft, weight=a, name=f"m{k}") for k, (ft, a) in enumerate(zip(fts, alphas))]
    fm.merge_sources(srcs, base, torch.device(DEV), layer_name="model.layers.0.x")
    assert len(fm.last_tree) == 2
    models = [dict(base=bits(base), ft=bits(ft), alpha=a, name=f"m{k}") for k, (ft, a) in enumerate(zip(fts, alphas))]
    info = {}
    O.merge_layer(bits(base), models, info=info, interp_imag=False)
    inter = info["intermediates"]
    assert len(inter) == 3                                  # two round-1 results and the final one
    round1 = {}
    for na, nb, t in fm.last_tree:
        key = next(k for k in inter if set(k.split("_")) == {na, nb})
        raw, resid, share = flip_accounted(t.cpu().numpy(), inter[key].reshape(R, C), k=16)
        print(f"\n[tree round 1 {key}] raw {raw:.3e} flip-accounted {resid:.3e}")
        assert resid <= 1e-5, (key, raw, resid)
        round1[key] = inter[key].reshape(R, C)
    # round 2 on the oracle's own round-1 results
    (ka, a), (kb, b) = sorted(round1.items(), key=lambda kv: -float(np.linalg.norm(kv[1])))
    t2 = 0.5                                                # both weights are (w_x + w_y) / 2 -> ratio of the two means
    wa = {k: (alphas[int(k.split("_")[0][1:])] + alphas[int(k.split("_")[1][1:])]) / 2 for k in round1}
    first, second = list(round1)                            # stack order of round 2 = order the pairs were produced
    t2 = wa[first] / (wa[first] + wa[second])
    ours, _, _ = F.merge_tensors_fft2_slerp(torch.from_numpy(a), torch.from_numpy(b), t=t2, device=DEV, t_sum=1.0,
                                            cutoff_pct=0.08, cull_pct=0.10)
    ref, n0, n1 = O.merge_tensors_fft2_slerp(a, b, t2, t_sum=1.0, cutoff_pct=0.08, cull_pct=0.10, interp_imag=False)
    So, Sr = np.fft.rfft2(ours.numpy().astype(np.float64)), np.fft.rfft2(np.asarray(ref, dtype=np.float64))
    A, B = np.fft.rfft2(a.astype(np.float64) / n0), np.fft.rfft2(b.astype(np.float64) / n1)
    floor = 1e-3 * np.median(np.abs(A.real))
    solid = (np.abs(A.real) > floor) & (np.abs(B.real) > floor)           # bins not decided by rounding noise
    frac_solid = float(solid.mean())
    # The cull statistic of round 2 (rank 0.10 N) sits where the noise-decided bins end and the solid ones begin, so its
    # VALUE depends on how many noise bins came out tiny -- a binomial count.  Bins next to either threshold are left out too.
    med = np.median(np.abs(Sr.real[solid]))
    thr_r = np.abs(Sr.real[solid & (np.abs(Sr.real) > 1e-4 * med)]).min()
    thr_o = np.abs(So.real[solid & (np.abs(So.real) > 1e-4 * med)]).min()
    tau = 1.25 * max(thr_r, thr_o)
    cmp = solid & (np.abs(Sr.real) > tau) & (np.abs(So.real) > tau)
    d = (So.real - Sr.real)[cmp]
    # a handful of decisions next to the thresholds may still flip: set the largest differences aside like flip_accounted
    e = np.sort(d ** 2)[::-1]
    resid = float(np.sqrt(e[64:].sum() / (Sr.real[cmp] ** 2).sum()))
    print(f"[tree round 2] bins above the noise floor {frac_solid:.3f}, compared {float(cmp.mean()):.3f}; cull thresholds "
          f"{thr_o:.4e} (ours) {thr_r:.4e} (oracle); Re rel-L2 {np.sqrt(e.sum() / (Sr.real[cmp] ** 2).sum()):.3e}, without the 64 largest {resid:.3e}")
    assert 0.55 < frac_solid < 0.75                         # two inputs with 20 % culled bins each: ~0.64 solid
    assert float(cmp.mean()) > 0.45
    # what remains is carried by the blend's scalars: a bin whose re0 is rounding noise and whose signs happen to agree
    # still adds re1^2 to the SLERP sum s11, so dot / ||rel|| carry a binomial ~1/sqrt(N) term (1e-3 at 1 Mi elements)
    assert resid <= 5e-3, resid
    assert rel_l2(So.imag, Sr.imag) <= 1e-5                 # imaginary part: Im X0, untouched by the blend
