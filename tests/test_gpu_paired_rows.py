"""The paired forward row pass (sm_fwd_rows_bf16_pair): both finetunes of a pair merge over one shared base in one pass.
Its spectra are those of two single-model passes bit for bit, its last CTA writes the scalar block k_prepare writes from
the same sums, and a pair with two different base tensors keeps the two single-model passes.  Run with `pytest -m gpu`."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import oracle_np as O
from tests.parity_util import bf16_ulp_distance, flip_accounted

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


@pytest.fixture(scope="module")
def E():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from shardmerge_b200 import engine
    return engine


def bits(t):
    return t.contiguous().view(torch.int16).cpu().numpy().view(np.uint16)


def _inputs(shape, seed, sig=(0.002, 0.0026)):
    g = torch.Generator(device=DEV).manual_seed(seed)
    base = (0.02 * torch.randn(shape, generator=g, device=DEV)).to(torch.bfloat16)
    fts = [(base.float() + s * torch.randn(shape, generator=g, device=DEV)).to(torch.bfloat16) for s in sig]
    return base, fts


@pytest.mark.parametrize("shape", [(4096, 4096), (14336, 4096), (4096, 14336), (1024, 4096)])
def test_paired_pass_equals_two_single_passes(E, shape):
    """q/o, gate/up, down_proj and k/v of Llama-3.1-8B."""
    from shardmerge_b200 import _lib
    R, C = shape
    pl = E.get_plan(R, C, DEV)
    lib, st = pl.lib, E._stream(pl.device)
    assert lib.sm_fwd_rows_pair_supported(pl.handle) == 1
    base, (ft0, ft1) = _inputs(shape, seed=R + C)
    planes = [torch.zeros((R, pl.P), dtype=torch.float32, device=DEV) for _ in range(8)]
    re0, im0, re1, im1, rr0, ri0, rr1, ri1 = planes
    ref_ss = torch.zeros(2, dtype=torch.float64, device=DEV)
    for ft, re, im, k in ((ft0, rr0, ri0, 0), (ft1, rr1, ri1, 1)):
        _lib.check(lib.sm_fwd_rows_bf16(pl.handle, pl.tables.data_ptr(), base.data_ptr(), ft.data_ptr(), re.data_ptr(),
                                        im.data_ptr(), ref_ss.data_ptr() + 8 * k, st), "sm_fwd_rows_bf16")
    ctl = torch.zeros(_lib.SM_CTL_BYTES, dtype=torch.uint8, device=DEV)
    _lib.check(lib.sm_fwd_rows_bf16_pair(pl.handle, pl.tables.data_ptr(), base.data_ptr(), ft0.data_ptr(), ft1.data_ptr(),
                                         re0.data_ptr(), im0.data_ptr(), re1.data_ptr(), im1.data_ptr(), ctl.data_ptr(),
                                         1e-10, 0.0, st), "sm_fwd_rows_bf16_pair")
    torch.cuda.synchronize()
    for got, want in ((re0, rr0), (im0, ri0), (re1, rr1), (im1, ri1)):
        assert torch.equal(got.view(torch.int32), want.view(torch.int32))
    ss = ctl[_lib.SM_CTL_SUMSQ:_lib.SM_CTL_SUMSQ + 16].view(torch.float64).cpu()
    # per-CTA partials are added in a different order: the two sums agree to fp64 rounding
    assert torch.allclose(ss, ref_ss.cpu(), rtol=1e-12, atol=0.0), (ss, ref_ss)
    # ...and to torch's fp64 sum of squares of the fp32 deltas up to the fp32 per-thread partials of every row pass
    for k, ft in enumerate((ft0, ft1)):
        d = (ft.float() - base.float()).double()
        assert abs(float(ss[k]) / float((d * d).sum()) - 1) < 1e-6


def _scalars(ctl, L):
    """the part of the scalar block the pair merge's decisions write: scales, out scale, norms, swap, branch, target_norm"""
    h = ctl.cpu()
    flt = h[L.SM_CTL_FLT:L.SM_CTL_FLT + 64].view(torch.int32)
    ints = h[L.SM_CTL_INT:L.SM_CTL_INT + 16].view(torch.int32)
    tn = h[L.SM_CTL_TN:L.SM_CTL_TN + 8].view(torch.int64)
    f = [int(flt[i]) for i in (L.SM_F_SCALE_X, L.SM_F_SCALE_Y, L.SM_F_OUT_SCALE, L.SM_F_NORM_X, L.SM_F_NORM_Y)]
    return f + [int(ints[L.SM_I_SWAP]), int(ints[L.SM_I_BRANCH]), int(tn[0])]


def _tiny(base, idx, v):
    ft = base.clone()
    ft.view(-1)[idx] = base.view(-1)[idx] + v
    return ft


@pytest.mark.parametrize("case,branch,target_norm", [
    ("equal", "slerp", 0.0), ("zero_delta", "arith", 0.0), ("ratio_below_0.1", "arith", 0.0),
    ("both_zero", "add", 0.0), ("small_norms", "slerp-early", 0.0), ("swapped_given_tn", "slerp", 0.37),
])
def test_paired_pass_scalar_block_equals_k_prepare(E, case, branch, target_norm):
    """The whole chain on a shared base (paired row pass, decisions in its last CTA) against the chain that is handed the
    same two sums and runs k_prepare (rows_done): the same scalar block, bit for bit."""
    from shardmerge_b200 import _lib as L
    R, C = 1024, 4096
    base, (ft0, ft1) = _inputs((R, C), seed=7)
    if case == "equal":
        ft1 = ft0.clone()
    elif case == "zero_delta":
        ft1 = base.clone()
    elif case == "ratio_below_0.1":
        g = torch.Generator(device=DEV).manual_seed(8)
        ft0 = (base.float() + 0.05 * torch.randn((R, C), generator=g, device=DEV)).to(torch.bfloat16)
    elif case == "both_zero":
        ft0, ft1 = base.clone(), base.clone()
    elif case == "small_norms":
        base = torch.zeros((R, C), dtype=torch.bfloat16, device=DEV)
        ft0, ft1 = _tiny(base, 12345, 5e-5), _tiny(base, 777, 4e-5)
    elif case == "swapped_given_tn":
        ft0, ft1 = ft1, ft0
    out = torch.empty((R, C), dtype=torch.bfloat16, device=DEV)
    ws_a = E.get_workspace(R, C, DEV, lane="paired-a")
    ws_b = E.get_workspace(R, C, DEV, lane="paired-b")
    s0, s1 = E.make_source(base, ft0, weight=0.3), E.make_source(base, ft1, weight=0.5)
    kw = dict(t=0.3 / 0.8, target_norm=target_norm)
    E.pair_merge_async(ws_a, s0, s1, base, out, **kw).resolve()
    sumsq = ws_a.ctl[L.SM_CTL_SUMSQ:L.SM_CTL_SUMSQ + 16].view(torch.float64).cpu().tolist()
    E.pair_merge_async(ws_b, s0, s1, base, out, rows_done=True, sumsq=sumsq, **kw).resolve()
    got, want = _scalars(ws_a.ctl, L), _scalars(ws_b.ctl, L)
    assert got == want, (case, got, want)
    assert L.BRANCH_NAMES[want[6]] == branch


def _profiled(lib, fn):
    """per kernel class of the fused chain: (launches, algorithmic bytes) of what fn() enqueues"""
    from shardmerge_b200 import _lib
    n = len(_lib.CLS_NAMES)
    lib.sm_profile_enable(1)
    try:
        fn()
        torch.cuda.synchronize()
    finally:
        ms, by, la = (ctypes.c_double * n)(), (ctypes.c_double * n)(), (ctypes.c_int * n)()
        lib.sm_profile_collect(ms, by, la, n)
        lib.sm_profile_enable(0)
    return {name: (int(la[i]), float(by[i])) for i, name in enumerate(_lib.CLS_NAMES)}


def test_two_bases_keep_two_row_passes_and_match_the_oracle(E):
    """merge_sources with two different base tensors (equal values, separate storage) runs two single-model row passes
    and k_prepare, and matches the oracle as before; with one shared base it runs the paired pass, and the two give the
    same bf16 result."""
    from shardmerge_b200 import _lib
    from shardmerge_b200.config import MergeConfig
    from shardmerge_b200.index import InMemoryIndex
    from shardmerge_b200.merge.fast_fourier import FourierMerge
    shape = (1024, 4096)
    N = shape[0] * shape[1]
    base, fts = _inputs(shape, seed=99)
    base1 = base.clone()
    fm = FourierMerge(MergeConfig(finetune_merge=[], output_base_model="org/base", output_dir="/tmp/unused"),
                      index_manager=InMemoryIndex({}))
    lib = _lib.load()
    res = {}

    def run(key, b1):
        srcs = [E.make_source(base, fts[0], weight=0.3, name="m0"), E.make_source(b1, fts[1], weight=0.5, name="m1")]
        res[key] = fm.merge_sources(srcs, base, torch.device(DEV), layer_name="model.layers.0.x")
        assert fm.last_info["branches"] == ["slerp"]
    two = _profiled(lib, lambda: run("two", base1))
    one = _profiled(lib, lambda: run("one", base))
    assert two["row_fwd"] == (2, 16.0 * N) and two["scalars"][0] == 1
    assert one["row_fwd"] == (1, 14.0 * N) and one["scalars"][0] == 0
    assert torch.equal(res["one"].view(torch.int16), res["two"].view(torch.int16))
    models = [dict(base=bits(b), ft=bits(fts[k]), alpha=a, name=f"m{k}") for k, (b, a) in enumerate(((base, 0.3), (base1, 0.5)))]
    info = {}
    oo = O.merge_layer(bits(base), models, info=info)
    assert abs(fm.last_info["target_norm"] / info["target_norm"] - 1) < 1e-6
    basef = O.bf16_to_f32(bits(base))
    raw, resid, share = flip_accounted(O.bf16_to_f32(bits(res["two"])) - basef, O.bf16_to_f32(oo) - basef, k=16)
    frac1 = float((bf16_ulp_distance(bits(res["two"]), oo) <= 1).mean())
    assert resid < 0.05 and frac1 >= 0.98, (raw, resid, share, frac1)
