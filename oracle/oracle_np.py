"""oracle_np.py -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

A CPU (numpy) restatement of the reference's per-tensor spectral merge path, used only as
the checker in tests/, in __graft_entry__.smoke() and as bench.py's `cpu_baseline` /
`--impl reference` arm.  Nothing under shardmerge_b200/ imports this module.

Every function cites the reference span it restates (paths relative to the reference root).
Where the arithmetic lives in a third-party dependency (torch >= 2.9.1, pyproject.toml:11;
torch.fft -> MKL/cuFFT, torch.sort, torch.norm), the published semantics are restated with
numpy: np.fft in single precision (numpy >= 2.0 keeps float32/complex64), np.sort, and
norms accumulated in float64 then rounded to float32 -- deliberately NOT reproducing the
low bias of torch's CPU fp32 `.norm()` at large N (SURVEY.md section 0 / 7.3-0).

Pinning: tests/test_oracle_golden.py checks this file against tests/golden/*.npz, which
oracle/make_golden.py produced by importing the reference itself from /root/reference
(stage taps and final bf16 outputs, CPU, seeded inputs).  The reference's own tests hold no
numeric golden values for this path (SURVEY.md section 8c), so those fixtures are the pin.

bf16 tensors are carried as uint16 bit patterns (numpy has no bfloat16).
"""
from __future__ import annotations

import numpy as np

F32 = np.float32


# --------------------------------------------------------------------------- bf16 helpers
def bf16_to_f32(u16: np.ndarray) -> np.ndarray:
    return (u16.astype(np.uint32) << 16).view(np.float32)


def f32_to_bf16(x: np.ndarray) -> np.ndarray:
    """round-to-nearest-even, NaN kept quiet (what torch's .to(torch.bfloat16) does)."""
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)
    nan = (u & 0x7FFFFFFF) > 0x7F800000
    r = ((u.astype(np.uint64) + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint16)
    r[nan] = ((u[nan] >> 16) | 0x0040).astype(np.uint16)
    return r


def widen(x: np.ndarray) -> np.ndarray:
    """A stored tensor as fp32, exactly: uint16 arrays are bf16 bit patterns, float16 and float32 arrays are taken as
    they are (what `.to(torch.float32)` does to a bf16, fp16 or fp32 tensor)."""
    x = np.asarray(x)
    if x.dtype == np.uint16:
        return bf16_to_f32(x)
    if x.dtype in (np.float16, np.float32):
        return x.astype(np.float32)
    raise TypeError(f"no stored tensor dtype is carried as {x.dtype} (uint16 = bf16 bits, float16, float32)")


def norm32(x: np.ndarray) -> float:
    """torch.norm of an fp32 tensor, restated with an accurate (fp64) accumulation and the
    fp32 result torch would hand back through .item()."""
    x = np.asarray(x, dtype=np.float32).ravel()
    return float(np.float32(np.sqrt(np.dot(x.astype(np.float64), x.astype(np.float64)))))


# --------------------------------------------------------------------------- shard/tensor/functions.py
def slerp(v0: np.ndarray, v1: np.ndarray, t: float) -> np.ndarray:
    """shard/tensor/functions.py:24-43 on 1-D fp32 vectors."""
    n0, n1 = norm32(v0), norm32(v1)
    with np.errstate(invalid="ignore", divide="ignore"):
        s01 = np.float32(np.dot(v0.astype(np.float64), v1.astype(np.float64)))
        dot = np.float32(s01 / (np.float32(n0) * np.float32(n1)))          # :36
        dot = np.float32(np.clip(dot, -1.0, 1.0))                           # :37
        theta = np.float32(np.arccos(dot) * np.float32(t))                  # :39
        rel = (v1 - v0 * dot).astype(np.float32)                            # :40
        rn = np.float32(max(norm32(rel), 1e-12)) if np.isfinite(dot) else np.float32(np.nan)
        rel = (rel / rn).astype(np.float32)                                 # :41 F.normalize(eps=1e-12)
        return (v0 * np.float32(np.cos(theta)) + rel * np.float32(np.sin(theta))).astype(np.float32)   # :43


def fft_transform(x: np.ndarray) -> np.ndarray:
    """shard/tensor/functions.py:45-58 -> complex64."""
    x = np.asarray(x, dtype=np.float32)
    if x.ndim == 1:
        return np.fft.fft(x).astype(np.complex64)
    return np.fft.fftn(x, axes=(-2, -1)).astype(np.complex64)


def ifft_transform(z: np.ndarray) -> np.ndarray:
    """shard/tensor/functions.py:60-73 -> float32 (real part of the inverse transform)."""
    z = np.asarray(z)
    if z.dtype != np.complex64:
        z = z.astype(np.complex64)
    if z.ndim == 1:
        return np.fft.ifft(z).real.astype(np.float32)
    return np.fft.ifftn(z, axes=(-2, -1)).real.astype(np.float32)


def normalize_tensor(x: np.ndarray):
    """shard/tensor/functions.py:75-88.  `tensor / norm` with a Python scalar."""
    n = norm32(x)
    if n == 0:
        return x, n
    return (x / np.float32(n)).astype(np.float32), n


def kth_abs(values: np.ndarray, k: int) -> float:
    """sorted(values.ravel())[k] as done with torch.sort at functions.py:114-120 and :139-141."""
    flat = np.sort(values.ravel(), kind="stable")
    if k >= flat.size:
        return float(flat[-1])
    return float(flat[k])


def interpolate_fft_components(v0_fft, v1_fft, t, t_sum=1.0, cutoff_pct=0.0, cull_pct=0.0, interp_imag=True,
                               taps=None):
    """shard/tensor/functions.py:90-162."""
    re0 = np.ascontiguousarray(v0_fft.real, dtype=np.float32)
    re1 = np.ascontiguousarray(v1_fft.real, dtype=np.float32)
    a0, a1 = np.abs(re0), np.abs(re1)
    if cutoff_pct > 0:                                                      # :113-120
        allr = np.concatenate([a0.ravel(), a1.ravel()])
        thr = np.float32(kth_abs(allr, int(allr.size * cutoff_pct)))
    else:
        thr = np.float32(0)
    sign = np.sign(re0) == np.sign(re1)                                     # :124
    small = a1 < thr                                                        # :125-126 (re1 tested twice)
    slerp_mask = sign & ~small                                              # :127
    sum_mask = sign & ~slerp_mask                                           # :128
    rest_mask = ~slerp_mask & ~sum_mask                                     # :129
    larger = a0 > a1                                                        # :131
    out = np.zeros_like(re0)
    out[slerp_mask] = slerp(re0[slerp_mask], re1[slerp_mask], t)            # :134
    out[sum_mask] = (re0[sum_mask] + np.float32(t_sum) * re1[sum_mask]).astype(np.float32)   # :135
    out[rest_mask] = np.where(larger[rest_mask], re0[rest_mask], re1[rest_mask])             # :136
    cull_thr = np.float32(0)
    if cull_pct > 0:                                                        # :138-148
        ao = np.abs(out)
        cull_thr = np.float32(kth_abs(ao, int(ao.size * cull_pct)))
        out[ao < cull_thr] = 0
    if taps is not None:
        taps.update(thr_cut=float(thr), thr_cull=float(cull_thr), real=out.copy(),
                    frac_slerp=float(slerp_mask.mean()), frac_sum=float(sum_mask.mean()))
    if interp_imag:                                                         # :150-158 nested imaginary path
        i0 = fft_transform(np.ascontiguousarray(v0_fft.imag, dtype=np.float32))
        i1 = fft_transform(np.ascontiguousarray(v1_fft.imag, dtype=np.float32))
        j = interpolate_fft_components(i0, i1, t, cutoff_pct=0, cull_pct=0, interp_imag=False)
        imag = ifft_transform(j)
    else:
        imag = np.ascontiguousarray(v0_fft.imag, dtype=np.float32)          # :160
    return (out + 1j * imag).astype(np.complex64)


def merge_tensors_fft2_slerp(v0, v1, t, b=0.1, t_sum=1.0, cutoff_pct=0.0, cull_pct=0.0, interp_imag=True,
                             taps=None):
    """shard/tensor/functions.py:164-221 -> (merged fp32, norm_v0, norm_v1)."""
    v0, n0 = normalize_tensor(np.asarray(v0, dtype=np.float32))             # :181-182
    v1, n1 = normalize_tensor(np.asarray(v1, dtype=np.float32))
    if n1 < 0.0001:                                                          # :184-185
        return v0, n0, n1
    if n0 < 0.0001:                                                          # :187-190
        return v0, n0, n1
    f0, f1 = fft_transform(v0), fft_transform(v1)                            # :193-194
    if taps is not None:
        taps.update(fft0=f0, fft1=f1)
    ratio = n1 / (n0 + 1e-10)
    if ratio < b:                                                            # :199-202
        res = (f0 + f1 * np.complex64(t)).astype(np.complex64)
    else:                                                                    # :205
        res = interpolate_fft_components(f0, f1, t, t_sum=t_sum, cutoff_pct=cutoff_pct, cull_pct=cull_pct,
                                         interp_imag=interp_imag, taps=taps)
    m = ifft_transform(res)                                                  # :208
    m = np.where(np.isnan(m), np.float32(0), m).astype(np.float32)           # :211-213
    if np.any(np.isinf(m)):                                                  # :215-217
        raise ValueError("Inf in ifft output")
    return m, n0, n1


def arithmetic_fft_components(v0_fft, v1_fft, t, agreement, do_imag=True):
    """shard/tensor/functions.py:256-302."""
    re0 = np.ascontiguousarray(v0_fft.real, dtype=np.float32)
    re1 = np.ascontiguousarray(v1_fft.real, dtype=np.float32)
    sign = (np.sign(re0) == np.sign(re1)) if agreement else np.ones(re0.shape, dtype=bool)   # :273-276
    out = np.zeros_like(re0)
    out[sign] = (re0[sign] + np.float32(t) * re1[sign]).astype(np.float32)   # :279
    # :282 compares v0 with itself -> the "larger" mask is all False -> always v1
    out[~sign] = re1[~sign]                                                  # :284
    if do_imag:                                                              # :291-299
        i0 = fft_transform(np.ascontiguousarray(v0_fft.imag, dtype=np.float32))
        i1 = fft_transform(np.ascontiguousarray(v1_fft.imag, dtype=np.float32))
        j = arithmetic_fft_components(i0, i1, t, agreement, do_imag=False)
        imag = ifft_transform(j)
    else:
        imag = np.ascontiguousarray(v0_fft.imag, dtype=np.float32)
    return (out + 1j * imag).astype(np.complex64)


def task_arithmetic_fft2(v0, v1, t, agreement=True):
    """shard/tensor/functions.py:224-254."""
    f0 = fft_transform(np.asarray(v0, dtype=np.float32))
    f1 = fft_transform(np.asarray(v1, dtype=np.float32))
    return ifft_transform(arithmetic_fft_components(f0, f1, t, agreement))


def correlated_pairs(corr: np.ndarray, way: str = "least"):
    """shard/tensor/functions.py:316-365 (greedy pairing on |corr| of the upper triangle)."""
    n = corr.shape[0]
    avail = np.triu(np.ones((n, n), dtype=bool), k=1)
    items = list(range(n))
    out = []
    while avail.any():
        valid = np.where(avail, corr, np.inf)
        finite = np.abs(valid[valid != np.inf])
        if way == "least":
            m = finite.min()
        elif way == "most":
            m = finite.max()
        else:
            raise ValueError("Invalid way. Choose 'least' or 'most'.")
        idx = np.argwhere(np.abs(valid) == m)
        if len(idx) == 0:
            break
        x, y = int(idx[0][0]), int(idx[0][1])
        out.append((x, y, float(corr[x, y])))
        avail[x, :] = False; avail[:, x] = False; avail[y, :] = False; avail[:, y] = False
        items.remove(x); items.remove(y)
    for i in items:
        out.append((i, -1, float(corr[i, i])))
    return out


# --------------------------------------------------------------------------- shard/merge/fast_fourier.py
def merge_layer(base_out_bf16, models, target_norm_offset=1e-10, cull_start_pct=0.20, interp_imag=True,
                info=None):
    """FourierMerge._merge_layer for a regular (model.layers.*) tensor,
    shard/merge/fast_fourier.py:132-276, with the disk cache replaced by a dict.

    base_out_bf16: the output-base tensor -- uint16 bf16 bit patterns, or a float16 / float32 array (see `widen`).
    models: list of dicts {base: array, ft: array, alpha: float, name: str}, arrays stored as base_out_bf16 may be
            (already filtered by use_layer_index, :135).
    Returns uint16 bit patterns of the merged bf16 tensor.
    """
    cache = {}
    norms, stack, weights = [], [], []
    for m in models:                                                         # :147-158
        delta = (widen(m["ft"]) - widen(m["base"])).astype(np.float32)   # base.py:128-132
        norms.append(np.float32(norm32(delta)))
        cache[m["name"]] = delta
        stack.append(m["name"]); weights.append(float(m["alpha"]))
    target_norm = float(np.float32(np.mean(np.array(norms, dtype=np.float32)))) + target_norm_offset   # :165
    cull_pct = cull_start_pct
    branches = []
    while len(stack) > 1:                                                    # :171-254
        n = len(stack)
        corr = np.zeros((n, n), dtype=np.float32)
        for i in range(n):
            for j in range(i + 1, n):
                corr[i, j] = norms[i] * norms[j]                             # :180-184 (stale norms in later rounds)
        nxt, nxt_w = [], []
        for x, y, _ in correlated_pairs(corr, "least"):
            if y < 0:
                nxt.append(stack[x]); nxt_w.append(weights[x]); continue
            a_name, b_name = stack[x], stack[y]
            a_w, b_w = weights[x], weights[y]
            a, b = cache[a_name], cache[b_name]
            na, nb = norm32(a), norm32(b)
            if abs(na) < abs(nb):                                            # :212-215 (weights are NOT swapped)
                a, b = b, a; a_name, b_name = b_name, a_name; na, nb = nb, na
            cnorm_a = abs(na / target_norm); cnorm_b = abs(nb / target_norm)
            n_ratio = cnorm_b / (cnorm_a + 1e-10)
            if cnorm_a < 1e-6:                                               # :223-225
                merged = (a + b).astype(np.float32); branches.append("add")
            elif cnorm_b < 1e-6 or n_ratio < 0.1:                            # :226-232
                norm_scale = target_norm / na
                sa = (a * np.float32(norm_scale)).astype(np.float32)
                w_scale = b_w / (a_w + 1e-10)
                sb = ((b * np.float32(w_scale)).astype(np.float32) * np.float32(norm_scale)).astype(np.float32)
                merged = task_arithmetic_fft2(sa, sb, t=1.0, agreement=True); branches.append("arith")
            else:                                                            # :233-243
                a_prop = a_w / (a_w + b_w)
                merged, _, _ = merge_tensors_fft2_slerp(a, b, t=a_prop, t_sum=1.0, cutoff_pct=0.08,
                                                        cull_pct=cull_pct, interp_imag=interp_imag)
                merged = (merged * np.float32(target_norm)).astype(np.float32); branches.append("slerp")
            name = f"{a_name}_{b_name}"
            nxt.append(name); nxt_w.append((a_w + b_w) / 2.0)
            cache[name] = merged
        stack, weights = nxt, nxt_w
        cull_pct = cull_pct / 2.0                                            # :254
    result = cache[stack[0]]                                                 # :256-257
    with np.errstate(invalid="ignore"):
        result = (widen(base_out_bf16) + result).astype(np.float32)          # :269
    result = np.where(np.isnan(result), np.float32(0), result).astype(np.float32)   # :270-271
    if np.any(np.isinf(result)):                                             # :273-274
        raise ValueError("Inf in merged tensor")
    if info is not None:
        info.update(branches=branches, target_norm=target_norm, norms=[float(x) for x in norms],
                    merged_f32=cache[stack[0]], intermediates={k: v for k, v in cache.items() if "_" in k})          # the fp32 tree result before the base is added (:256-257)
    return f32_to_bf16(result)                                               # :276


# --------------------------------------------------------------------------- element-wise strategies (SURVEY 8f N3)
def _bf16_round(x: np.ndarray) -> np.ndarray:
    """fp32 values rounded to bf16 and widened again (one bf16 rounding, as after every torch bf16 op)."""
    return bf16_to_f32(f32_to_bf16(np.asarray(x, dtype=np.float32)))


def _elem_codec(dtype: str):
    """(widen to fp32, round fp32 to the storage dtype and widen again, narrow to storage) for the element-wise strategies:
    'bf16' tensors travel as uint16 bit patterns, 'f16' as np.float16, 'f32' as np.float32."""
    if dtype == "bf16":
        return bf16_to_f32, _bf16_round, f32_to_bf16
    if dtype == "f16":
        return (lambda a: np.asarray(a, dtype=np.float16).astype(np.float32),
                lambda x: np.asarray(x, dtype=np.float32).astype(np.float16).astype(np.float32),
                lambda x: np.asarray(x, dtype=np.float32).astype(np.float16))
    if dtype == "f32":
        ident = lambda a: np.asarray(a, dtype=np.float32)
        return ident, ident, ident
    raise ValueError(dtype)


def _cascade_sum_rows(x: np.ndarray) -> np.ndarray:
    """torch.sum(x, dim=0) of a CPU float tensor [M, ...] (ATen SumKernel.cpp, cascade_sum -> multi_row_sum over the outer
    dimension, fp32 accumulators): rows are added one by one into a level-0 accumulator; after every 16 rows it is
    folded into level 1 (after 256 into level 2, ...), and the levels are added at the end.  Up to 15 rows this is the plain
    sequential sum; from 16 rows on the association differs."""
    M = x.shape[0]
    acc = [np.zeros(x.shape[1:], dtype=np.float32) for _ in range(4)]
    i = 0
    while i + 16 <= M:
        for _ in range(16):
            acc[0] = acc[0] + x[i]
            i += 1
        for j in range(1, 4):
            acc[j] = acc[j] + acc[j - 1]
            acc[j - 1] = np.zeros_like(acc[0])
            if i & (15 << (4 * j)):
                break
    while i < M:
        acc[0] = acc[0] + x[i]
        i += 1
    for j in range(1, 4):
        acc[0] = acc[0] + acc[j]
    return acc[0]


def addition_merge(base, fts, dtype: str = "bf16") -> np.ndarray:
    """AdditionMerge._merge_layer (shard/merge/addition.py:44-83): out = 0; out += (ft - base) per model, every
    operation in the tensors' own dtype (bf16 / fp16: computed in fp32, rounded to the dtype after each op).  The summed
    delta is returned -- the base is NOT added back.  Storage as in _elem_codec (bf16: uint16 bit patterns in and out)."""
    widen, rnd, narrow = _elem_codec(dtype)
    with np.errstate(invalid="ignore", over="ignore"):
        b = widen(base)
        out = np.zeros(b.shape, dtype=np.float32)
        for ft in fts:
            delta = rnd(widen(ft) - b)                             # :72
            out = rnd(out + delta)                                 # :73
    return narrow(out)


def taskaddition_merge(base, fts, dtype: str = "bf16") -> np.ndarray:
    """TaskAdditionMerge._merge_layer (shard/merge/taskaddition.py:44-83): deltas in the tensors' dtype, majority sign over
    the models (sign of the sum of signs), deltas whose sign differs from it zeroed, the rest summed (torch.sum on CPU:
    fp32 accumulators in model order -- cascaded from 16 models on, _cascade_sum_rows -- one rounding at the end)."""
    widen, rnd, narrow = _elem_codec(dtype)
    with np.errstate(invalid="ignore", over="ignore"):
        b = widen(base)
        d = np.stack([rnd(widen(ft) - b) for ft in fts], axis=0)   # :68
        sgn = np.sign(d)                                            # :71   (NaN stays NaN)
        w = np.sign(_cascade_sum_rows(sgn))                        # :73   (small integers: exact in any order)
        mask = (sgn == w[None]).astype(np.float32)                 # :75   (NaN == NaN is False)
        masked = rnd(d * mask)                                     # :76
        acc = _cascade_sum_rows(masked)                            # :78
    return narrow(acc)
