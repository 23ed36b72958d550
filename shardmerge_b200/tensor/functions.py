"""Tensor-level spectral merge operators with the signatures of shard/tensor/functions.py.

Every function keeps the reference's name, argument meaning, return convention (results come
back on the CPU, like the reference which ends every transform with `.to("cpu")`,
functions.py:56,58,71,73) and error behaviour, but the arithmetic runs in the sm_100a kernels
behind include/shardmerge_b200.h.  `device` must name a CUDA device: there is no CPU path.

Scope notes (documented deviations, all below FFT rounding except where stated):
  * Spectra handed to interpolate_fft_components / arithmetic_fft_components / ifft_transform
    are treated as spectra of REAL tensors (Hermitian); that is how the reference produces and
    consumes them.  ifft_transform keeps `.real` semantics exactly (Hermitian projection).
  * The nested "imaginary part" path (functions.py:152-158, :291-299) feeds FFT rounding noise
    through a SLERP and returns Im X0 up to ~2e-7 relative (SURVEY.md 7.3-2, re-measured in
    tests/test_oracle_golden.py); here the imaginary part of the result is Im X0.
"""
from __future__ import annotations

import logging
from typing import Generator, Literal

import torch

from .. import engine as E

logger = logging.getLogger(__name__)


# ------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------
def _dev(device) -> torch.device:
    return E._require_cuda(device)


def _as_rows(t: torch.Tensor):
    """rows x columns of `t` laid out as one matrix (leading dimensions stack [R][C] slices, engine.Plan)."""
    R, C = E.shape_rc(t)
    return R, C


def _spectrum_of(x32: torch.Tensor, dev, scale: float = 1.0):
    """real fp32 tensor (on dev) -> workspace whose slot 0 holds its half-planar spectrum * scale."""
    R, C = _as_rows(x32)
    ws = E.ws_for(x32, dev)
    ws.ctl.zero_()
    E.fwd_rows(ws, 0, E.Source(x32=x32), E.D_SUMSQ0)
    E.fwd_cols(ws, 0, scale=scale)
    return ws


def _expand(ws: E.Workspace, slot: int, shape) -> torch.Tensor:
    """half-planar spectrum -> full complex64 tensor (Hermitian mirror), slice by slice for a stack."""
    pl = ws.plan
    out = torch.empty((pl.R, pl.C), dtype=torch.complex64, device=pl.device)
    for b in range(pl.batch):
        off = b * pl.slice_bytes
        E._lib.check(pl.lib.sm_expand_full(pl.col_handle, ws.re[slot].data_ptr() + off, ws.im[slot].data_ptr() + off,
                                          out.data_ptr() + b * pl.Rin * pl.C * 8, E._stream(pl.device)), "sm_expand_full")
    return out.reshape(shape)


def _pack(ws: E.Workspace, slot: int, z: torch.Tensor):
    pl = ws.plan
    z = z.to(device=pl.device, dtype=torch.complex64).contiguous()
    for b in range(pl.batch):
        off = b * pl.slice_bytes
        E._lib.check(pl.lib.sm_pack_half(pl.col_handle, z.data_ptr() + b * pl.Rin * pl.C * 8, ws.re[slot].data_ptr() + off,
                                        ws.im[slot].data_ptr() + off, E._stream(pl.device)), "sm_pack_half")


# ------------------------------------------------------------------------------------------
# reference API
# ------------------------------------------------------------------------------------------
def slerp(v0: torch.Tensor, v1: torch.Tensor, t: float) -> torch.Tensor:
    """Global-dot spherical interpolation of two vectors (shard/tensor/functions.py:24-43).
    Inside the merge this is fused into sm_slerp_reduce / sm_blend; the stand-alone form runs
    as torch element-wise ops on the tensors' CUDA device."""
    if v0.device.type != "cuda":
        raise RuntimeError("shardmerge_b200.slerp needs CUDA tensors; there is no CPU path")
    dot = torch.clamp(torch.sum(v0 * v1) / (v0.norm() * v1.norm()), -1.0, 1.0)
    theta = torch.acos(dot) * t
    rel = torch.nn.functional.normalize(v1 - v0 * dot, dim=-1)
    return v0 * torch.cos(theta) + rel * torch.sin(theta)


def fft_transform(tensor: torch.Tensor, device: str) -> torch.Tensor:
    """1-D / 2-D FFT of a real tensor -> complex64 on the CPU (functions.py:45-58).
    Complex input (only the nested imaginary path of the reference does that) is not supported."""
    dev = _dev(device)
    if tensor.is_complex():
        raise TypeError("fft_transform expects a real tensor")
    x = tensor.to(dev).to(torch.float32).contiguous()
    ws = _spectrum_of(x, dev)
    return _expand(ws, 0, tuple(tensor.shape)).to("cpu")


def ifft_transform(tensor: torch.Tensor, device: str) -> torch.Tensor:
    """Real part of the inverse 1-D / 2-D FFT -> fp32 on the CPU (functions.py:60-73)."""
    dev = _dev(device)
    R, C = _as_rows(tensor)
    ws = E.ws_for(tensor, dev)
    ws.ctl.zero_()
    _pack(ws, 0, tensor.reshape(R, C))
    out = torch.empty((R, C), dtype=torch.float32, device=dev)
    E.inv_cols(ws, ws.re[0], ws.im[0], cull=False)
    E.inv_rows(ws, ws.re[0], ws.im[0], False, 1.0, None, out, check_ifft=False)
    return out.reshape(tuple(tensor.shape)).to("cpu")


def normalize_tensor(tensor: torch.Tensor, device: str) -> tuple[torch.Tensor, float]:
    """(tensor / ||tensor||, ||tensor||); a zero tensor is returned unchanged (functions.py:75-88)."""
    dev = _dev(device)
    norm = tensor.to(device=dev).norm().item()
    return (tensor / norm if norm != 0 else tensor), norm


def retry_on_select_miss(run, where: str, safe: bool = False):
    """run(safe) -> (result, sticky status of its order statistics).  A non-zero status means a sampled select window
    missed (or overflowed): the thresholds were NaN and the result is not the merge.  Then it is run again with the
    exhaustive select (safe=True), which must not miss.  `where` names the function or tensor in the messages."""
    while True:
        result, sticky = run(safe)
        if sticky == 0:
            return result
        if safe:
            raise RuntimeError(f"order-statistic select failed in safe mode {where}")
        logger.warning(f"select window miss {where}; re-running with the exhaustive select")
        safe = True


def _blend_planes(ws: E.Workspace, mode: str, t: float, t_sum: float, cutoff_pct: float, cull_pct: float,
                  agreement: bool):
    """Blend Re(slot 0) with Re(slot 1) in place into Re(slot 0), cull applied (not deferred)."""
    pl = ws.plan
    N = pl.R * pl.C
    re0, re1 = ws.re[0], ws.re[1]
    if mode == "slerp":
        if cutoff_pct > 0:
            E.select_kth(ws, re0, re1, int((2 * N) * cutoff_pct), E.F_THR_CUT, which=0)
        else:
            ws.flt[E.F_THR_CUT] = 0.0
        E.slerp_reduce(ws, re0, re1)
        E.slerp_scalars(ws, t)
        E.blend(ws, 0, True, re0, re1, t_sum, re0)
        if cull_pct > 0:
            E.select_kth(ws, re0, None, int(N * cull_pct), E.F_THR_CULL, which=1)
            thr = ws.flt[E.F_THR_CULL]
            valid = re0[:, : pl.Ch + 1]
            valid.masked_fill_(valid.abs() < thr, 0.0)        # functions.py:146
    else:
        E.blend(ws, 1, agreement, re0, re1, t, re0)


def interpolate_fft_components(v0_fft: torch.Tensor, v1_fft: torch.Tensor, t: float, device: str, t_sum: float = 1.0,
                               cutoff_pct: float = 0.0, cull_pct: float = 0.0, interp_imag: bool = True) -> torch.Tensor:
    """Three-way masked blend of the real parts of two spectra, cutoff / cull order statistics
    (functions.py:90-162).  Returns complex64 on `device` like the reference (whose result is
    allocated with torch.zeros_like(v0_fft, device=device))."""
    dev = _dev(device)
    R, C = _as_rows(v0_fft)

    def blend(safe):
        ws = E.ws_for(v0_fft, dev, safe_select=safe)
        ws.ctl.zero_()
        _pack(ws, 0, v0_fft.reshape(R, C))
        _pack(ws, 1, v1_fft.reshape(R, C))
        _blend_planes(ws, "slerp", t, t_sum, cutoff_pct, cull_pct, True)
        ws.read_ctl()
        return ws, ws.select_sticky()

    ws = retry_on_select_miss(blend, "in interpolate_fft_components")
    full = _expand(ws, 0, tuple(v0_fft.shape))
    # imaginary part: Im X0 (exact for interp_imag=False, functions.py:160; within rounding noise of
    # the nested path otherwise, see module docstring)
    out = torch.complex(full.real.contiguous(), v0_fft.imag.to(dev).to(torch.float32).contiguous())
    return out


def merge_tensors_fft2_slerp(v0: torch.Tensor, v1: torch.Tensor, t: float, device: str, b: float = .1,
                             t_sum: float = 1.0, cutoff_pct: float = 0.0, cull_pct: float = 0.0, _result_device=None
                             ) -> tuple[torch.Tensor, float, float]:
    """Normalise, FFT, blend, inverse FFT (functions.py:164-221) -> (merged fp32 on CPU, ||v0||, ||v1||).
    `_result_device` (not in the reference): leave the result there instead of copying it to the CPU."""
    dev = _dev(device)
    _cpu = "cpu" if _result_device is None else _result_device
    R, C = _as_rows(v0)
    ws = E.ws_for(v0, dev)
    ws.ctl.zero_()
    if v0.dtype != torch.float32 or v1.dtype != torch.float32:
        # normalize_tensor works in the tensors' OWN dtype (functions.py:85-88: a bf16 norm, a bf16 quotient -- what the
        # earlier FourierMerge feeds in, shard/merge/fourier.py:120,179); only fft_transform widens to fp32 (:55).  Those
        # roundings are 2^-9 relative per element, far above FFT rounding, so they are reproduced with the same torch ops.
        d0, d1 = v0.to(dev), v1.to(dev)
        n0, n1 = d0.norm().item(), d1.norm().item()
        x0 = (d0 / n0 if n0 != 0 else d0).to(torch.float32).contiguous()
        x1 = (d1 / n1 if n1 != 0 else d1).to(torch.float32).contiguous()
        E.fwd_rows(ws, 0, E.Source(x32=x0), E.D_SUMSQ0)
        E.fwd_rows(ws, 1, E.Source(x32=x1), E.D_SUMSQ1)
        v0n, inv0, inv1 = x0, 1.0, 1.0
    else:
        x0 = v0.to(dev).contiguous()
        x1 = v1.to(dev).contiguous()
        E.fwd_rows(ws, 0, E.Source(x32=x0), E.D_SUMSQ0)
        E.fwd_rows(ws, 1, E.Source(x32=x1), E.D_SUMSQ1)
        dbl, _, _, _ = ws.read_ctl()
        n0 = E.f32(float(dbl[E.D_SUMSQ0]) ** 0.5)
        n1 = E.f32(float(dbl[E.D_SUMSQ1]) ** 0.5)
        v0n = (x0 * E.inv_norm_f32(n0)) if n0 != 0 else x0
        inv0, inv1 = E.inv_norm_f32(n0), E.inv_norm_f32(n1)
    if n1 < .0001:                                            # functions.py:184-185
        return v0n.reshape(v0.shape).to(_cpu), n0, n1
    if n0 < .0001:                                            # functions.py:187-190
        logger.info(f"Warning: Small norm v0 ({n0})")
        return v0n.reshape(v0.shape).to(_cpu), n0, n1
    ratio = n1 / (n0 + 1e-10)
    out = torch.empty((R, C), dtype=torch.float32, device=dev)
    if ratio < b:                                             # functions.py:199-202 (linear: no blend needed)
        logger.info(f"Small norm v1 ({n1})")
        E.fwd_cols(ws, 0, scale=inv0)
        E.fwd_cols(ws, 1, scale=inv1)
        ws.re[0].add_(ws.re[1], alpha=float(t)); ws.im[0].add_(ws.im[1], alpha=float(t))
        E.inv_cols(ws, ws.re[0], ws.im[0], cull=False)
        E.inv_rows(ws, ws.re[0], ws.im[0], False, 1.0, None, out, check_ifft=True)
        _, _, flags, _ = ws.read_ctl()
    else:
        def blend(safe):
            w = ws
            if safe:
                # the blend ran in place: the row spectra are gone, redo them in the exhaustive select's workspace
                w = E.ws_for(v0, dev, safe_select=True)
                w.ctl.zero_()
                E.fwd_rows(w, 0, E.Source(x32=x0), E.D_SUMSQ0)
                E.fwd_rows(w, 1, E.Source(x32=x1), E.D_SUMSQ1)
            E.spectral_pair(w, 0, 1, scale0=inv0, scale1=inv1, mode="slerp", t=t,
                            t_sum=t_sum, cutoff_pct=cutoff_pct, cull_pct=cull_pct, out_scale=1.0, out=out)
            _, _, flags, _ = w.read_ctl()
            return flags, w.select_sticky()

        flags = retry_on_select_miss(blend, "in merge_tensors_fft2_slerp")
    if int(flags[0]) > 0:
        logger.info(f"Warning: NaN in ifft output: {int(flags[0])}")
    if int(flags[1]) > 0:                                     # functions.py:215-217
        logger.info(f"Warning: Inf in ifft output: {int(flags[1])}")
        raise ValueError("Inf in ifft output")
    return out.reshape(v0.shape).to(_cpu), n0, n1


def task_arithmetic_fft2(v0: torch.Tensor, v1: torch.Tensor, t: float, device: str, agreement: bool = True,
                         _result_device=None) -> torch.Tensor:
    """Sign-agreement arithmetic in the frequency domain (functions.py:224-254) -> fp32 on CPU."""
    dev = _dev(device)
    _cpu = "cpu" if _result_device is None else _result_device
    R, C = _as_rows(v0)
    x0 = v0.to(dev).to(torch.float32).contiguous()
    x1 = v1.to(dev).to(torch.float32).contiguous()
    ws = E.ws_for(v0, dev)
    ws.ctl.zero_()
    E.fwd_rows(ws, 0, E.Source(x32=x0), E.D_SUMSQ0)
    E.fwd_rows(ws, 1, E.Source(x32=x1), E.D_SUMSQ1)
    out = torch.empty((R, C), dtype=torch.float32, device=dev)
    E.spectral_pair(ws, 0, 1, scale0=1.0, scale1=1.0, mode="arith", t=t, agreement=agreement, out_scale=1.0,
                    out=out, check_ifft=False)
    return out.reshape(v0.shape).to(_cpu)


def arithmetic_fft_components(v0_fft: torch.Tensor, v1_fft: torch.Tensor, t: float, agreement: bool, device: str,
                              do_imag: bool = True) -> torch.Tensor:
    """Real parts: sign agreement -> v0 + t*v1, else v1 (functions.py:256-302; the reference's
    "larger value" mask compares v0 with itself and is always False).  Returns complex64 on the CPU."""
    dev = _dev(device)
    R, C = _as_rows(v0_fft)
    ws = E.ws_for(v0_fft, dev)
    ws.ctl.zero_()
    _pack(ws, 0, v0_fft.reshape(R, C))
    _pack(ws, 1, v1_fft.reshape(R, C))
    _blend_planes(ws, "arith", t, 1.0, 0.0, 0.0, agreement)
    full = _expand(ws, 0, tuple(v0_fft.shape))
    out = torch.complex(full.real.contiguous(), v0_fft.imag.to(dev).to(torch.float32).contiguous())
    return out.to("cpu")


def correlate_pairs(tensors: torch.Tensor, work_device: str, store_device: str) -> torch.Tensor:
    """Symmetric matrix of mean cosine similarities (along dim 0) between stacked tensors (functions.py:304-314).
    One streaming kernel per pair on `work_device` (sm_cosine_cols); fp32 and bf16 stacks, anything else is upcast."""
    dev = _dev(work_device)
    lib = E._lib.load()
    n = tensors.shape[0]
    m = torch.zeros(n, n, device=store_device)
    items = []
    for i in range(n):
        t = tensors[i].to(dev)
        if t.dtype not in (torch.float32, torch.bfloat16):
            t = t.to(torch.float32)
        items.append(t.contiguous())
    acc = torch.zeros(1, dtype=torch.float64, device=dev)
    for i in range(n):
        a = items[i]
        R, C = (a.shape[0], a[0].numel()) if a.ndim >= 2 else (a.shape[0], 1)
        for j in range(i + 1, n):
            b = items[j] if items[j].dtype == a.dtype else items[j].to(a.dtype)
            E._lib.check(lib.sm_cosine_cols(0 if a.dtype == torch.float32 else 1, int(R), int(C), a.data_ptr(), b.data_ptr(),
                                            acc.data_ptr(), E._stream(dev)), "sm_cosine_cols")
            c = acc.item() / C
            m[i, j] = m[j, i] = c
    return m


def correlated_pairs(correlation_matrix: torch.Tensor, way: Literal['least', 'most'] = 'least'
                     ) -> Generator[tuple[int, int, float], None, None]:
    """Greedy pairing over the upper triangle by least / most |correlation|; every index is used
    once, leftovers are yielded as (i, -1, corr[i, i]) (functions.py:316-365)."""
    if way not in ("least", "most"):
        raise ValueError("Invalid way. Choose 'least' or 'most'.")
    c = correlation_matrix.detach().to("cpu", torch.float64)
    n = c.size(0)
    free = list(range(n))
    while len(free) >= 2:
        best = None
        for ii, x in enumerate(free):                         # row-major scan = first match of torch.nonzero
            for y in free[ii + 1:]:
                v = abs(c[x, y].item())
                if best is None or (v < best[0] if way == "least" else v > best[0]):
                    best = (v, x, y)
        _, x, y = best
        yield (x, y, correlation_matrix[x, y].item())
        free.remove(x); free.remove(y)
    for i in free:
        yield (i, -1, correlation_matrix[i, i].item())
