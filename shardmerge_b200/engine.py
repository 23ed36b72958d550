"""Device-resident spectral merge pipeline on top of the C ABI (include/shardmerge_b200.h).

This module owns plans, twiddle tables and workspaces (all torch-allocated: the C library
never allocates) and strings the kernels together for one pair merge:

    rows(A), rows(B)            delta + row FFT + sum of squares          (k_row_fwd)
    -- one host read of the two sums: norms decide order / branch (fast_fourier.py:209-232)
    cols(A), cols(B)            column sweeps, spectrum scaled by 1/norm  (k_col)
    select(cutoff)              exact order statistic of |Re X0|,|Re X1|  (k_count_collect ...)
    reduce + scalars            masked SLERP sums, dot/theta              (k_slerp_reduce)
    blend                       three-way masked blend of the real parts  (k_blend)
    select(cull)                exact order statistic of |Re R|
    inverse cols + rows         cull on load, iFFT, x target_norm, + base, bf16 (k_col, k_row_inv)

Tensors stay on the GPU from the bf16 inputs to the bf16 output; the reference's
TensorDiskCache round trips (shard/merge/fast_fourier.py:46-77) have no equivalent here.
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass, field
from typing import Optional

import torch

from . import _lib

# slots of the scalar block (_lib mirrors its layout from include/shardmerge_b200.h): float64 from SM_CTL_SUMSQ ...
D_SUMSQ0, D_SUMSQ1 = 0, 1
D_S00 = (_lib.SM_CTL_SUMS - _lib.SM_CTL_SUMSQ) // 8
D_S11, D_S01 = D_S00 + 1, D_S00 + 2
# ... and float32 from SM_CTL_FLT (cos, sin, relnorm follow dot: scal4 of sm_slerp_scalars)
F_THR_CUT, F_THR_CULL, F_DOT = _lib.SM_F_THR_CUT, _lib.SM_F_THR_CULL, _lib.SM_F_DOT
F_COS, F_SIN, F_RELNORM = F_DOT + 1, F_DOT + 2, F_DOT + 3


class UnsupportedShape(ValueError):
    pass


def _require_cuda(device) -> torch.device:
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError(
            f"shardmerge_b200 only runs on CUDA devices (got device={device!r}); there is no CPU path"
        )
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    return dev


def _stream(dev) -> int:
    return torch.cuda.current_stream(dev).cuda_stream


def _p(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


class Profiler:
    """Optional per-kernel-class accounting: launch counts always, CUDA-event timing and
    algorithmic bytes (SURVEY.md 8d / DESIGN.md) when `timing` is on.  bench.py uses it for the
    `roofline` and `gpu_launches` fields; it is off (None) by default."""

    def __init__(self, timing: bool = False):
        self.timing = timing
        self.launches = 0
        self.fused_calls = 0
        self.calls: dict = {}          # tag -> [n_calls, n_launches, bytes, [(start, end), ...]]
        _lib.load().sm_profile_enable(1 if timing else 0)

    def record(self, tag, launches, nbytes, dev, fn):
        ent = self.calls.setdefault(tag, [0, 0, 0, []])
        ent[0] += 1; ent[1] += launches; ent[2] += nbytes
        self.launches += launches
        if self.timing:
            st = torch.cuda.current_stream(dev)
            a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
            a.record(st); rc = fn(); b.record(st)
            ent[3].append((a, b))
            return rc
        return fn()

    def summary(self):
        out = {}
        for tag, (n, l, by, evs) in self.calls.items():
            ms = sum(a.elapsed_time(b) for a, b in evs) if evs else None
            out[tag] = dict(calls=n, launches=l, bytes=by, ms=ms)
        # classes timed inside the fused C chain (sm_profile_collect)
        lib = _lib.load()
        n = len(_lib.CLS_NAMES)
        ms = (ctypes.c_double * n)(); by = (ctypes.c_double * n)(); la = (ctypes.c_int * n)()
        lib.sm_profile_collect(ms, by, la, n)
        for i, name in enumerate(_lib.CLS_NAMES):
            if la[i] == 0:
                continue
            ent = out.setdefault(name, dict(calls=0, launches=0, bytes=0, ms=0.0))
            ent["calls"] += self.fused_calls
            ent["launches"] += int(la[i]); ent["bytes"] += float(by[i])
            ent["ms"] = (ent["ms"] or 0.0) + float(ms[i])
        return out


PROFILER: Optional[Profiler] = None


def _run(tag, launches, nbytes, dev, fn):
    if PROFILER is None:
        return fn()
    return PROFILER.record(tag, launches, nbytes, dev, fn)


class Plan:
    """FFT plan + twiddle tables for tensors of shape [R][C] on one device, or for a stack of `batch` such matrices
    (a tensor with leading dimensions: the reference's fftn(dim=(-2, -1)) transforms every [R][C] slice on its own while
    norms, order statistics and SLERP sums run over the WHOLE tensor, shard/tensor/functions.py:58,85,113-141).  A stack
    is laid out as one [batch * R][C] matrix: row passes and statistics use a plan over all its rows, the column sweeps a
    plan over R rows applied to every slice in turn."""

    def __init__(self, R: int, C: int, device, batch: int = 1):
        self.lib = _lib.load()
        self.device = _require_cuda(device)
        self.Rin, self.batch = R, batch
        self.R, self.C, self.Ch = R * batch, C, C // 2
        self.handle = self.lib.sm_plan_create(self.R, C)
        if not self.handle:
            raise UnsupportedShape(self.lib.sm_last_error().decode())
        self.P = self.lib.sm_plan_pitch(self.handle)
        with torch.cuda.device(self.device):
            self.tables = torch.empty(self.lib.sm_plan_table_bytes(self.handle), dtype=torch.uint8, device=self.device)
            _lib.check(self.lib.sm_plan_init_tables(self.handle, self.tables.data_ptr(), _stream(self.device)), "init_tables")
            self.col_handle, self.col_tables = self.handle, self.tables
            if batch > 1:
                self.col_handle = self.lib.sm_plan_create(R, C)
                if not self.col_handle:
                    raise UnsupportedShape(self.lib.sm_last_error().decode())
                self.col_tables = torch.empty(self.lib.sm_plan_table_bytes(self.col_handle), dtype=torch.uint8, device=self.device)
                _lib.check(self.lib.sm_plan_init_tables(self.col_handle, self.col_tables.data_ptr(), _stream(self.device)),
                           "init_tables")
        self.col_passes = self.lib.sm_plan_col_passes(self.col_handle)
        self.slice_bytes = R * self.P * 4                          # one [R][P] fp32 plane slice

    def describe(self) -> str:
        buf = ctypes.create_string_buffer(1024)
        self.lib.sm_plan_describe(self.col_handle, buf, 1024)
        return buf.value.decode() + (f" x {self.batch} slices" if self.batch > 1 else "")

    def row_freq(self) -> torch.Tensor:
        """stored row -> frequency index within its slice (CPU int64 tensor, one slice)."""
        return torch.tensor([self.lib.sm_plan_row_freq(self.col_handle, i) for i in range(self.Rin)], dtype=torch.int64)

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                if getattr(self, "col_handle", None) and self.col_handle != self.handle:
                    self.lib.sm_plan_destroy(self.col_handle)
                self.lib.sm_plan_destroy(self.handle)
                self.handle = self.col_handle = None
        except Exception:
            pass


class Workspace:
    """Spectrum planes, scalar block and select scratch for one plan (re-used across tensors)."""

    def __init__(self, plan: Plan, n_spectra: int = 2, safe_select: bool = False):
        self.plan = plan
        dev = plan.device
        self.n_spectra = n_spectra
        # zero-filled: no kernel writes the padding columns (Ch+1 .. P-1) with anything but blend(0, 0) = 0, and the
        # fused statistics pass relies on them being zero
        self.re = [torch.zeros((plan.R, plan.P), dtype=torch.float32, device=dev) for _ in range(n_spectra)]
        self.im = [torch.zeros((plan.R, plan.P), dtype=torch.float32, device=dev) for _ in range(n_spectra)]
        self.re_out = torch.zeros((plan.R, plan.P), dtype=torch.float32, device=dev)   # blend output of the fused chain
        self.ctl = torch.zeros(_lib.SM_CTL_BYTES, dtype=torch.uint8, device=dev)
        self.dbl, self.flt, self.flags, _, _, self.sel = ctl_views(self.ctl)
        self.safe_select = safe_select
        mode = 1 if safe_select else 0
        # select scratch in front, the fused statistics' persistent histograms behind it (sm_fstats_* uses the LAST
        # sm_fstats_ws_bytes of the buffer and wants them zero-filled once)
        nbytes = max(plan.lib.sm_select_ws_bytes(plan.handle, 2, mode), plan.lib.sm_select_ws_bytes(plan.handle, 1, mode))
        nbytes = (nbytes + 255) // 256 * 256 + plan.lib.sm_fstats_ws_bytes(plan.handle)
        self.sel_ws = torch.zeros(nbytes, dtype=torch.uint8, device=dev)
        # pinned landing zone for the scalar block
        self.ctl_host = torch.empty(_lib.SM_CTL_BYTES, dtype=torch.uint8).pin_memory()

    # typed pointers into the scalar block
    def dptr(self, slot): return self.dbl.data_ptr() + 8 * slot
    def fptr(self, slot): return self.flt.data_ptr() + 4 * slot
    def selptr(self, which): return self.sel.data_ptr() + _lib.SM_SELECT_STATE_BYTES * which
    def fsptr(self, which): return self.ctl.data_ptr() + _lib.SM_CTL_FS + _lib.SM_FS_STATE_BYTES * which

    def fs_status(self):
        """(sticky word of the fused cutoff state, sticky word of the fused blend/cull state) -- synchronous."""
        h = self.ctl.cpu()
        return tuple(_word(h, o) for o in _FS_STICKY)

    def select_sticky(self) -> int:
        """Sticky status of every order statistic since `ctl` was zeroed, as of the last read_ctl(): non-zero when a sampled
        window missed, was too wide or overflowed, i.e. a threshold came out NaN and the tensor has to be redone with
        safe_select."""
        return select_sticky_of(self.ctl_host)

    def read_ctl(self):
        """Synchronous read-back of the scalar block -> (float64[8], float32[16], int32[4], sel bytes)."""
        self.ctl_host.copy_(self.ctl, non_blocking=True)
        torch.cuda.current_stream(self.plan.device).synchronize()
        dbl, flt, flags, _, _, sel = ctl_views(self.ctl_host)
        return dbl, flt, flags, sel


def ctl_views(h: torch.Tensor):
    """Views of a scalar block `h` (uint8, on the device or a host copy) as include/shardmerge_b200.h lays it out:
    (float64 from SM_CTL_SUMSQ: the sums of squares of x and y, then the SLERP sums (D_*); float32 slots SM_F_*; the u32
    nan / inf counters as int32; int32 slots SM_I_*; float64 target_norm; the bytes of the two select states)."""
    L = _lib
    return (h[L.SM_CTL_SUMSQ:L.SM_CTL_FLT].view(torch.float64), h[L.SM_CTL_FLT:L.SM_CTL_FLAGS].view(torch.float32),
            h[L.SM_CTL_FLAGS:L.SM_CTL_INT].view(torch.int32), h[L.SM_CTL_INT:L.SM_CTL_TN].view(torch.int32),
            h[L.SM_CTL_TN:L.SM_CTL_TN + 8].view(torch.float64), h[L.SM_CTL_SEL:L.SM_CTL_SEL + 2 * L.SM_SELECT_STATE_BYTES])


# byte offsets of the sticky words of the two select states and of the two fused statistics states
_SEL_STICKY = [_lib.SM_CTL_SEL + k * _lib.SM_SELECT_STATE_BYTES + _lib.SM_SELECT_STICKY_OFF for k in (0, 1)]
_FS_STICKY = [_lib.SM_CTL_FS + k * _lib.SM_FS_STATE_BYTES + _lib.SM_FS_STICKY_OFF for k in (0, 1)]


def _word(h: torch.Tensor, off: int) -> int:
    return int(h[off:off + 4].view(torch.int32)[0])


def select_sticky_of(h: torch.Tensor) -> int:
    """OR of the sticky words of the two select states and of the two fused statistics states in a host copy `h`
    (uint8) of a scalar block."""
    sticky = 0
    for off in _SEL_STICKY + _FS_STICKY:
        sticky |= _word(h, off)
    return sticky


_plans: dict = {}
_workspaces: dict = {}


def get_plan(R: int, C: int, device, batch: int = 1) -> Plan:
    dev = _require_cuda(device)
    key = (dev.index, R, C, batch)
    pl = _plans.get(key)
    if pl is None:
        pl = _plans[key] = Plan(R, C, dev, batch)
    return pl


def get_workspace(R: int, C: int, device, n_spectra: int = 2, safe_select: bool = False, lane=0, batch: int = 1) -> Workspace:
    """Workspaces are cached per (device, shape, select mode, lane); a lane is one of the streams FourierMerge
    spreads consecutive tensors over, and two tensors in flight must not share planes.  `batch` > 1: a stack of
    [R][C] matrices (see Plan)."""
    dev = _require_cuda(device)
    key = (dev.index, R, C, batch, safe_select, lane)
    ws = _workspaces.get(key)
    if ws is None or ws.n_spectra < n_spectra:
        if ws is not None:
            # the planes being replaced may still be read by kernels enqueued on another stream
            torch.cuda.synchronize(dev)
        ws = _workspaces[key] = Workspace(get_plan(R, C, dev, batch), n_spectra, safe_select)
    return ws


def ws_for(t: torch.Tensor, device, **kw) -> Workspace:
    """Workspace for a tensor's shape: 1-D -> one row, 2-D -> [R][C], more dimensions -> a stack of [R][C] slices."""
    R, C, B = shape_rcb(t)
    return get_workspace(R, C, device, batch=B, **kw)


def clear_caches():
    _workspaces.clear()
    _plans.clear()


def shape_rcb(t: torch.Tensor):
    """-> (rows, columns, slices) of the matrices the reference's fft / fftn(dim=(-2, -1)) transforms (functions.py:55-58)."""
    if t.ndim == 0:
        raise UnsupportedShape("a 0-d tensor has nothing to transform")
    if t.ndim == 1:
        return 1, t.shape[0], 1
    b = 1
    for d in t.shape[:-2]:
        b *= d
    return t.shape[-2], t.shape[-1], b


def shape_rc(t: torch.Tensor):
    """rows x columns of the tensor seen as ONE matrix (a stack of slices counts all its rows)."""
    R, C, B = shape_rcb(t)
    return R * B, C


# ------------------------------------------------------------------------------------------
# sources: what a row pass can read
# ------------------------------------------------------------------------------------------
@dataclass
class Source:
    """Either a (base, finetune) pair of bf16 tensors (delta is formed in the kernel) or an
    fp32 tensor that already is a delta / intermediate merge result."""
    base: Optional[torch.Tensor] = None
    ft: Optional[torch.Tensor] = None
    x32: Optional[torch.Tensor] = None
    weight: float = 1.0
    name: str = ""
    norm: float = float("nan")     # filled after the row pass

    @property
    def is_bf16(self) -> bool:
        return self.x32 is None

    def delta_f32(self) -> torch.Tensor:
        """fp32 delta as a torch tensor (only used by the rare FFT-free fallbacks)."""
        if self.x32 is not None:
            return self.x32
        return self.ft.to(torch.float32) - self.base.to(torch.float32)


def make_source(base: Optional[torch.Tensor], ft: Optional[torch.Tensor], x32: Optional[torch.Tensor] = None,
                weight: float = 1.0, name: str = "") -> Source:
    if x32 is not None:
        return Source(x32=x32.contiguous().to(torch.float32), weight=weight, name=name)
    if base.dtype == torch.bfloat16 and ft.dtype == torch.bfloat16:
        return Source(base=base.contiguous(), ft=ft.contiguous(), weight=weight, name=name)
    # other storage dtypes: form the fp32 delta with torch (exact upcast + one rounding, base.py:128-132)
    return Source(x32=(ft.to(torch.float32) - base.to(torch.float32)).contiguous(), weight=weight, name=name)


# ------------------------------------------------------------------------------------------
# kernel wrappers
# ------------------------------------------------------------------------------------------
def fwd_rows(ws: Workspace, slot: int, src: Source, sumsq_slot: int, m1: float = 1.0, m2: float = 1.0):
    fwd_rows_ptr(ws, slot, src, ws.dptr(sumsq_slot), m1, m2)


def fwd_rows_ptr(ws: Workspace, slot: int, src: Source, sumsq_ptr: int, m1: float = 1.0, m2: float = 1.0):
    pl, lib = ws.plan, ws.plan.lib
    st = _stream(pl.device)
    N = pl.R * pl.C
    if src.is_bf16:
        rc = _run("row_fwd", 1, 8 * N, pl.device, lambda: lib.sm_fwd_rows_bf16(
            pl.handle, pl.tables.data_ptr(), src.base.data_ptr(), src.ft.data_ptr(),
            ws.re[slot].data_ptr(), ws.im[slot].data_ptr(), sumsq_ptr, st))
    else:
        rc = _run("row_fwd_f32", 1, 8 * N, pl.device, lambda: lib.sm_fwd_rows_f32(
            pl.handle, pl.tables.data_ptr(), src.x32.data_ptr(), m1, m2,
            ws.re[slot].data_ptr(), ws.im[slot].data_ptr(), sumsq_ptr, st))
    _lib.check(rc, "sm_fwd_rows")


def fwd_cols(ws: Workspace, slot: int, scale: float = 1.0, scale_slot: Optional[int] = None, write_im: bool = True):
    pl, lib = ws.plan, ws.plan.lib
    N = pl.R * pl.C
    sweeps = max(1, pl.col_passes)
    nbytes = 8 * N * sweeps - (0 if write_im else 2 * N)
    sptr = None if scale_slot is None else ws.fptr(scale_slot)

    def run():
        for b in range(pl.batch):
            off = b * pl.slice_bytes
            rc = lib.sm_fwd_cols(pl.col_handle, pl.col_tables.data_ptr(), ws.re[slot].data_ptr() + off,
                                 ws.im[slot].data_ptr() + off, sptr, float(scale), 1 if write_im else 0, _stream(pl.device))
            if rc:
                return rc
        return 0

    _lib.check(_run("col_fwd", pl.batch * lib.sm_plan_col_launches(pl.col_handle), nbytes, pl.device, run), "sm_fwd_cols")


def select_kth(ws: Workspace, plane0: torch.Tensor, plane1: Optional[torch.Tensor], rank: int, out_slot: int,
               which: int = 0):
    pl, lib = ws.plan, ws.plan.lib
    N = pl.R * pl.C
    rc = _run("select2" if plane1 is not None else "select1", 16, (4 if plane1 is not None else 2) * N, pl.device,
              lambda: lib.sm_select_kth_abs(pl.handle, plane0.data_ptr(), _p(plane1), int(rank), 1 if ws.safe_select else 0,
                                            ws.selptr(which), ws.sel_ws.data_ptr(), ws.sel_ws.numel(), ws.fptr(out_slot),
                                            _stream(pl.device)))
    _lib.check(rc, "sm_select_kth_abs")


def slerp_reduce(ws: Workspace, re0: torch.Tensor, re1: torch.Tensor):
    pl, lib = ws.plan, ws.plan.lib
    _lib.check(_run("reduce", 1, 4 * pl.R * pl.C, pl.device, lambda: lib.sm_slerp_reduce(
        pl.handle, re0.data_ptr(), re1.data_ptr(), ws.fptr(F_THR_CUT), ws.dptr(D_S00), _stream(pl.device))), "sm_slerp_reduce")


def slerp_scalars(ws: Workspace, t: float):
    pl, lib = ws.plan, ws.plan.lib
    _lib.check(_run("scalars", 1, 0, pl.device, lambda: lib.sm_slerp_scalars(
        ws.dptr(D_S00), float(t), ws.fptr(F_DOT), _stream(pl.device))), "sm_slerp_scalars")


def blend(ws: Workspace, mode: int, agreement: bool, re0: torch.Tensor, re1: torch.Tensor, t_sum: float,
          out: torch.Tensor):
    pl, lib = ws.plan, ws.plan.lib
    _lib.check(_run("blend", 1, 6 * pl.R * pl.C, pl.device, lambda: lib.sm_blend(
        pl.handle, mode, 1 if agreement else 0, re0.data_ptr(), re1.data_ptr(), ws.fptr(F_THR_CUT),
        ws.fptr(F_DOT), float(t_sum), out.data_ptr(), _stream(pl.device))), "sm_blend")


def fstats_cutoff(ws: Workspace, reX: torch.Tensor, reY: torch.Tensor, rank: int, t: float, sel_ptr: Optional[int] = None):
    """Fused cutoff statistic + SLERP sums + scalars (csrc/kernels_fstats.cu): writes F_THR_CUT, F_DOT.., D_S00.."""
    pl, lib = ws.plan, ws.plan.lib
    _lib.check(_run("stats_cutoff", 3, 4 * pl.R * pl.C, pl.device, lambda: lib.sm_fstats_cutoff(
        pl.handle, reX.data_ptr(), reY.data_ptr(), sel_ptr, int(rank), float(t),
        ws.fsptr(0), ws.sel_ws.data_ptr(), ws.sel_ws.numel(), ws.fptr(F_THR_CUT), ws.fptr(F_DOT), ws.dptr(D_S00),
        _stream(pl.device))), "sm_fstats_cutoff")


def fstats_blend_cull(ws: Workspace, reX: torch.Tensor, reY: torch.Tensor, t_sum: float, out: torch.Tensor, rank: int,
                      sel_ptr: Optional[int] = None):
    """Fused SLERP blend + cull statistic of its output: writes `out` and F_THR_CULL."""
    pl, lib = ws.plan, ws.plan.lib
    _lib.check(_run("blend_cull", 3, 6 * pl.R * pl.C, pl.device, lambda: lib.sm_fstats_blend_cull(
        pl.handle, reX.data_ptr(), reY.data_ptr(), sel_ptr, ws.fptr(F_THR_CUT), ws.fptr(F_DOT), float(t_sum),
        out.data_ptr(), int(rank), ws.fsptr(1), ws.sel_ws.data_ptr(), ws.sel_ws.numel(),
        ws.fptr(F_THR_CULL), _stream(pl.device))), "sm_fstats_blend_cull")


def inv_cols(ws: Workspace, re: torch.Tensor, im: torch.Tensor, cull: bool):
    pl, lib = ws.plan, ws.plan.lib
    sweeps = pl.col_passes
    if sweeps == 0:
        return
    cptr = ws.fptr(F_THR_CULL) if cull else None

    def run():
        for b in range(pl.batch):
            off = b * pl.slice_bytes
            rc = lib.sm_inv_cols(pl.col_handle, pl.col_tables.data_ptr(), re.data_ptr() + off, im.data_ptr() + off, cptr,
                                 _stream(pl.device))
            if rc:
                return rc
        return 0

    _lib.check(_run("col_inv", pl.batch * lib.sm_plan_col_launches(pl.col_handle), 8 * pl.R * pl.C * sweeps, pl.device, run),
               "sm_inv_cols")


def inv_rows(ws: Workspace, re: torch.Tensor, im: torch.Tensor, cull: bool, scale: float,
             base: Optional[torch.Tensor], out: torch.Tensor, check_ifft: bool = True):
    pl, lib = ws.plan, ws.plan.lib
    st = _stream(pl.device)
    cptr = ws.fptr(F_THR_CULL) if cull else None
    N = pl.R * pl.C
    scale = float(scale) * pl.batch          # the kernel's 1 / (rows * C) counts all rows of a stack; one slice has rows / batch
    if out.dtype == torch.bfloat16:
        rc = _run("row_inv", 1, 8 * N, pl.device, lambda: lib.sm_inv_rows_bf16(
            pl.handle, pl.tables.data_ptr(), re.data_ptr(), im.data_ptr(), cptr, base.data_ptr(),
            out.data_ptr(), None, float(scale), 1 if check_ifft else 0, ws.flags.data_ptr(), st))
    else:
        rc = _run("row_inv_f32", 1, 8 * N, pl.device, lambda: lib.sm_inv_rows_f32(
            pl.handle, pl.tables.data_ptr(), re.data_ptr(), im.data_ptr(), cptr, out.data_ptr(),
            None, float(scale), 1 if check_ifft else 0, ws.flags.data_ptr(), st))
    _lib.check(rc, "sm_inv_rows")


def delta_axpby_bf16(base_out, s0: Source, ca: float, s1: Optional[Source], cb: float, scale: float,
                     out: torch.Tensor, flags: torch.Tensor):
    lib = _lib.load()
    dev = out.device
    rc = _run("axpby", 1, out.numel() * (8 if s1 is None else 12), dev, lambda: lib.sm_delta_axpby_bf16(
        out.numel(), base_out.data_ptr(), s0.base.data_ptr(), s0.ft.data_ptr(), float(ca),
        None if s1 is None else s1.base.data_ptr(), None if s1 is None else s1.ft.data_ptr(),
        float(cb), float(scale), out.data_ptr(), flags.data_ptr(), _stream(dev)))
    _lib.check(rc, "sm_delta_axpby_bf16")


# ------------------------------------------------------------------------------------------
# pair merge
# ------------------------------------------------------------------------------------------
def f32(x: float) -> float:
    """round a Python float to fp32 (what torch does when a Python scalar meets an fp32 tensor)."""
    return torch.tensor(x, dtype=torch.float32).item()


def inv_norm_f32(norm: float) -> float:
    """`tensor / norm` with a Python scalar on CUDA is tensor * (1/norm) evaluated in fp32."""
    nf = f32(norm)
    return f32(1.0 / nf) if nf != 0.0 else 1.0


@dataclass
class PairResult:
    out: torch.Tensor
    flags: Optional[torch.Tensor] = None     # int32[4] device counters (nan_ifft, inf_ifft, nan_final, inf_final)
    branch: str = ""
    scalars: dict = field(default_factory=dict)


def spectral_pair(ws: Workspace, slot0: int, slot1: int, *, scale0: float, scale1: float, mode: str, t: float,
                  t_sum: float = 1.0, cutoff_pct: float = 0.0, cull_pct: float = 0.0, agreement: bool = True,
                  out_scale: float = 1.0, base: Optional[torch.Tensor] = None, out: torch.Tensor = None,
                  check_ifft: bool = True):
    """Everything after the row passes for one pair whose row spectra sit in slot0 (role v0) and
    slot1 (role v1): column sweeps, statistics, blend, inverse, epilogue into `out`."""
    pl = ws.plan
    N = pl.R * pl.C
    fwd_cols(ws, slot0, scale=scale0, write_im=True)
    fwd_cols(ws, slot1, scale=scale1, write_im=False)
    re0, im0, re1 = ws.re[slot0], ws.im[slot0], ws.re[slot1]
    fused_stats = (mode == "slerp" and not ws.safe_select and cutoff_pct > 0 and cull_pct > 0
                   and pl.lib.sm_fstats_supported(pl.handle))
    if fused_stats:
        # one pass for the cutoff statistic + SLERP sums + scalars, one for the blend + cull statistic
        # (csrc/kernels_fstats.cu); a missed window shows up in ws.fs_status() and the caller redoes the tensor
        fstats_cutoff(ws, re0, re1, int((2 * N) * cutoff_pct), t)
        fstats_blend_cull(ws, re0, re1, t_sum, re0, int(N * cull_pct))
        cull = True
    elif mode == "slerp":
        if cutoff_pct > 0:
            # functions.py:113-120: sorted(cat(|re0|,|re1|))[int(2N*cutoff_pct)]
            select_kth(ws, re0, re1, int((2 * N) * cutoff_pct), F_THR_CUT, which=0)
        else:
            ws.flt[F_THR_CUT] = 0.0
        slerp_reduce(ws, re0, re1)
        slerp_scalars(ws, t)
        blend(ws, 0, True, re0, re1, t_sum, re0)
        cull = cull_pct > 0
        if cull:
            # functions.py:138-141: sorted(|R.real|)[int(N*cull_pct)]
            select_kth(ws, re0, None, int(N * cull_pct), F_THR_CULL, which=1)
    elif mode == "arith":
        blend(ws, 1, agreement, re0, re1, t, re0)
        cull = False
    else:
        raise ValueError(mode)
    inv_cols(ws, re0, im0, cull)
    inv_rows(ws, re0, im0, cull, out_scale, base, out, check_ifft=check_ifft)


# ------------------------------------------------------------------------------------------
# fused, host-sync-free pair merge (csrc/pipeline.cu)
# ------------------------------------------------------------------------------------------
class _PinnedPool:
    """Pinned landing slots for scalar blocks whose check is deferred.  A slot is handed out by take() and comes
    back through give() when its PendingPair has been resolved (or dropped); the pool grows by a chunk when every
    slot is out, so any number of tensors can be in flight before resolve_all()."""

    CHUNK = 256

    def __init__(self):
        self.chunks: list = []
        self.free: list = []

    def take(self) -> torch.Tensor:
        if not self.free:
            buf = torch.empty((self.CHUNK, _lib.SM_CTL_BYTES), dtype=torch.uint8).pin_memory()
            self.chunks.append(buf)
            self.free.extend(buf[i] for i in range(self.CHUNK))
        return self.free.pop()

    def give(self, slot: torch.Tensor):
        self.free.append(slot)


_ring: Optional[_PinnedPool] = None


def take_pinned_slot() -> torch.Tensor:
    """A 1 KiB pinned host block (uint8) from the scalar-block pool; hand it back with give_pinned_slot()."""
    global _ring
    if _ring is None:
        _ring = _PinnedPool()
    return _ring.take()


def give_pinned_slot(slot: torch.Tensor):
    if _ring is not None:
        _ring.give(slot)


class PendingPair:
    """Result of pair_merge_async: the output tensor is already enqueued; `resolve()` waits for the
    scalar block, and reports what the device decided."""

    def __init__(self, out, host_ctl, event, layer_name=""):
        self.out, self.host_ctl, self.event, self.layer_name = out, host_ctl, event, layer_name
        self.redo = None
        self.info: dict = {}

    def __del__(self):
        # a handle dropped without resolve(): the copy may still be in flight, wait before the slot is reused
        if self.host_ctl is not None and _ring is not None:
            try:
                self.event.synchronize()
                _ring.give(self.host_ctl)
            except Exception:
                pass
            self.host_ctl = None

    def resolve(self) -> dict:
        if self.host_ctl is None:
            return self.info
        self.event.synchronize()
        h = self.host_ctl
        _, flt, flags, ints, tn, _ = ctl_views(h)
        self.info = dict(norms=[float(flt[_lib.SM_F_NORM_X]), float(flt[_lib.SM_F_NORM_Y])], target_norm=float(tn[0]),
                         swap=int(ints[_lib.SM_I_SWAP]), branch=_lib.BRANCH_NAMES.get(int(ints[_lib.SM_I_BRANCH]), "?"),
                         select_sticky=select_sticky_of(h), flags=[int(v) for v in flags],
                         thr_cut=float(flt[F_THR_CUT]), thr_cull=float(flt[F_THR_CULL]), dot=float(flt[F_DOT]))
        _ring.give(h)
        self.host_ctl = None
        return self.info


def pair_merge_async(ws: Workspace, s0: Source, s1: Source, base_out: Optional[torch.Tensor], out: torch.Tensor, *, t: float,
                     t_sum: float = 1.0, cutoff_pct: float = 0.08, cull_pct: float = 0.20,
                     target_norm_offset: float = 1e-10, layer_name: str = "", slots=(0, 1), rows_done: bool = False,
                     sumsq=None, target_norm: float = 0.0) -> PendingPair:
    """Enqueue one pair merge as a single stream-ordered chain (csrc/pipeline.cu).  `out` is bf16 (base_out is added,
    the end of _merge_layer) or fp32 (merged * target_norm: an intermediate of the pair tree, base_out unused).  A source
    is a bf16 (base, finetune) pair or an fp32 tensor; with rows_done the row spectra already sit in `slots` and `sumsq`
    carries their sums of squares.  target_norm > 0 overrides the mean of the two norms (tree: mean over all models)."""
    global _ring
    pl, lib = ws.plan, ws.plan.lib
    dev = pl.device
    a = _lib.PairArgs()
    if s0.is_bf16:
        a.base0, a.ft0 = s0.base.data_ptr(), s0.ft.data_ptr()
    else:
        a.x32_0 = s0.x32.data_ptr()
    if s1.is_bf16:
        a.base1, a.ft1 = s1.base.data_ptr(), s1.ft.data_ptr()
    else:
        a.x32_1 = s1.x32.data_ptr()
    if out.dtype == torch.bfloat16:
        a.base_out, a.out_bf16 = base_out.data_ptr(), out.data_ptr()
    else:
        a.out_f32 = out.data_ptr()
    a.rows_done = 1 if rows_done else 0
    if rows_done:
        a.sumsq[0], a.sumsq[1] = float(sumsq[0]), float(sumsq[1])
    a.target_norm = float(target_norm)
    a.re[0], a.re[1], a.re[2] = ws.re[slots[0]].data_ptr(), ws.re[slots[1]].data_ptr(), ws.re_out.data_ptr()
    a.im[0], a.im[1] = ws.im[slots[0]].data_ptr(), ws.im[slots[1]].data_ptr()
    a.ctl = ws.ctl.data_ptr()
    a.sel_ws, a.sel_ws_bytes = ws.sel_ws.data_ptr(), ws.sel_ws.numel()
    a.t, a.t_sum, a.cutoff_pct, a.cull_pct = float(t), float(t_sum), float(cutoff_pct), float(cull_pct)
    a.target_norm_offset = float(target_norm_offset)
    a.select_mode = 1 if ws.safe_select else 0
    sweeps = lib.sm_plan_col_passes(pl.handle)
    if PROFILER is not None:
        fs = lib.sm_fstats_supported(pl.handle) and not ws.safe_select
        cl = lib.sm_plan_col_launches(pl.handle)          # launches of one column transform (column bands x sweeps)
        # two finetunes of one base: one paired row pass that also makes the scalar decisions (csrc/pipeline.cu)
        paired = (not rows_done and s0.is_bf16 and s1.is_bf16 and s0.base.data_ptr() == s1.base.data_ptr()
                  and lib.sm_fwd_rows_pair_supported(pl.handle))
        PROFILER.launches += (1 if paired else (0 if rows_done else 2) + 1) + 2 * cl + ((2 + 2) if fs else (11 + 2 + 1 + 11)) + (cl if sweeps else 0) + 1
        PROFILER.fused_calls += 1
    _lib.check(lib.sm_pair_merge_async(pl.handle, pl.tables.data_ptr(), ctypes.byref(a), _stream(dev)), "sm_pair_merge_async")
    if _ring is None:
        _ring = _PinnedPool()
    host = _ring.take()
    host.copy_(ws.ctl, non_blocking=True)
    ev = torch.cuda.Event()
    ev.record(torch.cuda.current_stream(dev))
    return PendingPair(out, host, ev, layer_name)
