"""ctypes binding of libshardmerge_b200.so (C ABI declared in include/shardmerge_b200.h).

There is no CPU fallback: if the shared library is missing or a call fails, the caller
gets an exception.  Build the library with `make` (or `__graft_entry__.build()`).
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_LIB_PATH = Path(__file__).resolve().parent / "libshardmerge_b200.so"
_lib = None

# name -> (restype, [argtypes]); mirrors include/shardmerge_b200.h one to one
_vp, _f, _d, _i, _sz, _u64 = C.c_void_p, C.c_float, C.c_double, C.c_int, C.c_size_t, C.c_uint64
SIGNATURES = {
    "sm_version": (_i, []),
    "sm_last_error": (C.c_char_p, []),
    "sm_plan_create": (_vp, [_i, _i]),
    "sm_plan_destroy": (None, [_vp]),
    "sm_plan_pitch": (_i, [_vp]),
    "sm_plan_row_freq": (_i, [_vp, _i]),
    "sm_plan_col_passes": (_i, [_vp]),
    "sm_plan_col_launches": (_i, [_vp]),
    "sm_plan_describe": (_i, [_vp, C.c_char_p, _i]),
    "sm_plan_table_bytes": (_sz, [_vp]),
    "sm_plan_init_tables": (_i, [_vp, _vp, _vp]),
    "sm_fwd_rows_bf16": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sm_fwd_rows_f32": (_i, [_vp, _vp, _vp, _f, _f, _vp, _vp, _vp, _vp]),
    "sm_fwd_cols": (_i, [_vp, _vp, _vp, _vp, _vp, _f, _i, _vp]),
    "sm_inv_norm": (_i, [_vp, _vp, _vp]),
    "sm_select_ws_bytes": (_sz, [_vp, _i, _i]),
    "sm_select_kth_abs": (_i, [_vp, _vp, _vp, _u64, _i, _vp, _vp, _sz, _vp, _vp]),
    "sm_slerp_reduce": (_i, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "sm_slerp_scalars": (_i, [_vp, _d, _vp, _vp]),
    "sm_blend": (_i, [_vp, _i, _i, _vp, _vp, _vp, _vp, _f, _vp, _vp]),
    "sm_fstats_supported": (_i, [_vp]),
    "sm_fstats_ws_bytes": (_sz, [_vp]),
    "sm_fstats_cutoff": (_i, [_vp, _vp, _vp, _vp, _u64, _d, _vp, _vp, _sz, _vp, _vp, _vp, _vp]),
    "sm_fstats_blend_cull": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _f, _vp, _u64, _vp, _vp, _sz, _vp, _vp]),
    "sm_inv_cols": (_i, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "sm_inv_rows_bf16": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _f, _i, _vp, _vp]),
    "sm_inv_rows_f32": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _f, _i, _vp, _vp]),
    "sm_delta_axpby_bf16": (_i, [_sz, _vp, _vp, _vp, _f, _vp, _vp, _f, _f, _vp, _vp, _vp]),
    "sm_elem_merge": (_i, [_i, _i, _sz, _vp, _vp, _i, _vp, _vp]),
    "sm_elem_merge_bf16": (_i, [_i, _sz, _vp, _vp, _i, _vp, _vp]),
    "sm_cosine_cols": (_i, [_i, _i, _i, _vp, _vp, _vp, _vp]),
    "sm_lora_materialize": (_i, [_i, _i, _i, _i, _vp, _i, _vp, _vp, _f, _vp, _vp]),
    "sm_lowrank_ws_bytes": (_sz, [_i, _i, _i]),
    "sm_lowrank_right": (_i, [_i, _i, _i, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "sm_lowrank_left": (_i, [_i, _i, _i, _i, _vp, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "sm_copy_bytes": (_i, [_vp, _vp, _sz, _vp]),
    "sm_expand_full": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "sm_pack_half": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "sm_pair_merge_slerp_async": (_i, [_vp, _vp, _vp, _vp]),
    "sm_pair_merge_tree_async": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "sm_profile_enable": (_i, [_i]),
    "sm_profile_collect": (_i, [_vp, _vp, _vp, _i]),
}


class PairArgs(C.Structure):
    """sm_pair_args of include/shardmerge_b200.h"""
    _fields_ = [("base0", _vp), ("ft0", _vp), ("base1", _vp), ("ft1", _vp), ("base_out", _vp), ("out_bf16", _vp),
                ("re", _vp * 3), ("im", _vp * 2), ("ctl", _vp), ("sel_ws", _vp), ("sel_ws_bytes", _sz),
                ("t", _d), ("t_sum", _f), ("cutoff_pct", _d), ("cull_pct", _d), ("target_norm_offset", _d),
                ("select_mode", _i)]


class PairExt(C.Structure):
    """sm_pair_ext of include/shardmerge_b200.h"""
    _fields_ = [("x32_0", _vp), ("x32_1", _vp), ("rows_done", _i), ("sumsq", _d * 2), ("target_norm", _d), ("out_f32", _vp)]


CLS_NAMES = ["row_fwd", "col_fwd", "stats_cutoff", "reduce", "scalars", "blend_cull", "select1", "col_inv", "row_inv"]
BRANCH_NAMES = {0: "slerp", 1: "add", 2: "arith", 3: "slerp-early", 4: "slerp-linear"}
SELECT_STATE_BYTES = 64
FS_STATE_BYTES, FS_STATUS_OFF, FS_STICKY_OFF, CTL_FS_OFF, CTL_BYTES = 128, 28, 72, 512, 1024


class ShardMergeLibraryError(RuntimeError):
    pass


def lib_path() -> Path:
    return Path(os.environ.get("SHARDMERGE_B200_LIB", str(_LIB_PATH)))


def load():
    """Load the shared library (once) and set every prototype."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not path.exists():
        raise ShardMergeLibraryError(
            f"{path} not found: the sm_100a extension is not built (run `make` in the repo root). "
            "shardmerge_b200 has no CPU fallback."
        )
    lib = C.CDLL(str(path))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here = header/library mismatch
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc != 0:
        msg = load().sm_last_error()
        raise ShardMergeLibraryError(f"{what} failed (rc={rc}): {msg.decode() if msg else ''}")
