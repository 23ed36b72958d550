"""The C-ABI library loads on a machine without a GPU and exports exactly what the header declares."""
import ctypes
import re
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


def _declared():
    header = (ROOT / "include" / "shardmerge_b200.h").read_text()
    return set(re.findall(r"\b(sm_[a-z0-9_]+)\s*\(", header))


def test_library_exports_every_declared_symbol():
    from shardmerge_b200 import _lib
    lib = _lib.load()
    declared = _declared()
    assert len(declared) >= 25
    for name in declared:
        assert hasattr(lib, name), name
    # and the ctypes prototype table covers the header one to one
    assert set(_lib.SIGNATURES) == declared


def test_plan_queries_need_no_gpu():
    from shardmerge_b200 import _lib
    lib = _lib.load()
    assert lib.sm_version() >= 100
    p = lib.sm_plan_create(4096, 14336)
    assert p
    assert lib.sm_plan_pitch(p) == 7200 and lib.sm_plan_col_passes(p) == 2
    freq = sorted(lib.sm_plan_row_freq(p, i) for i in range(4096))
    assert freq == list(range(4096))                     # stored order is a permutation
    # W_C + W_R tables plus the first-stage quad table (Ch / first radix entries of 32 bytes)
    assert lib.sm_plan_table_bytes(p) >= (4096 + 14336) * 8 + (7168 // 7) * 32
    buf = ctypes.create_string_buffer(512)
    assert lib.sm_plan_describe(p, buf, 512) > 0 and b"R=4096" in buf.value
    lib.sm_plan_destroy(p)
    # awkward lengths get a plan with generic radix stages (embed_tokens: 128256 = 2^8 * 3 * 167; Qwen2.5: 18944 = 2^9 * 37)
    for R, C, want in ((128256, 8192, b"3 167"), (18944, 3584, b"37"), (3584, 18944, b"37")):
        p = lib.sm_plan_create(R, C)
        assert p, (R, C)
        assert sorted(lib.sm_plan_row_freq(p, i) for i in range(0, R, 97)) == sorted(set(lib.sm_plan_row_freq(p, i) for i in range(0, R, 97)))
        assert lib.sm_plan_describe(p, buf, 512) > 0 and want in buf.value, buf.value
        lib.sm_plan_destroy(p)
    # unsupported shapes are refused with a message, not mangled
    assert not lib.sm_plan_create(16, 7)                 # odd C
    assert b"unsupported" in lib.sm_last_error()
    assert not lib.sm_plan_create(2 * 1031, 64)          # prime factor above 1021


def test_hot_shape_plans_unchanged():
    """The specialised kernels are chosen by factorisation: the plans of the BASELINE shapes must stay what the GPU parity
    report was measured with (tests/golden/plans_baseline.json: the plan strings of that run, one per shape)."""
    import json
    from pathlib import Path
    from shardmerge_b200 import _lib
    lib = _lib.load()
    rep = json.loads((Path(__file__).resolve().parent / "golden" / "plans_baseline.json").read_text())
    assert len(rep) == 12
    buf = ctypes.create_string_buffer(1024)
    for key, plan in rep.items():
        R, C = (int(v) for v in key.split("x"))
        p = lib.sm_plan_create(R, C)
        lib.sm_plan_describe(p, buf, 1024)
        assert buf.value.decode() == plan, key
        lib.sm_plan_destroy(p)


@pytest.mark.parametrize("R,C", [(4096, 4096), (1024, 4096), (14336, 4096), (4096, 14336), (8192, 8192), (1024, 8192),
                                 (28672, 8192), (8192, 28672), (2048, 2048), (256, 2048), (5632, 2048), (2048, 5632),
                                 (1, 2048), (1, 4096), (1, 8192)])
def test_every_baseline_shape_has_a_plan(R, C):
    from shardmerge_b200 import _lib
    lib = _lib.load()
    p = lib.sm_plan_create(R, C)
    assert p, (R, C)
    lib.sm_plan_destroy(p)


def test_no_cpu_fallback():
    import torch
    from shardmerge_b200 import engine
    from shardmerge_b200.tensor import functions as F
    with pytest.raises(RuntimeError):
        engine._require_cuda("cpu")
    with pytest.raises(RuntimeError):
        F.fft_transform(torch.randn(8, 8), "cpu")
    with pytest.raises(RuntimeError):
        F.merge_tensors_fft2_slerp(torch.randn(8, 8), torch.randn(8, 8), 0.5, "cpu")


def test_scalar_block_mirror_matches_header():
    """_lib's copy of the scalar-block layout is the header's #defines, name for name."""
    from shardmerge_b200 import _lib
    header = (ROOT / "include" / "shardmerge_b200.h").read_text()
    prefix = r"SM_(?:CTL|F|I|BRANCH|FS|SELECT)_\w+"
    declared = {name: int(v) for name, v in re.findall(rf"^#define ({prefix})\s+(\d+)", header, re.M)}
    assert len(declared) >= 29
    mirrored = {name: getattr(_lib, name) for name in dir(_lib) if re.fullmatch(prefix, name)}
    assert mirrored == declared
    assert set(_lib.BRANCH_NAMES) == {v for k, v in declared.items() if k.startswith("SM_BRANCH_")}


def test_pair_args_layout_matches_header(tmp_path):
    """sizeof and every field offset of sm_pair_args, compiled from the header, equal those of _lib.PairArgs."""
    import os
    import subprocess
    from shardmerge_b200 import _lib
    fields = [f[0] for f in _lib.PairArgs._fields_]
    src = tmp_path / "pair_args.c"
    src.write_text("#include <stdio.h>\n#include <stddef.h>\n#include \"shardmerge_b200.h\"\nint main(void) {\n"
                   "  printf(\"sizeof %zu\\n\", sizeof(sm_pair_args));\n"
                   + "".join(f"  printf(\"{f} %zu\\n\", offsetof(sm_pair_args, {f}));\n" for f in fields) + "  return 0;\n}\n")
    exe = tmp_path / "pair_args"
    subprocess.run([os.environ.get("CC", "gcc"), "-I", str(ROOT / "include"), "-o", str(exe), str(src)], check=True)
    got = dict(line.split() for line in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    assert int(got.pop("sizeof")) == ctypes.sizeof(_lib.PairArgs)
    assert {f: int(v) for f, v in got.items()} == {f: getattr(_lib.PairArgs, f).offset for f in fields}
