"""Which plans get the paired forward row pass (sm_fwd_rows_bf16_pair): host logic, no GPU needed."""
from shardmerge_b200 import _lib


def test_pair_support_follows_the_row_kernels():
    """Only row lengths whose single-model pass runs a kernel with a paired variant get one (C = 4096 with an even row
    count, C = 14336); elsewhere the paired call fails with a message and launches nothing."""
    lib = _lib.load()
    for (R, C), want in (((1024, 4096), 1), ((4096, 4096), 1), ((1023, 4096), 0), ((4096, 14336), 1), ((1, 14336), 1),
                         ((8192, 28672), 0), ((1024, 8192), 0), ((2048, 2048), 0), ((512, 5632), 0), ((64, 128), 0)):
        p = lib.sm_plan_create(R, C)
        assert p, (R, C)
        try:
            assert lib.sm_fwd_rows_pair_supported(p) == want, (R, C)
            if not want:
                rc = lib.sm_fwd_rows_bf16_pair(p, None, None, None, None, None, None, None, None, None, 1e-10, 0.0, None)
                assert rc != 0 and b"no paired row kernel" in lib.sm_last_error(), (R, C)
        finally:
            lib.sm_plan_destroy(p)
