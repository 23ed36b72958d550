"""oracle_np.merge_layer on fp16 and fp32 checkpoints (CPU only).

merge_layer takes each stored tensor in its own dtype -- uint16 bf16 bit patterns, float16, float32 -- and widens it
exactly, as `.to(torch.float32)` does in the reference (base.py:128-132, fast_fourier.py:269).  So a value stored in any of
the three dtypes merges to the same bits, and a delta is formed in fp32 whatever the storage dtype."""
import numpy as np
import pytest

from oracle import oracle_np as O


def _stored(x):
    """bf16 bit patterns of fp32 values `x`, rounded so that float16 holds them exactly too: bf16 keeps 8 significant
    bits, a normal float16 11, so only magnitudes below float16's smallest normal (2^-14) have to go."""
    x = O.bf16_to_f32(O.f32_to_bf16(np.asarray(x, dtype=np.float32)))
    u = O.f32_to_bf16(np.where(np.abs(x) < 2.0 ** -14, np.float32(0), x).astype(np.float32))
    assert np.array_equal(O.bf16_to_f32(u).astype(np.float16).astype(np.float32), O.bf16_to_f32(u))
    return u


def _case(kind, seed):
    """(output base, [(base, finetune, alpha)]) as bf16 bit patterns, drawn so that merge_layer takes `kind`."""
    rng = np.random.default_rng(seed)
    shape = (64, 128)
    base = _stored(0.02 * rng.standard_normal(shape))
    sig = {"slerp": (0.002, 0.0026), "arith": (0.0026, 0.0001), "tree": (0.002, 0.0026, 0.0023), "single": (0.002,)}[kind]
    fts = [_stored(O.bf16_to_f32(base) + s * rng.standard_normal(shape)) for s in sig]
    return base, [(base, ft, a) for ft, a in zip(fts, (0.3, 0.5, 0.4))]


def _as(u16, dtype):
    return u16 if dtype == "bf16" else O.bf16_to_f32(u16).astype({"fp16": np.float16, "fp32": np.float32}[dtype])


BRANCHES = {"slerp": ["slerp"], "arith": ["arith"], "tree": ["slerp", "slerp"], "single": []}


@pytest.mark.parametrize("kind", sorted(BRANCHES))
@pytest.mark.parametrize("base_dt,ft_dt,out_dt", [("fp16", "fp16", "fp16"), ("fp32", "fp32", "fp32"), ("bf16", "fp32", "bf16"),
                                                   ("fp16", "bf16", "fp16"), ("fp32", "fp16", "bf16")])
def test_bf16_representable_values_merge_alike_in_every_dtype(kind, base_dt, ft_dt, out_dt):
    base_out, models = _case(kind, seed=len(kind))
    info_ref, info = {}, {}
    want = O.merge_layer(base_out, [dict(base=b, ft=f, alpha=a, name=f"m{k}") for k, (b, f, a) in enumerate(models)], info=info_ref)
    got = O.merge_layer(_as(base_out, out_dt), [dict(base=_as(b, base_dt), ft=_as(f, ft_dt), alpha=a, name=f"m{k}")
                                                for k, (b, f, a) in enumerate(models)], info=info)
    assert info_ref["branches"] == info["branches"] == BRANCHES[kind]
    assert info["target_norm"] == info_ref["target_norm"]
    assert got.dtype == np.uint16 and np.array_equal(got, want)


def test_fp16_delta_beyond_the_fp16_range_is_formed_in_fp32():
    """base -60000 and finetune +60000 (both fp16) differ by 120000, which fp16 cannot hold (max 65504): the delta, its
    norm and the merged tensor stay finite."""
    rng = np.random.default_rng(5)
    shape = (32, 64)
    base = (0.02 * rng.standard_normal(shape)).astype(np.float16)
    fts = [(base.astype(np.float32) + s * rng.standard_normal(shape)).astype(np.float16) for s in (0.002, 0.0026)]
    base[3, 5], fts[0][3, 5], fts[1][3, 5] = -60000, 60000, 50000
    info = {}
    one = O.merge_layer(base, [dict(base=base, ft=fts[0], alpha=0.3, name="m0")], info=info)
    assert info["branches"] == [] and info["norms"][0] >= 120000
    # one model: the output is base + delta, so the spike comes back as the finetune's value
    assert O.bf16_to_f32(one)[3, 5] == O.bf16_to_f32(O.f32_to_bf16(np.float32(60000)))
    assert np.array_equal(one, O.f32_to_bf16(fts[0].astype(np.float32)))
    info = {}
    two = O.merge_layer(base, [dict(base=base, ft=ft, alpha=a, name=f"m{k}") for k, (ft, a) in enumerate(zip(fts, (0.3, 0.5)))],
                        info=info)
    assert info["branches"] == ["slerp"] and min(info["norms"]) >= 100000         # 50000 is 49984 in fp16
    assert np.isfinite(O.bf16_to_f32(two)).all()


def test_other_storage_dtypes_are_refused():
    with pytest.raises(TypeError):
        O.widen(np.zeros(4, dtype=np.float64))
    with pytest.raises(TypeError):
        O.widen(np.zeros(4, dtype=np.int16))


@pytest.mark.parametrize("norms", [(np.inf, 0.4), (np.inf, 0.4, 0.5), (0.3, np.inf, 0.5, 0.6)])
def test_infinite_norm_products_are_not_paired(norms):
    """The delta of a finetune holding an Inf has an infinite norm, and so do its norm products.  The product's pairing,
    like the oracle's, runs over the finite products and raises ValueError when only infinite ones are left."""
    import torch
    from shardmerge_b200.tensor.functions import correlated_pairs

    def outcome(pairs):
        try:
            return [(x, y) for x, y, _ in pairs()]
        except ValueError:
            return ValueError

    c = np.triu(np.outer(norms, norms), 1).astype(np.float32)
    for way in ("least", "most"):
        want = outcome(lambda: O.correlated_pairs(c, way))
        assert outcome(lambda: list(correlated_pairs(torch.from_numpy(c), way))) == want
        assert (want is ValueError) == (len(norms) != 3)
