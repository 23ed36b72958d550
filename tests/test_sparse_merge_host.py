"""TIES / DARE, host side: the oracle's Philox against Random123's known answers, the DARE and magnitude keep masks, one
small case worked out by hand for each strategy, and the refusals of initialize().  No GPU."""
import asyncio

import numpy as np
import pytest
import torch

from shardmerge_b200.config import MergeConfig, MergeModel
from shardmerge_b200.index import LocalSafetensorsIndex
from shardmerge_b200.lora import UnsupportedAdapter
from shardmerge_b200.merge import DareLinearMerge, DareTiesMerge, TiesMerge
from shardmerge_b200.merge import ties as T
from tests import sparse_oracle as O
from tests.lora_util import adapter_tensors, llama_shapes, random_model, write_adapter, write_model

f32 = np.float32


@pytest.mark.parametrize("ctr,key,want", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_known_answers(ctr, key, want):
    assert tuple(int(w) for w in O.philox4x32_10(ctr, key)) == want


def test_dare_key_is_the_strategy_key():
    for seed, i, name in [(0, 0, "a"), (7, 3, "model.layers.1.mlp.up_proj.weight"), (2 ** 40, 63, "x")]:
        assert T.dare_key(seed, i, name) == O.dare_key(seed, i, name)


@pytest.mark.parametrize("density", [0.01, 0.1, 0.5, 0.9])
def test_dare_kept_fraction(density):
    n = 1 << 20
    kept = int(O.dare_keep_mask(n, density, 0, 0, "model.layers.0.self_attn.q_proj.weight").sum())
    p = O.keep24(density) / 2 ** 24
    assert abs(kept - n * p) <= 5 * (n * p * (1 - p)) ** 0.5


def test_dare_mask_depends_on_seed_model_and_name_only():
    n, name = 4099, "model.layers.3.mlp.down_proj.weight"
    m2 = O.dare_keep_mask(n, 0.3, 5, 2, name)
    O.dare_keep_mask(n, 0.3, 5, 0, "model.layers.0.mlp.down_proj.weight")     # other tensors / models in between
    assert np.array_equal(O.dare_keep_mask(n, 0.3, 5, 2, name), m2)
    assert np.array_equal(O.dare_keep_mask(2 * n, 0.3, 5, 2, name)[:n], m2)   # a prefix does not depend on n
    # model 2 merged alone and next to zero-weight models: the same result, so its mask ignores who else takes part
    rng = np.random.default_rng(0)
    W = rng.standard_normal(n).astype(f32)
    F = [W + rng.standard_normal(n).astype(f32) for _ in range(3)]
    alone = O.ties_family_merge("dare_linear", W, [F[2]], [1.0], 0.3, seed=5, tensor_name=name, model_indices=[2])
    joint = O.ties_family_merge("dare_linear", W, F, [0.0, 0.0, 1.0], 0.3, seed=5, tensor_name=name)
    assert np.array_equal(alone.view(np.uint32), joint.view(np.uint32))
    assert not np.array_equal(O.dare_keep_mask(n, 0.5, 5, 0, name), O.dare_keep_mask(n, 0.5, 5, 1, name))
    assert O.dare_keep_mask(n, 1.0, 5, 0, name).all()


@pytest.mark.parametrize("k", [0, 1, 37, 500, 999, 1000])
def test_magnitude_keep_all_equal_keeps_the_first_k(k):
    d = np.where(np.random.default_rng(k).random(1000) < 0.5, f32(-0.25), f32(0.25))
    keep = O.magnitude_keep_mask(d, k)
    assert keep.sum() == k and keep[:k].all() and not keep[k:].any()


@pytest.mark.parametrize("k", [0, 1, 200, 1234, 3000, 4096])
def test_magnitude_keep_five_values(k):
    d = np.random.default_rng(k + 1).choice(np.array([-2, -1, 0.5, 1, 2], dtype=f32), 4096)
    keep = O.magnitude_keep_mask(d, k)
    assert keep.sum() == k
    K, J = O.magnitude_threshold(d, k)
    mag = d.view(np.uint32) & np.uint32(0x7FFFFFFF)
    assert np.array_equal(keep, (mag > K) | ((mag == K) & (np.arange(d.size) <= J)))
    if 0 < k < d.size:      # every dropped magnitude is at most every kept one, and ties go to the lower index
        assert mag[~keep].max() <= mag[keep].min()
        tied = np.flatnonzero(mag == mag[keep].min())
        assert keep[tied].sum() == 0 or np.flatnonzero(keep[tied]).max() < np.flatnonzero(~keep[tied]).min(initial=tied.size)


# one tensor of 8 elements, 3 models with weights 1, 1, 2, base 1.0, density 0.5, scale 1
D3 = np.array([[4, -2, 0, 1, -3, 2, 0.5, -1],
               [-1, 3, 2, -1, -3, 0, 0.5, 2],
               [2, 2, -4, 0, 1, -2, -0.5, 1]], dtype=f32)
NAME3 = "model.layers.0.mlp.up_proj.weight"


def _by_hand_case(mode):
    W = np.ones(8, dtype=f32)
    return O.ties_family_merge(mode, W, [W + d for d in D3], [1.0, 1.0, 2.0], 0.5, scale=1.0, seed=7, tensor_name=NAME3)


def test_ties_by_hand():
    # k = 4 per model; model 2 has |d| = 2 at j = 0, 1, 5 (all kept after the 4 at j = 2)
    # v0 = [4,-2,0,0,-3,2,0,0]  v1 = [0,3,2,0,-3,0,0,2]  v2 = 2*[2,2,-4,0,0,-2,0,0]
    # S = [8,5,-6,0,-6,-2,0,2]: majority + - + (S = 0 counts as +) ...
    want = [f32(1) + f32(8) / f32(3), f32(1) + f32(7) / f32(3), -3, 1, -2, -1, 1, 3]
    assert np.array_equal(_by_hand_case("ties"), np.array(want, dtype=f32))


def test_dare_masks_of_the_by_hand_case():
    got = [O.dare_keep_mask(8, 0.5, 7, i, NAME3).astype(int).tolist() for i in range(3)]
    assert got == [[0, 1, 1, 0, 0, 1, 1, 1], [0, 1, 0, 1, 0, 0, 1, 1], [1, 0, 0, 0, 1, 1, 0, 0]]


def test_dare_ties_by_hand():
    # t_i = kept ? 2 d_i : 0 -> v0 = [0,-4,0,0,0,4,1,-2]  v1 = [0,6,0,-2,0,0,1,4]  v2 = 2*[4,0,0,0,2,-4,0,0]
    # S = [8,2,0,-2,4,-4,2,2]
    assert np.array_equal(_by_hand_case("dare_ties"), np.array([5, 7, 1, -1, 3, -3, 2, 5], dtype=f32))


def test_dare_linear_by_hand():
    # m = S, D = 1 + 1 + 2 = 4 everywhere
    assert np.array_equal(_by_hand_case("dare_linear"), np.array([3, 1.5, 1, 0.5, 2, 0, 1.5, 1.5], dtype=f32))


def test_round_to_is_torch_rne():
    x = np.random.default_rng(3).standard_normal(10000).astype(f32) * f32(1e3)
    for name, dt in (("bfloat16", torch.bfloat16), ("float16", torch.float16)):
        want = torch.from_numpy(x).to(dt).view(torch.int16).numpy().view(np.uint16)
        assert np.array_equal(O.round_to(x, name), want)


# ---- refusals of initialize(): raised before any tensor data is read or output written
SHAPES = llama_shapes(layers=2)


@pytest.fixture
def storage(tmp_path):
    write_model(tmp_path / "org" / "base", random_model(SHAPES, 0))
    write_model(tmp_path / "org" / "base2", random_model(SHAPES, 1))
    write_model(tmp_path / "org" / "ft", random_model(SHAPES, 2))
    write_model(tmp_path / "org" / "ft64", random_model(SHAPES, 3, dtype=torch.float64))
    write_adapter(tmp_path / "org" / "ad", adapter_tensors(SHAPES, ("q_proj",), 4, seed=9), r=4)
    return tmp_path


def _strategy(storage, cls, models, **kw):
    cfg = MergeConfig(finetune_merge=models, output_base_model="org/base", output_dir=str(storage / "out"),
                      storage_dir=str(storage))
    return cls(cfg, index_manager=LocalSafetensorsIndex(cfg.storage_path), **kw)


def _refused(storage, strategy, exc=ValueError, match=None):
    with pytest.raises(exc, match=match):
        asyncio.run(strategy.merge("cuda:0"))
    out = storage / "out"
    assert not out.exists() or not any(out.iterdir())


@pytest.mark.parametrize("cls", [TiesMerge, DareTiesMerge, DareLinearMerge])
@pytest.mark.parametrize("density", [0.0, -0.1, 1.0000001, 2.0, float("nan")])
def test_refuses_density(storage, cls, density):
    _refused(storage, _strategy(storage, cls, [MergeModel(model="org/ft", base="org/base")], density=density), match="density")


@pytest.mark.parametrize("cls", [TiesMerge, DareTiesMerge, DareLinearMerge])
def test_refuses_other_bases(storage, cls):
    models = [MergeModel(model="org/ft", base="org/base"), MergeModel(model="org/ft", base="org/base2")]
    _refused(storage, _strategy(storage, cls, models, density=0.5), match="base")


@pytest.mark.parametrize("cls", [TiesMerge, DareTiesMerge, DareLinearMerge])
def test_refuses_adapters(storage, cls):
    assert cls.merges_adapters is False
    _refused(storage, _strategy(storage, cls, [MergeModel(model="org/ad", base="org/base")], density=0.5), UnsupportedAdapter)


@pytest.mark.parametrize("cls", [TiesMerge, DareTiesMerge, DareLinearMerge])
def test_refuses_more_than_64_models_in_a_tensor(storage, cls):
    models = [MergeModel(model="org/ft", base="org/base", start_layer=0, end_layer=0) for _ in range(33)]
    models += [MergeModel(model="org/ft", base="org/base", start_layer=0, end_layer=-1) for _ in range(32)]
    _refused(storage, _strategy(storage, cls, models, density=0.5), match="at most 64")
    # 65 entries, but never more than 64 in one tensor: accepted by initialize()
    models[0] = MergeModel(model="org/ft", base="org/base", start_layer=5, end_layer=5)
    asyncio.run(_strategy(storage, cls, models, density=0.5).initialize())


@pytest.mark.parametrize("cls", [TiesMerge, DareTiesMerge, DareLinearMerge])
def test_refuses_other_dtypes(storage, cls):
    _refused(storage, _strategy(storage, cls, [MergeModel(model="org/ft64", base="org/base")], density=0.5),
             match="float32, bfloat16 and float16")


def test_readme_names_method_and_parameters(storage):
    s = _strategy(storage, DareTiesMerge, [MergeModel(model="org/ft", base="org/base", alpha=0.7)], density=0.3, seed=11)
    text = s.get_readme()
    assert "DARE-TIES" in text and "density 0.3" in text and "seed 11" in text and "org/ft (weight 0.7)" in text
