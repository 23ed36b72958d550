"""Host-side logic that needs no GPU: config schema, layer classification, canonical tensor order,
writer (write-once shards, resume, finalize), pairing, name hashing, work partition, and a
world_size-2 gloo run of the shard-granular multi-GPU merge driver with a CPU stand-in strategy."""
import asyncio
import json
import os
import subprocess
import sys
import textwrap
from pathlib import Path

import click
import numpy as np
import pytest
import torch

from oracle import oracle_np as O
from shardmerge_b200 import schedule
from shardmerge_b200.config import MergeConfig, MergeModel
from shardmerge_b200.constants import INPUT_LAYER, OUTPUT_LAYER
from shardmerge_b200.index import InMemoryIndex, LocalSafetensorsIndex, canonical_layer_order
from shardmerge_b200.merge.fast_fourier import clamp, name_hash, task_arithmetic, tree_plan
from shardmerge_b200.tensor.functions import correlated_pairs
from shardmerge_b200.writer import ModelWriter, ShardLayer

ROOT = Path(__file__).resolve().parent.parent


def test_config_yaml_roundtrip(tmp_path):
    y = tmp_path / "c.yaml"
    y.write_text(textwrap.dedent("""
        output_base_model: "org/base"
        finetune_merge:
          - { model: "org/a", base: "org/base", alpha: 0.3, is_input: true }
          - { model: "org/b", base: "org/base", alpha: 0.5, is_output: true, start_layer: 2, end_layer: 5 }
        output_dir: "out"
        device: "cuda"
    """))
    cfg = MergeConfig.from_yaml(y)
    assert cfg.output_astype == torch.bfloat16 and cfg.device == "cuda"
    assert cfg.input_model.model == "org/a" and cfg.output_model.model == "org/b"
    b = cfg.finetune_merge[1]
    assert [b.use_layer_index(i) for i in (1, 2, 5, 6)] == [False, True, True, False]
    assert cfg.finetune_merge[0].use_layer_index(10**6)
    cfg.update({"device": "cuda:1"}, cache_dir="x", bogus=1)
    assert cfg.device == "cuda:1" and cfg.cache_dir == "x" and not hasattr(cfg, "bogus")
    (tmp_path / "bad.yaml").write_text("output_dir: x\n")
    with pytest.raises(click.BadParameter):
        MergeConfig.from_yaml(tmp_path / "bad.yaml")
    with pytest.raises(TypeError):
        MergeModel(model="a", base="b", unknown_key=1)


def test_layer_number():
    L = lambda n: ShardLayer(0, "s", n, False).layer_number
    assert L("model.embed_tokens.weight") == INPUT_LAYER
    assert L("model.norm.weight") == OUTPUT_LAYER and L("lm_head.weight") == OUTPUT_LAYER
    assert L("model.layers.17.mlp.up_proj.weight") == 17
    for bad in ("model.layers.07.x", "transformer.h.0.w"):
        with pytest.raises(ValueError):
            L(bad)


def test_canonical_layer_order():
    names = ["lm_head.weight", "model.layers.10.a.weight", "model.layers.2.b.weight", "model.layers.2.a.weight",
             "model.layers.0.b.weight", "model.layers.0.a.weight", "model.layers.10.b.weight", "model.norm.weight",
             "model.embed_tokens.weight", "rotary.inv_freq"]
    assert canonical_layer_order(names) == [
        "model.embed_tokens.weight", "model.layers.0.a.weight", "model.layers.0.b.weight", "model.layers.2.a.weight",
        "model.layers.2.b.weight", "model.layers.10.a.weight", "model.layers.10.b.weight", "model.norm.weight",
        "lm_head.weight", "rotary.inv_freq"]


def test_name_hash_and_helpers():
    h = name_hash("org/model-a_org/model-b")
    assert h.startswith("org/_org/::") and len(h.split("::")[1]) == 8
    assert name_hash("x") == name_hash("x") != name_hash("y")
    assert clamp(5, 0, 3) == 3 and clamp(-1, 0, 3) == 0 and clamp(2, 0, 3) == 2
    t = task_arithmetic(torch.tensor([1.0, -1.0, 2.0]), torch.tensor([2.0, 3.0, -1.0]))
    assert t.tolist() == [3.0, -1.0, 2.0]


def test_correlated_pairs_matches_oracle():
    rng = np.random.default_rng(0)
    for n in (2, 3, 4, 5, 7):
        norms = rng.uniform(0.2, 0.9, n).astype(np.float32)
        c = np.zeros((n, n), np.float32)
        for i in range(n):
            for j in range(i + 1, n):
                c[i, j] = norms[i] * norms[j]
        for way in ("least", "most"):
            mine = [(x, y) for x, y, _ in correlated_pairs(torch.from_numpy(c), way)]
            assert mine == [(x, y) for x, y, _ in O.correlated_pairs(c, way)]
            used = [v for p in mine for v in p if v >= 0]
            assert sorted(used) == list(range(n))
    with pytest.raises(ValueError):
        list(correlated_pairs(torch.zeros(3, 3), "sideways"))


def _oracle_tree(norms, weights, cull_start_pct):
    """The rounds of oracle_np.merge_layer's pair loop (the stale-norm products, :171-254 of the reference) as
    (x, y, a_w, b_w, cull_pct, last) with (x, -1, w, 0.0, cull_pct, False) for a model carried to the next round."""
    rounds, w, cull = [], list(weights), cull_start_pct
    while len(w) > 1:
        n = len(w)
        corr = np.zeros((n, n), dtype=np.float32)
        for i in range(n):
            for j in range(i + 1, n):
                corr[i, j] = norms[i] * norms[j]
        pairs = O.correlated_pairs(corr, "least")
        rnd = [(x, y, w[x], w[y] if y >= 0 else 0.0, cull, y >= 0 and len(pairs) == 1) for x, y, _ in pairs]
        rounds.append(rnd)
        w = [a_w if y < 0 else (a_w + b_w) / 2.0 for _, y, a_w, b_w, _, _ in rnd]
        cull = cull / 2.0
    return rounds


@pytest.mark.parametrize("kind", ["equal", "random"])
def test_tree_plan_matches_oracle_loop(kind):
    rng = np.random.default_rng(5)
    for m in range(1, 13):
        sumsq = [0.04] * m if kind == "equal" else list(rng.uniform(1e-4, 2.0, m))
        weights = list(rng.uniform(0.1, 1.0, m))
        norms, target_norm, rounds = tree_plan(sumsq, weights, 0.20, 1e-10)
        want_norms = [np.float32(v ** 0.5) for v in sumsq]
        assert norms == [float(v) for v in want_norms]
        assert abs(target_norm / (float(np.mean(np.array(want_norms, dtype=np.float32))) + 1e-10) - 1) < 1e-6
        assert [[tuple(st) for st in rnd] for rnd in rounds] == _oracle_tree(want_norms, weights, 0.20), m
        assert len(rounds) == (m - 1).bit_length() and sum(st.last for rnd in rounds for st in rnd) == (m > 1)


def _toy_model(seed, L=3, H=16):
    g = torch.Generator().manual_seed(seed)
    t = {"model.embed_tokens.weight": torch.randn(32, H, generator=g).to(torch.bfloat16),
         "model.norm.weight": torch.randn(H, generator=g).to(torch.bfloat16),
         "lm_head.weight": torch.randn(32, H, generator=g).to(torch.bfloat16)}
    for i in range(L):
        t[f"model.layers.{i}.mlp.up_proj.weight"] = torch.randn(2 * H, H, generator=g).to(torch.bfloat16)
        t[f"model.layers.{i}.input_layernorm.weight"] = torch.randn(H, generator=g).to(torch.bfloat16)
    return t


def test_writer_write_once_resume_finalize(tmp_path):
    from safetensors import safe_open
    idx = InMemoryIndex({"m": _toy_model(0)})
    asyncio.run(idx.add_model("m"))
    order = idx.get_layer_order("m")
    doc = idx.model_indexes["m"]
    w = ModelWriter(base_index=doc, output_path=tmp_path / "out", layer_order=order, output_astype=torch.float16)
    assert json.loads((tmp_path / "out" / "model.safetensors.index.json").read_text())["weight_map"] == doc["weight_map"]
    groups = list(w.shard_layers())
    assert [g[0].shard_name for g in groups] == sorted({v for v in doc["weight_map"].values()})
    first = groups[0]
    # nothing is written until the shard is complete
    w.add_tensor(first[0].layer_name, idx.models["m"][first[0].layer_name])
    assert not (tmp_path / "out" / first[0].shard_name).exists()
    for sl in first[1:]:
        w.add_tensor(sl.layer_name, idx.models["m"][sl.layer_name])
    path = tmp_path / "out" / first[0].shard_name
    w.wait()                                               # the file is written by the writer thread
    assert path.exists() and not list((tmp_path / "out").glob("*.tmp*"))
    with safe_open(path, framework="pt") as f:
        assert set(f.keys()) == {sl.layer_name for sl in first} and f.metadata() == {"format": "pt"}
        t = f.get_tensor(first[0].layer_name)
        assert t.dtype == torch.float16
        assert torch.equal(t, idx.models["m"][first[0].layer_name].to(torch.float16))
    with pytest.raises(RuntimeError):
        w.finalize()                                       # other shards are missing
    # resume: a new writer sees the finished shard as written and skips it
    w2 = ModelWriter(base_index=doc, output_path=tmp_path / "out", layer_order=order, output_astype=torch.float16)
    assert all(sl.written for sl in list(w2.shard_layers())[0])
    mtime = path.stat().st_mtime_ns
    w2.add_tensor(first[0].layer_name, idx.models["m"][first[0].layer_name])
    assert path.stat().st_mtime_ns == mtime
    for g in list(w2.shard_layers())[1:]:
        for sl in g:
            w2.add_tensor(sl.layer_name, idx.models["m"][sl.layer_name])
    w2.finalize()


def test_write_safetensors_matches_save_file(tmp_path):
    """The writer's own container code must produce the bytes safetensors.torch.save_file produces."""
    from safetensors.torch import save_file
    from shardmerge_b200.writer import write_safetensors
    g = torch.Generator().manual_seed(3)
    t = {"model.layers.1.b": torch.randn(5, 7, generator=g).to(torch.bfloat16),
         "model.layers.0.a": torch.randn(3, generator=g),
         "model.norm.weight": torch.randn(4, 2, 3, generator=g).to(torch.float16),
         "x.i64": torch.arange(5), "x.u8": torch.arange(7, dtype=torch.uint8), "x.scalar": torch.tensor(1.5),
         "x.empty": torch.zeros((0, 4), dtype=torch.bfloat16), "x.bool": torch.tensor([True, False, True])}
    for meta in ({"format": "pt"}, None):
        save_file(t, str(tmp_path / "a.safetensors"), metadata=meta)
        write_safetensors(tmp_path / "b.safetensors", t, metadata=meta)
        assert (tmp_path / "a.safetensors").read_bytes() == (tmp_path / "b.safetensors").read_bytes()
    with pytest.raises(ValueError):
        write_safetensors(tmp_path / "c.safetensors", {"nc": torch.zeros(4, 4).t()[1:]})
    # the parallel path (shared mapping + chunk copies by a thread pool) for files above 4 MB
    from concurrent.futures import ThreadPoolExecutor
    big = {"w.b": torch.randn(1100, 1024, generator=g).to(torch.bfloat16), "w.a": torch.randn(700, 1024, generator=g),
           "w.c": torch.randn(3, generator=g)}
    save_file(big, str(tmp_path / "a.safetensors"), metadata={"format": "pt"})
    with ThreadPoolExecutor(4) as pool:
        write_safetensors(tmp_path / "b.safetensors", big, metadata={"format": "pt"}, io_pool=pool)
    assert (tmp_path / "a.safetensors").read_bytes() == (tmp_path / "b.safetensors").read_bytes()


def test_writer_flush_partial_resumes_at_tensor_granularity(tmp_path):
    """A merge that aborts mid-shard keeps the tensors it already produced (ADVICE r1: resume granularity)."""
    from safetensors import safe_open
    idx = InMemoryIndex({"m": _toy_model(0)})
    asyncio.run(idx.add_model("m"))
    order, doc = idx.get_layer_order("m"), idx.model_indexes["m"]
    w = ModelWriter(base_index=doc, output_path=tmp_path / "out", layer_order=order, output_astype=torch.bfloat16)
    group = next(g for g in w.shard_layers() if len(g) > 1)
    w.add_tensor(group[0].layer_name, idx.models["m"][group[0].layer_name])
    w.flush_partial()
    with safe_open(tmp_path / "out" / group[0].shard_name, framework="pt") as f:
        assert set(f.keys()) == {group[0].layer_name}
    w2 = ModelWriter(base_index=doc, output_path=tmp_path / "out", layer_order=order, output_astype=torch.bfloat16)
    g2 = next(g for g in w2.shard_layers() if g[0].shard_name == group[0].shard_name)
    assert [sl.written for sl in g2] == [True] + [False] * (len(g2) - 1)
    for sl in g2[1:]:
        w2.add_tensor(sl.layer_name, idx.models["m"][sl.layer_name])
    w2.wait()
    with safe_open(tmp_path / "out" / group[0].shard_name, framework="pt") as f:
        assert set(f.keys()) == {sl.layer_name for sl in g2}
        assert torch.equal(f.get_tensor(group[0].layer_name), idx.models["m"][group[0].layer_name])


def test_process_layers_finalizes_each_tensor_before_the_writer_sees_it():
    """ADVICE r1 (high): deferred results must be resolved by identity before writer.add_tensor, whatever mix of
    deferred and immediate tensors is in flight (fused chain followed by pass-through tensors)."""
    from shardmerge_b200.merge.base import MergeTensorsBase
    log = []

    class Deferred(MergeTensorsBase):
        pipeline_depth = 1

        def __init__(self):
            self.pending = []

        def get_readme(self):
            return ""

        async def _merge_layer(self, shard_layer, device):
            t = torch.zeros(1)
            if shard_layer.layer_name.startswith("model.layers."):     # "fused": result is final only after _finalize
                self.pending.append(t)
            return t

        def _finalize(self, tensor):
            for i, p in enumerate(self.pending):
                if p is tensor:
                    del self.pending[: i + 1]
                    tensor += 1
                    return

    class Sink:
        def add_tensor(self, name, tensor):
            log.append((name, float(tensor)))

    names = ["model.layers.0.a", "model.norm.weight", "lm_head.weight", "model.layers.1.a", "model.layers.1.b",
             "model.embed_tokens.weight", "model.layers.2.a"]
    m = Deferred()
    asyncio.run(m._process_layers(Sink(), [ShardLayer(i, "s", n, False) for i, n in enumerate(names)], "cpu"))
    assert [n for n, _ in log] == names
    assert all(v == (1.0 if n.startswith("model.layers.") else 0.0) for n, v in log) and not m.pending


def test_fourier_merge_validates_shapes_up_front(tmp_path):
    """ADVICE r1: a tensor whose shape has no FFT plan (both dimensions odd here) is reported by initialize(), before
    any output exists; awkward but supported lengths (37, 167 as prime factors) pass."""
    from shardmerge_b200.engine import UnsupportedShape
    from shardmerge_b200.merge.fast_fourier import FourierMerge
    ok = {"model.embed_tokens.weight": torch.zeros(7, 3, dtype=torch.bfloat16),          # pass-through: never transformed
          "model.layers.0.mlp.up_proj.weight": torch.zeros(74, 334, dtype=torch.bfloat16),
          "model.layers.0.mlp.down_proj.weight": torch.zeros(16, 7, dtype=torch.bfloat16),  # odd rows: merged as the transpose
          "model.layers.0.input_layernorm.weight": torch.zeros(74, dtype=torch.bfloat16)}
    cfg = MergeConfig(finetune_merge=[MergeModel(model="org/a", base="org/base")], output_base_model="org/base",
                      output_dir=str(tmp_path / "out"))
    asyncio.run(FourierMerge(cfg, index_manager=InMemoryIndex({"org/base": ok, "org/a": ok})).initialize())
    bad = dict(ok)
    bad["model.layers.0.self_attn.q_proj.weight"] = torch.zeros(15, 7, dtype=torch.bfloat16)
    with pytest.raises(UnsupportedShape) as exc:
        asyncio.run(FourierMerge(cfg, index_manager=InMemoryIndex({"org/base": bad, "org/a": bad})).initialize())
    assert "q_proj" in str(exc.value) and not (tmp_path / "out").exists()


def test_verify_output_and_copy_model_files(tmp_path):
    """SURVEY 8f N4: the index / file alignment check of scripts/verify_safetensors.py plus dtype / shape / finiteness,
    and the local counterpart of `shard copy-model`."""
    from safetensors.torch import save_file
    from shardmerge_b200.validate import copy_model_files, verify_output
    out = tmp_path / "out"
    out.mkdir()
    a, b = torch.ones(4, 4, dtype=torch.bfloat16), torch.ones(8, dtype=torch.bfloat16)
    save_file({"model.layers.0.a": a, "model.layers.0.b": b}, str(out / "s1.safetensors"), metadata={"format": "pt"})
    save_file({"model.layers.1.a": a}, str(out / "s2.safetensors"), metadata={"format": "pt"})
    wm = {"model.layers.0.a": "s1.safetensors", "model.layers.0.b": "s1.safetensors", "model.layers.1.a": "s2.safetensors"}
    (out / "model.safetensors.index.json").write_text(json.dumps({"metadata": {}, "weight_map": wm}))
    rep = verify_output(out, expected_dtype=torch.bfloat16, expected_shapes={"model.layers.0.a": (4, 4)})
    assert rep.ok and rep.tensors == 3 and "align" in rep.summary()
    # break it: a NaN, a wrong dtype, a key the index does not know, a shard the index names but that is gone, an extra file
    bad = a.clone(); bad[0, 0] = float("nan")
    save_file({"model.layers.0.a": bad, "model.layers.0.b": b.float(), "stray": a}, str(out / "s1.safetensors"))
    (out / "s2.safetensors").unlink()
    save_file({"x": a}, str(out / "s9.safetensors"))
    rep = verify_output(out, expected_dtype=torch.bfloat16, expected_shapes={"model.layers.0.a": (2, 8)})
    assert not rep.ok
    assert rep.missing_files == ["s2.safetensors"] and rep.extra_files == ["s9.safetensors"]
    assert rep.extra_keys == {"s1.safetensors": ["stray"]} and rep.non_finite == {"model.layers.0.a": 1}
    assert rep.wrong_dtype == {"model.layers.0.b": "torch.float32"} and rep.wrong_shape == {"model.layers.0.a": (4, 4)}
    # copy-model: configuration / tokenizer files only
    src = tmp_path / "org" / "m"
    src.mkdir(parents=True)
    for n in ("config.json", "tokenizer.json", "generation_config.json", "model-00001-of-00001.safetensors",
              "model.safetensors.index.json", "pytorch_model.bin"):
        (src / n).write_text("{}")
    assert copy_model_files(src, out) == ["config.json", "generation_config.json", "tokenizer.json"]
    assert copy_model_files(src, out) == []                 # nothing is overwritten
    with pytest.raises(FileNotFoundError):
        copy_model_files(tmp_path / "nope", out)


def test_local_safetensors_index(tmp_path):
    from safetensors.torch import save_file
    model = _toy_model(1)
    d = tmp_path / "org" / "m"
    d.mkdir(parents=True)
    names = list(model)
    shards = {"model-00001-of-00002.safetensors": names[:4], "model-00002-of-00002.safetensors": names[4:]}
    wm = {}
    for fn, ns in shards.items():
        save_file({n: model[n] for n in ns}, str(d / fn), metadata={"format": "pt"})
        wm.update({n: fn for n in ns})
    (d / "model.safetensors.index.json").write_text(json.dumps({"metadata": {}, "weight_map": wm}))
    idx = LocalSafetensorsIndex(tmp_path)
    asyncio.run(idx.add_model("org/m"))
    assert idx.get_model_keys("org/m") == set(names)
    t = asyncio.run(idx.get_tensor("org/m", names[5]).get())
    assert torch.equal(t, model[names[5]])
    assert idx.tensor_numels("org/m") == {n: v.numel() for n, v in model.items()}
    with pytest.raises(FileNotFoundError):
        asyncio.run(idx.add_model("org/missing"))


def test_lpt_partition_llama70b_balance():
    H, I, KV, L = 8192, 28672, 1024, 80
    numels = {}
    for l in range(L):
        for nm, n in (("q", H * H), ("k", KV * H), ("v", KV * H), ("o", H * H), ("gate", I * H), ("up", I * H),
                      ("down", H * I), ("ln1", H), ("ln2", H)):
            numels[f"model.layers.{l}.{nm}"] = n
    parts = schedule.tensor_partition(numels, 8, n_models=2)
    assert sorted(n for p in parts for n in p) == sorted(numels)
    cost = {n: schedule.merge_cost(v, 2) for n, v in numels.items()}
    assert schedule.imbalance(parts, cost) < 0.03          # SURVEY 8e: < 3 %
    assert schedule.tensor_partition(numels, 8, 2) == parts  # deterministic
    assert schedule.lpt([("a", 3), ("b", 3), ("c", 2)], 2) == [["a", "c"], ["b"]]


WORKER = textwrap.dedent("""
    import asyncio, os, sys, torch, torch.distributed as dist
    sys.path.insert(0, %(root)r)
    from shardmerge_b200.config import MergeConfig, MergeModel
    from shardmerge_b200.index import InMemoryIndex
    from shardmerge_b200.merge.base import MergeTensorsBase
    from shardmerge_b200 import schedule
    sys.path.insert(0, os.path.join(%(root)r, "tests"))
    from test_host_logic import _toy_model

    class CpuStandIn(MergeTensorsBase):           # TEST stand-in: exercises partition + writer only
        def get_readme(self): return "readme"
        async def _merge_layer(self, shard_layer, device):
            t = await self.index_manager.get_tensor("org/a", shard_layer.layer_name).get()
            return (t.float() * 2).to(torch.bfloat16)

    dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%(port)d", rank=int(sys.argv[1]), world_size=2)
    models = {"org/base": _toy_model(0, L=6), "org/a": _toy_model(1, L=6)}
    cfg = MergeConfig(finetune_merge=[MergeModel(model="org/a", base="org/base")], output_base_model="org/base",
                      output_dir=sys.argv[2])
    m = CpuStandIn(cfg, index_manager=InMemoryIndex(models))
    mine = asyncio.run(schedule.merge_distributed(m, "cpu", dist.get_rank(), 2, barrier=dist.barrier))
    print("RANK", dist.get_rank(), "SHARDS", ",".join(mine), flush=True)
    dist.barrier()                                # nobody tears the store down while the other rank still talks to it
    dist.destroy_process_group()
""")


def test_merge_distributed_world2_gloo(tmp_path):
    from safetensors import safe_open
    import shutil
    import socket
    script = tmp_path / "worker.py"
    out = tmp_path / "out"
    for attempt in range(3):                      # a rendezvous port can be taken between the probe and the bind: retry
        with socket.socket() as sk:
            sk.bind(("127.0.0.1", 0))
            port = sk.getsockname()[1]
        script.write_text(WORKER % dict(root=str(ROOT), port=port))
        shutil.rmtree(out, ignore_errors=True)
        procs = [subprocess.Popen([sys.executable, str(script), str(r), str(out)], stdout=subprocess.PIPE,
                                  stderr=subprocess.STDOUT, text=True) for r in range(2)]
        logs = [p.communicate(timeout=180)[0] for p in procs]
        if all(p.returncode == 0 for p in procs):
            break
    assert all(p.returncode == 0 for p in procs), logs
    owned = [set(l.split("SHARDS")[1].strip().split(",")) for l in logs]
    assert owned[0] and owned[1] and not (owned[0] & owned[1])
    ref = _toy_model(1, L=6)
    seen = set()
    for f in out.glob("*.safetensors"):
        with safe_open(f, framework="pt") as sf:
            for k in sf.keys():
                assert torch.equal(sf.get_tensor(k), (ref[k].float() * 2).to(torch.bfloat16))
                seen.add(k)
    assert seen == set(ref) and (out / "README.md").read_text() == "readme"


SELECT_WORKER = textwrap.dedent("""
    import sys, numpy as np, torch, torch.distributed as dist
    sys.path.insert(0, %(root)r)
    from shardmerge_b200.rowsplit import dist_select_kth
    rank = int(sys.argv[1])
    dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%(port)d", rank=rank, world_size=2)
    rng = np.random.default_rng(5)
    full = rng.standard_normal((64, 96)).astype(np.float32)
    full[3, 7] = 0.0; full[10, 80] = np.float32(1e-30); full[20, 5] = full[21, 6]        # zero, tiny, a tie
    Ch = 90                                                   # columns 0..Ch valid, 91..95 padding
    full[:, Ch + 1:] = 0.0
    w = 48                                                    # two column slabs of 48
    mine = torch.from_numpy(full[:, rank * w:(rank + 1) * w].copy())
    col = rank * w + torch.arange(w)
    mult = torch.where(col <= Ch, torch.where((col == 0) | (col == Ch), 1, 2), 0).to(torch.int64)
    keys = mine.view(torch.int32) & 0x7FFFFFFF
    # reference: every valid bin with its multiplicity, sorted
    allmult = np.where(np.arange(96) <= Ch, np.where((np.arange(96) == 0) | (np.arange(96) == Ch), 1, 2), 0)
    ref = np.sort(np.repeat(np.abs(full), allmult, axis=1).ravel())
    ok = True
    for k in (0, 1, 17, len(ref) // 5, len(ref) // 2, len(ref) - 1):
        bits = dist_select_kth([keys], mult, k)
        val = np.array([bits], dtype=np.int32).view(np.float32)[0]
        ok = ok and (val == ref[k])
    # two planes at once (the cutoff statistic runs over cat(|re0|, |re1|))
    ref2 = np.sort(np.concatenate([ref, ref * np.float32(0.5)]))
    bits = dist_select_kth([keys, (mine * 0.5).view(torch.int32) & 0x7FFFFFFF], mult, len(ref2) // 12)
    ok = ok and (np.array([bits], dtype=np.int32).view(np.float32)[0] == ref2[len(ref2) // 12])
    print("RANK", rank, "OK" if ok else "MISMATCH", flush=True)
    dist.barrier(); dist.destroy_process_group()
""")


def test_distributed_order_statistic_world2_gloo(tmp_path):
    """The exact radix select the row-split merge uses for its two global order statistics (shardmerge_b200/rowsplit.py:
    weighted histograms per rank, all-reduce, three rounds), two ranks over gloo on CPU against a sort."""
    import socket
    script = tmp_path / "sel_worker.py"
    for attempt in range(3):
        with socket.socket() as sk:
            sk.bind(("127.0.0.1", 0))
            port = sk.getsockname()[1]
        script.write_text(SELECT_WORKER % dict(root=str(ROOT), port=port))
        procs = [subprocess.Popen([sys.executable, str(script), str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
                 for r in range(2)]
        logs = [p.communicate(timeout=180)[0] for p in procs]
        if all(p.returncode == 0 for p in procs):
            break
    assert all(p.returncode == 0 for p in procs), logs
    assert all("OK" in l and "MISMATCH" not in l for l in logs), logs
