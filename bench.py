#!/usr/bin/env python
"""bench.py -- throughput of the per-tensor spectral merge hot path (BASELINE.json metric:
merged params/sec, weight GB/s; % of HBM roofline for the dominant kernel).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload llama8b|llama70b|tinyllama] [--layers L] [--finetunes M] [--dump-outputs DIR]

A "step" is one pass of the hot path over the workload's merged tensors: for every
`model.layers.*` tensor of the named architecture, base + M finetunes (synthetic random-init
bf16, SURVEY.md 8d) -> merged bf16 tensor, through FourierMerge.merge_sources (the body of
`_merge_layer`).  Pass-through tensors (embed / norm / lm_head) are plain copies in the
reference and are not part of the timed work.

  value : whole-job merged params/s with inputs resident in HBM (device-timed, CUDA events,
          max over ranks).  N > 1: ONE model's tensor list is split over the ranks by
          shardmerge_b200.schedule.tensor_partition (longest-processing-time-first, whole tensors,
          no collective on the data path) -> strong scaling.
  e2e   : same metric through MergeTensorsBase._process_layers = FourierMerge._merge_layer +
          ModelWriter.add_tensor per tensor, on HOST (pinned) tensors: the H2D copies of base +
          finetunes, the D2H copy of every result into the writer's pinned staging and the
          safetensors shard files (tmpfs) are inside the timed region.
  roofline : dominant kernel class (column FFT sweeps): SURVEY 8(d) algorithmic bytes (8N per
          column transform, three transforms per pair) / CUDA-event time of its launches vs
          MEASURED_PEAKS.json hbm_gbs; `per_sweep` keeps the bytes the two sweeps really move.
  cpu_baseline / --impl reference : the REFERENCE ITSELF (oracle/_ref, a git-ignored copy of the
          reference's Python package: FourierMerge._merge_layer(device="cpu"),
          shard/merge/fast_fourier.py:103-276) on this box's host cores with all torch threads, on
          a bounded sample of the same workload; the numpy port only if oracle/_ref is absent.
"""
from __future__ import annotations

import argparse
import asyncio
import json
import os
import statistics
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

ARCH = {
    "tinyllama": dict(H=2048, I=5632, KV=256, L=22),
    "llama8b": dict(H=4096, I=14336, KV=1024, L=32),
    "llama70b": dict(H=8192, I=28672, KV=1024, L=80),
}
ALPHAS = (0.3, 0.5, 0.4, 0.2)
SIGMAS = (0.002, 0.0026, 0.0023, 0.0029)


def workload_name(workload, n_ft):
    return (f"{workload}-shaped base + {n_ft} finetunes (bf16), alpha {'/'.join(str(x) for x in ALPHAS[:n_ft])}, "
            "SLERP-FFT merge of every model.layers.* tensor")


def layer_tensors(a):
    H, I, KV = a["H"], a["I"], a["KV"]
    return [("self_attn.q_proj.weight", (H, H)), ("self_attn.k_proj.weight", (KV, H)),
            ("self_attn.v_proj.weight", (KV, H)), ("self_attn.o_proj.weight", (H, H)),
            ("mlp.gate_proj.weight", (I, H)), ("mlp.up_proj.weight", (I, H)), ("mlp.down_proj.weight", (H, I)),
            ("input_layernorm.weight", (H,)), ("post_attention_layernorm.weight", (H,))]


def numel(shape):
    n = 1
    for s in shape:
        n *= s
    return n


def synth_tensor(torch, shape, idx, n_ft, device):
    """SURVEY.md 8d synthetic weights, generated on `device`."""
    g = torch.Generator(device=device).manual_seed(1234 + idx)
    if len(shape) == 1:
        base = (1.0 + 0.1 * torch.randn(shape, generator=g, device=device)).to(torch.bfloat16)
        sig = [0.01 * (1 + 0.3 * k) for k in range(n_ft)]
    else:
        base = (0.02 * torch.randn(shape, generator=g, device=device)).to(torch.bfloat16)
        sig = SIGMAS
    fts = []
    for k in range(n_ft):
        gk = torch.Generator(device=device).manual_seed(100000 * (k + 1) + idx)
        fts.append((base.float() + sig[k] * torch.randn(shape, generator=gk, device=device)).to(torch.bfloat16))
    return base, fts


class ClockSampler:
    """SM clock and clock-event (throttle) reasons sampled through NVML every 10 ms during the timed region
    (B200_PROFILING.md recipe; nvidia-smi -lms is too coarse for a region of a few hundred ms)."""

    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.sm, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None

    def _loop(self, nv, h):
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons", None)
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                if get_reasons is not None:
                    bits = int(get_reasons(h))
                    for bit, name in self.REASONS.items():
                        if bits & bit:
                            self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.01)

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.gpu_index]) if vis and vis.split(",")[self.gpu_index].isdigit() else self.gpu_index
            h = nv.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self._thread = threading.Thread(target=self._loop, args=(nv, h), daemon=True)
            self._thread.start()
        except Exception:
            self._thread = None

    def stop(self):
        self._stop.set()
        if self._thread is not None:
            self._thread.join(timeout=1)
        return dict(sm_mhz=statistics.median(self.sm) if self.sm else None, sm_max_mhz=self.max_mhz,
                    reasons=sorted(self.reasons), samples=len(self.sm))


# ------------------------------------------------------------------------------------------
def cpu_port_rate(shape, n_ft, threads, repeats=1):
    """oracle merge_layer on `threads` concurrent tensors of `shape` -> (params/s, seconds)."""
    import numpy as np
    from concurrent.futures import ThreadPoolExecutor
    from oracle import oracle_np as O

    def make(i):
        rng = np.random.default_rng(1234 + i)
        base32 = (0.02 * rng.standard_normal(shape)).astype(np.float32)
        base = O.f32_to_bf16(base32)
        models = []
        for k in range(n_ft):
            ft = O.f32_to_bf16((O.bf16_to_f32(base) + SIGMAS[k] * rng.standard_normal(shape)).astype(np.float32))
            models.append(dict(base=base, ft=ft, alpha=ALPHAS[k], name=f"m{k}"))
        return base, models

    jobs = [make(i) for i in range(threads)]
    t0 = time.perf_counter()
    for _ in range(repeats):
        if threads == 1:
            O.merge_layer(*jobs[0])
        else:
            with ThreadPoolExecutor(max_workers=threads) as ex:
                list(ex.map(lambda j: O.merge_layer(*j), jobs))
    dt = time.perf_counter() - t0
    return threads * repeats * numel(shape) / dt, dt


def cpu_reference_rate(shapes, n_ft, repeats=1):
    """The unmodified reference's FourierMerge._merge_layer(device="cpu") (oracle/ref_runner.py) on one tensor per
    shape in `shapes` -> (params/s, seconds, threads, kind, per-shape seconds).  Falls back to the numpy port."""
    from oracle import ref_runner as RR
    if not RR.available():
        r, dt = cpu_port_rate(shapes[0], n_ft, 1, repeats=repeats)
        return r, dt, 1, "port", {f"{shapes[0][0]}x{shapes[0][1]}": dt}
    import torch
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    jobs = []
    for i, shape in enumerate(shapes):
        base, fts = synth_tensor(torch, shape, 7000 + i, n_ft, "cpu")
        jobs.append((shape, base, fts))
    per = {}
    t0 = time.perf_counter()
    for _ in range(repeats):
        for shape, base, fts in jobs:
            t1 = time.perf_counter()
            RR.merge_layer(base, fts, list(ALPHAS[:n_ft]), device="cpu")
            per[f"{shape[0]}x{shape[1]}"] = round(time.perf_counter() - t1, 2)
    dt = time.perf_counter() - t0
    return repeats * sum(numel(sh) for sh in shapes) / dt, dt, threads, "reference", per


def reference_sample_shapes(a):
    """one k_proj-shaped and one q_proj-shaped tensor: ~15 s of the reference on 8 host cores at Llama-8B shapes."""
    return [(a["KV"], a["H"]), (a["H"], a["H"])]


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    a = ARCH[args.workload]
    shapes = reference_sample_shapes(a)
    for _ in range(min(args.warmup, 1)):
        cpu_reference_rate(shapes[:1], args.finetunes)
    params, secs, per = 0, 0.0, {}
    for _ in range(args.steps):
        r, dt, threads, kind, per = cpu_reference_rate(shapes, args.finetunes)
        params += sum(numel(sh) for sh in shapes); secs += dt
    value = params / secs
    what = ("the reference's FourierMerge._merge_layer(device='cpu') (oracle/_ref)" if kind == "reference"
            else "numpy port of the reference (oracle/_ref absent)")
    sample = (f"per step one tensor each of {' and '.join(f'{s[0]}x{s[1]}' for s in shapes)} through {what}, "
              f"torch threads = {threads}; seconds per tensor {per}; at most one warm-up step")
    line = dict(impl="reference", metric="merged_params_per_sec", value=value, unit="params/s", n_gpus=args.gpus,
                steps=args.steps, warmup=min(args.warmup, 1), ms_per_step=1000 * secs / args.steps, higher_is_better=True,
                scaling="strong", vs_baseline=None, dtype="f32", data="synthetic",
                config=dict(workload=workload_name(args.workload, args.finetunes), sample=sample),
                cpu_baseline=dict(value=value, unit="params/s", cores=threads, kind=kind, sample=sample),
                e2e=dict(value=value, unit="params/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                gpu_launches=0)
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------
DUMP_BYTES = 60 << 20                   # sampled values of all tensors together; the .npy headers stay well inside 64 MB


def dump_outputs(torch, out_dir, outputs, catalog):
    """Write this rank's merged tensors as out_dir/<name>.npy (float32, flattened).  A tensor larger than its share of
    DUMP_BYTES is sampled at sorted flat indices drawn from a generator seeded with its catalog index, so the same
    arguments give the same positions in every run and two builds can be compared value for value."""
    import numpy as np
    out_dir.mkdir(parents=True, exist_ok=True)
    per_tensor = DUMP_BYTES // 4 // len(catalog)
    seeds = {name: idx for name, _, idx in catalog}
    total = 0
    for name, t in outputs.items():
        flat = t.reshape(-1)
        n = flat.numel()
        if n > per_tensor:
            pos = np.sort(np.random.default_rng(seeds[name]).choice(n, size=per_tensor, replace=False))
            flat = flat[torch.from_numpy(pos).to(flat.device)]
        arr = flat.float().cpu().numpy()
        np.save(out_dir / f"{name}.npy", arr)
        total += arr.nbytes
    print(f"[bench] wrote {len(outputs)} merged tensors ({total / 2**20:.1f} MiB of float32) to {out_dir}", file=sys.stderr)


# ------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="llama8b", choices=sorted(ARCH))
    ap.add_argument("--layers", type=int, default=0, help="layers of the model (0 = all L, or as many as fit on the ranks together)")
    ap.add_argument("--finetunes", type=int, default=2)
    ap.add_argument("--e2e-layers", type=int, default=8)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-files", type=int, default=1, help="0: skip the second e2e measurement that writes the shard files")
    ap.add_argument("--prefetch-depth", type=int, default=-1, help="tensors whose uploads run ahead in the e2e loop (-1: the strategy's default)")
    ap.add_argument("--profile-json", default="", help="write the per-kernel-class summary here")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the merged tensors of the last timed step to DIR/<tensor name>.npy (float32; a fixed, "
                         "seeded sample of each tensor, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl=ours) needs a CUDA device: shardmerge_b200 has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from shardmerge_b200 import engine as E
    from shardmerge_b200 import schedule
    from shardmerge_b200.config import MergeConfig, MergeModel
    from shardmerge_b200.index import InMemoryIndex
    from shardmerge_b200.merge.fast_fourier import FourierMerge
    from shardmerge_b200.writer import ModelWriter, ShardLayer

    a = ARCH[args.workload]
    M = args.finetunes
    per_layer = layer_tensors(a)
    params_layer = sum(numel(s) for _, s in per_layer)
    free_b, _ = torch.cuda.mem_get_info(dev)
    bytes_layer = params_layer * 2 * (M + 2)                      # base + M finetunes + output, bf16
    max_params = max(numel(s) for _, s in per_layer)
    ws_bytes = 5 * 4 * 4 * max_params                             # workspaces of the distinct shapes (generous)
    fit = (free_b * 0.85 - ws_bytes) / bytes_layer                # layers of this architecture one GPU can hold
    L = a["L"] if args.layers <= 0 else min(args.layers, a["L"])
    L = max(1, min(L, int(fit * world * 0.97)))                   # ONE model of L layers, split over the ranks

    # ---- the model's merged tensors, and this rank's share (whole tensors, LPT; same answer on every rank) ------
    catalog = []                                                  # (name, shape, seed index)
    for layer in range(L):
        for nm, shape in per_layer:
            catalog.append((f"model.layers.{layer}.{nm}", shape, len(catalog)))
    numels = {name: numel(shape) for name, shape, _ in catalog}
    parts = schedule.tensor_partition(numels, world, n_models=M)
    mine = set(parts[rank])
    cost = {n: schedule.merge_cost(v, M) for n, v in numels.items()}
    imbalance = schedule.imbalance(parts, cost) if world > 1 else 0.0
    tensors = []                                                  # (name, base, [fts]) resident on this rank
    for name, shape, idx in catalog:
        if name in mine:
            base, fts = synth_tensor(torch, shape, idx, M, dev)
            tensors.append((name, base, fts))
    torch.cuda.synchronize(dev)
    merged_params = sum(numels.values())                          # whole job, all ranks
    my_params = sum(numels[n] for n in mine)

    cfg = MergeConfig(finetune_merge=[MergeModel(model=f"synth/ft{k}", base="synth/base", alpha=ALPHAS[k],
                                                 is_input=(k == 0), is_output=(k == 1)) for k in range(M)],
                      output_base_model="synth/base", output_dir="/tmp/unused", device=str(dev))
    fm = FourierMerge(cfg, index_manager=InMemoryIndex({}))
    outputs = {}

    def step():
        outputs.clear()
        for name, base, fts in tensors:
            srcs = [E.make_source(base, ft, weight=ALPHAS[k], name=f"synth/ft{k}") for k, ft in enumerate(fts)]
            outputs[name] = fm.merge_sources(srcs, base, dev, layer_name=name, defer=True)
        fm.resolve_all()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x):
        if world > 1:
            t = torch.tensor([x], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return x

    for _ in range(args.warmup):
        step()
    barrier()
    # ---- timed region: production configuration (consecutive tensors spread over fm.lanes streams) -------------
    sampler = ClockSampler(local_rank)
    sampler.start()
    E.PROFILER = E.Profiler(timing=False)                          # counts launches only
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    t_wall0 = time.perf_counter()
    for s0, s1 in ev:
        s0.record(); step(); s1.record()
    barrier()
    wall = time.perf_counter() - t_wall0
    gpu_launches = E.PROFILER.launches
    E.PROFILER = None
    clocks = sampler.stop()
    if args.dump_outputs:                                         # before the serial pass below overwrites `outputs`
        dump_outputs(torch, Path(args.dump_outputs), outputs, catalog)
    elapsed_ms = max_over_ranks(sum(s0.elapsed_time(s1) for s0, s1 in ev))
    value = merged_params * args.steps / (elapsed_ms / 1000.0)
    if world > 1:
        t = torch.tensor([float(gpu_launches)], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        gpu_launches = int(t.item())

    # ---- per-kernel pass: the same steps on ONE stream with a CUDA-event pair around every kernel class ----------
    # (with several lanes the kernels of different tensors overlap, and an event pair around one of them would also
    # time its neighbours; the roofline figures therefore come from this serial pass, `value` from the region above)
    lanes_used = fm.lanes
    fm.lanes = 1
    step()
    barrier()
    E.PROFILER = E.Profiler(timing=True)
    pv = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for s0, s1 in pv:
        s0.record(); step(); s1.record()
    barrier()
    prof = E.PROFILER
    E.PROFILER = None
    fm.lanes = lanes_used
    serial_ms = sum(s0.elapsed_time(s1) for s0, s1 in pv)
    value_serial = my_params * args.steps / (serial_ms / 1000.0)

    # ---- roofline of the dominant kernel class ---------------------------------------------
    summ = prof.summary()
    peaks_path = ROOT / "MEASURED_PEAKS.json"
    if peaks_path.exists():
        peak, peak_src = float(json.loads(peaks_path.read_text())["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    col_moved = sum(summ[t]["bytes"] for t in ("col_fwd", "col_inv") if t in summ)     # what the sweeps really move
    col_ms = sum(summ[t]["ms"] for t in ("col_fwd", "col_inv") if t in summ)
    col_launch = sum(summ[t]["launches"] for t in ("col_fwd", "col_inv") if t in summ)
    # SURVEY 8(d): a column transform is 8N bytes (read + write the 4N-byte half spectrum once); a pair merge has three
    # (two forward, one inverse).  Tensors with a single sweep or none (R <= 256, 1-D) move exactly that already.
    n2d = sum(numels[n] for n in mine if len(next(sh for nm, sh, _ in catalog if nm == n)) == 2)
    col_alg = 24.0 * n2d * (M - 1) * args.steps                  # M - 1 pair merges per tensor (pair tree for M > 2)
    achieved = col_alg / (col_ms / 1000.0) / 1e9 if col_ms else None
    per_sweep = col_moved / (col_ms / 1000.0) / 1e9 if col_ms else None
    kernel_ms_total = sum(v["ms"] or 0.0 for v in summ.values())
    traffic, traffic_note = None, None
    tpath = ROOT / "profiles" / "r02_traffic.json"
    if tpath.exists():                                            # dram__bytes_read + dram__bytes_write of one captured launch
        tj = json.loads(tpath.read_text())
        traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
        traffic_note = dict(launch=tj["kernel"], algorithmic_bytes_of_that_launch=tj["algorithmic_bytes"],
                            survey_8d_bytes_of_that_launch=tj.get("algorithmic_bytes_survey_8d_share"), source=tj["source"])
    pipeline_alg = 64.0 * n2d * (M - 1) * args.steps              # SURVEY 8(d): 64N bytes per pair merge
    roofline = dict(bound="hbm", kernel="k_col_p3 / k_col_p (column FFT sweeps, forward+inverse)", achieved=achieved, peak=peak,
                    unit="GB/s", frac=(achieved / peak if achieved else None), traffic=traffic, traffic_note=traffic_note,
                    peak_source=peak_src,
                    bytes_model="SURVEY 8(d): 8N per column transform x 3 transforms per pair = 24N; the two-sweep "
                                "four-step kernels move 16N per transform (per_sweep)",
                    per_sweep=dict(gbs=per_sweep, frac=(per_sweep / peak if per_sweep else None),
                                   bytes_per_launch=(col_moved / col_launch if col_launch else None)),
                    bytes_per_launch=(col_alg / col_launch if col_launch else None),
                    share_of_kernel_time=(col_ms / kernel_ms_total if kernel_ms_total else None),
                    whole_pipeline=dict(gbs=(pipeline_alg / (serial_ms / 1000.0) / 1e9),
                                        frac=(pipeline_alg / (serial_ms / 1000.0) / 1e9 / peak),
                                        note="64N algorithmic bytes per pair merge over the serial pass"),
                    measured="CUDA events around every kernel class during a serial (one stream) pass of the same steps "
                             "inside this run (rank 0's share of the tensors); the timed region overlaps kernels of "
                             "consecutive tensors on several streams",
                    serial_pass=dict(ms_per_step=serial_ms / args.steps, params_per_s_per_gpu=value_serial),
                    per_class={k: dict(calls=v["calls"], launches=v["launches"], ms=v["ms"],
                                       gbs=(v["bytes"] / (v["ms"] / 1000.0) / 1e9 if v["ms"] else None),
                                       frac=(v["bytes"] / (v["ms"] / 1000.0) / 1e9 / peak if v["ms"] and v["bytes"] else None))
                               for k, v in summ.items()})

    # ---- e2e: host tensors through _process_layers + ModelWriter ---------------------------------
    e2e = None
    if not args.no_e2e:
        import shutil
        import tempfile
        Le = max(1, min(args.e2e_layers, L))
        # this rank's tensors among the first Le layers (the same partition as above restricted to those layers)
        e2e_catalog = [(n, sh, i) for n, sh, i in catalog if int(n.split(".")[2]) < Le]
        e2e_parts = schedule.tensor_partition({n: numel(sh) for n, sh, _ in e2e_catalog}, world, n_models=M)
        e2e_mine = set(e2e_parts[rank])
        del tensors[:]
        outputs.clear()
        E.clear_caches()
        torch.cuda.empty_cache()
        host = {"synth/base": {}, **{f"synth/ft{k}": {} for k in range(M)}}
        names = []
        for name, shape, idx in e2e_catalog:
            if name not in e2e_mine:
                continue
            base, fts = synth_tensor(torch, shape, idx, M, dev)
            host["synth/base"][name] = base.cpu().pin_memory()
            for k, ft in enumerate(fts):
                host[f"synth/ft{k}"][name] = ft.cpu().pin_memory()
            names.append(name)
            del base, fts
        # one output shard per transformer layer (as HF checkpoints roughly do), files on tmpfs when there is one
        index = InMemoryIndex(host)
        fm2 = FourierMerge(cfg, index_manager=index)
        weight_map = {n: f"model-{int(n.split('.')[2]) + 1:05d}-of-{Le:05d}.safetensors" for n in names}
        # shard files of the with_files measurement: tmpfs if it has room for the steps' output (twice over), else the default
        # temp directory, else that measurement is skipped (it must never take the bench line down)
        need_bytes = 2 * max(args.steps, 2) * sum(host["synth/base"][n].numel() * 2 for n in names)
        tmp_root, files_ok = None, False
        for cand in ("/dev/shm", tempfile.gettempdir()):
            try:
                if os.path.isdir(cand) and os.access(cand, os.W_OK) and shutil.disk_usage(cand).free > need_bytes * (world if cand == "/dev/shm" else 1):
                    tmp_root, files_ok = cand, True
                    break
            except OSError:
                pass
        out_root = Path(tempfile.mkdtemp(prefix=f"shardmerge_bench_r{rank}_", dir=tmp_root))
        h2d = sum(t.numel() * 2 for n in names for t in [host["synth/base"][n]] + [host[f"synth/ft{k}"][n] for k in range(M)])
        d2h = sum(host["synth/base"][n].numel() * 2 for n in names)
        layers_e2e = [ShardLayer(i, weight_map[n], n, False) for i, n in enumerate(names)]
        fm2.defer_checks = True                    # what MergeTensorsBase.merge() sets: checks settle one tensor behind
        pool = {}                                  # the writer's pinned pool survives from step to step, like within one merge

        writers = []

        class StagingOnlyWriter(ModelWriter):      # the whole hand-over (pinned pool, side-stream D2H, shard assembly) minus the file
            def _write_shard(self, shard_name, staged):
                with self._lock:
                    for n_ in staged:
                        self.written_shard_layers.add((shard_name, n_))

        if args.prefetch_depth >= 0:
            fm2.prefetch_depth = args.prefetch_depth
        loop = asyncio.new_event_loop()

        def measure(WriterCls, tag):
            """-> (ms until every result of every timed step sits in pinned host memory, ms until all files are complete)"""

            async def e2e_step(k):
                # the reference's hot loop (shard/merge/base.py:212-223): _merge_layer + writer.add_tensor per tensor; here
                # the uploads of the next tensors, this tensor's kernels, the previous tensor's download and the shard
                # assembly (writer threads) overlap.  The step ends when every result sits in the writer's pinned host memory.
                out = out_root / f"{tag}{k}"
                writer = WriterCls(base_index={"metadata": {}, "weight_map": weight_map}, output_path=out, layer_order=names,
                                   output_astype=torch.bfloat16, pinned_pool=pool.get("pool"), queue_depth=2 * Le,
                                   writer_threads=min(8, Le), io_threads=min(16, os.cpu_count() or 8))
                pool["pool"] = writer._pool
                await fm2._process_layers(writer, layers_e2e, str(dev))
                writer.wait_staged()
                torch.cuda.synchronize(dev)
                writers.append(writer)

            def finish_files():
                for w in writers:
                    w.finalize()                   # waits until the last shard file is complete, checks completeness
                del writers[:]

            # warm-up: as many steps as will be timed, their files finished only afterwards, so that the writer's pinned
            # pool ends up holding the staging buffers of that many steps (no cudaHostAlloc inside the timed region)
            n_warm = max(args.steps, min(args.warmup, 2), 1)
            for k in range(n_warm):
                loop.run_until_complete(e2e_step(-1 - k))
            finish_files()
            for k in range(n_warm):
                shutil.rmtree(out_root / f"{tag}{-1 - k}", ignore_errors=True)     # bench housekeeping, outside the timed region
            barrier()
            e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            e0.record()
            for k in range(args.steps):
                loop.run_until_complete(e2e_step(k))
            e1.record()
            finish_files()
            e2.record()
            barrier()
            for k in range(args.steps):
                shutil.rmtree(out_root / f"{tag}{k}", ignore_errors=True)
            return e0.elapsed_time(e1), e0.elapsed_time(e2)

        t_e2e0 = time.perf_counter()
        index.copy_events = []                     # (start, end) events of every upload: how busy the H2D copy engine is
        my_ems, _ = measure(StagingOnlyWriter, "s")
        copy_pairs, index.copy_events = index.copy_events, None
        # the last args.steps * len(uploads per step) pairs belong to the timed steps (warm-up steps come first)
        per_step = len(names) * (M + 1)
        timed = copy_pairs[-args.steps * per_step:] if per_step else []
        h2d_busy_ms = sum(a_.elapsed_time(b_) for a_, b_ in timed)
        ems = max_over_ranks(my_ems)
        ems_files = None
        if world > 1:                                   # every rank must take the same branch: all measure, or none
            t = torch.tensor([1.0 if files_ok else 0.0], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            files_ok = bool(t.item() > 0.5)
        if args.e2e_files and files_ok:
            try:
                _, my_files = measure(ModelWriter, "f")
            except Exception as exc:                    # a full file system must not take the bench line down
                print(f"[bench] with_files measurement failed: {exc}", file=sys.stderr)
                my_files = float("nan")
            ems_files = max_over_ranks(my_files)
            if ems_files != ems_files:
                ems_files = None
        e2e_wall = time.perf_counter() - t_e2e0
        shutil.rmtree(out_root, ignore_errors=True)
        # what plain pinned copies achieve on this box, both directions at once (the e2e path moves 6 B in and 2 B out
        # per merged parameter, so it is bounded by the host link, not by the kernels); all ranks probe at the same time
        pin_in = torch.empty(1 << 29, dtype=torch.uint8).pin_memory(); dev_in = torch.empty(1 << 29, dtype=torch.uint8, device=dev)
        pin_out = torch.empty(1 << 28, dtype=torch.uint8).pin_memory(); dev_out = torch.empty(1 << 28, dtype=torch.uint8, device=dev)
        s_in, s_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
        barrier()
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record()
        s_in.wait_event(p0); s_out.wait_event(p0)
        with torch.cuda.stream(s_in):
            for _ in range(2):
                dev_in.copy_(pin_in, non_blocking=True)
        with torch.cuda.stream(s_out):
            for _ in range(2):
                pin_out.copy_(dev_out, non_blocking=True)
        torch.cuda.current_stream(dev).wait_stream(s_in); torch.cuda.current_stream(dev).wait_stream(s_out)
        p1.record(); torch.cuda.synchronize(dev)
        link_ms = p0.elapsed_time(p1)
        link = dict(h2d_gbs=2 * (1 << 29) / link_ms / 1e6, d2h_gbs=2 * (1 << 28) / link_ms / 1e6,
                    note="per rank, all ranks at once: 1 GiB in + 0.5 GiB out, pinned, concurrent (the 3:1 ratio of the merge)")
        del pin_in, dev_in, pin_out, dev_out
        e2e_params = sum(numel(sh) for _, sh, _ in e2e_catalog)         # whole job
        h2d_all, d2h_all = h2d, d2h
        if world > 1:
            t = torch.tensor([float(h2d), float(d2h)], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            h2d_all, d2h_all = int(t[0].item()), int(t[1].item())
        e2e = dict(value=e2e_params * args.steps / (ems / 1000.0), unit="params/s",
                   h2d_bytes_per_step=h2d_all, d2h_bytes_per_step=d2h_all, layers=Le, host_link_probe=link,
                   h2d_gbs_achieved_rank0=h2d * args.steps / (my_ems / 1000.0) / 1e9,
                   h2d_copy_engine_rank0=dict(busy_ms=h2d_busy_ms, busy_fraction_of_timed_region=h2d_busy_ms / my_ems if my_ems else None,
                                              gbs_while_busy=(h2d * args.steps / (h2d_busy_ms / 1000.0) / 1e9) if h2d_busy_ms else None),
                   with_files=(dict(value=e2e_params * args.steps / (ems_files / 1000.0), unit="params/s",
                                    note="a second set of the same steps with the unmodified ModelWriter, timed until finalize() has "
                                         "returned for every step: all safetensors shards (one per layer) complete on "
                                         + ("tmpfs (/dev/shm)" if tmp_root == "/dev/shm" else str(tmp_root))
                                         + "; the file copies compete with the DMA for host memory bandwidth")
                               if ems_files else None),
                   wall_s=e2e_wall, prefetch_depth=fm2.prefetch_depth,
                   api="MergeTensorsBase._process_layers (FourierMerge._merge_layer + ModelWriter.add_tensor per tensor) on pinned "
                       "host tensors: H2D of base + finetunes and D2H of every merged tensor into ModelWriter's pinned staging "
                       "(pool, side stream, shard assembly on the writer threads) are inside the timed region, which ends when "
                       "the last result has arrived in host memory; `value` leaves the file system out (the shard's file write is "
                       "skipped), `with_files` is the same through the unmodified ModelWriter until the files are complete")

    # ---- CPU baseline (rank 0, N = 1 only) -----------------------------------------------------
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        shapes = reference_sample_shapes(a)
        r, dt, threads, kind, per = cpu_reference_rate(shapes, M)
        cpu_baseline = dict(value=r, unit="params/s", cores=threads, kind=kind,
                            sample=f"one tensor each of {' and '.join(f'{s[0]}x{s[1]}' for s in shapes)} through "
                                   + ("the reference's FourierMerge._merge_layer(device='cpu') (oracle/_ref)" if kind == "reference"
                                      else "oracle/oracle_np.merge_layer (numpy port; oracle/_ref absent)")
                                   + f", torch threads = {threads}, {dt:.1f} s; seconds per tensor {per}")

    if rank == 0:
        line = dict(metric="merged_params_per_sec", value=value, unit="params/s", n_gpus=world, steps=args.steps,
                    warmup=args.warmup, ms_per_step=elapsed_ms / args.steps, higher_is_better=True, scaling="strong",
                    vs_baseline=None, dtype="f32", data="synthetic",
                    merged_gb_per_s=value * 2 / 1e9,
                    config=dict(workload=workload_name(args.workload, M),
                                layers_resident=L, layers_of_model=a["L"], merged_params_per_step=merged_params,
                                tensors_per_step=len(catalog), tensors_on_rank0=len(mine),
                                l2="inputs per step and rank (%.1f GB) exceed the 126 MB L2" % (my_params * 2 * (M + 1) / 1e9),
                                partition="whole tensors, longest-processing-time-first over the ranks "
                                          "(schedule.tensor_partition), no collective on the data path",
                                partition_imbalance=imbalance, streams_per_gpu=lanes_used),
                    roofline=roofline, cpu_baseline=cpu_baseline, e2e=e2e, gpu_launches=gpu_launches, clocks=clocks,
                    wall_s=wall)
        print(json.dumps(line))
        if args.profile_json:
            Path(args.profile_json).parent.mkdir(parents=True, exist_ok=True)
            Path(args.profile_json).write_text(json.dumps(dict(summary=summ, line=line), indent=1))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
