"""A checkpoint's difference from its base as a PEFT LoRA adapter: a randomized SVD of every delta on the GPU.

For every tensor name of a base W and a model M with the same names and shapes, Δ = fp32(M) − fp32(W) (one rounded fp32
subtraction per element, the delta the merges use) and the tensor is
  - a LoRA pair when it is a 2-D `model.layers.*.weight` or `lm_head.weight` in fp32 / bf16 / fp16 and Δ is not all zero:
    lora_B [R][r'] @ lora_A [r'][C] ≈ Δ with r' = min(rank, R, C), the balanced split of a rank-r' truncated SVD
    (lora_B = U·diag(√S), lora_A = diag(√S)·Vᵀ) and lora_alpha = r', so the scaling is exactly 1;
  - a full tensor (`modules_to_save`) when its bytes differ from the base's otherwise (embeddings, norms, biases, ...);
  - omitted when it is byte-identical to the base.

The SVD is randomized (Halko, Martinsson & Tropp) with k = min(r' + oversample, R, C) columns: Ω [C][k] from `omega`,
Y = Δ Ω; `power_iters` times Q = orth(Y), Q₂ = orth((QᵀΔ)ᵀ), Y = Δ Q₂; then Q = orth(Y), Bm = QᵀΔ, and the SVD of Bm as a
QR of Bmᵀ plus a k×k SVD.  The products with Δ are csrc/kernels_lowrank.cu (Δ formed on load, fp32 FMA); the
orthonormalisations and the small SVD are torch.linalg.
"""
from __future__ import annotations

import argparse
import asyncio
import contextlib
import hashlib
import math
import re
import sys
import time
from pathlib import Path
from typing import Dict, Optional, Tuple

import torch

from . import _lib, lora
from . import engine as E
from .index import LocalSafetensorsIndex

INDEX_FILE = "model.safetensors.index.json"
FACTOR_DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}
_LORA_TENSOR = re.compile(r"^(model\.layers\..+\.weight|lm_head\.weight)$")
_PREFETCH_AHEAD = 2          # tensors whose reads and uploads run ahead of the one being factorised


# ---- the kernels -----------------------------------------------------------------------------------------------------
def _operands(W: torch.Tensor, M: torch.Tensor, S: torch.Tensor, what: str) -> Tuple[int, int, int]:
    if W.device.type != "cuda" or M.device != W.device or S.device != W.device:
        raise RuntimeError(f"{what} needs W, M and its fp32 operand on one CUDA device (got {W.device}, {M.device}, "
                           f"{S.device}); there is no CPU path")
    if W.dtype not in lora._DTYPE_CODE or M.dtype not in lora._DTYPE_CODE:
        raise NotImplementedError(f"{what}: W and M in fp32 / bf16 / fp16 (got {W.dtype}, {M.dtype})")
    if W.ndim != 2 or W.shape != M.shape:
        raise ValueError(f"{what}: W and M are 2-D of one shape (got {tuple(W.shape)}, {tuple(M.shape)})")
    if S.dtype != torch.float32 or S.ndim != 2 or S.shape[1] < 1 or not S.is_contiguous():
        raise ValueError(f"{what}: the small operand is a contiguous fp32 [L][k] tensor with k >= 1")
    R, C = W.shape
    return int(R), int(C), int(S.shape[1])


def _workspace(R: int, C: int, k: int, device) -> torch.Tensor:
    return torch.empty(max(int(_lib.load().sm_lowrank_ws_bytes(R, C, k)), 16), dtype=torch.uint8, device=device)


def lowrank_right(W: torch.Tensor, M: torch.Tensor, X: torch.Tensor, *, sumsq: bool = False,
                  ws: Optional[torch.Tensor] = None):
    """(Y, s): Y [R][k] = Δ @ X in fp32 for X [C][k] fp32, Δ = fp32(M) − fp32(W); s is Σ fp32(δ²) summed in fp64 as a
    0-dim fp64 device tensor when `sumsq`, else None.  Enqueued on the current stream (sm_lowrank_right)."""
    R, C, k = _operands(W, M, X, "lowrank_right")
    if X.shape[0] != C:
        raise ValueError(f"lowrank_right: X is [C={C}][k], got {tuple(X.shape)}")
    W, M = W.contiguous(), M.contiguous()
    ws = _workspace(R, C, k, W.device) if ws is None else ws
    Y = torch.empty((R, k), dtype=torch.float32, device=W.device)
    s = torch.empty((), dtype=torch.float64, device=W.device) if sumsq else None
    rc = _lib.load().sm_lowrank_right(R, C, k, lora._DTYPE_CODE[W.dtype], W.data_ptr(), lora._DTYPE_CODE[M.dtype],
                                      M.data_ptr(), X.data_ptr(), Y.data_ptr(), None if s is None else s.data_ptr(),
                                      ws.data_ptr(), ws.numel(), E._stream(W.device))
    _lib.check(rc, "sm_lowrank_right")
    return Y, s


def lowrank_left(W: torch.Tensor, M: torch.Tensor, Q: torch.Tensor, *, ws: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Z [k][C] = Qᵀ @ Δ in fp32 for Q [R][k] fp32, Δ = fp32(M) − fp32(W).  Enqueued on the current stream
    (sm_lowrank_left)."""
    R, C, k = _operands(W, M, Q, "lowrank_left")
    if Q.shape[0] != R:
        raise ValueError(f"lowrank_left: Q is [R={R}][k], got {tuple(Q.shape)}")
    W, M = W.contiguous(), M.contiguous()
    ws = _workspace(R, C, k, W.device) if ws is None else ws
    Z = torch.empty((k, C), dtype=torch.float32, device=W.device)
    rc = _lib.load().sm_lowrank_left(R, C, k, lora._DTYPE_CODE[W.dtype], W.data_ptr(), lora._DTYPE_CODE[M.dtype],
                                     M.data_ptr(), Q.data_ptr(), Z.data_ptr(), ws.data_ptr(), ws.numel(),
                                     E._stream(W.device))
    _lib.check(rc, "sm_lowrank_left")
    return Z


# ---- the randomized SVD ----------------------------------------------------------------------------------------------
def omega(name: str, C: int, k: int, seed: int = 0) -> torch.Tensor:
    """The Gaussian test matrix Ω [C][k] (fp32, CPU) of tensor `name`: drawn from a generator seeded by (seed,
    sha256(name)), so it depends on neither the order in which tensors are processed nor the device."""
    digest = hashlib.sha256(str(int(seed)).encode() + b":" + hashlib.sha256(name.encode()).digest()).digest()
    g = torch.Generator().manual_seed(int.from_bytes(digest[:8], "little") >> 1)
    return torch.randn((C, k), generator=g, dtype=torch.float32)


def _orth(Y: torch.Tensor) -> torch.Tensor:
    return torch.linalg.qr(Y).Q.contiguous()            # the kernels take row-major operands; LAPACK's Q is column-major


class _Spans:
    """CUDA-event spans per phase, summed at the end (only when timings are asked for)."""

    def __init__(self):
        self.spans: Dict[str, list] = {}

    @contextlib.contextmanager
    def __call__(self, phase: str):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        yield
        e1.record()
        self.spans.setdefault(phase, []).append((e0, e1))

    def seconds(self) -> Dict[str, float]:
        torch.cuda.synchronize()
        return {p: sum(a.elapsed_time(b) for a, b in v) / 1e3 for p, v in self.spans.items()}


def _no_span(phase: str):
    return contextlib.nullcontext()


def _factorize(W, M, r, oversample, power_iters, Om, span=_no_span):
    """lora_A [r'][C], lora_B [R][r'] (fp32, device), the singular values S [k] and ‖Δ‖² (0-dim fp64, device)."""
    R, C = W.shape
    rr = min(r, R, C)
    ws = _workspace(R, C, Om.shape[1], W.device)
    with span("kernels"):
        Y, norm2 = lowrank_right(W, M, Om, sumsq=True, ws=ws)
    for _ in range(power_iters):
        with span("linalg"):
            Q = _orth(Y)
        with span("kernels"):
            Z = lowrank_left(W, M, Q, ws=ws)
        with span("linalg"):
            Q2 = _orth(Z.T)
        with span("kernels"):
            Y, _ = lowrank_right(W, M, Q2, ws=ws)
    with span("linalg"):
        Q = _orth(Y)
    with span("kernels"):
        Bm = lowrank_left(W, M, Q, ws=ws)
    with span("linalg"):
        Qb, Rb = torch.linalg.qr(Bm.T)               # Bm = Rbᵀ Qbᵀ
        Us, S, Vh = torch.linalg.svd(Rb.T)           # Rbᵀ = Us diag(S) Vh
        root = S[:rr].sqrt()
        B = (Q @ Us[:, :rr]) * root
        A = (root[:, None] * (Vh[:rr] @ Qb.T)).contiguous()
    return A, B, S, norm2


def _residual(norm2: float, S: torch.Tensor, rr: int) -> float:
    if not norm2 > 0.0:
        return 0.0
    kept = float((S[:rr].double() ** 2).sum())
    return math.sqrt(max(0.0, norm2 - kept) / norm2)


# ---- checkpoints in, adapter out -------------------------------------------------------------------------------------
def _sample(names, n: int = 4) -> str:
    names = sorted(names)
    return ", ".join(names[:n]) + (f", ... ({len(names)} in all)" if len(names) > n else "")


def _check_inputs(base_dir: Path, model_dir: Path, output_dir: Path, rank, dtype, oversample, power_iters):
    if int(rank) < 1:
        raise ValueError(f"extract_lora: rank must be >= 1 (got {rank})")
    if int(oversample) < 0 or int(power_iters) < 0:
        raise ValueError(f"extract_lora: oversample and power_iters must be >= 0 (got {oversample}, {power_iters})")
    if dtype not in FACTOR_DTYPES.values():
        raise ValueError(f"extract_lora: factor dtype fp32, bf16 or fp16 (got {dtype})")
    for what, d in (("base", base_dir), ("model", model_dir)):
        if not (d / INDEX_FILE).is_file():
            kind = "a LoRA adapter, not a full checkpoint" if lora.is_adapter_dir(d) else "not a full checkpoint"
            raise FileNotFoundError(f"extract_lora: {what} {d} has no {INDEX_FILE} ({kind})")
    if output_dir.exists() and (not output_dir.is_dir() or any(output_dir.iterdir())):
        raise FileExistsError(f"extract_lora: {output_dir} exists and is not an empty directory")


def extract_lora(base_dir, model_dir, output_dir, rank: int, *, dtype: torch.dtype = torch.float32, oversample: int = 8,
                 power_iters: int = 2, seed: int = 0, device="cuda:0",
                 timings: Optional[Dict[str, float]] = None) -> Dict[str, float]:
    """Write the difference of the checkpoint `model_dir` from `base_dir` as a PEFT LoRA adapter at `output_dir` (see the
    module docstring) with factors in `dtype` (fp32, bf16 or fp16) and return, for every LoRA pair, the relative residual
    sqrt(max(0, ‖Δ‖² − Σ_{i≤r'} S_i²)) / ‖Δ‖ of its rank-r' truncation, ‖Δ‖² accumulated in fp64.  The difference of two
    fp32 sums, it is accurate only to about 1e-3 absolute.

    Both directories hold `model.safetensors.index.json` (a merge's output does) with the same tensor names and shapes.
    Refused before any device work: rank < 1, oversample or power_iters < 0, a directory without that index (an adapter
    directory included), differing names or shapes (ValueError), an `output_dir` that exists and is not empty
    (FileExistsError).  A NaN or Inf in a Δ raises ValueError naming the tensor.  `output_dir` appears complete or not at
    all.  `timings`, if given, receives seconds spent waiting for file reads, in the kernels, in torch.linalg, writing,
    and in all."""
    base_dir, model_dir, output_dir = Path(base_dir).resolve(), Path(model_dir).resolve(), Path(output_dir).resolve()
    _check_inputs(base_dir, model_dir, output_dir, rank, dtype, oversample, power_iters)
    index = LocalSafetensorsIndex(base_dir.parent)      # storage_dir / "/abs/path" is the absolute path itself
    base_uri, model_uri = str(base_dir), str(model_dir)
    asyncio.run(index.add_model(base_uri))
    asyncio.run(index.add_model(model_uri))
    base_keys, model_keys = index.get_model_keys(base_uri), index.get_model_keys(model_uri)
    if base_keys != model_keys:
        raise ValueError(f"extract_lora: tensor names differ; only in the base: [{_sample(base_keys - model_keys)}]; "
                         f"only in the model: [{_sample(model_keys - base_keys)}]")
    base_shapes, model_shapes = index.tensor_shapes(base_uri), index.tensor_shapes(model_uri)
    for name in sorted(base_keys):
        if tuple(base_shapes[name]) != tuple(model_shapes[name]):
            raise ValueError(f"extract_lora: {name} has shape {tuple(base_shapes[name])} in the base, "
                             f"{tuple(model_shapes[name])} in the model")

    dev = E._require_cuda(device)
    t_start = time.perf_counter()
    spans = _Spans() if timings is not None else None
    clock = {"read_wait": 0.0}
    tensors: Dict[str, object] = {}
    residuals: Dict[str, float] = {}
    order = index.get_layer_order(base_uri)

    async def run():
        ahead = 0
        for i, name in enumerate(order):
            while ahead < len(order) and ahead <= i + _PREFETCH_AHEAD:
                index.prefetch(base_uri, order[ahead], str(dev))
                index.prefetch(model_uri, order[ahead], str(dev))
                ahead += 1
            t0 = time.perf_counter()
            W = await index.get_tensor(base_uri, name, device=str(dev)).get()
            M = await index.get_tensor(model_uri, name, device=str(dev)).get()
            clock["read_wait"] += time.perf_counter() - t0
            _one(name, W, M)

    def _one(name, W, M):
        if W.dtype == M.dtype and torch.equal(W.reshape(-1).view(torch.uint8), M.reshape(-1).view(torch.uint8)):
            return                                                        # byte-identical: omitted
        floats = W.dtype.is_floating_point and M.dtype.is_floating_point
        if (_LORA_TENSOR.match(name) and W.ndim == 2 and W.dtype in lora._DTYPE_CODE and M.dtype in lora._DTYPE_CODE):
            R, C = W.shape
            rr = min(int(rank), R, C)
            Om = omega(name, C, min(rr + int(oversample), R, C), seed).to(dev, non_blocking=True)
            A, B, S, norm2 = _factorize(W, M, int(rank), int(oversample), int(power_iters), Om,
                                        spans if spans is not None else _no_span)
            n2 = float(norm2)
            if not math.isfinite(n2):
                d = M.float() - W.float()
                if not bool(torch.isfinite(d).all()):
                    raise ValueError(f"extract_lora: the difference of {name} holds NaN or Inf")
                n2 = float(d.double().square().sum())                   # fp32 squares overflowed; Δ itself is finite
            if n2 > 0.0 or not torch.equal(M.float(), W.float()):
                tensors[name] = (A.to(dtype).cpu(), B.to(dtype).cpu())
                residuals[name] = _residual(n2, S, rr)
                return
        elif floats and not bool(torch.isfinite(M.float() - W.float()).all()):
            raise ValueError(f"extract_lora: the difference of {name} holds NaN or Inf")
        tensors[name] = M.contiguous().cpu()                              # stored whole

    with torch.cuda.device(dev):
        asyncio.run(run())
        torch.cuda.synchronize(dev)
        t_write = time.perf_counter()
        lora.save_adapter(output_dir, tensors, {"r": int(rank), "base_model_name_or_path": str(base_dir)})
        if timings is not None:
            timings.update(spans.seconds())
            timings.update({"read_wait": clock["read_wait"], "write": time.perf_counter() - t_write,
                            "total": time.perf_counter() - t_start})
    return residuals


def main(argv=None) -> int:
    p = argparse.ArgumentParser(prog="python -m shardmerge_b200.extract",
                                description="Write a checkpoint's difference from its base as a PEFT LoRA adapter.")
    p.add_argument("base", help="base checkpoint directory (with model.safetensors.index.json)")
    p.add_argument("model", help="finetuned or merged checkpoint directory with the same tensors")
    p.add_argument("out", help="adapter directory to create (absent or empty)")
    p.add_argument("--rank", type=int, required=True)
    p.add_argument("--dtype", choices=sorted(FACTOR_DTYPES), default="fp32", help="dtype of lora_A / lora_B")
    p.add_argument("--device", default="cuda:0")
    p.add_argument("--oversample", type=int, default=8)
    p.add_argument("--power-iters", type=int, default=2)
    p.add_argument("--seed", type=int, default=0)
    a = p.parse_args(argv)
    res = extract_lora(a.base, a.model, a.out, a.rank, dtype=FACTOR_DTYPES[a.dtype], oversample=a.oversample,
                       power_iters=a.power_iters, seed=a.seed, device=a.device)
    print(f"wrote {a.out}: {len(res)} LoRA pairs at rank {a.rank}")
    for name, r in sorted(res.items(), key=lambda kv: -kv[1])[:10]:
        print(f"  residual {r:.4f}  {name}")
    return 0


if __name__ == "__main__":
    sys.exit(main())
