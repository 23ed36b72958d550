"""numpy restatement of the TIES / DARE merges (DESIGN.md section 8, csrc/kernels_sparse.cu), the reference the tests
compare the device's bits against.  float32 throughout: one IEEE rounding per numpy operation (numpy never contracts
a * b + c into an FMA), sums in ascending model order starting from +0.0."""
from __future__ import annotations

import hashlib

import numpy as np

PHILOX_M = (np.uint64(0xD2511F53), np.uint64(0xCD9E8D57))
PHILOX_W = (0x9E3779B9, 0xBB67AE85)
MODES = ("ties", "dare_ties", "dare_linear")


def philox4x32_10(ctr, key):
    """Philox4x32-10 (Salmon et al. 2011, Random123 constants).  ctr: 4 uint32 arrays (broadcastable), key: (k0, k1).
    Returns the 4 output words as uint32 arrays."""
    c = [np.asarray(x, dtype=np.uint64) & np.uint64(0xFFFFFFFF) for x in ctr]
    k0, k1 = int(key[0]) & 0xFFFFFFFF, int(key[1]) & 0xFFFFFFFF
    mask = np.uint64(0xFFFFFFFF)
    for r in range(10):
        if r:
            k0, k1 = (k0 + PHILOX_W[0]) & 0xFFFFFFFF, (k1 + PHILOX_W[1]) & 0xFFFFFFFF
        p0, p1 = PHILOX_M[0] * c[0], PHILOX_M[1] * c[2]
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & mask, p1 >> np.uint64(32), p1 & mask
        c = [hi1 ^ c[1] ^ np.uint64(k0), lo1, hi0 ^ c[3] ^ np.uint64(k1), lo0]
    return [x.astype(np.uint32) for x in c]


def dare_key(seed: int, model_index: int, tensor_name: str):
    """(k0, k1): the first 8 bytes of sha256(f"{seed}/{i}/{name}"), little-endian, k0 = the low word."""
    v = int.from_bytes(hashlib.sha256(f"{seed}/{model_index}/{tensor_name}".encode()).digest()[:8], "little")
    return v & 0xFFFFFFFF, v >> 32


def keep24(density: float) -> int:
    return int(density * 2 ** 24)


def dare_keep_mask(n: int, density: float, seed: int, model_index: int, tensor_name: str) -> np.ndarray:
    """Element j is kept iff (word j & 3 of Philox at counter (c lo, c hi, 0, 0), c = j >> 2) >> 8 < int(density * 2^24)."""
    c = np.arange((n + 3) // 4, dtype=np.uint64)
    zero = np.zeros_like(c)
    words = np.stack(philox4x32_10((c & np.uint64(0xFFFFFFFF), c >> np.uint64(32), zero, zero),
                                   dare_key(seed, model_index, tensor_name)), axis=1).reshape(-1)[:n]
    return (words >> np.uint32(8)) < np.uint32(keep24(density))


def magnitude_keep_mask(d: np.ndarray, k: int) -> np.ndarray:
    """The k entries of largest |d| (by the fp32 bit pattern with the sign cleared), ties to the lower flat index."""
    d = np.ascontiguousarray(d, dtype=np.float32).reshape(-1)
    mag = (d.view(np.uint32) & np.uint32(0x7FFFFFFF)).astype(np.int64)
    order = np.argsort(-mag, kind="stable")
    keep = np.zeros(d.size, dtype=bool)
    keep[order[:k]] = True
    return keep


def magnitude_threshold(d: np.ndarray, k: int):
    """(K, J) of magnitude_keep_mask: kept iff mag > K or (mag == K and j <= J); k = 0 gives (0xffffffff, -1)."""
    d = np.ascontiguousarray(d, dtype=np.float32).reshape(-1)
    if k == 0:
        return 0xFFFFFFFF, -1
    mag = (d.view(np.uint32) & np.uint32(0x7FFFFFFF)).astype(np.int64)
    j = int(np.argsort(-mag, kind="stable")[k - 1])
    return int(mag[j]), j


def f32(x) -> np.float32:
    return np.float32(x)


def ties_family_merge(mode: str, base: np.ndarray, fts, weights, density: float, scale: float = 1.0, seed: int = 0,
                      tensor_name: str = "", model_indices=None) -> np.ndarray:
    """The merged tensor in fp32, before the rounding to the base's dtype (round_to below).  base and fts: float32 arrays
    holding the exact values of the stored tensors; model_indices: each model's position in finetune_merge (keys DARE)."""
    assert mode in MODES
    W = np.ascontiguousarray(base, dtype=np.float32).reshape(-1)
    n = W.size
    idx = list(range(len(fts))) if model_indices is None else list(model_indices)
    v = []
    for i, (F, w) in zip(idx, zip(fts, weights)):
        d = np.ascontiguousarray(F, dtype=np.float32).reshape(-1) - W
        if mode == "ties":
            t = np.where(magnitude_keep_mask(d, int(density * n)), d, f32(0))
        else:
            t = np.where(dare_keep_mask(n, density, seed, i, tensor_name), d / f32(density), f32(0))
        v.append(f32(w) * t)
    S = np.zeros(n, dtype=np.float32)
    for vi in v:
        S = S + vi
    pos = S >= f32(0)
    m = np.zeros(n, dtype=np.float32)
    D = np.zeros(n, dtype=np.float32)
    for vi, w in zip(v, weights):
        mask = np.ones(n, dtype=bool) if mode == "dare_linear" else np.where(pos, vi > 0, vi < 0)
        m = m + np.where(mask, vi, f32(0))
        D = D + np.where(mask, f32(w), f32(0))
    D = np.where(D == f32(0), f32(1), D)
    return (W + f32(scale) * (m / D)).reshape(np.shape(base))


def round_to(x: np.ndarray, dtype: str) -> np.ndarray:
    """Round-to-nearest-even of fp32 values to 'float32' / 'float16' / 'bfloat16', returned as the stored bit patterns
    (uint32 / uint16 / uint16)."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    if dtype == "float32":
        return x.view(np.uint32)
    if dtype == "float16":
        return x.astype(np.float16).view(np.uint16)
    u = x.view(np.uint32).astype(np.uint64)
    r = ((u + np.uint64(0x7FFF) + ((u >> np.uint64(16)) & np.uint64(1))) >> np.uint64(16)).astype(np.uint16)
    nan = (u & np.uint64(0x7FFFFFFF)) > np.uint64(0x7F800000)
    return np.where(nan, ((u >> np.uint64(16)) | np.uint64(0x40)).astype(np.uint16), r)
