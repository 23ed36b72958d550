// kernels_sparse.cu -- the task-vector merges TIES (Yadav et al. 2023) and DARE (Yu et al. 2023): per-model sparsification
// of the deltas d_i = fp32(F_i) - fp32(W), a weighted sign-elected (or plain) disjoint mean, added back onto the base.
// DESIGN.md section 8 states the definition; tests/sparse_oracle.py restates it in numpy and the GPU tests compare bits.
//
//   select (TIES only): per model, the exact k-th largest delta magnitude with ties taken by the lower flat index, as a
//          key K_i and a last kept index J_i: element j of model i is kept iff |d|bits > K_i || (|d|bits == K_i && j <= J_i).
//          Three radix passes over the flipped 31-bit magnitude key (0x7fffffff - |d|bits, so that ascending key order is
//          the descending magnitude order) fill the histograms of up to 8 models per launch from one read of the base;
//          sel_pick_digit (select_core.cuh) picks each model's digit; a fourth pass counts the elements equal to K_i per
//          tile of kTile elements, and one CTA per model scans those counts and finds J_i inside its tile.  k depends only
//          on n, so nothing is read back to the host in between.
//   merge: one streaming pass over W and every F_i that re-forms d_i, keeps it by the thresholds or by a Philox4x32-10
//          mask keyed per (seed, model, tensor), weights, elects the sign, takes the disjoint mean, scales, adds the base
//          and rounds to W's dtype.  Non-finite deltas are counted per model.
//
// Every fp32 operation is one IEEE rounding (explicit __f*_rn intrinsics: no contraction).  Inputs are fp32, bf16 or fp16
// each; all tensors 16-byte aligned; any n (the last partial group of 8 is read element by element); 64-bit indices.
#include <algorithm>
#include "sm_internal.h"
#include "elem_codec.cuh"
#include "select_core.cuh"

namespace {

constexpr int kMaxModels = SM_SPARSE_MAX_MODELS;
constexpr int kGroup = 8;                // models whose histograms one select launch fills (8 x 8 KB of shared memory)
constexpr int kTile = 16384;             // elements per tie-count tile
constexpr int kThreads = 256;

// 8 adjacent elements j0..j0+7 of a tensor of dtype DT (-1: dtype given at run time), zeros past n
template <int DT>
__device__ __forceinline__ void load8(int dt, const void* p, size_t j0, size_t n, float (&f)[8]) {
  const int d = DT >= 0 ? DT : dt;
  if (j0 + 8 <= n) {
    if (d == 0) ElemCodec<0>::load8(p, j0, f);
    else if (d == 1) ElemCodec<1>::load8(p, j0, f);
    else ElemCodec<2>::load8(p, j0, f);
  } else {
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const size_t j = j0 + e;
      f[e] = 0.f;
      if (j < n) f[e] = d == 0 ? ElemCodec<0>::load(p, j) : (d == 1 ? ElemCodec<1>::load(p, j) : ElemCodec<2>::load(p, j));
    }
  }
}

template <int DT>
__device__ __forceinline__ void store8(int dt, void* p, size_t j0, size_t n, const float (&o)[8]) {
  const int d = DT >= 0 ? DT : dt;
  if (j0 + 8 <= n) {
    if (d == 0) ElemCodec<0>::store8(p, j0, o);
    else if (d == 1) ElemCodec<1>::store8(p, j0, o);
    else ElemCodec<2>::store8(p, j0, o);
  } else {
    for (int e = 0; e < 8 && j0 + e < n; ++e) {
      if (d == 0) ElemCodec<0>::store(p, j0 + e, o[e]);
      else if (d == 1) ElemCodec<1>::store(p, j0 + e, o[e]);
      else ElemCodec<2>::store(p, j0 + e, o[e]);
    }
  }
}

__device__ __forceinline__ unsigned int magbits(float d) { return __float_as_uint(d) & 0x7fffffffu; }

struct Thr { unsigned int key; unsigned int status; long long last; };     // sm_sparse_thr
static_assert(sizeof(Thr) == sizeof(sm_sparse_thr), "sm_sparse_thr layout");

struct SelArgs {
  const void* base; const void* ft[kMaxModels]; unsigned char ft_dt[kMaxModels];
  int base_dt, M; size_t n;
  SelState* st; unsigned int* hist; unsigned int* counts; size_t n_tiles; Thr* thr;
};

// ---------------------------------------------------------------- select: one radix digit of every model of a group
template <int DT>
__global__ void __launch_bounds__(kThreads) k_sparse_hist(const __grid_constant__ SelArgs a, int pass) {
  extern __shared__ unsigned int sh[];                 // [kGroup][kHistBins]
  const int g0 = blockIdx.y * kGroup, G = min(kGroup, a.M - g0);
  for (int i = threadIdx.x; i < G * kHistBins; i += blockDim.x) sh[i] = 0u;
  unsigned int prefix[kGroup];
#pragma unroll
  for (int g = 0; g < kGroup; ++g) prefix[g] = g < G ? a.st[g0 + g].prefix : 0u;
  __syncthreads();
  const size_t n8 = (a.n + 7) / 8, stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += stride) {
    float b[8];
    load8<DT>(a.base_dt, a.base, i * 8, a.n, b);
    const int valid = (int)min((size_t)8, a.n - i * 8);
#pragma unroll
    for (int g = 0; g < kGroup; ++g) {
      if (g >= G) break;
      float f[8];
      load8<DT>(a.ft_dt[g0 + g], a.ft[g0 + g], i * 8, a.n, f);
      unsigned int* h = sh + g * kHistBins;
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        if (e >= valid) break;
        const unsigned int key = 0x7fffffffu - magbits(__fsub_rn(f[e], b[e]));
        if (pass == 0) atomicAdd(&h[key >> 20], 1u);
        else if (pass == 1) { if ((key >> 20) == (prefix[g] >> 20)) atomicAdd(&h[(key >> 10) & 1023u], 1u); }
        else { if ((key >> 10) == (prefix[g] >> 10)) atomicAdd(&h[key & 1023u], 1u); }
      }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < G * kHistBins; i += blockDim.x)
    if (sh[i]) atomicAdd(&a.hist[(size_t)g0 * kHistBins + i], sh[i]);
}

__global__ void k_sparse_init(SelState* st, int M, unsigned long long rank) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < M) {
    SelState s{};
    s.rank = rank; s.hi = 0x7fffffffu;
    st[i] = s;
  }
}

// one CTA of 1024 threads per model
__global__ void __launch_bounds__(1024) k_sparse_pick(unsigned int* hist, SelState* st, int pass) {
  sel_pick_digit(hist + (size_t)blockIdx.x * kHistBins, st + blockIdx.x, pass, pass == 2 ? PICK_FINISH : PICK_NONE, nullptr);
}

// ---------------------------------------------------------------- select: elements equal to the statistic, per tile
template <int DT>
__global__ void __launch_bounds__(kThreads) k_sparse_ties(const __grid_constant__ SelArgs a) {
  __shared__ unsigned int s_key[kMaxModels], s_cnt[kMaxModels];
  for (int m = threadIdx.x; m < a.M; m += blockDim.x) s_key[m] = 0x7fffffffu - a.st[m].prefix;
  const int lane = threadIdx.x & 31;
  for (size_t tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    for (int m = threadIdx.x; m < a.M; m += blockDim.x) s_cnt[m] = 0u;
    __syncthreads();
    // every thread runs the same trip count, so the warp ballots below see all 32 lanes
    for (int step = 0; step < kTile / (8 * kThreads); ++step) {
      const size_t j0 = tile * kTile + (size_t)step * 8 * kThreads + threadIdx.x * 8;
      const int valid = j0 < a.n ? (int)min((size_t)8, a.n - j0) : 0;
      float b[8];
      if (valid) load8<DT>(a.base_dt, a.base, j0, a.n, b);
      for (int m = 0; m < a.M; ++m) {
        unsigned int c = 0u;
        if (valid) {
          float f[8];
          load8<DT>(a.ft_dt[m], a.ft[m], j0, a.n, f);
#pragma unroll
          for (int e = 0; e < 8; ++e) c += (e < valid && magbits(__fsub_rn(f[e], b[e])) == s_key[m]) ? 1u : 0u;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
        if (lane == 0 && c) atomicAdd(&s_cnt[m], c);
      }
    }
    __syncthreads();
    for (int m = threadIdx.x; m < a.M; m += blockDim.x) a.counts[(size_t)m * a.n_tiles + tile] = s_cnt[m];
    __syncthreads();
  }
}

// exclusive block scan of one value per thread (1024 threads); returns the block total through *total
__device__ __forceinline__ unsigned long long block_excl_scan(unsigned long long v, unsigned long long* total) {
  __shared__ unsigned long long wsum[32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  unsigned long long incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned long long x = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += x;
  }
  if (lane == 31) wsum[wid] = incl;
  __syncthreads();
  if (wid == 0) {
    const unsigned long long w = wsum[lane];
    unsigned long long wi = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long x = __shfl_up_sync(0xffffffffu, wi, o);
      if (lane >= o) wi += x;
    }
    wsum[lane] = wi - w;
    if (lane == 31) *total = wi;
  }
  __syncthreads();
  const unsigned long long r = wsum[wid] + incl - v;
  __syncthreads();
  return r;
}

// one CTA of 1024 threads per model: the (rank + 1)-th element equal to the statistic, in index order, is the last kept
template <int DT>
__global__ void __launch_bounds__(1024) k_sparse_resolve(const __grid_constant__ SelArgs a) {
  __shared__ unsigned long long s_total;
  __shared__ long long s_tile, s_last;
  __shared__ unsigned long long s_rank;
  const int m = blockIdx.x;
  const SelState* st = a.st + m;
  const unsigned int key = 0x7fffffffu - st->prefix;
  const unsigned long long rank = st->rank;            // ties in index order that precede the last kept one
  const unsigned int* cnt = a.counts + (size_t)m * a.n_tiles;
  if (threadIdx.x == 0) { s_tile = -1; s_last = -1; }
  // tiles: each thread sums a contiguous run of them
  const size_t per = (a.n_tiles + blockDim.x - 1) / blockDim.x;
  const size_t t0 = min(a.n_tiles, per * threadIdx.x), t1 = min(a.n_tiles, t0 + per);
  unsigned long long mine = 0ull;
  for (size_t t = t0; t < t1; ++t) mine += cnt[t];
  const unsigned long long before = block_excl_scan(mine, &s_total);
  if (rank >= before && rank < before + mine) {
    unsigned long long acc = before;
    for (size_t t = t0; t < t1; ++t) {
      if (rank < acc + cnt[t]) { s_tile = (long long)t; s_rank = rank - acc; break; }
      acc += cnt[t];
    }
  }
  __syncthreads();
  if (s_tile >= 0) {
    // inside the tile: kTile / 1024 = 16 consecutive elements per thread
    const size_t j0 = (size_t)s_tile * kTile + (size_t)threadIdx.x * (kTile / 1024);
    float b[8], f[8];
    unsigned int c = 0u;
    unsigned int hit = 0u;                              // bit e: element j0 + e equals the statistic
#pragma unroll
    for (int h = 0; h < kTile / 1024; h += 8) {
      if (j0 + h < a.n) {
        load8<DT>(a.base_dt, a.base, j0 + h, a.n, b);
        load8<DT>(a.ft_dt[m], a.ft[m], j0 + h, a.n, f);
#pragma unroll
        for (int e = 0; e < 8; ++e)
          if (j0 + h + e < a.n && magbits(__fsub_rn(f[e], b[e])) == key) { hit |= 1u << (h + e); ++c; }
      }
    }
    unsigned long long tot;
    const unsigned long long pre = block_excl_scan(c, &tot);
    const unsigned long long r = s_rank;
    if (r >= pre && r < pre + c) {
      unsigned long long q = r - pre;
      for (int e = 0; e < kTile / 1024; ++e)
        if ((hit >> e) & 1u) { if (q == 0ull) { s_last = (long long)(j0 + e); break; } --q; }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    Thr t;
    t.key = key; t.last = s_last;
    t.status = (st->status != 0u || s_last < 0) ? 1u : 0u;
    a.thr[m] = t;
  }
}

__global__ void k_sparse_keep_none(Thr* thr, int M) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < M) { Thr t; t.key = 0xffffffffu; t.status = 0u; t.last = -1; thr[i] = t; }
}

// ---------------------------------------------------------------- merge
// Philox4x32-10 (Salmon, Moraes, Dror & Shaw 2011), the Random123 round and key-schedule constants
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r) { k.x += 0x9E3779B9u; k.y += 0xBB67AE85u; }
    const unsigned int lo0 = 0xD2511F53u * c.x, hi0 = __umulhi(0xD2511F53u, c.x);
    const unsigned int lo1 = 0xCD9E8D57u * c.z, hi1 = __umulhi(0xCD9E8D57u, c.z);
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
  }
  return c;
}

struct MergeArgs {
  const void* base; const void* ft[kMaxModels]; unsigned char ft_dt[kMaxModels];
  float w[kMaxModels]; uint2 key[kMaxModels];
  const Thr* thr; unsigned int* nonfinite; void* out;
  size_t n; int M, base_dt; float density, scale; unsigned int keep24;
};

enum { MODE_TIES = 0, MODE_DARE_TIES = 1, MODE_DARE_LINEAR = 2 };

// v_i = fp32(w_i) * t_i for the 8 elements j0..j0+7 of model m, given d = its deltas; counts non-finite deltas
template <int MODE>
__device__ __forceinline__ void weighted8(const MergeArgs& a, int m, size_t j0, int valid, const float (&d)[8], float (&v)[8]) {
  bool keep[8];
  if (MODE == MODE_TIES) {
    const Thr t = a.thr[m];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const unsigned int k = magbits(d[e]);
      keep[e] = k > t.key || (k == t.key && (long long)(j0 + e) <= t.last);
    }
  } else {
    const unsigned long long c = j0 >> 2;
    const uint4 r0 = philox4x32_10(make_uint4((unsigned int)c, (unsigned int)(c >> 32), 0u, 0u), a.key[m]);
    const uint4 r1 = philox4x32_10(make_uint4((unsigned int)(c + 1), (unsigned int)((c + 1) >> 32), 0u, 0u), a.key[m]);
    const unsigned int w[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
#pragma unroll
    for (int e = 0; e < 8; ++e) keep[e] = (w[e] >> 8) < a.keep24;
  }
  unsigned int bad = 0u;
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const float t = keep[e] ? (MODE == MODE_TIES ? d[e] : __fdiv_rn(d[e], a.density)) : 0.f;
    v[e] = __fmul_rn(a.w[m], t);
    bad += (e < valid && magbits(d[e]) >= 0x7f800000u) ? 1u : 0u;
  }
  if (bad) atomicAdd(a.nonfinite + m, bad);
}

// consensus: mask_i = sign(v_i) == majority, majority = +1 iff S = sum v_i >= 0; sums in ascending i from +0.0
template <int MODE>
__device__ __forceinline__ void accumulate8(const MergeArgs& a, int m, const float (&v)[8], const bool (&pos)[8], float (&num)[8],
                                            float (&den)[8]) {
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const bool in = MODE == MODE_DARE_LINEAR || (pos[e] ? v[e] > 0.f : v[e] < 0.f);
    if (in) { num[e] = __fadd_rn(num[e], v[e]); den[e] = __fadd_rn(den[e], a.w[m]); }
  }
}

__device__ __forceinline__ void finish8(const MergeArgs& a, const float (&b)[8], const float (&num)[8], const float (&den)[8],
                                        float (&o)[8]) {
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const float dd = den[e] == 0.f ? 1.f : den[e];
    o[e] = __fadd_rn(b[e], __fmul_rn(a.scale, __fdiv_rn(num[e], dd)));
  }
}

// MC > 0: MC models known at compile time, all tensors of dtype DT; each thread issues the loads of every model before it
// consumes the first and keeps the weighted deltas in registers.  MC = 0: any model count and per-tensor dtypes; the
// consensus modes re-form the weighted deltas in a second sweep over the models (the reloads hit L1 / L2).
template <int MODE, int MC, int DT>
__global__ void __launch_bounds__(kThreads) k_sparse_merge(const __grid_constant__ MergeArgs a) {
  const size_t n8 = (a.n + 7) / 8, stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += stride) {
    const size_t j0 = i * 8;
    const int valid = (int)min((size_t)8, a.n - j0);
    float b[8], num[8], den[8], o[8];
    bool pos[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) { num[e] = 0.f; den[e] = 0.f; }
    load8<DT>(a.base_dt, a.base, j0, a.n, b);
    if (MC > 0) {
      constexpr int K = MC > 0 ? MC : 1;
      float v[K][8];
#pragma unroll
      for (int m = 0; m < K; ++m) load8<DT>(DT, a.ft[m], j0, a.n, v[m]);
#pragma unroll
      for (int m = 0; m < K; ++m) {
        float d[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) d[e] = __fsub_rn(v[m][e], b[e]);
        weighted8<MODE>(a, m, j0, valid, d, v[m]);
      }
      if (MODE != MODE_DARE_LINEAR) {
        float s[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) s[e] = 0.f;
#pragma unroll
        for (int m = 0; m < K; ++m)
#pragma unroll
          for (int e = 0; e < 8; ++e) s[e] = __fadd_rn(s[e], v[m][e]);
#pragma unroll
        for (int e = 0; e < 8; ++e) pos[e] = s[e] >= 0.f;
      }
#pragma unroll
      for (int m = 0; m < K; ++m) accumulate8<MODE>(a, m, v[m], pos, num, den);
    } else {
      float f[8], d[8], v[8];
      if (MODE != MODE_DARE_LINEAR) {
        float s[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) s[e] = 0.f;
        for (int m = 0; m < a.M; ++m) {
          load8<DT>(a.ft_dt[m], a.ft[m], j0, a.n, f);
#pragma unroll
          for (int e = 0; e < 8; ++e) d[e] = __fsub_rn(f[e], b[e]);
          weighted8<MODE>(a, m, j0, valid, d, v);
#pragma unroll
          for (int e = 0; e < 8; ++e) s[e] = __fadd_rn(s[e], v[e]);
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) pos[e] = s[e] >= 0.f;
      }
      for (int m = 0; m < a.M; ++m) {
        load8<DT>(a.ft_dt[m], a.ft[m], j0, a.n, f);
#pragma unroll
        for (int e = 0; e < 8; ++e) d[e] = __fsub_rn(f[e], b[e]);
        // valid = 0 in the consensus modes: the first sweep counted the non-finite deltas already
        weighted8<MODE>(a, m, j0, MODE == MODE_DARE_LINEAR ? valid : 0, d, v);
        accumulate8<MODE>(a, m, v, pos, num, den);
      }
    }
    finish8(a, b, num, den, o);
    store8<DT>(a.base_dt, a.out, j0, a.n, o);
  }
}

int grid_for(size_t items, int per_sm) {
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) sms = 148;
  size_t need = (items + kThreads - 1) / kThreads;
  if (need < 1) need = 1;
  const size_t cap = (size_t)sms * per_sm;
  return (int)(need < cap ? need : cap);
}

size_t align256(size_t x) { return (x + 255) / 256 * 256; }
size_t n_tiles_of(size_t n) { return (n + kTile - 1) / kTile; }

// workspace layout: thresholds, select states, histograms, tie counts
struct WsLayout { size_t thr, st, hist, counts, total; };
WsLayout ws_layout(size_t n, int M) {
  WsLayout l;
  l.thr = 0;
  l.st = align256(sizeof(Thr) * M);
  l.hist = l.st + align256(sizeof(SelState) * M);
  l.counts = l.hist + align256((size_t)kHistBins * 4 * M);
  l.total = l.counts + align256(n_tiles_of(n) * 4 * M);
  return l;
}

int check_inputs(const char* who, int base_dtype, const void* base, const int* ft_dtypes, const void* const* fts, int n_models,
                 const void* out) {
  if (n_models < 1 || n_models > kMaxModels) { sm_set_error("%s: 1..%d models, got %d", who, kMaxModels, n_models); return -2; }
  if (base_dtype < 0 || base_dtype > 2) { sm_set_error("%s: base dtype 0 (fp32), 1 (bf16) or 2 (fp16), got %d", who, base_dtype); return -2; }
  bool aligned = (uintptr_t)base % 16 == 0 && (uintptr_t)out % 16 == 0;
  for (int m = 0; m < n_models; ++m) {
    if (ft_dtypes[m] < 0 || ft_dtypes[m] > 2) { sm_set_error("%s: model %d dtype %d is not 0, 1 or 2", who, m, ft_dtypes[m]); return -2; }
    aligned = aligned && (uintptr_t)fts[m] % 16 == 0;
  }
  if (!aligned) { sm_set_error("%s: tensors must be 16-byte aligned", who); return -2; }
  return 0;
}

}  // namespace

extern "C" size_t sm_sparse_ws_bytes(size_t n, int n_models) {
  if (n_models < 1) n_models = 1;
  return ws_layout(n, n_models).total;
}

extern "C" int sm_sparse_select(size_t n, uint64_t k, int base_dtype, const void* base, const int* ft_dtypes,
                                const void* const* fts, int n_models, void* ws, size_t ws_bytes, void* stream) {
  const int rc = check_inputs("sparse_select", base_dtype, base, ft_dtypes, fts, n_models, base);
  if (rc) return rc;
  if (k > n) { sm_set_error("sparse_select: k = %llu exceeds n = %llu", (unsigned long long)k, (unsigned long long)n); return -2; }
  const WsLayout l = ws_layout(n, n_models);
  if (ws_bytes < l.total || (uintptr_t)ws % 256 != 0) { sm_set_error("sparse_select: workspace too small or not 256-byte aligned"); return -3; }
  cudaStream_t s = (cudaStream_t)stream;
  unsigned char* w = static_cast<unsigned char*>(ws);
  SelArgs a{};
  a.base = base; a.base_dt = base_dtype; a.M = n_models; a.n = n;
  bool same = base_dtype == 1;
  for (int m = 0; m < n_models; ++m) { a.ft[m] = fts[m]; a.ft_dt[m] = (unsigned char)ft_dtypes[m]; same = same && ft_dtypes[m] == 1; }
  a.st = reinterpret_cast<SelState*>(w + l.st); a.hist = reinterpret_cast<unsigned int*>(w + l.hist);
  a.counts = reinterpret_cast<unsigned int*>(w + l.counts); a.n_tiles = n_tiles_of(n); a.thr = reinterpret_cast<Thr*>(w + l.thr);
  if (k == 0 || n == 0) {                               // nothing kept
    k_sparse_keep_none<<<(n_models + 63) / 64, 64, 0, s>>>(a.thr, n_models);
    SM_LAUNCH_CHECK();
    return 0;
  }
  SM_CUDA_CHECK(cudaMemsetAsync(a.hist, 0, (size_t)kHistBins * 4 * n_models, s));
  k_sparse_init<<<1, 64, 0, s>>>(a.st, n_models, (unsigned long long)(k - 1));
  SM_LAUNCH_CHECK();
  const size_t smem = (size_t)kGroup * kHistBins * 4;
  const dim3 hg((unsigned int)grid_for((n + 7) / 8, 3), (unsigned int)((n_models + kGroup - 1) / kGroup));
  auto hist = same ? k_sparse_hist<1> : k_sparse_hist<-1>;
  SM_CUDA_CHECK(cudaFuncSetAttribute(hist, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  for (int pass = 0; pass < 3; ++pass) {
    hist<<<hg, kThreads, smem, s>>>(a, pass);
    SM_LAUNCH_CHECK();
    k_sparse_pick<<<n_models, 1024, 0, s>>>(a.hist, a.st, pass);
    SM_LAUNCH_CHECK();
  }
  const unsigned int tg = (unsigned int)std::min<size_t>(a.n_tiles, (size_t)148 * 8);
  if (same) k_sparse_ties<1><<<tg, kThreads, 0, s>>>(a);
  else k_sparse_ties<-1><<<tg, kThreads, 0, s>>>(a);
  SM_LAUNCH_CHECK();
  if (same) k_sparse_resolve<1><<<n_models, 1024, 0, s>>>(a);
  else k_sparse_resolve<-1><<<n_models, 1024, 0, s>>>(a);
  SM_LAUNCH_CHECK();
  return 0;
}

extern "C" int sm_sparse_merge(int mode, size_t n, int base_dtype, const void* base, const int* ft_dtypes, const void* const* fts,
                               int n_models, const float* weights, const uint32_t* keys, float density, uint32_t keep24,
                               float scale, const void* thr, uint32_t* nonfinite, void* out, void* stream) {
  if (mode < 0 || mode > 2) { sm_set_error("sparse_merge: unknown mode %d", mode); return -2; }
  const int rc = check_inputs("sparse_merge", base_dtype, base, ft_dtypes, fts, n_models, out);
  if (rc) return rc;
  if (mode == MODE_TIES && !thr) { sm_set_error("sparse_merge: TIES needs the thresholds of sm_sparse_select"); return -2; }
  if (mode != MODE_TIES && !keys) { sm_set_error("sparse_merge: DARE needs one Philox key per model"); return -2; }
  cudaStream_t s = (cudaStream_t)stream;
  SM_CUDA_CHECK(cudaMemsetAsync(nonfinite, 0, sizeof(uint32_t) * n_models, s));
  if (n == 0) return 0;
  MergeArgs a{};
  a.base = base; a.base_dt = base_dtype; a.M = n_models; a.n = n; a.out = out; a.nonfinite = nonfinite;
  a.thr = reinterpret_cast<const Thr*>(thr); a.density = density; a.scale = scale; a.keep24 = keep24;
  bool same = base_dtype == 1;
  for (int m = 0; m < n_models; ++m) {
    a.ft[m] = fts[m]; a.ft_dt[m] = (unsigned char)ft_dtypes[m]; a.w[m] = weights[m];
    a.key[m] = keys ? make_uint2(keys[2 * m], keys[2 * m + 1]) : make_uint2(0u, 0u);
    same = same && ft_dtypes[m] == 1;
  }
  const unsigned int grid = (unsigned int)grid_for((n + 7) / 8, 16);
#define SM_SPARSE_MODES(MC, DT)                                                       \
  if (mode == MODE_TIES) k_sparse_merge<MODE_TIES, MC, DT><<<grid, kThreads, 0, s>>>(a);  \
  else if (mode == MODE_DARE_TIES) k_sparse_merge<MODE_DARE_TIES, MC, DT><<<grid, kThreads, 0, s>>>(a); \
  else k_sparse_merge<MODE_DARE_LINEAR, MC, DT><<<grid, kThreads, 0, s>>>(a);
#define SM_SPARSE_CASE(MC) case MC: { SM_SPARSE_MODES(MC, 1) } break;
  if (same && n_models <= 8) {                          // the common case: bf16 throughout, compile-time model count
    switch (n_models) {
      SM_SPARSE_CASE(1) SM_SPARSE_CASE(2) SM_SPARSE_CASE(3) SM_SPARSE_CASE(4)
      SM_SPARSE_CASE(5) SM_SPARSE_CASE(6) SM_SPARSE_CASE(7) SM_SPARSE_CASE(8)
    }
  } else {
    SM_SPARSE_MODES(0, -1)
  }
#undef SM_SPARSE_CASE
#undef SM_SPARSE_MODES
  SM_LAUNCH_CHECK();
  return 0;
}
