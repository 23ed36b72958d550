// kernels_stats.cu -- sm_100a kernels for everything between the forward and the inverse
// FFT: exact order statistics (replacing the two torch.sort calls of
// interpolate_fft_components, shard/tensor/functions.py:113-122 and :138-148), the masked
// SLERP reductions (functions.py:36-41 under the masks of :124-129), the three-way blend
// (:134-136) and its arithmetic sibling (:273-284), plus the FFT-free element-wise paths of
// FourierMerge._merge_layer (shard/merge/fast_fourier.py:223-225, :256-257, :269-276) and
// the API-level spectrum format conversions.
//
// All of these are streaming, HBM-bound kernels over the valid part of the half-planar
// spectrum: rows x (Ch+1) columns at pitch P, read as 16-byte vectors; a stored bin
// counts once in columns 0 and Ch and twice elsewhere (Hermitian multiplicity).
#include "sm_internal.h"
#include "select_core.cuh"

namespace {

__device__ __forceinline__ unsigned int absbits(float v) { return __float_as_uint(v) & 0x7fffffffu; }
__device__ __forceinline__ int sgn(float v) { return (v > 0.f) - (v < 0.f); }   // torch.sign: NaN -> 0

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ unsigned long long warp_sum_u64(unsigned long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// launch geometry shared by the plane kernels: x = chunk of 1024 columns, y strides rows
inline dim3 ew_grid(const SmPlan& p, int max_y) {
  int gx = (p.Ch + 1 + SM_EW_COLS - 1) / SM_EW_COLS;
  int gy = p.R < max_y ? p.R : max_y;
  if (gy < 1) gy = 1;
  return dim3(gx, gy);
}
inline int ew_max_y(const SmPlan& p) {
  int gx = (p.Ch + 1 + SM_EW_COLS - 1) / SM_EW_COLS;
  int y = (148 * 8 + gx - 1) / gx;      // ~8 CTAs of 256 threads per SM
  return y < 1 ? 1 : y;
}

// ------------------------------------------------------------------ select: bookkeeping
__global__ void k_sel_init(SelState* st, unsigned long long rank, unsigned int lo, unsigned int hi,
                           unsigned int cap) {
  st->rank = rank; st->below = 0ull; st->prefix = 0u; st->lo = lo; st->hi = hi;
  st->ncand = 0u; st->cap = cap; st->status = 0u; st->value = 0.f;
}

__device__ __forceinline__ unsigned long long mix64(unsigned long long x) {
  x += 0x9e3779b97f4a7c15ull;
  x = (x ^ (x >> 30)) * 0xbf58476d1ce4e5b9ull;
  x = (x ^ (x >> 27)) * 0x94d049bb133111ebull;
  return x ^ (x >> 31);
}

// uniform random sample of the FULL (mirrored) spectrum of 1 or 2 planes
__global__ void k_sample(SmPlan pl, const float* __restrict__ p0, const float* __restrict__ p1, int n_planes,
                         unsigned int ns, unsigned int* __restrict__ keys) {
  const unsigned long long per_plane = (unsigned long long)pl.R * (unsigned long long)pl.C;
  const unsigned long long total = per_plane * (unsigned long long)n_planes;
  for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < ns; i += gridDim.x * blockDim.x) {
    unsigned long long j = __umul64hi(mix64(i), total);
    const float* pp = p0;
    if (j >= per_plane) { j -= per_plane; pp = p1; }
    const unsigned int row = (unsigned int)(j / (unsigned long long)pl.C);
    unsigned int c = (unsigned int)(j - (unsigned long long)row * pl.C);
    if (c > (unsigned int)pl.Ch) c = pl.C - c;
    keys[i] = absbits(pp[(size_t)row * pl.P + c]);
  }
}

// ------------------------------------------------------------------ select: radix passes over flat keys
__global__ void __launch_bounds__(256) k_hist_flat(const unsigned int* __restrict__ keys,
                                                   const unsigned int* __restrict__ n_dev, unsigned int n_host,
                                                   const SelState* __restrict__ st, int pass,
                                                   unsigned int* __restrict__ hist) {
  __shared__ unsigned int sh[kHistBins];
  for (int i = threadIdx.x; i < kHistBins; i += blockDim.x) sh[i] = 0u;
  __syncthreads();
  unsigned int n = n_host;
  if (n_dev) { n = *n_dev; if (n > st->cap) n = st->cap; }
  const unsigned int prefix = st->prefix;
  const bool dead = (st->status != 0u);
  if (!dead) {
    for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
      const unsigned int k = keys[i];
      if (pass == 0) atomicAdd(&sh[k >> 20], 1u);
      else if (pass == 1) { if ((k >> 20) == (prefix >> 20)) atomicAdd(&sh[(k >> 10) & 1023u], 1u); }
      else { if ((k >> 10) == (prefix >> 10)) atomicAdd(&sh[k & 1023u], 1u); }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < kHistBins; i += blockDim.x)
    if (sh[i]) atomicAdd(&hist[i], sh[i]);
}

// single CTA, 1024 threads: extend the prefix of `st` by one radix digit
__global__ void __launch_bounds__(1024) k_pick(unsigned int* __restrict__ hist, SelState* st, int pass, int action,
                                               float* thr_out) {
  sel_pick_digit(hist, st, pass, action, thr_out);
}

// single CTA, 1024 threads: order statistics of the SAMPLE at ranks k_lo and k_hi, resolved to 21 key
// bits (two sweeps over the sample, both ranks per sweep), give the key window [lo, hi] that the
// full-data pass will count against / collect from.  k_lo < 0 -> lo = 0, k_hi >= ns -> hi = all keys.
__global__ void __launch_bounds__(1024) k_sample_window(const unsigned int* __restrict__ keys, unsigned int ns,
                                                        SelState* st, long long k_lo, long long k_hi,
                                                        unsigned long long rank_full) {
  __shared__ unsigned int sh[kHistBins];
  __shared__ PickOut out_a, out_b;
  const bool want_a = (k_lo >= 0 && k_lo < (long long)ns), want_b = (k_hi >= 0 && k_hi < (long long)ns);
  for (int i = threadIdx.x; i < kHistBins; i += blockDim.x) sh[i] = 0u;
  __syncthreads();
  for (unsigned int i = threadIdx.x; i < ns; i += blockDim.x) atomicAdd(&sh[keys[i] >> 20], 1u);
  __syncthreads();
  block_pick(sh, want_a ? (unsigned long long)k_lo : 0ull, &out_a, kHistBins, false);
  block_pick(sh, want_b ? (unsigned long long)k_hi : 0ull, &out_b, kHistBins, true);
  const unsigned int bin_a = (unsigned int)(out_a.bin < 0 ? 0 : out_a.bin);
  const unsigned int bin_b = (unsigned int)(out_b.bin < 0 ? 0 : out_b.bin);
  const unsigned long long ra = out_a.rank_in_bin, rb = out_b.rank_in_bin;
  __syncthreads();
  // second digit: two 1024-bin histograms in the two halves of sh
  for (unsigned int i = threadIdx.x; i < ns; i += blockDim.x) {
    const unsigned int key = keys[i], top = key >> 20, sub = (key >> 10) & 1023u;
    if (top == bin_a) atomicAdd(&sh[sub], 1u);
    if (top == bin_b) atomicAdd(&sh[1024 + sub], 1u);
  }
  __syncthreads();
  block_pick(sh, ra, &out_a, 1024, false);
  block_pick(sh + 1024, rb, &out_b, 1024, false);
  if (threadIdx.x == 0) {
    const unsigned int sub_a = (unsigned int)(out_a.bin < 0 ? 0 : out_a.bin);
    const unsigned int sub_b = (unsigned int)(out_b.bin < 0 ? 1023 : out_b.bin);
    st->lo = want_a ? ((bin_a << 20) | (sub_a << 10)) : 0u;
    st->hi = want_b ? ((bin_b << 20) | (sub_b << 10) | 1023u) : 0x7fffffffu;
    st->rank = rank_full; st->below = 0ull; st->ncand = 0u; st->prefix = 0u;
  }
}

// ------------------------------------------------------------------ select: count below the window, collect inside
constexpr int kStage = 8192;       // smem staging entries per CTA
// kSafe = false (sampled window, candidates are ~1 % of the keys): a CTA stages everything it finds
//         and flushes once at the end -- no barrier inside the streaming loop; if the stage overflows
//         the select is flagged (status bit 1) and the caller falls back to the safe mode.
// kSafe = true  (window = all keys): barrier + flush test after every row.
template <bool kSafe>
__global__ void __launch_bounds__(SM_EW_THREADS) k_count_collect(const __grid_constant__ SmPlan pl,
                                                                 const float* __restrict__ p0,
                                                                 const float* __restrict__ p1, SelState* st,
                                                                 unsigned int* __restrict__ cand) {
  __shared__ unsigned int s_buf[kStage];
  __shared__ unsigned int s_cnt, s_base;
  __shared__ unsigned long long s_below[SM_EW_THREADS / 32];
  if (threadIdx.x == 0) s_cnt = 0u;
  __syncthreads();
  const unsigned int lo = st->lo, hi = st->hi, cap = st->cap;
  const int c0 = blockIdx.x * SM_EW_COLS + threadIdx.x * 4;
  const bool active = (c0 <= pl.Ch);
  unsigned long long below = 0ull;
  const int n_planes = p1 ? 2 : 1;
  auto scan4 = [&](const float4 v) {
    const float e[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int c = c0 + i;
      if (c <= pl.Ch) {
        const unsigned int w = (c == 0 || c == pl.Ch) ? 1u : 2u;
        const unsigned int k = absbits(e[i]);
        if (k < lo) below += w;
        else if (k <= hi) {
          const unsigned int pos = atomicAdd(&s_cnt, w);
          if (pos + w <= (unsigned int)kStage) { s_buf[pos] = k; if (w == 2u) s_buf[pos + 1] = k; }
        }
      }
    }
  };
  if (!kSafe) {
    if (active) {
      int row = blockIdx.y;
      for (; row + gridDim.y < pl.R; row += 2 * gridDim.y) {          // two rows in flight per plane
        float4 v[4];
        for (int pi = 0; pi < n_planes; ++pi) {
          const float* pp = pi == 0 ? p0 : p1;
          v[2 * pi] = *reinterpret_cast<const float4*>(pp + (size_t)row * pl.P + c0);
          v[2 * pi + 1] = *reinterpret_cast<const float4*>(pp + (size_t)(row + gridDim.y) * pl.P + c0);
        }
        for (int q = 0; q < 2 * n_planes; ++q) scan4(v[q]);
      }
      for (; row < pl.R; row += gridDim.y)
        for (int pi = 0; pi < n_planes; ++pi)
          scan4(*reinterpret_cast<const float4*>((pi == 0 ? p0 : p1) + (size_t)row * pl.P + c0));
    }
  } else {
    for (int row = blockIdx.y; row < pl.R; row += gridDim.y) {
      if (active)
        for (int pi = 0; pi < n_planes; ++pi)
          scan4(*reinterpret_cast<const float4*>((pi == 0 ? p0 : p1) + (size_t)row * pl.P + c0));
      __syncthreads();
      const unsigned int cnt_now = s_cnt;
      __syncthreads();                               // everyone has read it before anyone appends again
      // a CTA adds at most 256*4*2*2 = 4096 entries per row: flush once fewer than that remain
      if (cnt_now > (unsigned int)(kStage - 4096)) {
        if (threadIdx.x == 0) s_base = atomicAdd(&st->ncand, cnt_now);
        __syncthreads();
        const unsigned int base = s_base;
        for (unsigned int i = threadIdx.x; i < cnt_now; i += blockDim.x)
          if (base + i < cap) cand[base + i] = s_buf[i];
        __syncthreads();
        if (threadIdx.x == 0) s_cnt = 0u;
        __syncthreads();
      }
    }
  }
  __syncthreads();
  {
    unsigned int cnt = s_cnt;
    if (cnt > (unsigned int)kStage) {                // only possible in the fast variant
      if (threadIdx.x == 0) atomicOr(&st->status, 2u);
      cnt = kStage;
    }
    if (cnt) {
      if (threadIdx.x == 0) s_base = atomicAdd(&st->ncand, cnt);
      __syncthreads();
      const unsigned int base = s_base;
      for (unsigned int i = threadIdx.x; i < cnt; i += blockDim.x)
        if (base + i < cap) cand[base + i] = s_buf[i];
    }
  }
  below = warp_sum_u64(below);
  if ((threadIdx.x & 31) == 0) s_below[threadIdx.x >> 5] = below;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long b = 0ull;
    for (int i = 0; i < SM_EW_THREADS / 32; ++i) b += s_below[i];
    if (b) atomicAdd(&st->below, b);
  }
}

// ------------------------------------------------------------------ SLERP masked sums
__global__ void __launch_bounds__(SM_EW_THREADS) k_slerp_reduce(SmPlan pl, const float* __restrict__ reX,
                                                                const float* __restrict__ reY, const int* sel,
                                                                const float* __restrict__ thr_cut,
                                                                double* __restrict__ sums3) {
  __shared__ double s_part[3][SM_EW_THREADS / 32];
  const bool sw = (sel != nullptr && *sel != 0);      // device-side role pick: v0 is the larger-norm model
  const float* __restrict__ re0 = sw ? reY : reX;
  const float* __restrict__ re1 = sw ? reX : reY;
  const float thr = *thr_cut;
  const int c0 = blockIdx.x * SM_EW_COLS + threadIdx.x * 4;
  double s00 = 0.0, s11 = 0.0, s01 = 0.0;
  if (c0 <= pl.Ch) {
    for (int row = blockIdx.y; row < pl.R; row += gridDim.y) {
      const float4 a4 = *reinterpret_cast<const float4*>(re0 + (size_t)row * pl.P + c0);
      const float4 b4 = *reinterpret_cast<const float4*>(re1 + (size_t)row * pl.P + c0);
      const float a[4] = {a4.x, a4.y, a4.z, a4.w}, b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int c = c0 + i;
        if (c <= pl.Ch) {
          const float w = (c == 0 || c == pl.Ch) ? 1.f : 2.f;
          const bool in = (sgn(a[i]) == sgn(b[i])) && !(fabsf(b[i]) < thr);
          if (in) {
            s00 += (double)w * (double)a[i] * (double)a[i];
            s11 += (double)w * (double)b[i] * (double)b[i];
            s01 += (double)w * (double)a[i] * (double)b[i];
          }
        }
      }
    }
  }
  s00 = warp_sum_d(s00); s11 = warp_sum_d(s11); s01 = warp_sum_d(s01);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) { s_part[0][wid] = s00; s_part[1][wid] = s11; s_part[2][wid] = s01; }
  __syncthreads();
  if (threadIdx.x < 3) {
    double t = 0.0;
    for (int i = 0; i < SM_EW_THREADS / 32; ++i) t += s_part[threadIdx.x][i];
    atomicAdd(&sums3[threadIdx.x], t);
  }
}

__global__ void k_slerp_scalars(const double* __restrict__ sums3, double t, float* __restrict__ scal4) {
  const double s00 = sums3[0], s11 = sums3[1], s01 = sums3[2];
  // torch: dot = sum(v0*v1) / (v0.norm() * v1.norm()), all fp32 tensors (functions.py:36)
  const float n0 = (float)sqrt(s00), n1 = (float)sqrt(s11);
  float dot = (float)s01 / (n0 * n1);
  dot = fminf(fmaxf(dot, -1.0f), 1.0f);             // clamp keeps NaN as NaN
  if (!(dot == dot)) dot = __uint_as_float(0x7fc00000u);
  const float theta = (float)acos((double)dot) * (float)t;
  const float ct = (float)cos((double)theta), sn = (float)sin((double)theta);
  // || v1 - v0*dot ||^2 = s11 - 2 dot s01 + dot^2 s00   (dot as the fp32 value that is used element-wise)
  const double d = (double)dot;
  double rn2 = s11 - 2.0 * d * s01 + d * d * s00;
  if (rn2 < 0.0) rn2 = 0.0;
  float rn = (float)sqrt(rn2);
  if (rn < 1e-12f) rn = 1e-12f;                      // F.normalize eps
  if (!(d == d)) rn = __uint_as_float(0x7fc00000u);
  scal4[0] = dot; scal4[1] = ct; scal4[2] = sn; scal4[3] = rn;
}

// ------------------------------------------------------------------ blend
__global__ void __launch_bounds__(SM_EW_THREADS) k_blend(SmPlan pl, int mode, int agreement,
                                                         const float* reX, const float* reY, const int* sel,
                                                         const float* __restrict__ thr_cut,
                                                         const float* __restrict__ scal4, float t_sum,
                                                         float* out) {
  const int c0 = blockIdx.x * SM_EW_COLS + threadIdx.x * 4;
  if (c0 > pl.Ch) return;
  const bool sw = (sel != nullptr && *sel != 0);
  const float* re0 = sw ? reY : reX;
  const float* re1 = sw ? reX : reY;
  float thr = 0.f, dot = 0.f, ct = 0.f, sn = 0.f, rn = 1.f;
  if (mode == 0) { thr = *thr_cut; dot = scal4[0]; ct = scal4[1]; sn = scal4[2]; rn = scal4[3]; }
  for (int row = blockIdx.y; row < pl.R; row += gridDim.y) {
    const size_t off = (size_t)row * pl.P + c0;
    const float4 a4 = *reinterpret_cast<const float4*>(re0 + off);
    const float4 b4 = *reinterpret_cast<const float4*>(re1 + off);
    const float a[4] = {a4.x, a4.y, a4.z, a4.w}, b[4] = {b4.x, b4.y, b4.z, b4.w};
    float o[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const bool same = (sgn(a[i]) == sgn(b[i]));
      if (mode == 0) {
        const bool small = fabsf(b[i]) < thr;
        if (same && !small) {
          // v0*cos(theta) + normalize(v1 - v0*dot)*sin(theta), one rounding per torch op
          const float rel = __fsub_rn(b[i], __fmul_rn(a[i], dot));
          o[i] = __fadd_rn(__fmul_rn(a[i], ct), __fmul_rn(__fdiv_rn(rel, rn), sn));
        } else if (same) {
          o[i] = __fadd_rn(a[i], __fmul_rn(t_sum, b[i]));
        } else {
          o[i] = (fabsf(a[i]) > fabsf(b[i])) ? a[i] : b[i];
        }
      } else {
        o[i] = (same || !agreement) ? __fadd_rn(a[i], __fmul_rn(t_sum, b[i])) : b[i];
      }
    }
    *reinterpret_cast<float4*>(out + off) = make_float4(o[0], o[1], o[2], o[3]);
  }
}

// ------------------------------------------------------------------ FFT-free element-wise path
__device__ __forceinline__ float bf16lo(unsigned int u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf16hi(unsigned int u) { return __uint_as_float(u & 0xffff0000u); }
__device__ __forceinline__ unsigned int f2bf16(float f) {
  unsigned int u = __float_as_uint(f);
  if ((u & 0x7fffffffu) > 0x7f800000u) return (u >> 16) | 0x0040u;
  u += 0x7fffu + ((u >> 16) & 1u);
  return u >> 16;
}

__global__ void __launch_bounds__(256) k_delta_axpby(size_t n2, const unsigned int* __restrict__ bo,
                                                     const unsigned int* __restrict__ b0,
                                                     const unsigned int* __restrict__ f0, float ca,
                                                     const unsigned int* __restrict__ b1,
                                                     const unsigned int* __restrict__ f1, float cb, float scale,
                                                     unsigned int* __restrict__ out, unsigned int* flags4) {
  unsigned int nan_c = 0u, inf_c = 0u;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += (size_t)gridDim.x * blockDim.x) {
    const unsigned int ub = bo[i], u0b = b0[i], u0f = f0[i];
    float d0 = __fmul_rn(ca, __fsub_rn(bf16lo(u0f), bf16lo(u0b)));
    float d1 = __fmul_rn(ca, __fsub_rn(bf16hi(u0f), bf16hi(u0b)));
    if (f1) {
      const unsigned int u1b = b1[i], u1f = f1[i];
      d0 = __fadd_rn(d0, __fmul_rn(cb, __fsub_rn(bf16lo(u1f), bf16lo(u1b))));
      d1 = __fadd_rn(d1, __fmul_rn(cb, __fsub_rn(bf16hi(u1f), bf16hi(u1b))));
    }
    float y0 = __fadd_rn(bf16lo(ub), __fmul_rn(d0, scale));
    float y1 = __fadd_rn(bf16hi(ub), __fmul_rn(d1, scale));
    unsigned int k0 = absbits(y0), k1 = absbits(y1);
    if (k0 > 0x7f800000u) { ++nan_c; y0 = 0.f; } else if (k0 == 0x7f800000u) ++inf_c;
    if (k1 > 0x7f800000u) { ++nan_c; y1 = 0.f; } else if (k1 == 0x7f800000u) ++inf_c;
    out[i] = f2bf16(y0) | (f2bf16(y1) << 16);
  }
  if (nan_c) atomicAdd(flags4 + 2, nan_c);
  if (inf_c) atomicAdd(flags4 + 3, inf_c);
}

// ------------------------------------------------------------------ format conversion (API level)
__device__ __forceinline__ int stored_row(const SmPlan& pl, int k) {   // frequency -> stored row
  if (pl.col_passes < 2) return k;
  const int ka = k % pl.Ra, kb = k / pl.Ra;
  return pl.Rb * ka + kb;
}

__global__ void k_expand_full(SmPlan pl, const float* __restrict__ re, const float* __restrict__ im,
                              float2* __restrict__ out) {
  for (int kr = blockIdx.y; kr < pl.R; kr += gridDim.y)
  for (int kc = blockIdx.x * blockDim.x + threadIdx.x; kc < pl.C; kc += gridDim.x * blockDim.x) {
    float2 v;
    if (kc <= pl.Ch) {
      const size_t off = (size_t)stored_row(pl, kr) * pl.P + kc;
      v.x = re[off]; v.y = im[off];
    } else {
      const int mr = (pl.R - kr) % pl.R, mc = pl.C - kc;
      const size_t off = (size_t)stored_row(pl, mr) * pl.P + mc;
      v.x = re[off]; v.y = -im[off];
    }
    out[(size_t)kr * pl.C + kc] = v;
  }
}

__global__ void k_pack_half(SmPlan pl, const float2* __restrict__ in, float* __restrict__ re,
                            float* __restrict__ im) {
  for (int kr = blockIdx.y; kr < pl.R; kr += gridDim.y)
  for (int kc = blockIdx.x * blockDim.x + threadIdx.x; kc <= pl.Ch; kc += gridDim.x * blockDim.x) {
    const int mr = (pl.R - kr) % pl.R;
    const float2 a = in[(size_t)kr * pl.C + kc];
    const float2 b = in[(size_t)mr * pl.C + ((pl.C - kc) % pl.C)];
    const size_t off = (size_t)stored_row(pl, kr) * pl.P + kc;
    re[off] = 0.5f * (a.x + b.x);
    im[off] = 0.5f * (a.y - b.y);
  }
}

}  // namespace

// ================================================================== C ABI
static unsigned int fast_cap(const SmPlan& p, int n_planes) {
  unsigned long long total = (unsigned long long)p.R * p.C * n_planes;
  unsigned long long cap = total / 16;
  if (cap < (1ull << 20)) cap = 1ull << 20;
  if (cap > 0xfffffff0ull) cap = 0xfffffff0ull;
  return (unsigned int)cap;
}
static const unsigned int kSampleN = 1u << 16;
static bool use_safe(const SmPlan& p, int n_planes, int mode) {
  unsigned long long total = (unsigned long long)p.R * p.C * n_planes;
  return mode != 0 || total <= (4ull << 20);
}

extern "C" size_t sm_select_ws_bytes(const sm_plan* plan, int n_planes, int mode) {
  const SmPlan& p = plan->p;
  unsigned long long total = (unsigned long long)p.R * p.C * n_planes;
  size_t bytes = kHistBins * 4;
  if (use_safe(p, n_planes, mode)) bytes += (size_t)total * 4;
  else bytes += (size_t)kSampleN * 4 + (size_t)fast_cap(p, n_planes) * 4;
  return bytes + 256;
}

extern "C" int sm_select_kth_abs(const sm_plan* plan, const float* plane0, const float* plane1, uint64_t rank,
                                 int mode, void* sel_state, void* ws, size_t ws_bytes, float* thr_out,
                                 void* stream) {
  const SmPlan& p = plan->p;
  cudaStream_t s = (cudaStream_t)stream;
  const int n_planes = plane1 ? 2 : 1;
  const unsigned long long total = (unsigned long long)p.R * p.C * n_planes;
  if (total >= 0xfffffff0ull) { sm_set_error("select: more than 2^32 keys"); return -2; }
  if (ws_bytes < sm_select_ws_bytes(plan, n_planes, mode)) { sm_set_error("select: workspace too small"); return -3; }
  if (rank >= total) rank = total - 1;               // functions.py:116-117: past the end -> last element
  SelState* st = reinterpret_cast<SelState*>(sel_state);
  unsigned int* hist = reinterpret_cast<unsigned int*>(ws);
  unsigned int* buf = hist + kHistBins;
  SM_CUDA_CHECK(cudaMemsetAsync(hist, 0, kHistBins * 4, s));
  const bool safe = use_safe(p, n_planes, mode);
  const dim3 eg = ew_grid(p, ew_max_y(p));
  unsigned int* cand;
  if (safe) {
    cand = buf;
    k_sel_init<<<1, 1, 0, s>>>(st, rank, 0u, 0x7fffffffu, (unsigned int)total);
    SM_LAUNCH_CHECK();
  } else {
    unsigned int* sample = buf;
    cand = buf + kSampleN;
    // sample ranks that bracket `rank` of the full key set with ~6 sigma of binomial noise
    const double pq = (double)rank / (double)total;
    const double ks = pq * (double)kSampleN;
    const double delta = 6.0 * sqrt((double)kSampleN * pq * (1.0 - pq)) + 16.0;
    k_sel_init<<<1, 1, 0, s>>>(st, rank, 0u, 0u, fast_cap(p, n_planes));
    SM_LAUNCH_CHECK();
    k_sample<<<148, 256, 0, s>>>(p, plane0, plane1, n_planes, kSampleN, sample);
    SM_LAUNCH_CHECK();
    k_sample_window<<<1, 1024, 0, s>>>(sample, kSampleN, st, (long long)floor(ks - delta), (long long)ceil(ks + delta), rank);
    SM_LAUNCH_CHECK();
  }
  if (safe) k_count_collect<true><<<eg, SM_EW_THREADS, 0, s>>>(p, plane0, plane1, st, cand);
  else k_count_collect<false><<<eg, SM_EW_THREADS, 0, s>>>(p, plane0, plane1, st, cand);
  SM_LAUNCH_CHECK();
  for (int pass = 0; pass < 3; ++pass) {
    k_hist_flat<<<592, 256, 0, s>>>(cand, &st->ncand, 0u, st, pass, hist);
    SM_LAUNCH_CHECK();
    k_pick<<<1, 1024, 0, s>>>(hist, st, pass, pass == 0 ? PICK_ADJUST : (pass == 2 ? PICK_FINISH : PICK_NONE), thr_out);
    SM_LAUNCH_CHECK();
  }
  return 0;
}

int sm_slerp_reduce_sel(const sm_plan* plan, const float* reX, const float* reY, const int* sel,
                        const float* thr_cut, double* sums3, void* stream) {
  const SmPlan& p = plan->p;
  k_slerp_reduce<<<ew_grid(p, ew_max_y(p)), SM_EW_THREADS, 0, (cudaStream_t)stream>>>(p, reX, reY, sel, thr_cut, sums3);
  SM_LAUNCH_CHECK();
  return 0;
}
extern "C" int sm_slerp_reduce(const sm_plan* plan, const float* re0, const float* re1, const float* thr_cut,
                               double* sums3, void* stream) {
  return sm_slerp_reduce_sel(plan, re0, re1, nullptr, thr_cut, sums3, stream);
}

extern "C" int sm_slerp_scalars(const double* sums3, double t, float* scal4, void* stream) {
  k_slerp_scalars<<<1, 1, 0, (cudaStream_t)stream>>>(sums3, t, scal4);
  SM_LAUNCH_CHECK();
  return 0;
}

int sm_blend_sel(const sm_plan* plan, int mode, int agreement, const float* reX, const float* reY, const int* sel,
                 const float* thr_cut, const float* scal4, float t_sum, float* out_re, void* stream) {
  const SmPlan& p = plan->p;
  if (mode == 0 && (!thr_cut || !scal4)) { sm_set_error("blend: SLERP mode needs thr_cut and scal4"); return -2; }
  k_blend<<<ew_grid(p, ew_max_y(p)), SM_EW_THREADS, 0, (cudaStream_t)stream>>>(p, mode, agreement, reX, reY, sel,
                                                                               thr_cut, scal4, t_sum, out_re);
  SM_LAUNCH_CHECK();
  return 0;
}
extern "C" int sm_blend(const sm_plan* plan, int mode, int agreement, const float* re0, const float* re1,
                        const float* thr_cut, const float* scal4, float t_sum, float* out_re, void* stream) {
  return sm_blend_sel(plan, mode, agreement, re0, re1, nullptr, thr_cut, scal4, t_sum, out_re, stream);
}

extern "C" int sm_delta_axpby_bf16(size_t n, const void* base_out, const void* base0, const void* ft0, float ca,
                                   const void* base1, const void* ft1, float cb, float scale, void* out_bf16,
                                   uint32_t* flags4, void* stream) {
  if (n & 1) { sm_set_error("delta_axpby: element count must be even"); return -2; }
  const size_t n2 = n / 2;
  int blocks = (int)((n2 + 255) / 256);
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (blocks < 1) blocks = 1;
  k_delta_axpby<<<blocks, 256, 0, (cudaStream_t)stream>>>(
      n2, (const unsigned int*)base_out, (const unsigned int*)base0, (const unsigned int*)ft0, ca,
      (const unsigned int*)base1, (const unsigned int*)ft1, cb, scale, (unsigned int*)out_bf16, flags4);
  SM_LAUNCH_CHECK();
  return 0;
}

extern "C" int sm_copy_bytes(void* dst, const void* src, size_t n, void* stream) {
  SM_CUDA_CHECK(cudaMemcpyAsync(dst, src, n, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return 0;
}

extern "C" int sm_expand_full(const sm_plan* plan, const float* re, const float* im, float* out_c64, void* stream) {
  const SmPlan& p = plan->p;
  dim3 g((p.C + 255) / 256 > 64 ? 64 : (p.C + 255) / 256, p.R > 32768 ? 32768 : p.R);
  k_expand_full<<<g, 256, 0, (cudaStream_t)stream>>>(p, re, im, reinterpret_cast<float2*>(out_c64));
  SM_LAUNCH_CHECK();
  return 0;
}

extern "C" int sm_pack_half(const sm_plan* plan, const float* in_c64, float* re, float* im, void* stream) {
  const SmPlan& p = plan->p;
  dim3 g((p.Ch + 256) / 256 > 64 ? 64 : (p.Ch + 256) / 256, p.R > 32768 ? 32768 : p.R);
  k_pack_half<<<g, 256, 0, (cudaStream_t)stream>>>(p, reinterpret_cast<const float2*>(in_c64), re, im);
  SM_LAUNCH_CHECK();
  return 0;
}
