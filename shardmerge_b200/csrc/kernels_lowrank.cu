// kernels_lowrank.cu -- the dense products of a randomized SVD of a checkpoint's difference from its base.
//
//   right:  Y[R][k] = Δ · X[C][k]       (and optionally Σ δ² in fp64)
//   left:   Z[k][C] = Q[R][k]ᵀ · Δ       with Δ[i][j] = fp32(M[i][j]) − fp32(W[i][j]), one rounded fp32 subtraction
//
// Δ is formed in registers from the two checkpoints' tensors (fp32 / bf16 / fp16, each with its own dtype) and never
// written.  Both products are one form, P[m][n] = Σ_l S[l][m] · D[l][n], over the reduction index l: S is the small [L][k]
// operand (X with L = C, or Q with L = R), D is Δ (left: D = Δ, n = column; right: D = Δᵀ, n = row), m runs over k.
//
// A 256-thread CTA owns 64 m × 128 n of P, a thread 4 m × 8 adjacent n in four packed f32x2 column pairs (fma.rn.f32x2),
// the inner loop of kernels_lora.cu.  S and Δ go through shared memory in chunks of 32 l.  fp32 FMA only: a bf16 or TF32
// operand would round Δ to 2^-9 .. 2^-11 relative and lose the fp32-level recovery of an exact low-rank difference.
// The reduction is split over gridDim.z so that every shape gives ~6 CTAs per SM: split s covers the l range
// [s·G/S, (s+1)·G/S) · 8 of G = ceil(L / 8) granules (16-byte vectors along a row stay inside one split), writes its fp32
// partial P_s to the workspace, and k_lowrank_reduce adds P_0 .. P_{S-1} in that order: no atomics, bit-identical runs.
// gridDim.x runs over the m tiles, so the CTAs that read the same Δ tile are launched together and share it through L2.
#include <algorithm>
#include "elem_codec.cuh"
#include "fft_core.cuh"
#include "sm_internal.h"

namespace {

using smfft::pf;
using smfft::pf_fma;
using smfft::pf_hi;
using smfft::pf_lo;
using smfft::pf_make;

constexpr int kTm = 64, kTn = 128, kKc = 32, kThreads = 256;
constexpr int kRowsPerThread = 4, kColsPerThread = 8;
constexpr int kGranule = 8;                            // split boundaries along l: multiples of one 8-element vector
constexpr long long kTargetCtas = 6 * 148;             // two waves at 3 resident CTAs per SM on 148 SMs
constexpr int kReduceThreads = 256;

struct LowrankArgs {
  const void* W; const void* M; const float* S;
  float* part;             // [splits][k][N] fp32 partials
  double* ss_part;         // [splits][gridDim.y] Σ δ² of each (split, n tile), right only; null: not wanted
  int R, C, k;
  int L, N;                // reduction and output length: (C, R) right, (R, C) left
  int splits;
  int vec;                 // 1: W and M 16-byte aligned and every row a whole number of 16-byte vectors in both dtypes
};

// Shared slot of column c of a Δ chunk row (kernels_lora.cu's a_slot): a thread's two 4-column halves are contiguous
// across the 16 column groups of a half-warp.
__device__ __forceinline__ int a_slot(int c) { return ((c >> 3) << 2) + (c & 3) + (((c >> 2) & 1) << 6); }

// d[e] = fp32(M[off + e]) - fp32(W[off + e]) for e < cnt, 0 beyond
template <int WDT, int MDT>
__device__ __forceinline__ void delta8(const LowrankArgs& a, size_t off, int cnt, float (&d)[8]) {
  using Cw = ElemCodec<WDT>;
  using Cm = ElemCodec<MDT>;
  if (a.vec && cnt == 8) {
    float w[8], m[8];
    Cw::load8(a.W, off, w);
    Cm::load8(a.M, off, m);
#pragma unroll
    for (int e = 0; e < 8; ++e) d[e] = __fsub_rn(m[e], w[e]);
  } else {
#pragma unroll
    for (int e = 0; e < 8; ++e) d[e] = e < cnt ? __fsub_rn(Cm::load(a.M, off + e), Cw::load(a.W, off + e)) : 0.f;
  }
}

__device__ __forceinline__ int split_edge(int L, int splits, int s) {
  const long long g = ((long long)(L + kGranule - 1) / kGranule) * s / splits;
  return (int)min((long long)L, g * kGranule);
}

template <bool RIGHT, int WDT, int MDT>
__global__ void __launch_bounds__(kThreads) k_lowrank(const __grid_constant__ LowrankArgs a) {
  __shared__ __align__(16) float Ds[kKc][kTn];
  __shared__ __align__(16) float Ss[kKc][kTm];
  __shared__ double ss_warp[kThreads / 32];
  sm_pdl_enter();
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4, warp = tid >> 5;
  const int m0 = blockIdx.x * kTm, n0 = blockIdx.y * kTn, s = blockIdx.z;
  const int l_begin = split_edge(a.L, a.splits, s), l_end = split_edge(a.L, a.splits, s + 1);
  const bool want_ss = RIGHT && a.ss_part != nullptr && blockIdx.x == 0;
  const bool active = m0 + warp * 2 * kRowsPerThread < a.k;   // a warp's 8 rows of m: none valid -> it only stages
  double ss = 0.0;

  pf acc[kRowsPerThread][kColsPerThread / 2];
#pragma unroll
  for (int q = 0; q < kRowsPerThread; ++q)
#pragma unroll
    for (int p = 0; p < kColsPerThread / 2; ++p) acc[q][p] = pf_make(0.f, 0.f);

  for (int l0 = l_begin; l0 < l_end; l0 += kKc) {
    const int kc = min(kKc, l_end - l0);
    __syncthreads();                                   // the previous chunk has been consumed
    for (int idx = tid; idx < kKc * kTm; idx += kThreads) {
      const int kk = idx / kTm, mm = idx % kTm, m = m0 + mm;
      Ss[kk][mm] = (kk < kc && m < a.k) ? __ldg(a.S + (size_t)(l0 + kk) * a.k + m) : 0.f;
    }
    if (RIGHT) {
      // Δᵀ chunk: 128 rows of Δ × 32 columns; a warp reads one 8-column vector of 32 consecutive rows
      for (int idx = tid; idx < kTn * (kKc / 8); idx += kThreads) {
        const int i = idx % kTn, v = idx / kTn, row = n0 + i, c = l0 + v * 8;
        float d[8];
        const int cnt = row < a.R ? min(8, l0 + kc - c) : 0;
        if (cnt > 0) delta8<WDT, MDT>(a, (size_t)row * a.C + c, cnt, d);
        else {
#pragma unroll
          for (int e = 0; e < 8; ++e) d[e] = 0.f;
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) Ds[v * 8 + e][a_slot(i)] = d[e];
        if (want_ss) {
#pragma unroll
          for (int e = 0; e < 8; ++e) ss += (double)__fmul_rn(d[e], d[e]);
        }
      }
    } else {
      // Δ chunk: 32 rows × 128 columns; a warp reads two rows, 16 vectors each
      for (int idx = tid; idx < kKc * (kTn / 8); idx += kThreads) {
        const int kk = idx / (kTn / 8), v = idx % (kTn / 8), c = n0 + v * 8;
        float d[8];
        const int cnt = kk < kc ? min(8, a.C - c) : 0;
        if (cnt > 0) delta8<WDT, MDT>(a, (size_t)(l0 + kk) * a.C + c, cnt, d);
        else {
#pragma unroll
          for (int e = 0; e < 8; ++e) d[e] = 0.f;
        }
        *reinterpret_cast<float4*>(&Ds[kk][v * 4]) = make_float4(d[0], d[1], d[2], d[3]);
        *reinterpret_cast<float4*>(&Ds[kk][64 + v * 4]) = make_float4(d[4], d[5], d[6], d[7]);
      }
    }
    __syncthreads();
    if (active) {
      for (int kk = 0; kk < kc; ++kk) {
        const float4 s4 = *reinterpret_cast<const float4*>(&Ss[kk][ty * kRowsPerThread]);
        const float4 lo = *reinterpret_cast<const float4*>(&Ds[kk][tx * 4]);
        const float4 hi = *reinterpret_cast<const float4*>(&Ds[kk][64 + tx * 4]);
        const pf dv[4] = {pf_make(lo.x, lo.y), pf_make(lo.z, lo.w), pf_make(hi.x, hi.y), pf_make(hi.z, hi.w)};
        const float sv[4] = {s4.x, s4.y, s4.z, s4.w};
#pragma unroll
        for (int q = 0; q < kRowsPerThread; ++q) {
          const pf sb = pf_make(sv[q], sv[q]);
#pragma unroll
          for (int p = 0; p < 4; ++p) acc[q][p] = pf_fma(sb, dv[p], acc[q][p]);
        }
      }
    }
  }

  const int n = n0 + tx * kColsPerThread;
  if (n < a.N) {
    const bool full = (a.N % 4) == 0 && n + kColsPerThread <= a.N;
#pragma unroll
    for (int q = 0; q < kRowsPerThread; ++q) {
      const int m = m0 + ty * kRowsPerThread + q;
      if (m >= a.k) break;
      float* p = a.part + ((size_t)s * a.k + m) * a.N + n;
      const float o[8] = {pf_lo(acc[q][0]), pf_hi(acc[q][0]), pf_lo(acc[q][1]), pf_hi(acc[q][1]),
                          pf_lo(acc[q][2]), pf_hi(acc[q][2]), pf_lo(acc[q][3]), pf_hi(acc[q][3])};
      if (full) {
        reinterpret_cast<float4*>(p)[0] = make_float4(o[0], o[1], o[2], o[3]);
        reinterpret_cast<float4*>(p)[1] = make_float4(o[4], o[5], o[6], o[7]);
      } else {
#pragma unroll
        for (int e = 0; e < kColsPerThread; ++e)
          if (n + e < a.N) p[e] = o[e];
      }
    }
  }
  if (want_ss) {                                       // fixed-order tree over the CTA: lanes, then warps
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) ss += __shfl_down_sync(0xffffffffu, ss, off);
    if ((tid & 31) == 0) ss_warp[warp] = ss;
    __syncthreads();
    if (tid == 0) {
      double t = 0.0;
      for (int w = 0; w < kThreads / 32; ++w) t += ss_warp[w];
      a.ss_part[(size_t)s * gridDim.y + blockIdx.y] = t;
    }
  }
}

// out = P_0 + P_1 + ... + P_{splits-1} in that order (left: out[m][n] = [k][C]; right: out[n][m] = [R][k]); thread 0 of
// block 0 adds the n_ss sum-of-squares partials in index order.
template <bool RIGHT>
__global__ void __launch_bounds__(kReduceThreads) k_lowrank_reduce(const float* part, int splits, int k, int N,
                                                                   float* out, const double* ss_part, int n_ss,
                                                                   double* sumsq) {
  sm_pdl_enter();
  const size_t total = (size_t)k * N;
  for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
    float acc = part[e];
    for (int s = 1; s < splits; ++s) acc = __fadd_rn(acc, part[(size_t)s * total + e]);
    if (RIGHT) {
      const size_t m = e / N, n = e % N;
      out[n * k + m] = acc;
    } else {
      out[e] = acc;
    }
  }
  if (sumsq != nullptr && blockIdx.x == 0 && threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < n_ss; ++i) t += ss_part[i];
    *sumsq = t;
  }
}

struct LowrankGeom {
  int L, N, m_tiles, n_tiles, splits;
  size_t part_bytes, ss_bytes;
};

LowrankGeom lowrank_geom(bool right, int R, int C, int k) {
  LowrankGeom g{};
  g.L = right ? C : R;
  g.N = right ? R : C;
  g.m_tiles = (k + kTm - 1) / kTm;
  g.n_tiles = (g.N + kTn - 1) / kTn;
  const long long tiles = (long long)g.m_tiles * g.n_tiles;
  const long long granules = (g.L + kGranule - 1) / kGranule;
  g.splits = (int)std::max(1LL, std::min({(kTargetCtas + tiles - 1) / tiles, granules, 65535LL}));
  g.part_bytes = ((size_t)g.splits * k * g.N * sizeof(float) + 15) / 16 * 16;
  g.ss_bytes = right ? (size_t)g.splits * g.n_tiles * sizeof(double) : 0;
  return g;
}

int lowrank_check(const char* what, int R, int C, int k, int w_dtype, int m_dtype) {
  if (R < 1 || C < 1 || k < 1) { sm_set_error("%s: R, C and k must be >= 1 (got %d, %d, %d)", what, R, C, k); return -2; }
  if (w_dtype < 0 || w_dtype > 2 || m_dtype < 0 || m_dtype > 2) {
    sm_set_error("%s: dtype codes 0 (fp32), 1 (bf16) or 2 (fp16), got W %d, M %d", what, w_dtype, m_dtype);
    return -2;
  }
  // gridDim.y runs over the 128-wide tiles of the output length (R for right, C for left)
  if ((size_t)(R + kTn - 1) / kTn > 65535u || (size_t)(C + kTn - 1) / kTn > 65535u) {
    sm_set_error("%s: %d x %d exceeds the grid (at most %d rows and columns)", what, R, C, 65535 * kTn);
    return -2;
  }
  return 0;
}

template <bool RIGHT, int WDT>
void launch_m(int m_dtype, dim3 grid, cudaStream_t st, const LowrankArgs& a) {
  if (m_dtype == 0) sm_launch(k_lowrank<RIGHT, WDT, 0>, grid, dim3(kThreads), 0, st, a);
  else if (m_dtype == 1) sm_launch(k_lowrank<RIGHT, WDT, 1>, grid, dim3(kThreads), 0, st, a);
  else sm_launch(k_lowrank<RIGHT, WDT, 2>, grid, dim3(kThreads), 0, st, a);
}

template <bool RIGHT>
int lowrank_run(const char* what, int R, int C, int k, int w_dtype, const void* W, int m_dtype, const void* M,
                const float* S, float* out, double* sumsq, void* ws, size_t ws_bytes, void* stream) {
  if (int rc = lowrank_check(what, R, C, k, w_dtype, m_dtype)) return rc;
  const LowrankGeom g = lowrank_geom(RIGHT, R, C, k);
  const size_t need = g.part_bytes + g.ss_bytes;
  if (ws == nullptr || (uintptr_t)ws % 16 != 0 || ws_bytes < need) {
    sm_set_error("%s: needs a 16-byte aligned workspace of %zu bytes (got %p, %zu; sm_lowrank_ws_bytes)", what, need, ws,
                 ws_bytes);
    return -2;
  }
  LowrankArgs a{};
  a.W = W; a.M = M; a.S = S;
  a.part = static_cast<float*>(ws);
  a.ss_part = (RIGHT && sumsq != nullptr) ? reinterpret_cast<double*>(static_cast<char*>(ws) + g.part_bytes) : nullptr;
  a.R = R; a.C = C; a.k = k; a.L = g.L; a.N = g.N; a.splits = g.splits;
  const int wes = w_dtype == 0 ? 4 : 2, mes = m_dtype == 0 ? 4 : 2;
  a.vec = (uintptr_t)W % 16 == 0 && (uintptr_t)M % 16 == 0 && ((size_t)C * wes) % 16 == 0 && ((size_t)C * mes) % 16 == 0;
  cudaStream_t st = (cudaStream_t)stream;
  const dim3 grid((unsigned)g.m_tiles, (unsigned)g.n_tiles, (unsigned)g.splits);
  if (w_dtype == 0) launch_m<RIGHT, 0>(m_dtype, grid, st, a);
  else if (w_dtype == 1) launch_m<RIGHT, 1>(m_dtype, grid, st, a);
  else launch_m<RIGHT, 2>(m_dtype, grid, st, a);
  SM_LAUNCH_CHECK();
  const size_t total = (size_t)k * g.N;
  const unsigned blocks = (unsigned)std::min<size_t>((total + kReduceThreads - 1) / kReduceThreads, 148 * 16);
  sm_launch(k_lowrank_reduce<RIGHT>, dim3(blocks), dim3(kReduceThreads), 0, st, (const float*)a.part, g.splits, k, g.N,
            out, (const double*)a.ss_part, a.ss_part ? g.splits * g.n_tiles : 0, a.ss_part ? sumsq : nullptr);
  SM_LAUNCH_CHECK();
  return 0;
}

}  // namespace

extern "C" size_t sm_lowrank_ws_bytes(int R, int C, int k) {
  if (R < 1 || C < 1 || k < 1) return 0;
  const LowrankGeom r = lowrank_geom(true, R, C, k), l = lowrank_geom(false, R, C, k);
  return std::max(r.part_bytes + r.ss_bytes, l.part_bytes + l.ss_bytes);
}

extern "C" int sm_lowrank_right(int R, int C, int k, int w_dtype, const void* W, int m_dtype, const void* M,
                                const float* X, float* Y, double* sumsq, void* ws, size_t ws_bytes, void* stream) {
  return lowrank_run<true>("lowrank_right", R, C, k, w_dtype, W, m_dtype, M, X, Y, sumsq, ws, ws_bytes, stream);
}

extern "C" int sm_lowrank_left(int R, int C, int k, int w_dtype, const void* W, int m_dtype, const void* M,
                               const float* Q, float* Z, void* ws, size_t ws_bytes, void* stream) {
  return lowrank_run<false>("lowrank_left", R, C, k, w_dtype, W, m_dtype, M, Q, Z, nullptr, ws, ws_bytes, stream);
}
