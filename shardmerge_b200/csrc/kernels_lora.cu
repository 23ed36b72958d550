// kernels_lora.cu -- the finetuned weight of a PEFT LoRA adapter, formed on the device from its low-rank factors.
//
//   ft[i][j] = round_to_dtype(W)( fp32(W[i][j]) + s * acc[i][j] ),  acc[i][j] = sum_{k=0..r-1} fp32(B[i][k]) * fp32(A[k][j])
//
// W [R][C] is the base tensor, A = lora_A [r][C], B = lora_B [R][r], s the adapter's scaling.  acc is ONE fp32 FMA chain per
// element in ascending k starting from 0; s * acc and the add to W are rounded separately (no contraction), and the sum is
// rounded to W's dtype with RNE.  That is merge_and_unload on an fp32 copy of the base, up to the order of the fp32 sums.
//
// Each 256-thread CTA owns a 64-row x 128-column tile; a thread owns 4 rows x 8 adjacent columns (16 bytes of a bf16 / fp16
// row), carried as 4 rows x 4 column pairs in packed f32x2 registers (FFMA2).  The tile's B rows and A columns are staged in
// shared memory through chunks of kKc values of k, so any r >= 1 keeps the exact ascending chain.  HBM traffic is the base
// read and the result write (2N + 2N bytes for bf16) plus the factors, which the CTAs of a tile column share through L2;
// the kernel does r FMAs per element.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
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

template <int DT> struct LoraCodec;
template <> struct LoraCodec<0> {                    // fp32
  __device__ static float load(const void* p, size_t i) { return __ldg(reinterpret_cast<const float*>(p) + i); }
  __device__ static void load8(const void* p, size_t i, float (&f)[8]) {
    const float4* q = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p) + i);
    const float4 a = __ldg(q), b = __ldg(q + 1);
    f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
  }
  __device__ static void store(void* p, size_t i, float v) { reinterpret_cast<float*>(p)[i] = v; }
  __device__ static void store8(void* p, size_t i, const float (&o)[8]) {
    float4* q = reinterpret_cast<float4*>(reinterpret_cast<float*>(p) + i);
    q[0] = make_float4(o[0], o[1], o[2], o[3]); q[1] = make_float4(o[4], o[5], o[6], o[7]);
  }
};
template <> struct LoraCodec<1> {                    // bf16
  __device__ static float h2f(uint32_t u) { return __uint_as_float(u << 16); }
  __device__ static uint32_t f2h(float x) { __nv_bfloat16 h = __float2bfloat16_rn(x); return *reinterpret_cast<uint16_t*>(&h); }
  __device__ static float load(const void* p, size_t i) { return h2f(__ldg(reinterpret_cast<const uint16_t*>(p) + i)); }
  __device__ static void load8(const void* p, size_t i, float (&f)[8]) {
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(p) + i));
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) { f[2 * e] = h2f(w[e] & 0xffffu); f[2 * e + 1] = h2f(w[e] >> 16); }
  }
  __device__ static void store(void* p, size_t i, float v) { reinterpret_cast<uint16_t*>(p)[i] = (uint16_t)f2h(v); }
  __device__ static void store8(void* p, size_t i, const float (&o)[8]) {
    uint32_t w[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) w[e] = f2h(o[2 * e]) | (f2h(o[2 * e + 1]) << 16);
    *reinterpret_cast<uint4*>(reinterpret_cast<uint16_t*>(p) + i) = make_uint4(w[0], w[1], w[2], w[3]);
  }
};
template <> struct LoraCodec<2> {                    // fp16
  __device__ static float h2f(uint32_t u) { const uint16_t s = (uint16_t)u; return __half2float(*reinterpret_cast<const __half*>(&s)); }
  __device__ static uint32_t f2h(float x) { __half h = __float2half_rn(x); return *reinterpret_cast<uint16_t*>(&h); }
  __device__ static float load(const void* p, size_t i) { return h2f(__ldg(reinterpret_cast<const uint16_t*>(p) + i)); }
  __device__ static void load8(const void* p, size_t i, float (&f)[8]) {
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(p) + i));
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) { f[2 * e] = h2f(w[e] & 0xffffu); f[2 * e + 1] = h2f(w[e] >> 16); }
  }
  __device__ static void store(void* p, size_t i, float v) { reinterpret_cast<uint16_t*>(p)[i] = (uint16_t)f2h(v); }
  __device__ static void store8(void* p, size_t i, const float (&o)[8]) {
    uint32_t w[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) w[e] = f2h(o[2 * e]) | (f2h(o[2 * e + 1]) << 16);
    *reinterpret_cast<uint4*>(reinterpret_cast<uint16_t*>(p) + i) = make_uint4(w[0], w[1], w[2], w[3]);
  }
};

struct LoraArgs {
  const void* base; const void* A; const void* B; void* out;
  int R, C, r;
  float scaling;
  int vec;                 // 1: every 8-column group that lies inside the row is one 16-byte-aligned vector (or two for fp32)
};

// Shared layout of an A chunk row: column c of the tile sits at (c / 8) * 4 + (c % 4) + ((c % 8) / 4) * 64, so the two
// 4-column halves a thread reads are contiguous across the 16 column groups of a half-warp (conflict-free 16-byte loads).
__device__ __forceinline__ int a_slot(int c) { return ((c >> 3) << 2) + (c & 3) + (((c >> 2) & 1) << 6); }

template <int BDT, int ABDT>
__global__ void __launch_bounds__(kThreads) k_lora_materialize(const __grid_constant__ LoraArgs a) {
  __shared__ __align__(16) float As[kKc][kTn];
  __shared__ __align__(16) float Bs[kKc][kTm + 8];     // padded row: the transposing stores hit distinct banks
  sm_pdl_enter();
  using Ab = LoraCodec<ABDT>;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int r0 = blockIdx.y * kTm, c0 = blockIdx.x * kTn;

  pf acc[kRowsPerThread][kColsPerThread / 2];
#pragma unroll
  for (int q = 0; q < kRowsPerThread; ++q)
#pragma unroll
    for (int p = 0; p < kColsPerThread / 2; ++p) acc[q][p] = pf_make(0.f, 0.f);

  for (int k0 = 0; k0 < a.r; k0 += kKc) {
    const int kc = min(kKc, a.r - k0);
    __syncthreads();                                   // the previous chunk has been consumed
    for (int idx = tid; idx < kKc * kTn; idx += kThreads) {
      const int kk = idx / kTn, cc = idx % kTn, c = c0 + cc;
      As[kk][a_slot(cc)] = (kk < kc && c < a.C) ? Ab::load(a.A, (size_t)(k0 + kk) * a.C + c) : 0.f;
    }
    for (int idx = tid; idx < kKc * kTm; idx += kThreads) {
      // a warp stages 4 consecutive k of 8 rows: 8-byte runs of B in global memory, 32 distinct banks in Bs
      const int lane = idx & 31, grp = idx >> 5;
      const int kk = (lane & 3) + 4 * (grp & 7), rr = (lane >> 2) + 8 * (grp >> 3), row = r0 + rr;
      Bs[kk][rr] = (kk < kc && row < a.R) ? Ab::load(a.B, (size_t)row * a.r + k0 + kk) : 0.f;
    }
    __syncthreads();
    for (int kk = 0; kk < kc; ++kk) {                  // ascending k: one FMA per term, the exact chain of the definition
      const float4 b4 = *reinterpret_cast<const float4*>(&Bs[kk][ty * kRowsPerThread]);
      const float4 lo = *reinterpret_cast<const float4*>(&As[kk][tx * 4]);
      const float4 hi = *reinterpret_cast<const float4*>(&As[kk][64 + tx * 4]);
      const pf av[4] = {pf_make(lo.x, lo.y), pf_make(lo.z, lo.w), pf_make(hi.x, hi.y), pf_make(hi.z, hi.w)};
      const float bv[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int q = 0; q < kRowsPerThread; ++q) {
        const pf bb = pf_make(bv[q], bv[q]);
#pragma unroll
        for (int p = 0; p < 4; ++p) acc[q][p] = pf_fma(bb, av[p], acc[q][p]);
      }
    }
  }

  using Bc = LoraCodec<BDT>;
  const int col = c0 + tx * kColsPerThread;
  if (col >= a.C) return;
  const bool full = a.vec && col + kColsPerThread <= a.C;
#pragma unroll
  for (int q = 0; q < kRowsPerThread; ++q) {
    const int row = r0 + ty * kRowsPerThread + q;
    if (row >= a.R) break;
    const size_t off = (size_t)row * a.C + col;
    float w[8], o[8], d[8];
#pragma unroll
    for (int p = 0; p < 4; ++p) { d[2 * p] = pf_lo(acc[q][p]); d[2 * p + 1] = pf_hi(acc[q][p]); }
    if (full) {
      Bc::load8(a.base, off, w);
#pragma unroll
      for (int e = 0; e < 8; ++e) o[e] = __fadd_rn(w[e], __fmul_rn(a.scaling, d[e]));
      Bc::store8(a.out, off, o);
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e)
        if (col + e < a.C) Bc::store(a.out, off + e, __fadd_rn(Bc::load(a.base, off + e), __fmul_rn(a.scaling, d[e])));
    }
  }
}

template <int BDT>
void launch_ab(int ab_dtype, dim3 grid, cudaStream_t st, const LoraArgs& a) {
  if (ab_dtype == 0) sm_launch(k_lora_materialize<BDT, 0>, grid, dim3(kThreads), 0, st, a);
  else if (ab_dtype == 1) sm_launch(k_lora_materialize<BDT, 1>, grid, dim3(kThreads), 0, st, a);
  else sm_launch(k_lora_materialize<BDT, 2>, grid, dim3(kThreads), 0, st, a);
}

}  // namespace

extern "C" int sm_lora_materialize(int R, int C, int r, int base_dtype, const void* base, int ab_dtype, const void* lora_A,
                                   const void* lora_B, float scaling, void* ft_out, void* stream) {
  if (R < 1 || C < 1 || r < 1) { sm_set_error("lora_materialize: R, C and r must be >= 1 (got %d, %d, %d)", R, C, r); return -2; }
  if (base_dtype < 0 || base_dtype > 2 || ab_dtype < 0 || ab_dtype > 2) {
    sm_set_error("lora_materialize: dtype codes 0 (fp32), 1 (bf16) or 2 (fp16), got base %d, factors %d", base_dtype, ab_dtype);
    return -2;
  }
  if ((size_t)(R + kTm - 1) / kTm > 65535u) { sm_set_error("lora_materialize: %d rows exceed the grid", R); return -2; }
  LoraArgs a{};
  a.base = base; a.A = lora_A; a.B = lora_B; a.out = ft_out; a.R = R; a.C = C; a.r = r; a.scaling = scaling;
  const int esize = base_dtype == 0 ? 4 : 2;
  a.vec = ((uintptr_t)base % 16 == 0) && ((uintptr_t)ft_out % 16 == 0) && ((size_t)C * esize) % 16 == 0;
  const dim3 grid((unsigned)((C + kTn - 1) / kTn), (unsigned)((R + kTm - 1) / kTm));
  cudaStream_t st = (cudaStream_t)stream;
  if (base_dtype == 0) launch_ab<0>(ab_dtype, grid, st, a);
  else if (base_dtype == 1) launch_ab<1>(ab_dtype, grid, st, a);
  else launch_ab<2>(ab_dtype, grid, st, a);
  SM_LAUNCH_CHECK();
  return 0;
}
