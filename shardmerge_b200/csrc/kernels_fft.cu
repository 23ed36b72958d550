// kernels_fft.cu -- sm_100a kernels for the delta + forward real 2-D FFT and the inverse
// 2-D FFT + epilogue, and the plan part of the C ABI (include/shardmerge_b200.h).
//
// The arithmetic lives in fft_bodies.cuh (host/device); this file supplies the device
// execution policy, the launch geometry and the reductions that need CUDA intrinsics.
#include <cstdarg>
#include <mutex>
#include "fft_bodies.cuh"
#include "sm_internal.h"

using namespace smfft;

// ------------------------------------------------------------------ error plumbing
static thread_local char g_err[512] = "";
void sm_set_error(const char* fmt, ...) {
  va_list ap; va_start(ap, fmt); vsnprintf(g_err, sizeof(g_err), fmt, ap); va_end(ap);
}
extern "C" const char* sm_last_error(void) { return g_err; }
extern "C" int sm_version(void) { return 100; }

// ------------------------------------------------------------------ device exec policy
struct DeviceExec {
  __device__ __forceinline__ int nthreads() const { return (int)blockDim.x; }
  __device__ __forceinline__ int tid_begin() const { return (int)threadIdx.x; }
  __device__ __forceinline__ int tid_end() const { return (int)threadIdx.x + 1; }
  __device__ __forceinline__ void sync() const { __syncthreads(); }
};

extern __shared__ __align__(128) float2 g_dyn_smem[];

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ------------------------------------------------------------------ kernels
__global__ void __launch_bounds__(512) k_row_fwd(const __grid_constant__ SmPlan pl, const __grid_constant__ RowFwdArgs a, const cf* __restrict__ twC,
                                                 const cf* __restrict__ twQ, double* __restrict__ sumsq) {
  sm_pdl_enter();
  DeviceExec ex;
  float accf = 0.f;
  row_fwd_body(ex, pl, (int)blockIdx.x, a, twC, twQ, reinterpret_cast<cf*>(g_dyn_smem), &accf);
  __shared__ double wsum[16];
  double acc = warp_sum((double)accf);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) wsum[wid] = acc;
  __syncthreads();
  if (wid == 0) {
    const int nw = (blockDim.x + 31) >> 5;
    double v = lane < nw ? wsum[lane] : 0.0;
    v = warp_sum(v);
    if (lane == 0) atomicAdd(sumsq, v);
  }
}

__global__ void __launch_bounds__(512) k_row_inv(const __grid_constant__ SmPlan pl, const __grid_constant__ RowInvArgs a, const cf* __restrict__ twC,
                                                 const cf* __restrict__ twQ) {
  sm_pdl_enter();
  DeviceExec ex;
  row_inv_body(ex, pl, (int)blockIdx.x, a, twC, twQ, reinterpret_cast<cf*>(g_dyn_smem));
}

__global__ void __launch_bounds__(512) k_col(const __grid_constant__ SmPlan pl, const __grid_constant__ ColArgs a, const cf* __restrict__ twR) {
  sm_pdl_enter();
  DeviceExec ex;
  col_body(ex, pl, (int)blockIdx.x, (int)blockIdx.y, a, twR, reinterpret_cast<cf*>(g_dyn_smem));
}

// ---- compile-time specialised kernels for the hot shapes (Llama / TinyLlama factorizations)
// paired columns (two adjacent columns per thread, packed f32x2 arithmetic); capping registers for a 7th
// resident CTA was measured slower (spills), so the compiler's own allocation (<= 80 registers) stands
template <int R1, int R2, int NW, bool kInverse, bool kBigTw>
__global__ void __launch_bounds__(NW * 32) k_col_p(const __grid_constant__ ColCtArgs a, const cf* __restrict__ twR) {
  sm_pdl_enter();
  DeviceExec ex;
  col_ct_body_p<R1, R2, NW, kInverse, kBigTw>(ex, (int)blockIdx.x, (int)blockIdx.y, a, twR, reinterpret_cast<pf4*>(g_dyn_smem));
}

template <int R1, int R2, int R3, int NW, bool kInverse, bool kBigTw>
__global__ void __launch_bounds__(NW * 32) k_col_p3(const __grid_constant__ ColCtArgs a, const cf* __restrict__ twR) {
  sm_pdl_enter();
  DeviceExec ex;
  col_ct_body_p3<R1, R2, R3, NW, kInverse, kBigTw>(ex, (int)blockIdx.x, (int)blockIdx.y, a, twR, reinterpret_cast<pf4*>(g_dyn_smem));
}

// ---- mbarrier / bulk-copy primitives (cp.async.bulk, the 1-D TMA path) used by the bulk-copy fed row kernels below ----
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  } while (!ok);
}

template <int R1, int R2, int R3, int R4, int T, bool kPad>
__global__ void __launch_bounds__(T) k_row_fwd_ct(int C, int P, const RowFwdArgs a, const cf* __restrict__ twC,
                                                  const cf* __restrict__ twQ, double* __restrict__ sumsq) {
  sm_pdl_enter();
  DeviceExec ex;
  float accf = 0.f;
  row_fwd_ct_body<R1, R2, R3, R4, T, kPad>(ex, (int)blockIdx.x, C, P, a, twC, twQ, reinterpret_cast<cf*>(g_dyn_smem), &accf);
  __shared__ double wsum[16];
  double acc = warp_sum((double)accf);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) wsum[wid] = acc;
  __syncthreads();
  if (wid == 0) {
    double v = lane < (T + 31) / 32 ? wsum[lane] : 0.0;
    v = warp_sum(v);
    if (lane == 0) atomicAdd(sumsq, v);
  }
}

template <int R1, int R2, int R3, int R4, int T, bool kPad>
__global__ void __launch_bounds__(T) k_row_inv_ct(int C, int P, const RowInvArgs a, const cf* __restrict__ twC,
                                                  const cf* __restrict__ twQ) {
  sm_pdl_enter();
  DeviceExec ex;
  row_inv_ct_body<R1, R2, R3, R4, T, kPad>(ex, (int)blockIdx.x, C, P, a, twC, twQ, reinterpret_cast<cf*>(g_dyn_smem));
}

// ---- persistent row passes fed by bulk asynchronous copies (TMA 1-D, cp.async.bulk + mbarrier) ----
// One CTA walks rows blockIdx.x, blockIdx.x + gridDim.x, ...  The row it will transform next is
// copied global -> shared by the copy engine while it computes the current one: one elected thread
// issues the copy as soon as the stage-1 barrier has released the staging buffer, every thread waits
// on the mbarrier before stage 1 of the next row.  No thread ever stalls on a global load.
struct FwdStageHook {          // refill the input staging buffer with the CTA's next row
  const RowFwdArgs* a; int next_row, R, C; char* stage; uint64_t* bar;
  __device__ __forceinline__ void after_first_stage() const {
    if (threadIdx.x == 0 && next_row < R) {
      if (a->mode == 0) {
        mbar_expect_tx(bar, 4u * (uint32_t)C);
        bulk_g2s(stage, a->base + (size_t)next_row * C, 2u * (uint32_t)C, bar);
        bulk_g2s(stage + 2 * (size_t)C, a->ft + (size_t)next_row * C, 2u * (uint32_t)C, bar);
      } else {
        mbar_expect_tx(bar, 4u * (uint32_t)C);
        bulk_g2s(stage, a->x32 + (size_t)next_row * C, 4u * (uint32_t)C, bar);
      }
    }
  }
};

template <int R1, int R2, int R3, int R4, int T, bool kPad>
__global__ void __launch_bounds__(T) k_row_fwd_tma(int R, int C, int P, const __grid_constant__ RowFwdArgs a,
                                                   const cf* __restrict__ twC, const cf* __restrict__ twQ,
                                                   double* __restrict__ sumsq, int work_bytes) {
  sm_pdl_enter();
  DeviceExec ex;
  __shared__ uint64_t full;
  __shared__ double wsum[16];
  cf* work = reinterpret_cast<cf*>(g_dyn_smem);
  char* stage = reinterpret_cast<char*>(g_dyn_smem) + work_bytes;
  if (threadIdx.x == 0) { mbar_init(&full, 1); mbar_fence_init(); }
  __syncthreads();
  FwdStageHook hook{&a, (int)blockIdx.x, R, C, stage, &full};
  hook.after_first_stage();                       // first row of this CTA
  uint32_t phase = 0;
  double accd = 0.0;
  for (int row = blockIdx.x; row < R; row += gridDim.x) {
    mbar_wait(&full, phase); phase ^= 1u;
    float accf = 0.f;
    RowDeltaStagedSrc src;
    src.mode = a.mode;
    src.b32 = reinterpret_cast<const uint32_t*>(stage);
    src.f32 = reinterpret_cast<const uint32_t*>(stage + 2 * (size_t)C);
    src.x32 = reinterpret_cast<const cf*>(stage);
    src.m1 = a.m1; src.m2 = a.m2; src.acc = &accf;
    hook.next_row = row + gridDim.x;
    row_fwd_ct_stages<R1, R2, R3, R4, T, kPad>(ex, src, a.re + (size_t)row * P, a.im + (size_t)row * P, twC, twQ, work, hook);
    accd += (double)accf;                          // fp32 over one row's share, fp64 across rows
  }
  double acc = warp_sum(accd);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) wsum[wid] = acc;
  __syncthreads();
  if (wid == 0) {
    double v = lane < (T + 31) / 32 ? wsum[lane] : 0.0;
    v = warp_sum(v);
    if (lane == 0) atomicAdd(sumsq, v);
  }
}

struct InvStageHook {          // refill the spectrum staging (re, im rows) with the CTA's next row
  const float* re; const float* im; int next_row, R, P; char* st_re; char* st_im; uint64_t* bar;
  __device__ __forceinline__ void after_first_stage() const {
    if (threadIdx.x == 0 && next_row < R) {
      mbar_expect_tx(bar, 8u * (uint32_t)P);
      bulk_g2s(st_re, re + (size_t)next_row * P, 4u * (uint32_t)P, bar);
      bulk_g2s(st_im, im + (size_t)next_row * P, 4u * (uint32_t)P, bar);
    }
  }
};

template <int R1, int R2, int R3, int R4, int T, bool kPad>
__global__ void __launch_bounds__(T) k_row_inv_tma(int R, int C, int P, const __grid_constant__ RowInvArgs a,
                                                   const cf* __restrict__ twC, const cf* __restrict__ twQ, int work_bytes) {
  sm_pdl_enter();
  constexpr int CH = R1 * R2 * R3 * R4;
  DeviceExec ex;
  __shared__ uint64_t full_spec, full_base;
  cf* work = reinterpret_cast<cf*>(g_dyn_smem);
  char* st_re = reinterpret_cast<char*>(g_dyn_smem) + work_bytes;
  char* st_im = st_re + 4 * (size_t)P;
  char* st_base = st_im + 4 * (size_t)P;
  if (threadIdx.x == 0) { mbar_init(&full_spec, 1); mbar_init(&full_base, 1); mbar_fence_init(); }
  __syncthreads();
  const float* im = (a.sel != nullptr && *a.sel != 0) ? a.im_alt : a.im;
  InvStageHook hook{a.re, im, (int)blockIdx.x, R, P, st_re, st_im, &full_spec};
  hook.after_first_stage();
  auto load_base = [&](int row) {
    if (threadIdx.x == 0 && row < R && a.out_mode == 0) {
      mbar_expect_tx(&full_base, 2u * (uint32_t)C);
      bulk_g2s(st_base, a.base + (size_t)row * C, 2u * (uint32_t)C, &full_base);
    }
  };
  load_base((int)blockIdx.x);
  RowTangleStagedSrc gsrc;
  gsrc.re = reinterpret_cast<const float*>(st_re); gsrc.im = reinterpret_cast<const float*>(st_im);
  gsrc.twC = twC; gsrc.Ch = CH;
  gsrc.thr = (a.cull_thr != nullptr) ? *a.cull_thr : 0.f;
  RowEpilogueStagedDst gdst;
  gdst.out_mode = a.out_mode;
  gdst.base32 = reinterpret_cast<const uint32_t*>(st_base);
  gdst.inv_n = a.inv_n; gdst.check = a.check_ifft;
  gdst.scale = a.scale_ptr ? *a.scale_ptr : a.scale_host;
  gdst.flags = a.flags;
  uint32_t phase = 0;
  for (int row = blockIdx.x; row < R; row += gridDim.x) {
    gdst.out32 = a.out_mode == 0 ? reinterpret_cast<uint32_t*>(a.out_bf16 + (size_t)row * C) : nullptr;
    gdst.outf = a.out_mode != 0 ? reinterpret_cast<cf*>(a.out_f32 + (size_t)row * C) : nullptr;
    mbar_wait(&full_spec, phase);
    if (a.out_mode == 0) mbar_wait(&full_base, phase);
    phase ^= 1u;
    hook.next_row = row + gridDim.x;
    row_inv_ct_stages<R1, R2, R3, R4, T, kPad>(ex, gsrc, gdst, twC, twQ, work, hook);
    load_base(row + gridDim.x);                    // the last stage (the only reader of the base row) has passed its barrier
  }
}

// ---- paired-row forward pass: two adjacent rows per CTA, carried through the butterflies as the two lanes of
// packed f32x2 values (FADD2 / FMUL2 / FFMA2) ------------------------------------------------------------------
// k_row_fwd_tma is instruction-issue bound (63 % issue slots, 97 instructions per complex point,
// profiles/r01_ncu_full_rows_tma_raw.csv).  Here every FP, shared-memory and index instruction serves two rows,
// and the untangle is fused into the last stage: thread t owns the last-stage butterflies t and s - t, whose
// outputs are each other's mirror images (n <-> Ch - n), so the Hermitian half spectrum is formed in registers
// (one shared-memory write and two reads per point less, one barrier less, each mirror pair computed once).
// One work buffer: stage 1 fills it, stage 2 runs in place (a barrier between its loads and its stores), stage 3
// only reads it.  Shapes: Ch = R1*R2*R3 with Ch / R3 == 2 * T (C = 4096: 16 x 16 x 8, T = 128).  Each lane rounds
// exactly like the scalar kernel up to the untangle, which takes W^(Ch-n) = -conj(W^n) from the same table entry.
struct RowSmem2 {               // [phys(i)] of (re_row0, re_row1, im_row0, im_row1); 1-in-16 padding like RowSmem
  ulonglong2* buf;
  __device__ __forceinline__ static int phys(int i) { return i + (i >> 4); }
#if defined(__CUDA_ARCH__)      // pf is a 64-bit register pair on the device only
  __device__ __forceinline__ void load(int i, pf& re, pf& im) const { const ulonglong2 v = buf[phys(i)]; re.v = v.x; im.v = v.y; }
  __device__ __forceinline__ void store(int i, pf re, pf im) const { buf[phys(i)] = make_ulonglong2(re.v, im.v); }
#else
  void load(int, pf&, pf&) const {}
  void store(int, pf, pf) const {}
#endif
};

struct RowDeltaStaged2 {        // stage-1 source: staging = [base row0 | base row1 | ft row0 | ft row1], bf16
  const uint32_t* b32; const uint32_t* f32; int half; pf* acc;       // half = words per row
  __device__ __forceinline__ void load(int i, pf& re, pf& im) const {
    const uint32_t b0 = b32[i], b1 = b32[half + i], f0 = f32[i], f1 = f32[half + i];
    re = pf_make(bf16_bits_to_f32(f0 & 0xffffu), bf16_bits_to_f32(f1 & 0xffffu)) -
         pf_make(bf16_bits_to_f32(b0 & 0xffffu), bf16_bits_to_f32(b1 & 0xffffu));
    im = pf_make(bits_f32(f0 & 0xffff0000u), bits_f32(f1 & 0xffff0000u)) -
         pf_make(bits_f32(b0 & 0xffff0000u), bits_f32(b1 & 0xffff0000u));
    *acc = pf_fma(re, re, pf_fma(im, im, *acc));
  }
};

// X[n] and X[Ch - n] of both lanes from Z[n] = (ar, ai) and Z[Ch - n] = (br, bi); w = W_C^n; lane 0 -> (reA, imA),
// lane 1 -> (reB, imB)
__device__ __forceinline__ void untangle_pair2(pf ar, pf ai, pf br, pf bi, cf w, float* reA, float* imA, float* reB, float* imB,
                                               int n, int m) {
  const pf h = pf_bcast(0.5f);
  const pf er = h * (ar + br), ei = h * (ai - bi), pr = h * (ai + bi), qi = zero_of(ar) - h * (ar - br);
  const pf wx = pf_bcast(w.x), wy = pf_bcast(w.y);
  const pf tr = pf_fma(pr, wx, zero_of(ar) - qi * wy);       // pr * w.x - qi * w.y
  const pf ti = pf_fma(pr, wy, qi * wx);                      // pr * w.y + qi * w.x
  const pf xr = er + tr, xi = ei + ti;
  reA[n] = pf_lo(xr); reB[n] = pf_hi(xr); imA[n] = pf_lo(xi); imB[n] = pf_hi(xi);
  if (m != n) {
    const pf yr = er - tr, yi = ti - ei;
    reA[m] = pf_lo(yr); reB[m] = pf_hi(yr); imA[m] = pf_lo(yi); imB[m] = pf_hi(yi);
  }
}
// two adjacent rows: lane 1 is the row below lane 0's
__device__ __forceinline__ void untangle_pair2(pf ar, pf ai, pf br, pf bi, cf w, float* re0, float* im0, int P, int n, int m) {
  untangle_pair2(ar, ai, br, bi, w, re0, im0, re0 + P, im0 + P, n, m);
}

// ---- both finetunes of a pair merge over ONE base (sm_fwd_rows_bf16_pair): the same row of model 0 and model 1 in one
// CTA, so the base row is staged (k_row2_fwd) or fetched from HBM (k_row1_fwd_eo) once for both.  Per model the arithmetic
// is that of the single-model pass.  The second model's tensors and the pair merge's scalar block:
struct RowFwdPair {
  const uint16_t* ft1; float* re1; float* im1;
  unsigned char* ctl; double target_norm_offset, ext_tn;
};

struct RowDeltaStagedPair {     // stage-1 source: staging = [base row | ft0 row | ft1 row], bf16; lane k = ft_k - base
  const uint32_t* b32; const uint32_t* f0; const uint32_t* f1; pf* acc;
  __device__ __forceinline__ void load(int i, pf& re, pf& im) const {
    const uint32_t b = b32[i], g0 = f0[i], g1 = f1[i];
    const float br = bf16_bits_to_f32(b & 0xffffu), bi = bits_f32(b & 0xffff0000u);
    re = pf_make(bf16_bits_to_f32(g0 & 0xffffu), bf16_bits_to_f32(g1 & 0xffffu)) - pf_make(br, br);
    im = pf_make(bits_f32(g0 & 0xffff0000u), bits_f32(g1 & 0xffff0000u)) - pf_make(bi, bi);
    *acc = pf_fma(re, re, pf_fma(im, im, *acc));
  }
};

// End of a paired pass: the per-thread fp64 sums of squares of model 0 / model 1 -> sumsq[0], sumsq[1]; the last CTA to
// finish then makes the pair merge's decisions from the two totals, as k_prepare (pipeline.cu) does after two single-model
// passes.  The ticket word is zeroed with the rest of the scalar block before the pass.
template <int T>
__device__ __forceinline__ void row_pair_finish(double acc0, double acc1, double* sumsq, const RowFwdPair& pr) {
  constexpr int NW = (T + 31) / 32;
  __shared__ double wsum[2][NW];
  acc0 = warp_sum(acc0);
  acc1 = warp_sum(acc1);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) { wsum[0][wid] = acc0; wsum[1][wid] = acc1; }
  __syncthreads();
  if (wid != 0) return;
  double v0 = lane < NW ? wsum[0][lane] : 0.0, v1 = lane < NW ? wsum[1][lane] : 0.0;
  v0 = warp_sum(v0);
  v1 = warp_sum(v1);
  if (lane != 0) return;
  atomicAdd(sumsq, v0);
  atomicAdd(sumsq + 1, v1);
  __threadfence();
  if (atomicAdd(reinterpret_cast<unsigned int*>(pr.ctl + SM_CTL_TICKET), 1u) != gridDim.x - 1u) return;
  __threadfence();
  sm_prepare_scalars(pr.ctl, __ldcg(sumsq), __ldcg(sumsq + 1), pr.target_norm_offset, pr.ext_tn);
}

// kEO: the two lanes are the even / odd halves of ONE row instead of two rows (see k_row1_fwd_eo below): C = 8192 then has
// the staging and work-buffer footprint of a C = 4096 row pair and runs through this three-stage, bulk-copy fed kernel
__device__ __forceinline__ void untangle_pair1(float ar, float ai, float br, float bi, cf w, float* re0, float* im0, int n, int m);
__device__ __forceinline__ void combine_untangle4(pf xr, pf xi, pf yr, pf yi, const cf* __restrict__ twC, float* re0, float* im0,
                                                  int n, int H);
struct RowDeltaStagedEO {        // stage-1 source: complex elements 2i (lane 0) and 2i + 1 (lane 1) of one staged row
  const uint2* b64; const uint2* f64; pf* acc;
  __device__ __forceinline__ void load(int i, pf& re, pf& im) const {
    const uint2 b = b64[i], f = f64[i];
    re = pf_make(bf16_bits_to_f32(f.x & 0xffffu), bf16_bits_to_f32(f.y & 0xffffu)) -
         pf_make(bf16_bits_to_f32(b.x & 0xffffu), bf16_bits_to_f32(b.y & 0xffffu));
    im = pf_make(bits_f32(f.x & 0xffff0000u), bits_f32(f.y & 0xffff0000u)) -
         pf_make(bits_f32(b.x & 0xffff0000u), bits_f32(b.y & 0xffff0000u));
    *acc = pf_fma(re, re, pf_fma(im, im, *acc));
  }
};

// kPair: the lanes are row r of model 0 (a.ft, a.re, a.im) and row r of model 1 (pr): sm_fwd_rows_bf16_pair
template <int R1, int R2, int R3, int T, bool kEO, bool kPair = false>
__global__ void __launch_bounds__(T, 3) k_row2_fwd(int R, int C, int P, const __grid_constant__ RowFwdArgs a,
                                                const cf* __restrict__ twC, const cf* __restrict__ twQ,
                                                double* __restrict__ sumsq, int work_bytes, const __grid_constant__ RowFwdPair pr) {
  static_assert(!(kEO && kPair), "k_row2_fwd: the lanes are either even / odd halves or two models");
  sm_pdl_enter();
  constexpr int CH = R1 * R2 * R3;
  constexpr int S3 = CH / R3;                       // stride (and butterfly count) of the last stage
  static_assert(CH / R1 == T && CH / R2 == T && S3 == 2 * T, "k_row2_fwd: one butterfly per thread in stages 1-2, two in stage 3");
  __shared__ uint64_t full;
  __shared__ double wsum[16];
  RowSmem2 sm{reinterpret_cast<ulonglong2*>(g_dyn_smem)};
  char* stage = reinterpret_cast<char*>(g_dyn_smem) + work_bytes;
  const int tid = threadIdx.x;
  constexpr int kRows = (kEO || kPair) ? 1 : 2;     // rows per iteration, per tensor
  constexpr int kTw = kEO ? 4 : 2;                  // W_CH^e = twC[e * kTw]
  const int npairs = (kEO || kPair) ? R : (R >> 1);
  const uint32_t row_bytes = 2u * (uint32_t)C * kRows;    // bf16 bytes of one iteration's rows, per tensor
  if (tid == 0) { mbar_init(&full, 1); mbar_fence_init(); }
  __syncthreads();
  auto prefetch = [&](int pair) {                   // the rows of an iteration are contiguous: one bulk copy per tensor
    if (tid == 0 && pair < npairs) {
      mbar_expect_tx(&full, (kPair ? 3u : 2u) * row_bytes);
      bulk_g2s(stage, a.base + (size_t)pair * kRows * C, row_bytes, &full);
      bulk_g2s(stage + row_bytes, a.ft + (size_t)pair * kRows * C, row_bytes, &full);
      if constexpr (kPair) bulk_g2s(stage + 2 * row_bytes, pr.ft1 + (size_t)pair * C, row_bytes, &full);
    }
  };
  prefetch((int)blockIdx.x);
  uint32_t phase = 0;
  double accd = 0.0, accd1 = 0.0;                   // accd1: model 1 of a paired pass
  // every twiddle of this thread is the same for all row pairs; the loads are issued ahead of the barrier / wait that
  // precedes their use, so their latency is never exposed (the kernel is latency bound: 3 CTAs of 4 warps per SM)
  const int p2 = tid / R1, q2 = tid - p2 * R1;
  const int obase2 = q2 + R1 * R2 * p2, tstep2 = R1 * p2 * kTw;
  const int bA = tid, bB = tid == 0 ? S3 / 2 : S3 - tid;
  for (int pair = blockIdx.x; pair < npairs; pair += gridDim.x) {
    pf accp = pf_make(0.f, 0.f);
    {  // stage 1: delta + radix R1 (s = 1), first-stage quad twiddles (formed while the bulk copy lands)
      float wr[R1], wi[R1];
      quad_twiddles<R1>(twQ, tid, wr, wi, kEO ? 2 : 1);
      mbar_wait(&full, phase); phase ^= 1u;
      pf re[R1], im[R1];
      constexpr int Nr = CH / R1;
      if constexpr (kEO) {
        RowDeltaStagedEO src{reinterpret_cast<const uint2*>(stage), reinterpret_cast<const uint2*>(stage + row_bytes), &accp};
#pragma unroll
        for (int j = 0; j < R1; ++j) src.load(tid + j * Nr, re[j], im[j]);
      } else if constexpr (kPair) {
        RowDeltaStagedPair src{reinterpret_cast<const uint32_t*>(stage), reinterpret_cast<const uint32_t*>(stage + row_bytes),
                               reinterpret_cast<const uint32_t*>(stage + 2 * row_bytes), &accp};
#pragma unroll
        for (int j = 0; j < R1; ++j) src.load(tid + j * Nr, re[j], im[j]);
      } else {
        RowDeltaStaged2 src{reinterpret_cast<const uint32_t*>(stage), reinterpret_cast<const uint32_t*>(stage + row_bytes), C / 2, &accp};
#pragma unroll
        for (int j = 0; j < R1; ++j) src.load(tid + j * Nr, re[j], im[j]);
      }
      Dft<R1>::run(re, im);
      sm.store(R1 * tid, re[0], im[0]);
#pragma unroll
      for (int k = 1; k < R1; ++k) {
        pf xr = re[k], xi = im[k];
        cmul(xr, xi, wr[k], wi[k]);
        sm.store(R1 * tid + k, xr, xi);
      }
    }
    __syncthreads();
    prefetch(pair + (int)gridDim.x);                // the staging buffer is free again
    {  // stage 2: radix R2, s = R1, in place
      cf w[R2];
#pragma unroll
      for (int k = 1; k < R2; ++k) w[k] = ldg_cf(twC + tstep2 * k);
      pf re[R2], im[R2];
      constexpr int Nr = CH / R2;
#pragma unroll
      for (int j = 0; j < R2; ++j) sm.load(tid + j * Nr, re[j], im[j]);
      __syncthreads();
      Dft<R2>::run(re, im);
      sm.store(obase2, re[0], im[0]);
#pragma unroll
      for (int k = 1; k < R2; ++k) {
        pf xr = re[k], xi = im[k];
        cmul(xr, xi, w[k].x, w[k].y);
        sm.store(obase2 + k * R1, xr, xi);
      }
    }
    __syncthreads();
    if constexpr (kEO) {  // stage 3 on the butterflies t and S3 - t, then radix-2 combine + untangle (as in k_row1_fwd_eo)
      pf ar[R3], ai[R3], br[R3], bi[R3];
#pragma unroll
      for (int j = 0; j < R3; ++j) { sm.load(bA + j * S3, ar[j], ai[j]); sm.load(bB + j * S3, br[j], bi[j]); }
      __syncthreads();                              // the buffer has been read: the next row's stage 1 may overwrite it
      Dft<R3>::run(ar, ai);
      Dft<R3>::run(br, bi);
      float* re0 = a.re + (size_t)pair * P;
      float* im0 = a.im + (size_t)pair * P;
      if (tid != 0) {
#pragma unroll
        for (int k = 0; k < R3; ++k) combine_untangle4(ar[k], ai[k], br[R3 - 1 - k], bi[R3 - 1 - k], twC, re0, im0, bA + S3 * k, CH);
      } else {
        {  // n = 0: Z[0] = E0 + O0 -> X[0], X[Ch]; Z[CH] = E0 - O0 pairs with itself -> X[CH]
          const float e0r = pf_lo(ar[0]), e0i = pf_lo(ai[0]), o0r = pf_hi(ar[0]), o0i = pf_hi(ai[0]);
          const float zr = e0r + o0r, zi = e0i + o0i;
          re0[0] = zr + zi; im0[0] = 0.f; re0[2 * CH] = zr - zi; im0[2 * CH] = 0.f;
          untangle_pair1(e0r - o0r, e0i - o0i, e0r - o0r, e0i - o0i, ldg_cf(twC + CH), re0, im0, CH, CH);
        }
#pragma unroll
        for (int k = 1; k <= R3 / 2; ++k) combine_untangle4(ar[k], ai[k], ar[R3 - k], ai[R3 - k], twC, re0, im0, S3 * k, CH);
#pragma unroll
        for (int k = 0; k < R3 / 2; ++k) combine_untangle4(br[k], bi[k], br[R3 - 1 - k], bi[R3 - 1 - k], twC, re0, im0, S3 / 2 + S3 * k, CH);
      }
    } else {  // stage 3 (last, no twiddles) on the butterflies t and S3 - t (thread 0: 0 and S3 / 2) + untangle
      cf w[R3];
#pragma unroll
      for (int k = 0; k < R3; ++k) w[k] = ldg_cf(twC + (tid != 0 ? bA + S3 * k : (k <= R3 / 2 ? S3 * k : S3 / 2 + S3 * (k - R3 / 2 - 1))));
      pf ar[R3], ai[R3], br[R3], bi[R3];
#pragma unroll
      for (int j = 0; j < R3; ++j) { sm.load(bA + j * S3, ar[j], ai[j]); sm.load(bB + j * S3, br[j], bi[j]); }
      __syncthreads();                              // the buffer has been read: the next pair's stage 1 may overwrite it
      Dft<R3>::run(ar, ai);
      Dft<R3>::run(br, bi);
      // lane 0 -> (reA, imA), lane 1 -> (reB, imB): the next row of the same model (P floats further), or the same row of
      // model 1
      float* reA = a.re + (size_t)pair * kRows * P;
      float* imA = a.im + (size_t)pair * kRows * P;
      auto untangle = [&](pf ar_, pf ai_, pf br_, pf bi_, cf w_, int n) {
        if constexpr (kPair) untangle_pair2(ar_, ai_, br_, bi_, w_, reA, imA, pr.re1 + (size_t)pair * P, pr.im1 + (size_t)pair * P, n, CH - n);
        else untangle_pair2(ar_, ai_, br_, bi_, w_, reA, imA, P, n, CH - n);
      };
      if (tid != 0) {
#pragma unroll
        for (int k = 0; k < R3; ++k) {              // n = t + S3*k  <->  Ch - n = (S3 - t) + S3*(R3-1-k)
          const int n = bA + S3 * k;
          untangle(ar[k], ai[k], br[R3 - 1 - k], bi[R3 - 1 - k], w[k], n);
        }
      } else {
        // butterfly 0: n = S3*k <-> S3*(R3-k); n = 0 pairs with itself and also yields the Nyquist bin Ch
        {
          const pf h = ar[0], g = ai[0];
          const pf x0 = h + g, xn = h - g;
          float* reB = kPair ? pr.re1 + (size_t)pair * P : reA + P;
          float* imB = kPair ? pr.im1 + (size_t)pair * P : imA + P;
          reA[0] = pf_lo(x0); reB[0] = pf_hi(x0); imA[0] = 0.f; imB[0] = 0.f;
          reA[CH] = pf_lo(xn); reB[CH] = pf_hi(xn); imA[CH] = 0.f; imB[CH] = 0.f;
        }
#pragma unroll
        for (int k = 1; k <= R3 / 2; ++k) {         // w[k] = W^(S3*k)
          const int n = S3 * k;
          untangle(ar[k], ai[k], ar[R3 - k], ai[R3 - k], w[k], n);
        }
        // butterfly S3/2: n = S3/2 + S3*k <-> S3/2 + S3*(R3-1-k); w[R3/2 + 1 + k] = W^(S3/2 + S3*k)
#pragma unroll
        for (int k = 0; k < R3 / 2 - 1; ++k) {
          const int n = S3 / 2 + S3 * k;
          untangle(br[k], bi[k], br[R3 - 1 - k], bi[R3 - 1 - k], w[R3 / 2 + 1 + k], n);
        }
        {                                           // the last pair of that butterfly has no slot left in w[]
          const int k = R3 / 2 - 1, n = S3 / 2 + S3 * k;
          untangle(br[k], bi[k], br[R3 - 1 - k], bi[R3 - 1 - k], ldg_cf(twC + n), n);
        }
      }
    }
    // fp32 over one thread's share of one row, fp64 across
    if constexpr (kPair) { accd += (double)pf_lo(accp); accd1 += (double)pf_hi(accp); }
    else accd += (double)pf_lo(accp) + (double)pf_hi(accp);
  }
  if constexpr (kPair) { row_pair_finish<T>(accd, accd1, sumsq, pr); return; }
  double acc = warp_sum(accd);
  const int lane = tid & 31, wid = tid >> 5;
  if (lane == 0) wsum[wid] = acc;
  __syncthreads();
  if (wid == 0) {
    double v = lane < (T + 31) / 32 ? wsum[lane] : 0.0;
    v = warp_sum(v);
    if (lane == 0) atomicAdd(sumsq, v);
  }
}

// ---- paired-row forward pass, four stages (C = 2048: Ch = 8 x 8 x 4 x 4, T = 128) ----------------------------------
// Same idea as k_row2_fwd without a staging buffer: stage 1 reads the bf16 rows straight from global memory, and one
// thread asks the copy engine to pull the NEXT pair's rows into L2 (cp.async.bulk.prefetch.L2) so those loads are L2
// hits issued behind this pair's compute.  Stages 2 and 3 run in place, stage 4 forms the half spectrum in registers
// (butterflies t and S - t).  The work buffer is padded (RowSmem2X<true>).
__device__ __forceinline__ void bulk_prefetch_l2(const void* src_gmem, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src_gmem), "r"(bytes) : "memory");
}

// kPad = false: no padding (an odd first radix -- stride 7 -- and the later strides are conflict free as they are);
// kPad = true: one 16-byte element of padding per 8 (power-of-two radices: a quarter warp then covers all banks)
template <bool kPad>
struct RowSmem2X {
  ulonglong2* buf;
  __device__ __forceinline__ static int phys(int i) { return kPad ? i + (i >> 3) : i; }
#if defined(__CUDA_ARCH__)
  __device__ __forceinline__ void load(int i, pf& re, pf& im) const { const ulonglong2 v = buf[phys(i)]; re.v = v.x; im.v = v.y; }
  __device__ __forceinline__ void store(int i, pf re, pf im) const { buf[phys(i)] = make_ulonglong2(re.v, im.v); }
#else
  void load(int, pf&, pf&) const {}
  void store(int, pf, pf) const {}
#endif
};

struct RowDeltaGlobal2 {         // stage-1 source: bf16 words of both rows straight from global memory
  const uint32_t* b32; const uint32_t* f32; int half; pf* acc;       // half = words per row
  __device__ __forceinline__ void load(int i, pf& re, pf& im) const {
    const uint32_t b0 = ldg_u32(b32 + i), b1 = ldg_u32(b32 + half + i), f0 = ldg_u32(f32 + i), f1 = ldg_u32(f32 + half + i);
    re = pf_make(bf16_bits_to_f32(f0 & 0xffffu), bf16_bits_to_f32(f1 & 0xffffu)) -
         pf_make(bf16_bits_to_f32(b0 & 0xffffu), bf16_bits_to_f32(b1 & 0xffffu));
    im = pf_make(bits_f32(f0 & 0xffff0000u), bits_f32(f1 & 0xffff0000u)) -
         pf_make(bits_f32(b0 & 0xffff0000u), bits_f32(b1 & 0xffff0000u));
    *acc = pf_fma(re, re, pf_fma(im, im, *acc));
  }
};

template <int R1, int R2, int R3, int R4, int T, int kCtas>
__global__ void __launch_bounds__(T, kCtas) k_row2_fwd4(int R, int C, int P, const __grid_constant__ RowFwdArgs a,
                                                    const cf* __restrict__ twC, const cf* __restrict__ twQ,
                                                    double* __restrict__ sumsq) {
  sm_pdl_enter();
  constexpr int CH = R1 * R2 * R3 * R4;
  constexpr int NB1 = CH / R1, NB2 = CH / R2, NB3 = CH / R3, S4 = CH / R4;
  constexpr int s2 = R1, s3 = R1 * R2;
  constexpr int H2 = NB2 / T;
  static_assert(NB2 == H2 * T && H2 >= 1 && H2 <= 2 && NB3 == 2 * T && S4 == 2 * T, "k_row2_fwd4: 1-2 / 2 / 2 butterflies per thread in stages 2 / 3 / 4");
  __shared__ double wsum[16];
  RowSmem2X<true> sm{reinterpret_cast<ulonglong2*>(g_dyn_smem)};
  const int tid = threadIdx.x;
  const int npairs = R >> 1;
  double accd = 0.0;
  if (tid == 0 && (int)blockIdx.x < npairs) {
    bulk_prefetch_l2(a.base + (size_t)blockIdx.x * 2 * C, 4u * (uint32_t)C);
    bulk_prefetch_l2(a.ft + (size_t)blockIdx.x * 2 * C, 4u * (uint32_t)C);
  }
  for (int pair = blockIdx.x; pair < npairs; pair += gridDim.x) {
    pf accp = pf_make(0.f, 0.f);
    {  // stage 1: delta + radix R1 (s = 1) on the butterflies t, t + T, ... ; first-stage quad twiddles
      RowDeltaGlobal2 src{reinterpret_cast<const uint32_t*>(a.base + (size_t)pair * 2 * C),
                          reinterpret_cast<const uint32_t*>(a.ft + (size_t)pair * 2 * C), C / 2, &accp};
#pragma unroll 1
      for (int b = tid; b < NB1; b += T) stockham_bfly_first<R1, pf>(b, CH, twQ, src, sm);
    }
    __syncthreads();
    if (tid == 0 && pair + (int)gridDim.x < npairs) {   // next pair's rows -> L2 while this pair is transformed
      bulk_prefetch_l2(a.base + (size_t)(pair + gridDim.x) * 2 * C, 4u * (uint32_t)C);
      bulk_prefetch_l2(a.ft + (size_t)(pair + gridDim.x) * 2 * C, 4u * (uint32_t)C);
    }
    {  // stage 2: radix R2, s = R1, in place, butterflies t (and t + T)
      pf re[H2][R2], im[H2][R2];
#pragma unroll
      for (int h = 0; h < H2; ++h)
#pragma unroll
        for (int j = 0; j < R2; ++j) sm.load(tid + h * T + j * NB2, re[h][j], im[h][j]);
      __syncthreads();
#pragma unroll
      for (int h = 0; h < H2; ++h) {
        Dft<R2>::run(re[h], im[h]);
        const int b = tid + h * T;
        const int p = b / s2, q = b - p * s2;
        const int obase = q + s2 * R2 * p, tstep = s2 * p * 2;
        sm.store(obase, re[h][0], im[h][0]);
#pragma unroll
        for (int k = 1; k < R2; ++k) {
          const cf w = ldg_cf(twC + tstep * k);
          pf xr = re[h][k], xi = im[h][k];
          cmul(xr, xi, w.x, w.y);
          sm.store(obase + k * s2, xr, xi);
        }
      }
    }
    __syncthreads();
    {  // stage 3: radix R3, s = R1*R2, in place, butterflies t and t + T
      pf re[2][R3], im[2][R3];
#pragma unroll
      for (int h = 0; h < 2; ++h)
#pragma unroll
        for (int j = 0; j < R3; ++j) sm.load(tid + h * T + j * NB3, re[h][j], im[h][j]);
      __syncthreads();
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        Dft<R3>::run(re[h], im[h]);
        const int b = tid + h * T;
        const int p = b / s3, q = b - p * s3;
        const int obase = q + s3 * R3 * p, tstep = s3 * p * 2;
        sm.store(obase, re[h][0], im[h][0]);
#pragma unroll
        for (int k = 1; k < R3; ++k) {
          const cf w = ldg_cf(twC + tstep * k);
          pf xr = re[h][k], xi = im[h][k];
          cmul(xr, xi, w.x, w.y);
          sm.store(obase + k * s3, xr, xi);
        }
      }
    }
    __syncthreads();
    {  // stage 4 (last, no twiddles) on the butterflies t and S4 - t (thread 0: 0 and S4 / 2) + untangle
      const int bA = tid, bB = tid == 0 ? S4 / 2 : S4 - tid;
      pf ar[R4], ai[R4], br[R4], bi[R4];
#pragma unroll
      for (int j = 0; j < R4; ++j) { sm.load(bA + j * S4, ar[j], ai[j]); sm.load(bB + j * S4, br[j], bi[j]); }
      __syncthreads();                              // the buffer has been read: the next pair's stage 1 may overwrite it
      Dft<R4>::run(ar, ai);
      Dft<R4>::run(br, bi);
      float* re0 = a.re + (size_t)pair * 2 * P;
      float* im0 = a.im + (size_t)pair * 2 * P;
      if (tid != 0) {
#pragma unroll
        for (int k = 0; k < R4; ++k) {              // n = t + S4*k  <->  Ch - n = (S4 - t) + S4*(R4-1-k)
          const int n = bA + S4 * k;
          untangle_pair2(ar[k], ai[k], br[R4 - 1 - k], bi[R4 - 1 - k], ldg_cf(twC + n), re0, im0, P, n, CH - n);
        }
      } else {
        {
          const pf h = ar[0], g = ai[0];
          const pf x0 = h + g, xn = h - g;
          re0[0] = pf_lo(x0); re0[P] = pf_hi(x0); im0[0] = 0.f; im0[P] = 0.f;
          re0[CH] = pf_lo(xn); re0[P + CH] = pf_hi(xn); im0[CH] = 0.f; im0[P + CH] = 0.f;
        }
#pragma unroll
        for (int k = 1; k <= R4 / 2; ++k) {
          const int n = S4 * k;
          untangle_pair2(ar[k], ai[k], ar[R4 - k], ai[R4 - k], ldg_cf(twC + n), re0, im0, P, n, CH - n);
        }
#pragma unroll
        for (int k = 0; k < R4 / 2; ++k) {
          const int n = S4 / 2 + S4 * k;
          untangle_pair2(br[k], bi[k], br[R4 - 1 - k], bi[R4 - 1 - k], ldg_cf(twC + n), re0, im0, P, n, CH - n);
        }
      }
    }
    accd += (double)pf_lo(accp) + (double)pf_hi(accp);
  }
  double acc = warp_sum(accd);
  const int lane = tid & 31, wid = tid >> 5;
  if (lane == 0) wsum[wid] = acc;
  __syncthreads();
  if (wid == 0) {
    double v = lane < (T + 31) / 32 ? wsum[lane] : 0.0;
    v = warp_sum(v);
    if (lane == 0) atomicAdd(sumsq, v);
  }
}

// ---- longest rows (C = 28672, Ch = 14336): ONE row per CTA, the f32x2 lanes carry its even / odd halves ----------------
// Two such rows do not fit one SM (2 x 14336 x 16 B).  Instead the packed length-Ch transform of one row is split by
// decimation in time, Z[k] = E[k] + W_Ch^k O[k], Z[k + Ch/2] = E[k] - W_Ch^k O[k]: E and O are two independent
// transforms of length Ch/2 = 7 x 16 x 8 x 8 over the even / odd complex elements, i.e. exactly the two lanes of the
// four-stage paired engine (one 8-byte load per tensor feeds both).  The last stage then holds E, O at n and at
// Ch/2 - n, which is all the radix-2 combine plus the untangle of the four bins n, n + Ch/2, Ch/2 - n, Ch - n need.
// The one-row scalar kernel k_row_fwd_ct<7,16,16,8,512> moves 2.0 TB/s on these rows (no room for a staging buffer).
struct RowDeltaGlobalEO {        // stage-1 source: complex elements 2i (lane 0) and 2i + 1 (lane 1) of one row
  const uint2* b64; const uint2* f64; pf* acc;
  __device__ __forceinline__ void load(int i, pf& re, pf& im) const {
    const uint2 b = __ldg(b64 + i), f = __ldg(f64 + i);
    re = pf_make(bf16_bits_to_f32(f.x & 0xffffu), bf16_bits_to_f32(f.y & 0xffffu)) -
         pf_make(bf16_bits_to_f32(b.x & 0xffffu), bf16_bits_to_f32(b.y & 0xffffu));
    im = pf_make(bits_f32(f.x & 0xffff0000u), bits_f32(f.y & 0xffff0000u)) -
         pf_make(bits_f32(b.x & 0xffff0000u), bits_f32(b.y & 0xffff0000u));
    *acc = pf_fma(re, re, pf_fma(im, im, *acc));
  }
};

// X[n] and X[m] (m = full length - n) of one row from Z[n] = (ar, ai) and Z[m] = (br, bi); w = W_C^n
__device__ __forceinline__ void untangle_pair1(float ar, float ai, float br, float bi, cf w, float* re0, float* im0, int n, int m) {
  const float er = 0.5f * (ar + br), ei = 0.5f * (ai - bi), pr = 0.5f * (ai + bi), qi = -0.5f * (ar - br);
  const float tr = pr * w.x - qi * w.y, ti = pr * w.y + qi * w.x;
  re0[n] = er + tr; im0[n] = ei + ti;
  if (m != n) { re0[m] = er - tr; im0[m] = ti - ei; }
}

// the four bins n, n + H, H - n, 2H - n (H = Ch/2) from (E, O)[n] = lanes of (xr, xi) and (E, O)[H - n] = lanes of (yr, yi)
__device__ __forceinline__ void combine_untangle4(pf xr, pf xi, pf yr, pf yi, const cf* __restrict__ twC, float* re0, float* im0,
                                                  int n, int H) {
  const int m = H - n;                               // 0 < n < H
  const cf wn = ldg_cf(twC + 2 * n), wm = ldg_cf(twC + 2 * m);        // W_Ch^n, W_Ch^m (the table is W_C, C = 2 Ch)
  float onr = pf_hi(xr), oni = pf_hi(xi), omr = pf_hi(yr), omi = pf_hi(yi);
  cmul(onr, oni, wn.x, wn.y);
  cmul(omr, omi, wm.x, wm.y);
  const float enr = pf_lo(xr), eni = pf_lo(xi), emr = pf_lo(yr), emi = pf_lo(yi);
  // Z[n] = E + wO, Z[n + H] = E - wO; same at m
  untangle_pair1(enr + onr, eni + oni, emr - omr, emi - omi, ldg_cf(twC + n), re0, im0, n, 2 * H - n);      // (n, Ch - n = H + m)
  if (m != n) untangle_pair1(enr - onr, eni - oni, emr + omr, emi + omi, ldg_cf(twC + n + H), re0, im0, n + H, m);   // (n + H, m)
}

// kPair: one CTA transforms row r of model 0 (a.ft, a.re, a.im), then row r of model 1 (pr); the second read of the base
// row hits L2: sm_fwd_rows_bf16_pair
template <int R1, int R2, int R3, int R4, int T, int kCtas, bool kPair = false>
__global__ void __launch_bounds__(T, kCtas) k_row1_fwd_eo(int R, int C, int P, const __grid_constant__ RowFwdArgs a,
                                                      const cf* __restrict__ twC, const cf* __restrict__ twQ2,
                                                      double* __restrict__ sumsq, const __grid_constant__ RowFwdPair pr) {
  sm_pdl_enter();
  constexpr int CH = R1 * R2 * R3 * R4;             // length of the even / odd transforms = Ch / 2
  constexpr int NB1 = CH / R1, NB2 = CH / R2, NB3 = CH / R3, S4 = CH / R4;
  constexpr int s2 = R1, s3 = R1 * R2;
  constexpr int H2 = NB2 / T;
  static_assert(NB2 == H2 * T && H2 >= 1 && H2 <= 2 && NB3 == 2 * T && S4 == 2 * T, "k_row1_fwd_eo: 1-2 / 2 / 2 butterflies per thread in stages 2 / 3 / 4");
  __shared__ double wsum[16];
  RowSmem2X<false> sm{reinterpret_cast<ulonglong2*>(g_dyn_smem)};
  const int tid = threadIdx.x;
  double accd = 0.0, accd1 = 0.0;                   // accd1: model 1 of a paired pass
  if (tid == 0 && (int)blockIdx.x < R) {
    bulk_prefetch_l2(a.base + (size_t)blockIdx.x * C, 2u * (uint32_t)C);
    bulk_prefetch_l2(a.ft + (size_t)blockIdx.x * C, 2u * (uint32_t)C);
  }
  for (int row = blockIdx.x; row < R; row += gridDim.x) {
#pragma unroll 1
    for (int m = 0; m < (kPair ? 2 : 1); ++m) {      // the model of this iteration
      const uint16_t* ft = (kPair && m != 0) ? pr.ft1 : a.ft;
      pf accp = pf_make(0.f, 0.f);
      {  // stage 1: delta + radix R1 (s = 1); the sub-transforms have twiddles W_CH = W_C^4: twiddle tables are read at stride 4
        RowDeltaGlobalEO src{reinterpret_cast<const uint2*>(a.base + (size_t)row * C), reinterpret_cast<const uint2*>(ft + (size_t)row * C), &accp};
#pragma unroll 1
        for (int b = tid; b < NB1; b += T) stockham_bfly_first<R1, pf>(b, CH, twQ2, src, sm, 2);
      }
      __syncthreads();
      if (tid == 0) {                                 // the next iteration's rows -> L2 while this one is transformed
        if (kPair && m == 0) {
          bulk_prefetch_l2(pr.ft1 + (size_t)row * C, 2u * (uint32_t)C);
        } else if (row + (int)gridDim.x < R) {
          bulk_prefetch_l2(a.base + (size_t)(row + gridDim.x) * C, 2u * (uint32_t)C);
          bulk_prefetch_l2(a.ft + (size_t)(row + gridDim.x) * C, 2u * (uint32_t)C);
        }
      }
      {  // stage 2: radix R2, s = R1, in place, butterflies t (and t + T)
        pf re[H2][R2], im[H2][R2];
#pragma unroll
        for (int h = 0; h < H2; ++h)
#pragma unroll
          for (int j = 0; j < R2; ++j) sm.load(tid + h * T + j * NB2, re[h][j], im[h][j]);
        __syncthreads();
#pragma unroll
        for (int h = 0; h < H2; ++h) {
          Dft<R2>::run(re[h], im[h]);
          const int b = tid + h * T;
          const int p = b / s2, q = b - p * s2;
          const int obase = q + s2 * R2 * p, tstep = s2 * p * 4;
          sm.store(obase, re[h][0], im[h][0]);
#pragma unroll
          for (int k = 1; k < R2; ++k) {
            const cf w = ldg_cf(twC + tstep * k);
            pf xr = re[h][k], xi = im[h][k];
            cmul(xr, xi, w.x, w.y);
            sm.store(obase + k * s2, xr, xi);
          }
        }
      }
      __syncthreads();
      {  // stage 3: radix R3, s = R1*R2, in place, butterflies t and t + T
        pf re[2][R3], im[2][R3];
#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
          for (int j = 0; j < R3; ++j) sm.load(tid + h * T + j * NB3, re[h][j], im[h][j]);
        __syncthreads();
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          Dft<R3>::run(re[h], im[h]);
          const int b = tid + h * T;
          const int p = b / s3, q = b - p * s3;
          const int obase = q + s3 * R3 * p, tstep = s3 * p * 4;
          sm.store(obase, re[h][0], im[h][0]);
#pragma unroll
          for (int k = 1; k < R3; ++k) {
            const cf w = ldg_cf(twC + tstep * k);
            pf xr = re[h][k], xi = im[h][k];
            cmul(xr, xi, w.x, w.y);
            sm.store(obase + k * s3, xr, xi);
          }
        }
      }
      __syncthreads();
      {  // stage 4 (last) on the butterflies t and S4 - t (thread 0: 0 and S4 / 2), then combine + untangle
        const int bA = tid, bB = tid == 0 ? S4 / 2 : S4 - tid;
        pf ar[R4], ai[R4], br[R4], bi[R4];
#pragma unroll
        for (int j = 0; j < R4; ++j) { sm.load(bA + j * S4, ar[j], ai[j]); sm.load(bB + j * S4, br[j], bi[j]); }
        __syncthreads();                              // the buffer has been read: the next row's stage 1 may overwrite it
        Dft<R4>::run(ar, ai);
        Dft<R4>::run(br, bi);
        float* re0 = ((kPair && m != 0) ? pr.re1 : a.re) + (size_t)row * P;
        float* im0 = ((kPair && m != 0) ? pr.im1 : a.im) + (size_t)row * P;
        if (tid != 0) {
#pragma unroll
          for (int k = 0; k < R4; ++k)                // n = t + S4*k  <->  CH - n = (S4 - t) + S4*(R4-1-k)
            combine_untangle4(ar[k], ai[k], br[R4 - 1 - k], bi[R4 - 1 - k], twC, re0, im0, bA + S4 * k, CH);
        } else {
          {  // n = 0: Z[0] = E0 + O0 -> X[0], X[Ch]; Z[CH] = E0 - O0 pairs with itself -> X[CH]
            const float e0r = pf_lo(ar[0]), e0i = pf_lo(ai[0]), o0r = pf_hi(ar[0]), o0i = pf_hi(ai[0]);
            const float zr = e0r + o0r, zi = e0i + o0i;
            re0[0] = zr + zi; im0[0] = 0.f; re0[2 * CH] = zr - zi; im0[2 * CH] = 0.f;
            untangle_pair1(e0r - o0r, e0i - o0i, e0r - o0r, e0i - o0i, ldg_cf(twC + CH), re0, im0, CH, CH);
          }
#pragma unroll
          for (int k = 1; k <= R4 / 2; ++k)           // butterfly 0: n = S4*k <-> S4*(R4-k)
            combine_untangle4(ar[k], ai[k], ar[R4 - k], ai[R4 - k], twC, re0, im0, S4 * k, CH);
#pragma unroll
          for (int k = 0; k < R4 / 2; ++k)            // butterfly S4/2: n = S4/2 + S4*k <-> S4/2 + S4*(R4-1-k)
            combine_untangle4(br[k], bi[k], br[R4 - 1 - k], bi[R4 - 1 - k], twC, re0, im0, S4 / 2 + S4 * k, CH);
        }
      }
      if (kPair && m != 0) accd1 += (double)pf_lo(accp) + (double)pf_hi(accp);
      else accd += (double)pf_lo(accp) + (double)pf_hi(accp);
    }
  }
  if constexpr (kPair) { row_pair_finish<T>(accd, accd1, sumsq, pr); return; }
  double acc = warp_sum(accd);
  const int lane = tid & 31, wid = tid >> 5;
  if (lane == 0) wsum[wid] = acc;
  __syncthreads();
  if (wid == 0) {
    double v = lane < (T + 31) / 32 ? wsum[lane] : 0.0;
    v = warp_sum(v);
    if (lane == 0) atomicAdd(sumsq, v);
  }
}

// ---- paired-row inverse pass: the mirror image of k_row2_fwd ------------------------------------------------------
// Two adjacent spectrum rows per CTA as f32x2 lanes: tangle (from the staged re / im rows) + radix R1 with quad
// twiddles -> in-place radix R2 -> radix R3 straight into the epilogue (x 1/N, NaN -> 0 / Inf count, x target_norm,
// + base, NaN -> 0 / Inf count, bf16 RNE).  Only the spectrum is staged by bulk copies; the bf16 base words of a
// thread's outputs are plain loads issued before the last stage's shared-memory reads (their latency is covered by
// the stage), which keeps the CTA at 68 KB of shared memory: 3 CTAs per SM.  Same arithmetic per lane as
// k_row_inv_tma.  No cull on load here (2-D tensors cull in the first inverse column sweep).
struct RowTangleStaged2 {
  const float* re; const float* im; int P; int Ch;
  __device__ __forceinline__ void load(int k, cf w, pf& ore, pf& oim) const {
    pf xr = pf_make(re[k], re[P + k]), xi = pf_make(im[k], im[P + k]);
    pf mr = pf_make(re[Ch - k], re[P + Ch - k]), mi = pf_make(im[Ch - k], im[P + Ch - k]);
    if (k == 0) { xi = pf_make(0.f, 0.f); mi = xi; }    // .real semantics: bins 0 and Ch are real
    const pf Ar = xr + mr, Ai = xi - mi, Br = xr - mr, Bi = xi + mi;
    const pf wx = pf_bcast(w.x), wy = pf_bcast(w.y);
    const pf br = pf_fma(Br, wx, Bi * wy);              // B * conj(w)
    const pf bi = pf_fma(Bi, wx, zero_of(Br) - Br * wy);
    const pf zr = Ar - bi, zi = Ai + br;
    ore = zi; oim = zr;                                 // handed to the forward engine swapped
  }
};

__device__ __forceinline__ float epi_fix(float v, unsigned int* flags, int which) {
  return not_finite(v) ? sm_fix_nonfinite(v, flags, which) : v;
}
// one test for four values: the NaN-propagating maximum of the magnitudes is NaN / Inf iff any of them is
__device__ __forceinline__ float fmax_nan(float x, float y) { float r; asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(x), "f"(y)); return r; }
__device__ __forceinline__ bool any_not_finite4(float a, float b, float c, float d) {
  return not_finite(fmax_nan(fmax_nan(fabsf(a), fabsf(b)), fmax_nan(fabsf(c), fabsf(d))));
}

// y = x * scale (+ base) for four values with the reference's two checks -- ifft output (NaN -> 0, Inf counted: flags 0 / 1),
// merged value (flags 2 / 3).  ONE test on the results covers both in the common case: a non-finite x makes its y non-finite
// too (NaN and Inf propagate through x * scale + base, Inf * 0 = NaN), so only a non-finite y replays the checks in order.
__device__ __forceinline__ void epi_finish4(const RowInvArgs& a, float scale, bool add_base, float x0, float x1, float x2, float x3,
                                            float b0, float b1, float b2, float b3, float& y0, float& y1, float& y2, float& y3) {
  // __fmul_rn / __fadd_rn: one rounding per torch op, never contracted into an FMA
  y0 = __fmul_rn(x0, scale); y1 = __fmul_rn(x1, scale); y2 = __fmul_rn(x2, scale); y3 = __fmul_rn(x3, scale);
  if (add_base) { y0 = __fadd_rn(b0, y0); y1 = __fadd_rn(b1, y1); y2 = __fadd_rn(b2, y2); y3 = __fadd_rn(b3, y3); }
  if (any_not_finite4(y0, y1, y2, y3)) {                   // exceptional
    if (a.check_ifft && any_not_finite4(x0, x1, x2, x3)) {
      x0 = epi_fix(x0, a.flags, 0); x1 = epi_fix(x1, a.flags, 0); x2 = epi_fix(x2, a.flags, 0); x3 = epi_fix(x3, a.flags, 0);
    }
    y0 = __fmul_rn(x0, scale); y1 = __fmul_rn(x1, scale); y2 = __fmul_rn(x2, scale); y3 = __fmul_rn(x3, scale);
    if (add_base) {
      y0 = __fadd_rn(b0, y0); y1 = __fadd_rn(b1, y1); y2 = __fadd_rn(b2, y2); y3 = __fadd_rn(b3, y3);
      if (any_not_finite4(y0, y1, y2, y3)) {
        y0 = epi_fix(y0, a.flags, 2); y1 = epi_fix(y1, a.flags, 2); y2 = epi_fix(y2, a.flags, 2); y3 = epi_fix(y3, a.flags, 2);
      }
    }
  }
}

// element j of the pair: (a, b) = swapped engine output -> x[2j] = b / N, x[2j+1] = a / N for both rows
__device__ __forceinline__ void epilogue_store2(const RowInvArgs& a, float scale, uint32_t bb0, uint32_t bb1, uint32_t* out0,
                                                uint32_t* out1, float* of0, float* of1, int j, pf va, pf vb) {
  const pf n = pf_bcast(a.inv_n);
  pf x0 = vb * n, x1 = va * n;
  float x00 = pf_lo(x0), x01 = pf_hi(x0), x10 = pf_lo(x1), x11 = pf_hi(x1);   // xRC: element R of the pair, row C
  const bool add_base = a.out_mode == 0;
  const float b00 = add_base ? bf16_bits_to_f32(bb0 & 0xffffu) : 0.f, b10 = add_base ? bits_f32(bb0 & 0xffff0000u) : 0.f;
  const float b01 = add_base ? bf16_bits_to_f32(bb1 & 0xffffu) : 0.f, b11 = add_base ? bits_f32(bb1 & 0xffff0000u) : 0.f;
  float y00, y01, y10, y11;
  epi_finish4(a, scale, add_base, x00, x01, x10, x11, b00, b01, b10, b11, y00, y01, y10, y11);
  if (add_base) {
    out0[j] = pack_bf16x2_rne(y00, y10);
    out1[j] = pack_bf16x2_rne(y01, y11);
  } else {
    reinterpret_cast<float2*>(of0)[j] = make_float2(y00, y10);
    reinterpret_cast<float2*>(of1)[j] = make_float2(y01, y11);
  }
}

// Branch-free variants for the last stage's loop over its outputs: store what comes out and fold the magnitudes into `bad`
// (NaN-propagating maximum); the caller tests `bad` ONCE per batch of outputs and, if it is not finite, runs the exact
// epilogue above over the batch again (same addresses: the corrected values overwrite, the flags are counted there only).
// Keeps the batch one basic block: the per-value test of the exact epilogue cut the schedule into 16 pieces per iteration.
__device__ __forceinline__ float fmax3_nan(float x, float y, float z) { return fmax_nan(fmax_nan(x, y), z); }
__device__ __forceinline__ void epilogue_store2_fast(const RowInvArgs& a, float scale, uint32_t bb0, uint32_t bb1, uint32_t* out0,
                                                     uint32_t* out1, float* of0, float* of1, int j, pf va, pf vb, float& bad) {
  const pf n = pf_bcast(a.inv_n);
  const pf x0 = vb * n, x1 = va * n;
  float y00 = __fmul_rn(pf_lo(x0), scale), y01 = __fmul_rn(pf_hi(x0), scale), y10 = __fmul_rn(pf_lo(x1), scale), y11 = __fmul_rn(pf_hi(x1), scale);
  if (a.out_mode == 0) {
    y00 = __fadd_rn(bf16_bits_to_f32(bb0 & 0xffffu), y00); y10 = __fadd_rn(bits_f32(bb0 & 0xffff0000u), y10);
    y01 = __fadd_rn(bf16_bits_to_f32(bb1 & 0xffffu), y01); y11 = __fadd_rn(bits_f32(bb1 & 0xffff0000u), y11);
    out0[j] = pack_bf16x2_rne(y00, y10);
    out1[j] = pack_bf16x2_rne(y01, y11);
  } else {
    reinterpret_cast<float2*>(of0)[j] = make_float2(y00, y10);
    reinterpret_cast<float2*>(of1)[j] = make_float2(y01, y11);
  }
  bad = fmax3_nan(fmax3_nan(bad, fabsf(y00), fabsf(y01)), fabsf(y10), fabsf(y11));
}
__device__ __forceinline__ void epilogue_store_eo_fast(const RowInvArgs& a, float scale, uint2 bb, uint2* out64, float4* of, int m, pf va,
                                                       pf vb, float& bad) {
  const pf n = pf_bcast(a.inv_n);
  const pf x0 = vb * n, x1 = va * n;
  float y00 = __fmul_rn(pf_lo(x0), scale), y01 = __fmul_rn(pf_hi(x0), scale), y10 = __fmul_rn(pf_lo(x1), scale), y11 = __fmul_rn(pf_hi(x1), scale);
  if (a.out_mode == 0) {
    y00 = __fadd_rn(bf16_bits_to_f32(bb.x & 0xffffu), y00); y10 = __fadd_rn(bits_f32(bb.x & 0xffff0000u), y10);
    y01 = __fadd_rn(bf16_bits_to_f32(bb.y & 0xffffu), y01); y11 = __fadd_rn(bits_f32(bb.y & 0xffff0000u), y11);
    out64[m] = make_uint2(pack_bf16x2_rne(y00, y10), pack_bf16x2_rne(y01, y11));
  } else {
    of[m] = make_float4(y00, y10, y01, y11);
  }
  bad = fmax3_nan(fmax3_nan(bad, fabsf(y00), fabsf(y01)), fabsf(y10), fabsf(y11));
}

// kEO: the lanes are the even / odd halves of ONE row (decimation in frequency on the engine's input, see k_row1_inv_eo)
__device__ __forceinline__ void epilogue_store_eo(const RowInvArgs& a, float scale, uint2 bb, uint2* out64, float4* of, int m, pf va, pf vb);
struct RowTangleStagedEO {       // staged spectrum row (re, im), H = Ch / 2
  const float* re; const float* im; const cf* twC; int H;
  __device__ __forceinline__ void tangle(int k, float& ore, float& oim) const {
    float xr = re[k], xi = im[k], mr = re[2 * H - k], mi = im[2 * H - k];
    if (k == 0) { xi = 0.f; mi = 0.f; }
    const float Ar = xr + mr, Ai = xi - mi, Br = xr - mr, Bi = xi + mi;
    const cf w = ldg_cf(twC + k);
    const float br = Br * w.x + Bi * w.y, bi = Bi * w.x - Br * w.y;
    ore = Ai + br; oim = Ar - bi;
  }
  __device__ __forceinline__ void load(int n, pf& ore, pf& oim) const {
    float u1r, u1i, u2r, u2i;
    tangle(n, u1r, u1i);
    tangle(n + H, u2r, u2i);
    float dr = u1r - u2r, di = u1i - u2i;
    const cf w = ldg_cf(twC + 2 * n);                                     // W_Ch^n
    cmul(dr, di, w.x, w.y);
    ore = pf_make(u1r + u2r, dr); oim = pf_make(u1i + u2i, di);
  }
};

template <int R1, int R2, int R3, int T, bool kEO>
__global__ void __launch_bounds__(T, 3) k_row2_inv(int R, int C, int P, const __grid_constant__ RowInvArgs a,
                                                   const cf* __restrict__ twC, const cf* __restrict__ twQ, int work_bytes) {
  sm_pdl_enter();
  constexpr int CH = R1 * R2 * R3;
  constexpr int S3 = CH / R3;
  constexpr int kRows = kEO ? 1 : 2;
  constexpr int kTw = kEO ? 4 : 2;
  static_assert(CH / R1 == T && CH / R2 == T && S3 == 2 * T, "k_row2_inv: one butterfly per thread in stages 1-2, two in stage 3");
  __shared__ uint64_t full;
  RowSmem2 sm{reinterpret_cast<ulonglong2*>(g_dyn_smem)};
  char* st_re = reinterpret_cast<char*>(g_dyn_smem) + work_bytes;
  const uint32_t plane_bytes = 4u * (uint32_t)P * kRows;
  char* st_im = st_re + plane_bytes;
  const int tid = threadIdx.x;
  const int npairs = kEO ? R : (R >> 1);
  if (tid == 0) { mbar_init(&full, 1); mbar_fence_init(); }
  __syncthreads();
  const float* im_plane = (a.sel != nullptr && *a.sel != 0) ? a.im_alt : a.im;
  auto prefetch = [&](int pair) {                   // the rows of an iteration are contiguous in each plane
    if (tid == 0 && pair < npairs) {
      mbar_expect_tx(&full, 2u * plane_bytes);
      bulk_g2s(st_re, a.re + (size_t)pair * kRows * P, plane_bytes, &full);
      bulk_g2s(st_im, im_plane + (size_t)pair * kRows * P, plane_bytes, &full);
    }
  };
  prefetch((int)blockIdx.x);
  const float scale = a.scale_ptr ? *a.scale_ptr : a.scale_host;
  uint32_t phase = 0;
  const int p2 = tid / R1, q2 = tid - p2 * R1;
  const int obase2 = q2 + R1 * R2 * p2, tstep2 = R1 * p2 * kTw;
  for (int pair = blockIdx.x; pair < npairs; pair += gridDim.x) {
    {  // stage 1: tangle + radix R1 (s = 1), first-stage quad twiddles; all twiddles fetched while the bulk copy lands
      float wr[R1], wi[R1];
      quad_twiddles<R1>(twQ, tid, wr, wi, kEO ? 2 : 1);
      constexpr int Nr = CH / R1;
      pf re[R1], im[R1];
      if constexpr (kEO) {
        mbar_wait(&full, phase); phase ^= 1u;
        RowTangleStagedEO src{reinterpret_cast<const float*>(st_re), reinterpret_cast<const float*>(st_im), twC, CH};
#pragma unroll
        for (int j = 0; j < R1; ++j) src.load(tid + j * Nr, re[j], im[j]);
      } else {
        cf wt[R1];
#pragma unroll
        for (int j = 0; j < R1; ++j) wt[j] = ldg_cf(twC + tid + j * Nr);
        mbar_wait(&full, phase); phase ^= 1u;
        RowTangleStaged2 src{reinterpret_cast<const float*>(st_re), reinterpret_cast<const float*>(st_im), P, CH};
#pragma unroll
        for (int j = 0; j < R1; ++j) src.load(tid + j * Nr, wt[j], re[j], im[j]);
      }
      Dft<R1>::run(re, im);
      sm.store(R1 * tid, re[0], im[0]);
#pragma unroll
      for (int k = 1; k < R1; ++k) {
        pf xr = re[k], xi = im[k];
        cmul(xr, xi, wr[k], wi[k]);
        sm.store(R1 * tid + k, xr, xi);
      }
    }
    __syncthreads();
    prefetch(pair + (int)gridDim.x);                // the staging buffers are free again
    {  // stage 2: radix R2, s = R1, in place
      cf w[R2];
#pragma unroll
      for (int k = 1; k < R2; ++k) w[k] = ldg_cf(twC + tstep2 * k);
      pf re[R2], im[R2];
      constexpr int Nr = CH / R2;
#pragma unroll
      for (int j = 0; j < R2; ++j) sm.load(tid + j * Nr, re[j], im[j]);
      __syncthreads();
      Dft<R2>::run(re, im);
      sm.store(obase2, re[0], im[0]);
#pragma unroll
      for (int k = 1; k < R2; ++k) {
        pf xr = re[k], xi = im[k];
        cmul(xr, xi, w[k].x, w[k].y);
        sm.store(obase2 + k * R1, xr, xi);
      }
    }
    __syncthreads();
    if constexpr (kEO) {  // stage 3 (last): lane 0 / 1 of output m are the complex elements 2m / 2m + 1 of the row
      const uint2* base64 = reinterpret_cast<const uint2*>(a.base + (size_t)pair * C);
      uint2* out64 = a.out_mode == 0 ? reinterpret_cast<uint2*>(a.out_bf16 + (size_t)pair * C) : nullptr;
      float4* of = a.out_mode != 0 ? reinterpret_cast<float4*>(a.out_f32 + (size_t)pair * C) : nullptr;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int b = tid + h * T;
        uint2 bb[R3];
#pragma unroll
        for (int k = 0; k < R3; ++k) bb[k] = a.out_mode == 0 ? __ldg(base64 + b + k * S3) : make_uint2(0u, 0u);
        pf re[R3], im[R3];
#pragma unroll
        for (int j = 0; j < R3; ++j) sm.load(b + j * S3, re[j], im[j]);
        if (h == 1) __syncthreads();                // the buffer has been read: the next row's stage 1 may overwrite it
        Dft<R3>::run(re, im);
        float bad = 0.f;
#pragma unroll
        for (int k = 0; k < R3; ++k) epilogue_store_eo_fast(a, scale, bb[k], out64, of, b + k * S3, re[k], im[k], bad);
        if (not_finite(bad)) {                       // exceptional: the exact epilogue over the same outputs
#pragma unroll
          for (int k = 0; k < R3; ++k) epilogue_store_eo(a, scale, bb[k], out64, of, b + k * S3, re[k], im[k]);
        }
      }
    } else {  // stage 3 (last): butterflies t and t + T, outputs straight into the epilogue
      const size_t row0 = (size_t)pair * 2;
      const uint32_t* base0 = reinterpret_cast<const uint32_t*>(a.base + row0 * C);
      const uint32_t* base1 = base0 + C / 2;
      uint32_t* out0 = a.out_mode == 0 ? reinterpret_cast<uint32_t*>(a.out_bf16 + row0 * C) : nullptr;
      uint32_t* out1 = out0 + C / 2;
      float* of0 = a.out_mode != 0 ? a.out_f32 + row0 * C : nullptr;
      float* of1 = of0 + C;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int b = tid + h * T;
        uint32_t bb0[R3], bb1[R3];
#pragma unroll
        for (int k = 0; k < R3; ++k) {
          bb0[k] = a.out_mode == 0 ? ldg_u32(base0 + b + k * S3) : 0u;
          bb1[k] = a.out_mode == 0 ? ldg_u32(base1 + b + k * S3) : 0u;
        }
        pf re[R3], im[R3];
#pragma unroll
        for (int j = 0; j < R3; ++j) sm.load(b + j * S3, re[j], im[j]);
        if (h == 1) __syncthreads();                // the buffer has been read: the next pair's stage 1 may overwrite it
        Dft<R3>::run(re, im);
        float bad = 0.f;
#pragma unroll
        for (int k = 0; k < R3; ++k) epilogue_store2_fast(a, scale, bb0[k], bb1[k], out0, out1, of0, of1, b + k * S3, re[k], im[k], bad);
        if (not_finite(bad)) {                       // exceptional: the exact epilogue over the same outputs
#pragma unroll
          for (int k = 0; k < R3; ++k) epilogue_store2(a, scale, bb0[k], bb1[k], out0, out1, of0, of1, b + k * S3, re[k], im[k]);
        }
      }
    }
  }
}

// ---- paired-row inverse pass, four stages (C = 2048): the mirror image of k_row2_fwd4 -------------------------------
// No staging: the tangle reads the two spectrum rows straight from global memory, the
// next pair's rows are pulled into L2 by the copy engine in the meantime; stages 2-3 in place; the last stage feeds the
// epilogue with the bf16 base words loaded ahead of its shared-memory reads.
struct RowTangleGlobal2 {
  const float* re; const float* im; const cf* twC; int P; int Ch;
  __device__ __forceinline__ void load(int k, pf& ore, pf& oim) const {
    pf xr = pf_make(ldg_f32(re + k), ldg_f32(re + P + k)), xi = pf_make(ldg_f32(im + k), ldg_f32(im + P + k));
    pf mr = pf_make(ldg_f32(re + Ch - k), ldg_f32(re + P + Ch - k)), mi = pf_make(ldg_f32(im + Ch - k), ldg_f32(im + P + Ch - k));
    const cf w = ldg_cf(twC + k);
    if (k == 0) { xi = pf_make(0.f, 0.f); mi = xi; }    // .real semantics: bins 0 and Ch are real
    const pf Ar = xr + mr, Ai = xi - mi, Br = xr - mr, Bi = xi + mi;
    const pf wx = pf_bcast(w.x), wy = pf_bcast(w.y);
    const pf br = pf_fma(Br, wx, Bi * wy);              // B * conj(w)
    const pf bi = pf_fma(Bi, wx, zero_of(Br) - Br * wy);
    const pf zr = Ar - bi, zi = Ai + br;
    ore = zi; oim = zr;                                 // handed to the forward engine swapped
  }
};

template <int R1, int R2, int R3, int R4, int T, int kCtas>
__global__ void __launch_bounds__(T, kCtas) k_row2_inv4(int R, int C, int P, const __grid_constant__ RowInvArgs a,
                                                    const cf* __restrict__ twC, const cf* __restrict__ twQ) {
  sm_pdl_enter();
  constexpr int CH = R1 * R2 * R3 * R4;
  constexpr int NB1 = CH / R1, NB2 = CH / R2, NB3 = CH / R3, S4 = CH / R4;
  constexpr int s2 = R1, s3 = R1 * R2;
  constexpr int H2 = NB2 / T;
  static_assert(NB2 == H2 * T && H2 >= 1 && H2 <= 2 && NB3 == 2 * T && S4 == 2 * T, "k_row2_inv4: 1-2 / 2 / 2 butterflies per thread in stages 2 / 3 / 4");
  RowSmem2X<true> sm{reinterpret_cast<ulonglong2*>(g_dyn_smem)};
  const int tid = threadIdx.x;
  const int npairs = R >> 1;
  const float* im_plane = (a.sel != nullptr && *a.sel != 0) ? a.im_alt : a.im;
  const float scale = a.scale_ptr ? *a.scale_ptr : a.scale_host;
  auto prefetch = [&](int pair) {
    if (tid == 0 && pair < npairs) {
      bulk_prefetch_l2(a.re + (size_t)pair * 2 * P, 8u * (uint32_t)P);
      bulk_prefetch_l2(im_plane + (size_t)pair * 2 * P, 8u * (uint32_t)P);
      if (a.out_mode == 0) bulk_prefetch_l2(a.base + (size_t)pair * 2 * C, 4u * (uint32_t)C);
    }
  };
  prefetch((int)blockIdx.x);
  for (int pair = blockIdx.x; pair < npairs; pair += gridDim.x) {
    {  // stage 1: tangle + radix R1 (s = 1) on the butterflies t, t + T, ...
      RowTangleGlobal2 src{a.re + (size_t)pair * 2 * P, im_plane + (size_t)pair * 2 * P, twC, P, CH};
#pragma unroll 1
      for (int b = tid; b < NB1; b += T) stockham_bfly_first<R1, pf>(b, CH, twQ, src, sm);
    }
    __syncthreads();
    prefetch(pair + (int)gridDim.x);
    {  // stage 2: radix R2, s = R1, in place, butterflies t (and t + T)
      pf re[H2][R2], im[H2][R2];
#pragma unroll
      for (int h = 0; h < H2; ++h)
#pragma unroll
        for (int j = 0; j < R2; ++j) sm.load(tid + h * T + j * NB2, re[h][j], im[h][j]);
      __syncthreads();
#pragma unroll
      for (int h = 0; h < H2; ++h) {
        Dft<R2>::run(re[h], im[h]);
        const int b = tid + h * T;
        const int p = b / s2, q = b - p * s2;
        const int obase = q + s2 * R2 * p, tstep = s2 * p * 2;
        sm.store(obase, re[h][0], im[h][0]);
#pragma unroll
        for (int k = 1; k < R2; ++k) {
          const cf w = ldg_cf(twC + tstep * k);
          pf xr = re[h][k], xi = im[h][k];
          cmul(xr, xi, w.x, w.y);
          sm.store(obase + k * s2, xr, xi);
        }
      }
    }
    __syncthreads();
    {  // stage 3: radix R3, s = R1*R2, in place, butterflies t and t + T
      pf re[2][R3], im[2][R3];
#pragma unroll
      for (int h = 0; h < 2; ++h)
#pragma unroll
        for (int j = 0; j < R3; ++j) sm.load(tid + h * T + j * NB3, re[h][j], im[h][j]);
      __syncthreads();
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        Dft<R3>::run(re[h], im[h]);
        const int b = tid + h * T;
        const int p = b / s3, q = b - p * s3;
        const int obase = q + s3 * R3 * p, tstep = s3 * p * 2;
        sm.store(obase, re[h][0], im[h][0]);
#pragma unroll
        for (int k = 1; k < R3; ++k) {
          const cf w = ldg_cf(twC + tstep * k);
          pf xr = re[h][k], xi = im[h][k];
          cmul(xr, xi, w.x, w.y);
          sm.store(obase + k * s3, xr, xi);
        }
      }
    }
    __syncthreads();
    {  // stage 4 (last): butterflies t and t + T, outputs straight into the epilogue
      const size_t row0 = (size_t)pair * 2;
      const uint32_t* base0 = reinterpret_cast<const uint32_t*>(a.base + row0 * C);
      const uint32_t* base1 = base0 + C / 2;
      uint32_t* out0 = a.out_mode == 0 ? reinterpret_cast<uint32_t*>(a.out_bf16 + row0 * C) : nullptr;
      uint32_t* out1 = out0 + C / 2;
      float* of0 = a.out_mode != 0 ? a.out_f32 + row0 * C : nullptr;
      float* of1 = of0 + C;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int b = tid + h * T;
        uint32_t bb0[R4], bb1[R4];
#pragma unroll
        for (int k = 0; k < R4; ++k) {
          bb0[k] = a.out_mode == 0 ? ldg_u32(base0 + b + k * S4) : 0u;
          bb1[k] = a.out_mode == 0 ? ldg_u32(base1 + b + k * S4) : 0u;
        }
        pf re[R4], im[R4];
#pragma unroll
        for (int j = 0; j < R4; ++j) sm.load(b + j * S4, re[j], im[j]);
        if (h == 1) __syncthreads();                // the buffer has been read: the next pair's stage 1 may overwrite it
        Dft<R4>::run(re, im);
        float bad = 0.f;
#pragma unroll
        for (int k = 0; k < R4; ++k) epilogue_store2_fast(a, scale, bb0[k], bb1[k], out0, out1, of0, of1, b + k * S4, re[k], im[k], bad);
        if (not_finite(bad)) {                       // exceptional: the exact epilogue over the same outputs
#pragma unroll
          for (int k = 0; k < R4; ++k) epilogue_store2(a, scale, bb0[k], bb1[k], out0, out1, of0, of1, b + k * S4, re[k], im[k]);
        }
      }
    }
  }
}

// ---- longest rows, inverse: the mirror image of k_row1_fwd_eo -------------------------------------------------------------
// Decimation in frequency on the input of the length-Ch engine: u[2m] = FFT_{Ch/2}(U[n] + U[n + Ch/2])[m] and
// u[2m+1] = FFT_{Ch/2}((U[n] - U[n + Ch/2]) W_Ch^n)[m] are the two lanes; lane 0 / lane 1 of output m are the complex
// elements 2m / 2m+1 of the row, i.e. four consecutive real outputs: one 8-byte bf16 store (and base load) per m.
struct RowTangleGlobalEO {
  const float* re; const float* im; const cf* twC; int H;                // H = Ch / 2
  __device__ __forceinline__ void tangle(int k, float& ore, float& oim) const {     // RowTangleSrc::load without the cull
    float xr = ldg_f32(re + k), xi = ldg_f32(im + k), mr = ldg_f32(re + 2 * H - k), mi = ldg_f32(im + 2 * H - k);
    if (k == 0) { xi = 0.f; mi = 0.f; }
    const float Ar = xr + mr, Ai = xi - mi, Br = xr - mr, Bi = xi + mi;
    const cf w = ldg_cf(twC + k);
    const float br = Br * w.x + Bi * w.y, bi = Bi * w.x - Br * w.y;
    ore = Ai + br; oim = Ar - bi;
  }
  __device__ __forceinline__ void load(int n, pf& ore, pf& oim) const {
    float u1r, u1i, u2r, u2i;
    tangle(n, u1r, u1i);
    tangle(n + H, u2r, u2i);
    float dr = u1r - u2r, di = u1i - u2i;
    const cf w = ldg_cf(twC + 2 * n);                                     // W_Ch^n
    cmul(dr, di, w.x, w.y);
    ore = pf_make(u1r + u2r, dr); oim = pf_make(u1i + u2i, di);
  }
};

// output m of the even / odd engine: lane 0 -> x[4m], x[4m+1]; lane 1 -> x[4m+2], x[4m+3]
__device__ __forceinline__ void epilogue_store_eo(const RowInvArgs& a, float scale, uint2 bb, uint2* out64, float4* of, int m, pf va, pf vb) {
  const pf n = pf_bcast(a.inv_n);
  const pf x0 = vb * n, x1 = va * n;
  const float x00 = pf_lo(x0), x01 = pf_hi(x0), x10 = pf_lo(x1), x11 = pf_hi(x1);   // xEL: element E of the complex pair, lane L
  const bool add_base = a.out_mode == 0;
  const float b00 = add_base ? bf16_bits_to_f32(bb.x & 0xffffu) : 0.f, b10 = add_base ? bits_f32(bb.x & 0xffff0000u) : 0.f;
  const float b01 = add_base ? bf16_bits_to_f32(bb.y & 0xffffu) : 0.f, b11 = add_base ? bits_f32(bb.y & 0xffff0000u) : 0.f;
  float y00, y01, y10, y11;
  epi_finish4(a, scale, add_base, x00, x01, x10, x11, b00, b01, b10, b11, y00, y01, y10, y11);
  if (add_base) out64[m] = make_uint2(pack_bf16x2_rne(y00, y10), pack_bf16x2_rne(y01, y11));
  else of[m] = make_float4(y00, y10, y01, y11);
}

template <int R1, int R2, int R3, int R4, int T, int kCtas>
__global__ void __launch_bounds__(T, kCtas) k_row1_inv_eo(int R, int C, int P, const __grid_constant__ RowInvArgs a,
                                                      const cf* __restrict__ twC, const cf* __restrict__ twQ2) {
  sm_pdl_enter();
  constexpr int CH = R1 * R2 * R3 * R4;             // length of the two lane transforms = Ch / 2
  constexpr int NB1 = CH / R1, NB2 = CH / R2, NB3 = CH / R3, S4 = CH / R4;
  constexpr int s2 = R1, s3 = R1 * R2;
  constexpr int H2 = NB2 / T;
  static_assert(NB2 == H2 * T && H2 >= 1 && H2 <= 2 && NB3 == 2 * T && S4 == 2 * T, "k_row1_inv_eo: 1-2 / 2 / 2 butterflies per thread in stages 2 / 3 / 4");
  RowSmem2X<false> sm{reinterpret_cast<ulonglong2*>(g_dyn_smem)};
  const int tid = threadIdx.x;
  const float* im_plane = (a.sel != nullptr && *a.sel != 0) ? a.im_alt : a.im;
  const float scale = a.scale_ptr ? *a.scale_ptr : a.scale_host;
  auto prefetch = [&](int row) {
    if (tid == 0 && row < R) {
      bulk_prefetch_l2(a.re + (size_t)row * P, 4u * (uint32_t)P);
      bulk_prefetch_l2(im_plane + (size_t)row * P, 4u * (uint32_t)P);
      if (a.out_mode == 0) bulk_prefetch_l2(a.base + (size_t)row * C, 2u * (uint32_t)C);
    }
  };
  prefetch((int)blockIdx.x);
  for (int row = blockIdx.x; row < R; row += gridDim.x) {
    {  // stage 1: tangle + even / odd split + radix R1 (s = 1)
      RowTangleGlobalEO src{a.re + (size_t)row * P, im_plane + (size_t)row * P, twC, CH};
#pragma unroll 1
      for (int b = tid; b < NB1; b += T) stockham_bfly_first<R1, pf>(b, CH, twQ2, src, sm, 2);
    }
    __syncthreads();
    prefetch(row + (int)gridDim.x);
    {  // stage 2: radix R2, s = R1, in place, butterflies t (and t + T)
      pf re[H2][R2], im[H2][R2];
#pragma unroll
      for (int h = 0; h < H2; ++h)
#pragma unroll
        for (int j = 0; j < R2; ++j) sm.load(tid + h * T + j * NB2, re[h][j], im[h][j]);
      __syncthreads();
#pragma unroll
      for (int h = 0; h < H2; ++h) {
        Dft<R2>::run(re[h], im[h]);
        const int b = tid + h * T;
        const int p = b / s2, q = b - p * s2;
        const int obase = q + s2 * R2 * p, tstep = s2 * p * 4;
        sm.store(obase, re[h][0], im[h][0]);
#pragma unroll
        for (int k = 1; k < R2; ++k) {
          const cf w = ldg_cf(twC + tstep * k);
          pf xr = re[h][k], xi = im[h][k];
          cmul(xr, xi, w.x, w.y);
          sm.store(obase + k * s2, xr, xi);
        }
      }
    }
    __syncthreads();
    {  // stage 3: radix R3, s = R1*R2, in place, butterflies t and t + T
      pf re[2][R3], im[2][R3];
#pragma unroll
      for (int h = 0; h < 2; ++h)
#pragma unroll
        for (int j = 0; j < R3; ++j) sm.load(tid + h * T + j * NB3, re[h][j], im[h][j]);
      __syncthreads();
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        Dft<R3>::run(re[h], im[h]);
        const int b = tid + h * T;
        const int p = b / s3, q = b - p * s3;
        const int obase = q + s3 * R3 * p, tstep = s3 * p * 4;
        sm.store(obase, re[h][0], im[h][0]);
#pragma unroll
        for (int k = 1; k < R3; ++k) {
          const cf w = ldg_cf(twC + tstep * k);
          pf xr = re[h][k], xi = im[h][k];
          cmul(xr, xi, w.x, w.y);
          sm.store(obase + k * s3, xr, xi);
        }
      }
    }
    __syncthreads();
    {  // stage 4 (last): butterflies t and t + T, outputs straight into the epilogue
      const uint2* base64 = reinterpret_cast<const uint2*>(a.base + (size_t)row * C);
      uint2* out64 = a.out_mode == 0 ? reinterpret_cast<uint2*>(a.out_bf16 + (size_t)row * C) : nullptr;
      float4* of = a.out_mode != 0 ? reinterpret_cast<float4*>(a.out_f32 + (size_t)row * C) : nullptr;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int b = tid + h * T;
        uint2 bb[R4];
#pragma unroll
        for (int k = 0; k < R4; ++k) bb[k] = a.out_mode == 0 ? __ldg(base64 + b + k * S4) : make_uint2(0u, 0u);
        pf re[R4], im[R4];
#pragma unroll
        for (int j = 0; j < R4; ++j) sm.load(b + j * S4, re[j], im[j]);
        if (h == 1) __syncthreads();                // the buffer has been read: the next row's stage 1 may overwrite it
        Dft<R4>::run(re, im);
        float bad = 0.f;
#pragma unroll
        for (int k = 0; k < R4; ++k) epilogue_store_eo_fast(a, scale, bb[k], out64, of, b + k * S4, re[k], im[k], bad);
        if (not_finite(bad)) {                       // exceptional: the exact epilogue over the same outputs
#pragma unroll
          for (int k = 0; k < R4; ++k) epilogue_store_eo(a, scale, bb[k], out64, of, b + k * S4, re[k], im[k]);
        }
      }
    }
  }
}

// scale a 1-D spectrum (no column sweep exists to fold the normalisation into)
__global__ void k_scale_row(float* re, float* im, int n, const float* scale_dev, float scale_host, int write_im) {
  sm_pdl_enter();
  const float s = scale_dev ? *scale_dev : scale_host;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    re[i] *= s;
    if (write_im) im[i] *= s;
  }
}

__global__ void k_init_twiddles(cf* tw, int M) {
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < M; j += gridDim.x * blockDim.x) {
    double s, c;
    sincospi(2.0 * (double)j / (double)M, &s, &c);
    cf w; w.x = (float)c; w.y = (float)(-s);
    tw[j] = w;
  }
}

// quad[b] = {W^b, W^2b, W^4b, W^8b}, W = exp(-2*pi*i/N): first-stage twiddles of the row passes
__global__ void k_init_quads(cf* quad, int n_b, int N) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 4 * n_b; i += gridDim.x * blockDim.x) {
    const long long e = ((long long)(i >> 2) << (i & 3)) % N;
    double s, c;
    sincospi(2.0 * (double)e / (double)N, &s, &c);
    cf w; w.x = (float)c; w.y = (float)(-s);
    quad[i] = w;
  }
}

__global__ void k_inv_norm(const double* sumsq, float* out) {
  sm_pdl_enter();
  const double ss = *sumsq;
  const float nrm = (float)sqrt(ss);
  *out = (nrm != 0.f) ? (1.0f / nrm) : 1.0f;
}

// ------------------------------------------------------------------ host side
static std::once_flag g_attr_once;
static int g_attr_rc = 0;
static int ensure_attrs() {
  std::call_once(g_attr_once, [] {
    // opt in to the full 227 KB of shared memory per CTA (minus each kernel's static part)
    int dev = 0, optin = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    auto set = [&](const void* fn) {
      cudaFuncAttributes fa;
      if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, fn);
      if (e == cudaSuccess)
        e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, optin - (int)fa.sharedSizeBytes);
    };
    set((const void*)k_row_fwd);
    set((const void*)k_row_inv);
    set((const void*)k_col);
    if (e != cudaSuccess) { sm_set_error("shared-memory opt-in failed: %s", cudaGetErrorString(e)); g_attr_rc = -100; }
  });
  return g_attr_rc;
}

extern "C" sm_plan* sm_plan_create(int R, int C) {
  sm_plan* pl = new sm_plan;
  int rc = sm_make_plan(R, C, &pl->p);
  if (rc != 0) {
    sm_set_error("unsupported tensor shape [%d][%d] for the sm_100a FFT (rc=%d): C must be even, the prime factors of "
                 "C/2 and R at most %d, and R = a * b with one a-point and one b-point column instance of 32 columns "
                 "each fitting in shared memory", R, C, rc, SM_GENERIC_MAX);
    delete pl;
    return nullptr;
  }
  return pl;
}
extern "C" void sm_plan_destroy(sm_plan* plan) { delete plan; }
extern "C" int sm_plan_pitch(const sm_plan* plan) { return plan->p.P; }
extern "C" int sm_plan_col_passes(const sm_plan* plan) { return plan->p.col_passes; }
extern "C" int sm_plan_col_launches(const sm_plan* plan) {     // kernel launches of ONE column transform (one per sweep)
  return plan->p.col_passes == 2 ? 2 : 1;
}
extern "C" int sm_plan_row_freq(const sm_plan* plan, int stored) { return sm_row_freq(&plan->p, stored); }
extern "C" size_t sm_plan_table_bytes(const sm_plan* plan) {
  return sm_tab_bytes(plan->p);
}
extern "C" int sm_plan_describe(const sm_plan* plan, char* buf, int buflen) {
  const SmPlan& p = plan->p;
  int n = snprintf(buf, buflen, "R=%d C=%d P=%d row[%d thr, smem %d/%d, pad %d]:", p.R, p.C, p.P,
                   p.row_threads, p.row_smem_fwd, p.row_smem_inv, p.row_pad);
  for (int i = 0; i < p.n_row && n < buflen; ++i) n += snprintf(buf + n, buflen - n, " %d", p.row_rad[i]);
  if (n < buflen) n += snprintf(buf + n, buflen - n, " | col passes=%d Ra=%d[%d thr]:", p.col_passes, p.Ra, p.thrA);
  for (int i = 0; i < p.nA && n < buflen; ++i) n += snprintf(buf + n, buflen - n, " %d", p.radA[i]);
  if (p.col_passes == 2) {
    if (n < buflen) n += snprintf(buf + n, buflen - n, " Rb=%d[%d thr]:", p.Rb, p.thrB);
    for (int i = 0; i < p.nB && n < buflen; ++i) n += snprintf(buf + n, buflen - n, " %d", p.radB[i]);
  }
  return n;
}

extern "C" int sm_plan_init_tables(const sm_plan* plan, void* tables, void* stream) {
  const SmPlan& p = plan->p;
  cudaStream_t st = (cudaStream_t)stream;
  cf* twC = reinterpret_cast<cf*>(tables);
  cf* twR = reinterpret_cast<cf*>(reinterpret_cast<char*>(tables) + sm_tab_off_R(p));
  k_init_twiddles<<<(p.C + 255) / 256, 256, 0, st>>>(twC, p.C);
  SM_LAUNCH_CHECK();
  k_init_twiddles<<<(p.R + 255) / 256, 256, 0, st>>>(twR, p.R);
  SM_LAUNCH_CHECK();
  cf* twQ = reinterpret_cast<cf*>(reinterpret_cast<char*>(tables) + sm_tab_off_Q(p));
  const int nq = sm_quad_count(p);
  if (nq > 0) {
    k_init_quads<<<(4 * nq + 255) / 256, 256, 0, st>>>(twQ, nq, p.Ch);
    SM_LAUNCH_CHECK();
  }
  return 0;
}

static const cf* tabC(const SmPlan&, const void* tables) { return reinterpret_cast<const cf*>(tables); }
static const cf* tabQ(const SmPlan& p, const void* tables) {
  return reinterpret_cast<const cf*>(reinterpret_cast<const char*>(tables) + sm_tab_off_Q(p));
}
static const cf* tabR(const SmPlan& p, const void* tables) {
  return reinterpret_cast<const cf*>(reinterpret_cast<const char*>(tables) + sm_tab_off_R(p));
}

// ------------------------------------------------------------------ specialised dispatch
static int g_optin_smem = 0;
template <class K>
static cudaError_t opt_in(K kernel, bool* done) {
  if (*done) return cudaSuccess;
  if (g_optin_smem == 0) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&g_optin_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (e != cudaSuccess) return e;
  }
  cudaFuncAttributes fa;
  cudaError_t e = cudaFuncGetAttributes(&fa, (const void*)kernel);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute((const void*)kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             g_optin_smem - (int)fa.sharedSizeBytes);
  if (e == cudaSuccess) *done = true;
  return e;
}

template <int R1, int R2, int NW>
static int launch_col_p(bool inverse, bool big_tw, dim3 grid, const ColCtArgs& a, const cf* twR, cudaStream_t st) {
  static bool done[4] = {false, false, false, false};
  const int smem = (R2 > 1) ? R1 * R2 * SM_COL_TILE * 8 : 0;
  cudaError_t e;
#define SM_COLP_CASE(INV, BIG, IDX)                                                       \
  e = opt_in(k_col_p<R1, R2, NW, INV, BIG>, &done[IDX]);                                  \
  if (e != cudaSuccess) { sm_set_error("opt_in: %s", cudaGetErrorString(e)); return -100; } \
  sm_launch(k_col_p<R1, R2, NW, INV, BIG>, dim3(grid), dim3(NW * 32), (size_t)(smem), st, a, twR);
  if (!inverse && big_tw) { SM_COLP_CASE(false, true, 0) }
  else if (!inverse) { SM_COLP_CASE(false, false, 1) }
  else if (big_tw) { SM_COLP_CASE(true, true, 2) }
  else { SM_COLP_CASE(true, false, 3) }
#undef SM_COLP_CASE
  SM_LAUNCH_CHECK();
  return 0;
}

template <int R1, int R2, int R3, int NW>
static int launch_col_p3(bool inverse, bool big_tw, dim3 grid, const ColCtArgs& a, const cf* twR, cudaStream_t st) {
  static bool done[4] = {false, false, false, false};
  const int smem = R1 * R2 * R3 * SM_COL_TILE * 8;
  cudaError_t e;
#define SM_COLP3_CASE(INV, BIG, IDX)                                                      \
  e = opt_in(k_col_p3<R1, R2, R3, NW, INV, BIG>, &done[IDX]);                             \
  if (e != cudaSuccess) { sm_set_error("opt_in: %s", cudaGetErrorString(e)); return -100; } \
  sm_launch(k_col_p3<R1, R2, R3, NW, INV, BIG>, dim3(grid), dim3(NW * 32), (size_t)(smem), st, a, twR);
  if (!inverse && big_tw) { SM_COLP3_CASE(false, true, 0) }
  else if (!inverse) { SM_COLP3_CASE(false, false, 1) }
  else if (big_tw) { SM_COLP3_CASE(true, true, 2) }
  else { SM_COLP3_CASE(true, false, 3) }
#undef SM_COLP3_CASE
  SM_LAUNCH_CHECK();
  return 0;
}

static int try_col_p(int n_rad, const int* rad, bool inverse, bool big_tw, dim3 grid, const ColCtArgs& a,
                     const cf* twR, cudaStream_t st) {
  if (n_rad != 2) return 1;
  const int r1 = rad[0], r2 = rad[1];
  if (r1 == 8 && r2 == 8) return launch_col_p<8, 8, 4>(inverse, big_tw, grid, a, twR, st);
  // the long instances as three stages of radices <= 8 (~52 registers instead of 80: 32 resident warps per SM instead
  // of 24; measured col_fwd -6 %, col_inv -4 %); a Stockham transform is natural order in / out whatever its radices,
  // so the plan's (16, 8) / (7, 16) split may be re-factored (L = 256 as 8 x 8 x 4 with 512-thread CTAs measured 1 % slower
  // than its two-stage kernel and is not used).
  if (r1 == 16 && r2 == 8) return launch_col_p3<8, 8, 2, 8>(inverse, big_tw, grid, a, twR, st);
  if (r1 == 7 && r2 == 16) return launch_col_p3<7, 8, 2, 8>(inverse, big_tw, grid, a, twR, st);
  if (r1 == 16 && r2 == 16) return launch_col_p<16, 16, 8>(inverse, big_tw, grid, a, twR, st);
  if (r1 == 11 && r2 == 8) return launch_col_p<11, 8, 4>(inverse, big_tw, grid, a, twR, st);
  if (r1 == 8 && r2 == 4) return launch_col_p<8, 4, 2>(inverse, big_tw, grid, a, twR, st);
  return 1;
}

static int g_num_sms = 0;
static int num_sms() {
  if (g_num_sms == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
      g_num_sms = 148;
  }
  return g_num_sms;
}
// paired-row forward pass (k_row2_fwd); returns 1 if this shape / mode has none
template <int R1, int R2, int R3, int R4, int T, bool kPad>
static int try_row2_fwd(const SmPlan& p, const RowFwdArgs& fa, const cf* twC, const cf* twQ, double* sumsq, cudaStream_t st) {
  if constexpr (R4 == 1 && kPad && (R1 * R2 * R3) / R3 == 2 * T && (R1 * R2 * R3) / R1 == T && (R1 * R2 * R3) / R2 == T) {
    constexpr int CH = R1 * R2 * R3;
    if (fa.mode != 0 || (p.R & 1) || p.R < 2 || p.C % 8 != 0) return 1;
    static bool done = false;
    static int occ = 0;
    const int work_bytes = ((CH + (CH >> 4) + 1) * 16 + 127) / 128 * 128;
    const int smem = work_bytes + 8 * p.C;
    if (smem > 227 * 1024 - 256) return 1;
    cudaError_t e = opt_in(k_row2_fwd<R1, R2, R3, T, false>, &done);
    if (e == cudaSuccess && occ == 0) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_row2_fwd<R1, R2, R3, T, false>, T, smem);
    if (e != cudaSuccess) { sm_set_error("row2 setup: %s", cudaGetErrorString(e)); return -100; }
    int grid = num_sms() * (occ > 0 ? occ : 1);
    if (grid > p.R / 2) grid = p.R / 2;
    sm_launch(k_row2_fwd<R1, R2, R3, T, false>, dim3(grid), dim3(T), (size_t)(smem), st, p.R, p.C, p.P, fa, twC, twQ, sumsq, work_bytes, RowFwdPair{});
    SM_LAUNCH_CHECK();
    return 0;
  } else {
    return 1;
  }
}

// paired-row four-stage passes (k_row2_fwd4 / k_row2_inv4) with their own factorization Ch = R1*R2*R3*R4 (it need not be
// the plan's: the twiddle tables do not depend on it and the quad table covers first radices down to 8);
// return 1 if this mode has none
template <int R1, int R2, int R3, int R4, int T, int kCtas>
static int launch_row2_fwd4(const SmPlan& p, const RowFwdArgs& fa, const cf* twC, const cf* twQ, double* sumsq, cudaStream_t st) {
  constexpr int CH = R1 * R2 * R3 * R4;
  if (fa.mode != 0 || (p.R & 1) || p.R < 2 || p.C % 8 != 0 || p.Ch != CH) return 1;
  static bool done = false;
  const int smem = (CH + (CH >> 3) + 1) * 16;
  if (smem > 227 * 1024 - 256) return 1;
  cudaError_t e = opt_in(k_row2_fwd4<R1, R2, R3, R4, T, kCtas>, &done);
  if (e != cudaSuccess) { sm_set_error("row2 fwd4 setup: %s", cudaGetErrorString(e)); return -100; }
  int grid = num_sms() * kCtas;
  if (grid > p.R / 2) grid = p.R / 2;
  sm_launch(k_row2_fwd4<R1, R2, R3, R4, T, kCtas>, dim3(grid), dim3(T), (size_t)(smem), st, p.R, p.C, p.P, fa, twC, twQ, sumsq);
  SM_LAUNCH_CHECK();
  return 0;
}

template <int R1, int R2, int R3, int R4, int T, int kCtas>
static int launch_row2_inv4(const SmPlan& p, const RowInvArgs& ia, const cf* twC, const cf* twQ, cudaStream_t st) {
  constexpr int CH = R1 * R2 * R3 * R4;
  if (ia.cull_thr != nullptr || (p.R & 1) || p.R < 2 || p.C % 8 != 0 || p.P % 4 != 0 || p.Ch != CH) return 1;
  static bool done = false;
  const int smem = (CH + (CH >> 3) + 1) * 16;
  if (smem > 227 * 1024 - 256) return 1;
  cudaError_t e = opt_in(k_row2_inv4<R1, R2, R3, R4, T, kCtas>, &done);
  if (e != cudaSuccess) { sm_set_error("row2 inv4 setup: %s", cudaGetErrorString(e)); return -100; }
  int grid = num_sms() * kCtas;
  if (grid > p.R / 2) grid = p.R / 2;
  sm_launch(k_row2_inv4<R1, R2, R3, R4, T, kCtas>, dim3(grid), dim3(T), (size_t)(smem), st, p.R, p.C, p.P, ia, twC, twQ);
  SM_LAUNCH_CHECK();
  return 0;
}

// one row per CTA, lanes = even / odd halves (k_row1_fwd_eo): Ch = 2 * R1*R2*R3*R4; kPair: that row of both models (pr)
template <int R1, int R2, int R3, int R4, int T, int kCtas, bool kPair = false>
static int launch_row1_fwd_eo(const SmPlan& p, const RowFwdArgs& fa, const cf* twC, const cf* twQ, double* sumsq, cudaStream_t st,
                              const RowFwdPair& pr = RowFwdPair{}) {
  constexpr int CH = R1 * R2 * R3 * R4;
  if (fa.mode != 0 || p.R < 1 || p.C % 8 != 0 || p.Ch != 2 * CH) return 1;
  static bool done = false;
  const int smem = CH * 16;
  cudaError_t e = opt_in(k_row1_fwd_eo<R1, R2, R3, R4, T, kCtas, kPair>, &done);
  if (e != cudaSuccess) { sm_set_error("row1 fwd eo setup: %s", cudaGetErrorString(e)); return -100; }
  int grid = num_sms() * kCtas;
  if (grid > p.R) grid = p.R;
  sm_launch(k_row1_fwd_eo<R1, R2, R3, R4, T, kCtas, kPair>, dim3(grid), dim3(T), (size_t)(smem), st, p.R, p.C, p.P, fa, twC, twQ, sumsq, pr);
  SM_LAUNCH_CHECK();
  return 0;
}

// three-stage bulk-copy fed kernel with the lanes = even / odd halves of one row (k_row2_fwd<..., kEO = true>): Ch = 2 * R1*R2*R3
template <int R1, int R2, int R3, int T>
static int launch_row1_fwd_eo3(const SmPlan& p, const RowFwdArgs& fa, const cf* twC, const cf* twQ, double* sumsq, cudaStream_t st) {
  constexpr int CH = R1 * R2 * R3;
  if (fa.mode != 0 || p.R < 2 || p.C % 8 != 0 || p.Ch != 2 * CH) return 1;
  static bool done = false;
  static int occ = 0;
  const int work_bytes = ((CH + (CH >> 4) + 1) * 16 + 127) / 128 * 128;
  const int smem = work_bytes + 4 * p.C;
  cudaError_t e = opt_in(k_row2_fwd<R1, R2, R3, T, true>, &done);
  if (e == cudaSuccess && occ == 0) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_row2_fwd<R1, R2, R3, T, true>, T, smem);
  if (e != cudaSuccess) { sm_set_error("row1 fwd eo3 setup: %s", cudaGetErrorString(e)); return -100; }
  int grid = num_sms() * (occ > 0 ? occ : 1);
  if (grid > p.R) grid = p.R;
  sm_launch(k_row2_fwd<R1, R2, R3, T, true>, dim3(grid), dim3(T), (size_t)(smem), st, p.R, p.C, p.P, fa, twC, twQ, sumsq, work_bytes, RowFwdPair{});
  SM_LAUNCH_CHECK();
  return 0;
}

static int try_row2_fwd4(const SmPlan& p, const RowFwdArgs& fa, const cf* twC, const cf* twQ, double* sumsq, cudaStream_t st) {
  if (p.Ch == 4096) return launch_row1_fwd_eo3<16, 16, 8, 128>(p, fa, twC, twQ, sumsq, st);
  if (p.Ch == 14336) return launch_row1_fwd_eo<7, 16, 8, 8, 448, 1>(p, fa, twC, twQ, sumsq, st);
  if (p.Ch == 7168) return launch_row1_fwd_eo<7, 8, 8, 8, 224, 2>(p, fa, twC, twQ, sumsq, st);
  // TinyLlama shapes: C = 2048 as row pairs 8 x 8 x 4 x 4, C = 5632 as even / odd halves of 11 x 8 x 4 x 4
  if (p.Ch == 1024) return launch_row2_fwd4<8, 8, 4, 4, 128, 4>(p, fa, twC, twQ, sumsq, st);
  if (p.Ch == 2816) return launch_row1_fwd_eo<11, 8, 4, 4, 176, 2>(p, fa, twC, twQ, sumsq, st);
  return 1;
}
template <int R1, int R2, int R3, int R4, int T, int kCtas>
static int launch_row1_inv_eo(const SmPlan& p, const RowInvArgs& ia, const cf* twC, const cf* twQ, cudaStream_t st) {
  constexpr int CH = R1 * R2 * R3 * R4;
  if (ia.cull_thr != nullptr || p.R < 1 || p.C % 8 != 0 || p.Ch != 2 * CH) return 1;
  static bool done = false;
  const int smem = CH * 16;
  cudaError_t e = opt_in(k_row1_inv_eo<R1, R2, R3, R4, T, kCtas>, &done);
  if (e != cudaSuccess) { sm_set_error("row1 inv eo setup: %s", cudaGetErrorString(e)); return -100; }
  int grid = num_sms() * kCtas;
  if (grid > p.R) grid = p.R;
  sm_launch(k_row1_inv_eo<R1, R2, R3, R4, T, kCtas>, dim3(grid), dim3(T), (size_t)(smem), st, p.R, p.C, p.P, ia, twC, twQ);
  SM_LAUNCH_CHECK();
  return 0;
}

template <int R1, int R2, int R3, int T>
static int launch_row1_inv_eo3(const SmPlan& p, const RowInvArgs& ia, const cf* twC, const cf* twQ, cudaStream_t st) {
  constexpr int CH = R1 * R2 * R3;
  if (ia.cull_thr != nullptr || p.R < 2 || p.C % 8 != 0 || p.P % 4 != 0 || p.Ch != 2 * CH) return 1;
  static bool done = false;
  static int occ = 0;
  const int work_bytes = ((CH + (CH >> 4) + 1) * 16 + 127) / 128 * 128;
  const int smem = work_bytes + 8 * p.P;
  cudaError_t e = opt_in(k_row2_inv<R1, R2, R3, T, true>, &done);
  if (e == cudaSuccess && occ == 0) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_row2_inv<R1, R2, R3, T, true>, T, smem);
  if (e != cudaSuccess) { sm_set_error("row1 inv eo3 setup: %s", cudaGetErrorString(e)); return -100; }
  int grid = num_sms() * (occ > 0 ? occ : 1);
  if (grid > p.R) grid = p.R;
  sm_launch(k_row2_inv<R1, R2, R3, T, true>, dim3(grid), dim3(T), (size_t)(smem), st, p.R, p.C, p.P, ia, twC, twQ, work_bytes);
  SM_LAUNCH_CHECK();
  return 0;
}

static int try_row2_inv4(const SmPlan& p, const RowInvArgs& ia, const cf* twC, const cf* twQ, cudaStream_t st) {
  if (p.Ch == 4096) return launch_row1_inv_eo3<16, 16, 8, 128>(p, ia, twC, twQ, st);
  if (p.Ch == 14336) return launch_row1_inv_eo<7, 16, 8, 8, 448, 1>(p, ia, twC, twQ, st);
  if (p.Ch == 7168) return launch_row1_inv_eo<7, 8, 8, 8, 224, 2>(p, ia, twC, twQ, st);
  if (p.Ch == 1024) return launch_row2_inv4<8, 8, 4, 4, 128, 4>(p, ia, twC, twQ, st);
  if (p.Ch == 2816) return launch_row1_inv_eo<11, 8, 4, 4, 176, 2>(p, ia, twC, twQ, st);
  return 1;
}

// paired-row inverse pass (k_row2_inv); returns 1 if this shape / mode has none
template <int R1, int R2, int R3, int R4, int T, bool kPad>
static int try_row2_inv(const SmPlan& p, const RowInvArgs& ia, const cf* twC, const cf* twQ, cudaStream_t st) {
  if constexpr (R4 == 1 && kPad && (R1 * R2 * R3) / R3 == 2 * T && (R1 * R2 * R3) / R1 == T && (R1 * R2 * R3) / R2 == T) {
    constexpr int CH = R1 * R2 * R3;
    if (ia.cull_thr != nullptr || (p.R & 1) || p.R < 2 || p.C % 8 != 0 || p.P % 4 != 0) return 1;
    static bool done = false;
    static int occ = 0;
    const int work_bytes = ((CH + (CH >> 4) + 1) * 16 + 127) / 128 * 128;
    const int smem = work_bytes + 16 * p.P;
    if (smem > 227 * 1024 - 256) return 1;
    cudaError_t e = opt_in(k_row2_inv<R1, R2, R3, T, false>, &done);
    if (e == cudaSuccess && occ == 0) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_row2_inv<R1, R2, R3, T, false>, T, smem);
    if (e != cudaSuccess) { sm_set_error("row2 inv setup: %s", cudaGetErrorString(e)); return -100; }
    int grid = num_sms() * (occ > 0 ? occ : 1);
    if (grid > p.R / 2) grid = p.R / 2;
    sm_launch(k_row2_inv<R1, R2, R3, T, false>, dim3(grid), dim3(T), (size_t)(smem), st, p.R, p.C, p.P, ia, twC, twQ, work_bytes);
    SM_LAUNCH_CHECK();
    return 0;
  } else {
    return 1;
  }
}

template <int R1, int R2, int R3, int R4, int T, bool kPad>
static int launch_row_ct(bool inverse, const SmPlan& p, const RowFwdArgs* fa, const RowInvArgs* ia, const cf* twC,
                         const cf* twQ, double* sumsq, cudaStream_t st) {
  static bool done[4] = {false, false, false, false};
  static int occ[2] = {0, 0};
  constexpr int CH = R1 * R2 * R3 * R4;
  if (!inverse) {
    int rc = try_row2_fwd<R1, R2, R3, R4, T, kPad>(p, *fa, twC, twQ, sumsq, st);
    if (rc <= 0) return rc;
    rc = try_row2_fwd4(p, *fa, twC, twQ, sumsq, st);
    if (rc <= 0) return rc;
  }
  if (inverse) {
    int rc = try_row2_inv<R1, R2, R3, R4, T, kPad>(p, *ia, twC, twQ, st);
    if (rc <= 0) return rc;
    rc = try_row2_inv4(p, *ia, twC, twQ, st);
    if (rc <= 0) return rc;
  }
  constexpr int nst = (R2 > 1) + (R3 > 1) + (R4 > 1) + 1;
  constexpr int bufstride = kPad ? (CH + (CH >> 4) + 1) : CH;
  cudaError_t e;
  // persistent bulk-copy variant: rows must start 16-byte aligned and the staging must fit next to the work buffers
  const int work_bytes = (((!inverse ? (nst >= 2 ? 2 : 1) : (nst >= 3 ? 2 : 1)) * bufstride * 8) + 127) / 128 * 128;
  const int stage_bytes = !inverse ? 4 * p.C : 8 * p.P + ((ia->out_mode == 0) ? 2 * p.C : 0);
  const bool aligned = (p.C % 8 == 0);
  if (aligned && work_bytes + stage_bytes <= 227 * 1024 - 256 && p.R >= 2) {
    const int smem = work_bytes + stage_bytes;
    const int which = inverse ? 1 : 0;
    if (!inverse) {
      e = opt_in(k_row_fwd_tma<R1, R2, R3, R4, T, kPad>, &done[2]);
      if (e == cudaSuccess && occ[0] == 0)
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ[0], k_row_fwd_tma<R1, R2, R3, R4, T, kPad>, T, smem);
    } else {
      e = opt_in(k_row_inv_tma<R1, R2, R3, R4, T, kPad>, &done[3]);
      if (e == cudaSuccess && occ[1] == 0)
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ[1], k_row_inv_tma<R1, R2, R3, R4, T, kPad>, T, smem);
    }
    if (e != cudaSuccess) { sm_set_error("row tma setup: %s", cudaGetErrorString(e)); return -100; }
    int grid = num_sms() * (occ[which] > 0 ? occ[which] : 1);
    if (grid > p.R) grid = p.R;
    if (!inverse) sm_launch(k_row_fwd_tma<R1, R2, R3, R4, T, kPad>, dim3(grid), dim3(T), (size_t)(smem), st, p.R, p.C, p.P, *fa, twC, twQ, sumsq, work_bytes);
    else sm_launch(k_row_inv_tma<R1, R2, R3, R4, T, kPad>, dim3(grid), dim3(T), (size_t)(smem), st, p.R, p.C, p.P, *ia, twC, twQ, work_bytes);
    SM_LAUNCH_CHECK();
    return 0;
  }
  if (!inverse) {
    e = opt_in(k_row_fwd_ct<R1, R2, R3, R4, T, kPad>, &done[0]);
    if (e != cudaSuccess) { sm_set_error("opt_in: %s", cudaGetErrorString(e)); return -100; }
    sm_launch(k_row_fwd_ct<R1, R2, R3, R4, T, kPad>, dim3(p.R), dim3(T), (size_t)(p.row_smem_fwd), st, p.C, p.P, *fa, twC, twQ, sumsq);
  } else {
    e = opt_in(k_row_inv_ct<R1, R2, R3, R4, T, kPad>, &done[1]);
    if (e != cudaSuccess) { sm_set_error("opt_in: %s", cudaGetErrorString(e)); return -100; }
    sm_launch(k_row_inv_ct<R1, R2, R3, R4, T, kPad>, dim3(p.R), dim3(T), (size_t)(p.row_smem_inv), st, p.C, p.P, *ia, twC, twQ);
  }
  SM_LAUNCH_CHECK();
  return 0;
}

static bool row_radices_are(const SmPlan& p, int n, int a, int b, int c, int d) {
  if (p.n_row != n) return false;
  const int want[4] = {a, b, c, d};
  for (int i = 0; i < n; ++i) if (p.row_rad[i] != want[i]) return false;
  return true;
}

static int try_row_ct(bool inverse, const SmPlan& p, const RowFwdArgs* fa, const RowInvArgs* ia, const cf* twC,
                      const cf* twQ, double* sumsq, cudaStream_t st) {
  auto is = [&](int n, int a, int b, int c, int d) { return row_radices_are(p, n, a, b, c, d); };
  if (is(3, 16, 8, 8, 1) && p.row_threads == 64 && p.row_pad) return launch_row_ct<16, 8, 8, 1, 64, true>(inverse, p, fa, ia, twC, twQ, sumsq, st);
  if (is(3, 16, 16, 8, 1) && p.row_threads == 128 && p.row_pad) return launch_row_ct<16, 16, 8, 1, 128, true>(inverse, p, fa, ia, twC, twQ, sumsq, st);
  if (is(3, 16, 16, 16, 1) && p.row_threads == 256 && p.row_pad) return launch_row_ct<16, 16, 16, 1, 256, true>(inverse, p, fa, ia, twC, twQ, sumsq, st);
  if (is(3, 11, 16, 16, 1) && p.row_threads == 192 && p.row_pad) return launch_row_ct<11, 16, 16, 1, 192, true>(inverse, p, fa, ia, twC, twQ, sumsq, st);
  if (is(4, 7, 16, 8, 8) && p.row_threads == 448 && p.row_pad) return launch_row_ct<7, 16, 8, 8, 448, true>(inverse, p, fa, ia, twC, twQ, sumsq, st);
  if (is(4, 7, 16, 16, 8) && p.row_threads == 512 && !p.row_pad) return launch_row_ct<7, 16, 16, 8, 512, false>(inverse, p, fa, ia, twC, twQ, sumsq, st);
  return 1;
}

static int launch_row_fwd(const SmPlan& p, const void* tables, const RowFwdArgs& a, double* sumsq, cudaStream_t st) {
  if (ensure_attrs()) return -100;
  {
    const int rc = try_row_ct(false, p, &a, nullptr, tabC(p, tables), tabQ(p, tables), sumsq, st);
    if (rc <= 0) return rc;
  }
  sm_launch(k_row_fwd, dim3(p.R), dim3(p.row_threads), (size_t)(p.row_smem_fwd), st, p, a, tabC(p, tables), tabQ(p, tables), sumsq);
  SM_LAUNCH_CHECK();
  return 0;
}

extern "C" int sm_fwd_rows_bf16(const sm_plan* plan, const void* tables, const void* base_bf16, const void* ft_bf16,
                                float* re, float* im, double* sumsq, void* stream) {
  RowFwdArgs a{};
  a.mode = 0; a.base = (const uint16_t*)base_bf16; a.ft = (const uint16_t*)ft_bf16;
  a.m1 = 1.f; a.m2 = 1.f; a.re = re; a.im = im;
  return launch_row_fwd(plan->p, tables, a, sumsq, (cudaStream_t)stream);
}

// ---- both finetunes over one shared base in one pass (sm_fwd_rows_bf16_pair).  A plan gets the paired kernel only where
// sm_fwd_rows_bf16 runs the same kernel per model (try_row_ct -> try_row2_fwd / try_row2_fwd4), so each model's spectrum
// is bit for bit the single-model pass's: C = 4096 (k_row2_fwd: 24 KB staged per row instead of 32 KB per row pair; the
// CTA stays at 3 per SM, a 4th does not fit 228 KB with the 35 KB work buffer) and C = 14336 (k_row1_fwd_eo).  C = 28672
// through k_row1_fwd_eo<7,16,8,8,448,1,true> measured the same row-pass time as two single-model passes (B200, 1000 W:
// 6.86 / 6.87 against 6.81 / 6.94 ms per 2 Llama-70B layers) and C = 8192 has no paired kernel: both keep two passes.
enum RowPairKind { kRowPairNone = 0, kRowPairRow2, kRowPairEo7168 };
static RowPairKind row_pair_kind(const SmPlan& p) {
  if (p.C % 8 != 0 || p.R < 1) return kRowPairNone;
  if (row_radices_are(p, 3, 16, 16, 8, 1) && p.row_threads == 128 && p.row_pad && p.R % 2 == 0) return kRowPairRow2;
  if (row_radices_are(p, 4, 7, 16, 8, 8) && p.row_threads == 448 && p.row_pad && p.Ch == 7168) return kRowPairEo7168;
  return kRowPairNone;
}

template <int R1, int R2, int R3, int T>
static int launch_row2_fwd_pair(const SmPlan& p, const RowFwdArgs& fa, const RowFwdPair& pr, const cf* twC, const cf* twQ,
                                double* sumsq, cudaStream_t st) {
  constexpr int CH = R1 * R2 * R3;
  static bool done = false;
  static int occ = 0;
  const int work_bytes = ((CH + (CH >> 4) + 1) * 16 + 127) / 128 * 128;
  const int smem = work_bytes + 6 * p.C;           // staging: the base row and the row of each finetune
  cudaError_t e = opt_in(k_row2_fwd<R1, R2, R3, T, false, true>, &done);
  if (e == cudaSuccess && occ == 0) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_row2_fwd<R1, R2, R3, T, false, true>, T, smem);
  if (e != cudaSuccess) { sm_set_error("row2 pair setup: %s", cudaGetErrorString(e)); return -100; }
  int grid = num_sms() * (occ > 0 ? occ : 1);
  if (grid > p.R) grid = p.R;
  sm_launch(k_row2_fwd<R1, R2, R3, T, false, true>, dim3(grid), dim3(T), (size_t)(smem), st, p.R, p.C, p.P, fa, twC, twQ, sumsq, work_bytes, pr);
  SM_LAUNCH_CHECK();
  return 0;
}

extern "C" int sm_fwd_rows_pair_supported(const sm_plan* plan) { return row_pair_kind(plan->p) != kRowPairNone ? 1 : 0; }

extern "C" int sm_fwd_rows_bf16_pair(const sm_plan* plan, const void* tables, const void* base_bf16, const void* ft0_bf16,
                                     const void* ft1_bf16, float* re0, float* im0, float* re1, float* im1, void* ctl,
                                     double target_norm_offset, double target_norm, void* stream) {
  const SmPlan& p = plan->p;
  RowFwdArgs a{};
  a.mode = 0; a.base = (const uint16_t*)base_bf16; a.ft = (const uint16_t*)ft0_bf16;
  a.m1 = 1.f; a.m2 = 1.f; a.re = re0; a.im = im0;
  const RowFwdPair pr{(const uint16_t*)ft1_bf16, re1, im1, (unsigned char*)ctl, target_norm_offset, target_norm};
  double* sumsq = reinterpret_cast<double*>((unsigned char*)ctl + SM_CTL_SUMSQ);
  const cf* twC = tabC(p, tables);
  const cf* twQ = tabQ(p, tables);
  cudaStream_t st = (cudaStream_t)stream;
  switch (row_pair_kind(p)) {
    case kRowPairRow2: return launch_row2_fwd_pair<16, 16, 8, 128>(p, a, pr, twC, twQ, sumsq, st);
    case kRowPairEo7168: return launch_row1_fwd_eo<7, 8, 8, 8, 224, 2, true>(p, a, twC, twQ, sumsq, st, pr);
    default: break;
  }
  sm_set_error("sm_fwd_rows_bf16_pair: no paired row kernel for [%d][%d] (sm_fwd_rows_pair_supported)", p.R, p.C);
  return -102;
}

extern "C" int sm_fwd_rows_f32(const sm_plan* plan, const void* tables, const float* x, float m1, float m2,
                               float* re, float* im, double* sumsq, void* stream) {
  RowFwdArgs a{};
  a.mode = 1; a.x32 = x; a.m1 = m1; a.m2 = m2; a.re = re; a.im = im;
  return launch_row_fwd(plan->p, tables, a, sumsq, (cudaStream_t)stream);
}

static int launch_col(const SmPlan& p, const void* tables, int sweep, int inverse, float* re, float* im,
                      const float* cull_thr, const float* scale_dev, float scale_host, int use_scale,
                      int write_im, cudaStream_t st, float* im_alt = nullptr, const int* sel = nullptr,
                      const int* wsel = nullptr, int wskip = 0) {
  if (ensure_attrs()) return -100;
  ColArgs ca{};
  int n_inst = 0;
  sm_col_args(p, sweep, inverse, &ca, &n_inst);
  ca.re = re; ca.im = im; ca.cull_thr = cull_thr; ca.im_alt = im_alt; ca.sel = sel;
  ca.scale_ptr = scale_dev; ca.scale_host = scale_host; ca.use_scale = use_scale;
  ca.write_im = write_im; ca.wsel = wsel; ca.wskip = wskip;
  const int ntiles = sm_col_tiles(p);
  {
    ColCtArgs c{};
    c.p0 = inverse ? im : re; c.p1 = inverse ? re : im;
    c.p0_alt = inverse ? im_alt : nullptr; c.sel = inverse ? sel : nullptr;
    c.P = p.P; c.Ch = p.Ch; c.inst_mul = ca.inst_mul; c.elem_mul = ca.elem_mul; c.tw_mul = ca.tw_mul;
    c.thr_ptr = cull_thr; c.scale_ptr = use_scale ? scale_dev : nullptr;
    c.scale = use_scale ? scale_host : 1.0f; c.write_p1_fwd = write_im; c.wsel = wsel; c.wskip = wskip;
    const int rc = try_col_p(ca.n_rad, ca.rad, inverse != 0, ca.big_tw != 0, dim3(ntiles, n_inst), c, tabR(p, tables), st);
    if (rc <= 0) return rc;
  }
  const int threads = (sweep == 0) ? p.thrA : p.thrB;
  const int smem = (sweep == 0) ? p.smemA : p.smemB;
  sm_launch(k_col, dim3(dim3(ntiles, n_inst)), dim3(threads), (size_t)(smem), st, p, ca, tabR(p, tables));
  SM_LAUNCH_CHECK();
  return 0;
}

extern "C" int sm_fwd_cols(const sm_plan* plan, const void* tables, float* re, float* im,
                           const float* scale_dev, float scale_host, int write_im, void* stream) {
  return sm_fwd_cols_sel(plan, tables, re, im, scale_dev, scale_host, write_im, nullptr, 0, stream);
}

int sm_fwd_cols_sel(const sm_plan* plan, const void* tables, float* re, float* im, const float* scale_dev, float scale_host,
                    int write_im, const int* wsel, int wskip, void* stream) {
  const SmPlan& p = plan->p;
  cudaStream_t st = (cudaStream_t)stream;
  if (p.col_passes == 0) {
    sm_launch(k_scale_row, dim3((p.Ch + 1 + 255) / 256), dim3(256), (size_t)(0), st, re, im, p.Ch + 1, scale_dev, scale_host, write_im);
    SM_LAUNCH_CHECK();
    return 0;
  }
  for (int sweep = 0; sweep < p.col_passes; ++sweep) {
    const bool lastsweep = (sweep == p.col_passes - 1);
    int rc = launch_col(p, tables, sweep, 0, re, im, nullptr, scale_dev, scale_host, lastsweep ? 1 : 0,
                        lastsweep ? write_im : 1, st, nullptr, nullptr, lastsweep ? wsel : nullptr, wskip);
    if (rc) return rc;
  }
  return 0;
}

extern "C" int sm_inv_norm(const double* sumsq, float* out, void* stream) {
  sm_launch(k_inv_norm, dim3(1), dim3(1), (size_t)(0), (cudaStream_t)stream, sumsq, out);
  SM_LAUNCH_CHECK();
  return 0;
}

int sm_inv_cols_sel(const sm_plan* plan, const void* tables, float* re, float* im, float* im_alt, const int* sel,
                    const float* cull_thr, void* stream) {
  const SmPlan& p = plan->p;
  for (int i = 0; i < p.col_passes; ++i) {
    const int sweep = p.col_passes - 1 - i;   // undo sweep B first, then sweep A
    int rc = launch_col(p, tables, sweep, 1, re, im, i == 0 ? cull_thr : nullptr, nullptr, 1.f, 0, 1,
                        (cudaStream_t)stream, im_alt, sel);
    if (rc) return rc;
  }
  return 0;
}

extern "C" int sm_inv_cols(const sm_plan* plan, const void* tables, float* re, float* im, const float* cull_thr,
                           void* stream) {
  return sm_inv_cols_sel(plan, tables, re, im, nullptr, nullptr, cull_thr, stream);
}

static int launch_row_inv(const SmPlan& p, const void* tables, RowInvArgs& a, cudaStream_t st) {
  if (ensure_attrs()) return -100;
  a.inv_n = (float)(1.0 / ((double)p.R * (double)p.C));
  if (p.col_passes != 0) a.cull_thr = nullptr;
  {
    const int rc = try_row_ct(true, p, nullptr, &a, tabC(p, tables), tabQ(p, tables), nullptr, st);
    if (rc <= 0) return rc;
  }
  sm_launch(k_row_inv, dim3(p.R), dim3(p.row_threads), (size_t)(p.row_smem_inv), st, p, a, tabC(p, tables), tabQ(p, tables));
  SM_LAUNCH_CHECK();
  return 0;
}

int sm_inv_rows_bf16_sel(const sm_plan* plan, const void* tables, const float* re, const float* im,
                         const float* im_alt, const int* sel, const float* cull_thr, const void* base_bf16,
                         void* out_bf16, const float* scale_dev, float scale_host, int check_ifft, uint32_t* flags4,
                         void* stream) {
  RowInvArgs a{};
  a.check_ifft = check_ifft; a.im_alt = im_alt; a.sel = sel;
  a.re = re; a.im = im; a.cull_thr = cull_thr; a.out_mode = 0;
  a.base = (const uint16_t*)base_bf16; a.out_bf16 = (uint16_t*)out_bf16;
  a.scale_ptr = scale_dev; a.scale_host = scale_host; a.flags = flags4;
  return launch_row_inv(plan->p, tables, a, (cudaStream_t)stream);
}

int sm_inv_rows_f32_sel(const sm_plan* plan, const void* tables, const float* re, const float* im, const float* im_alt,
                        const int* sel, const float* cull_thr, float* out, const float* scale_dev, float scale_host,
                        int check_ifft, uint32_t* flags4, void* stream) {
  RowInvArgs a{};
  a.check_ifft = check_ifft; a.im_alt = im_alt; a.sel = sel;
  a.re = re; a.im = im; a.cull_thr = cull_thr; a.out_mode = 1; a.out_f32 = out;
  a.scale_ptr = scale_dev; a.scale_host = scale_host; a.flags = flags4;
  return launch_row_inv(plan->p, tables, a, (cudaStream_t)stream);
}

extern "C" int sm_inv_rows_bf16(const sm_plan* plan, const void* tables, const float* re, const float* im,
                                const float* cull_thr, const void* base_bf16, void* out_bf16,
                                const float* scale_dev, float scale_host, int check_ifft, uint32_t* flags4,
                                void* stream) {
  RowInvArgs a{};
  a.check_ifft = check_ifft;
  a.re = re; a.im = im; a.cull_thr = cull_thr; a.out_mode = 0;
  a.base = (const uint16_t*)base_bf16; a.out_bf16 = (uint16_t*)out_bf16;
  a.scale_ptr = scale_dev; a.scale_host = scale_host; a.flags = flags4;
  return launch_row_inv(plan->p, tables, a, (cudaStream_t)stream);
}

extern "C" int sm_inv_rows_f32(const sm_plan* plan, const void* tables, const float* re, const float* im,
                               const float* cull_thr, float* out, const float* scale_dev, float scale_host,
                               int check_ifft, uint32_t* flags4, void* stream) {
  RowInvArgs a{};
  a.check_ifft = check_ifft;
  a.re = re; a.im = im; a.cull_thr = cull_thr; a.out_mode = 1; a.out_f32 = out;
  a.scale_ptr = scale_dev; a.scale_host = scale_host; a.flags = flags4;
  return launch_row_inv(plan->p, tables, a, (cudaStream_t)stream);
}
