// sm_internal.h -- shared between the translation units of libshardmerge_b200.so
#pragma once
#include <cuda_runtime.h>
#include <cstdio>
#include <cstring>
#include "../../include/shardmerge_b200.h"
#include "plan.h"

struct sm_plan {
  SmPlan p;
};

void sm_set_error(const char* fmt, ...);

#define SM_CUDA_CHECK(expr)                                                            \
  do {                                                                                 \
    cudaError_t _e = (expr);                                                           \
    if (_e != cudaSuccess) {                                                           \
      sm_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return -100;                                                                     \
    }                                                                                  \
  } while (0)

#define SM_LAUNCH_CHECK()                                                              \
  do {                                                                                 \
    cudaError_t _e = cudaGetLastError();                                               \
    if (_e != cudaSuccess) {                                                           \
      sm_set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, __LINE__); \
      return -101;                                                                     \
    }                                                                                  \
  } while (0)

// ---- programmatic dependent launch (sm_90+): every kernel of the fused chain starts with sm_pdl_enter() -- wait until the
// preceding kernel of the stream has completed and its writes are visible -- and is launched through sm_launch(), which sets
// the programmatic stream serialization attribute.  Semantics are those of plain stream order (nothing is read before the
// wait); what is saved is the launch latency of kernel k+1, which is set up while kernel k still runs: ~2 us per boundary on
// B200 (tools/ubench_pdl.cu), 17 boundaries per pair merge.  No kernel issues griddepcontrol.launch_dependents: with an early
// trigger the next kernel's CTAs become resident and sit in the wait while the current one runs, which saves nothing more in
// a single stream (same ubench) and, with several lanes, takes the SM slots the OTHER lanes' kernels would have filled
// (value 53.0 -> 49.7 Gparam/s, profiles/r02_ab_pdl.log).
#ifdef __CUDACC__
__device__ __forceinline__ void sm_pdl_enter() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
}
template <class... KA, class... A>
static inline void sm_launch(void (*kernel)(KA...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, A&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  (void)cudaLaunchKernelEx(&cfg, kernel, static_cast<A&&>(args)...);      // errors surface in SM_LAUNCH_CHECK()
}

// The decisions the reference makes on the host from the two delta norms of a pair merge: which model is "a" (the larger
// norm, fast_fourier.py:212-215), which branch runs (:223-244) and target_norm (:165).  Writes the per-model spectrum
// scales 1/||delta||, the norms, target_norm, the role flag `swap` and the branch code into the scalar block.  One thread.
// ext_tn > 0: the target norm is given (the mean over ALL models of the layer in a pair tree, fast_fourier.py:165).
__device__ __forceinline__ void sm_prepare_scalars(unsigned char* ctl, double sumsq0, double sumsq1, double target_norm_offset,
                                                   double ext_tn) {
  float* flt = reinterpret_cast<float*>(ctl + SM_CTL_FLT);
  int* ints = reinterpret_cast<int*>(ctl + SM_CTL_INT);
  double* tn_out = reinterpret_cast<double*>(ctl + SM_CTL_TN);
  // torch.norm(delta) is an fp32 scalar; .item() widens it to a Python float
  const float nx = (float)sqrt(sumsq0), ny = (float)sqrt(sumsq1);
  const int swap = fabsf(nx) < fabsf(ny) ? 1 : 0;              // fast_fourier.py:212
  const double na = swap ? (double)ny : (double)nx, nb = swap ? (double)nx : (double)ny;
  const float mean32 = (nx + ny) / 2.0f;                        // torch.tensor(layer_norms).mean()  (:165)
  const double tn = ext_tn > 0.0 ? ext_tn : (double)mean32 + target_norm_offset;
  const double cnorm_a = fabs(na / tn), cnorm_b = fabs(nb / tn);
  const double n_ratio = cnorm_b / (cnorm_a + 1e-10);
  int branch = SM_BRANCH_SLERP;
  if (cnorm_a < 1e-6) branch = SM_BRANCH_ADD;                                   // :223
  else if (cnorm_b < 1e-6 || n_ratio < 0.1) branch = SM_BRANCH_ARITH;            // :226
  else if (nb < 1e-4 || na < 1e-4) branch = SM_BRANCH_EARLY;                     // functions.py:184-190
  else if (nb / (na + 1e-10) < 0.1) branch = SM_BRANCH_LINEAR;                   // functions.py:199-202
  flt[SM_F_SCALE_X] = nx != 0.f ? 1.0f / nx : 1.0f;             // normalize_tensor: x * (1/norm), fp32
  flt[SM_F_SCALE_Y] = ny != 0.f ? 1.0f / ny : 1.0f;
  flt[SM_F_OUT_SCALE] = (float)tn;
  flt[SM_F_NORM_X] = nx; flt[SM_F_NORM_Y] = ny;
  ints[SM_I_SWAP] = swap; ints[SM_I_BRANCH] = branch;
  *tn_out = tn;
}
#endif

// table layout inside the caller's buffer: [W_C : C entries][W_R : R entries][quads : 4 * (Ch / row_rad[0])]
// of float2; the quad table (fft_core.cuh: first-stage twiddles) starts 32-byte aligned.
static inline size_t sm_tab_off_R(const SmPlan& p) { return (size_t)p.C * 8; }
static inline size_t sm_tab_off_Q(const SmPlan& p) { return (((size_t)p.C + (size_t)p.R) * 8 + 31) / 32 * 32; }
static inline int sm_quad_count(const SmPlan& p) {     // entries b < Ch / r for the smallest first radix r any row kernel uses
  if (p.n_row <= 1) return 0;
  const int n = p.Ch / p.row_rad[0], n8 = (p.Ch % 8 == 0) ? p.Ch / 8 : 0;
  return n > n8 ? n : n8;
}
static inline size_t sm_tab_bytes(const SmPlan& p) { return sm_tab_off_Q(p) + 32 * (size_t)sm_quad_count(p); }
// column tiles (SM_COL_TILE columns each) over the Ch + 1 columns of the half spectrum
static inline int sm_col_tiles(const SmPlan& p) { return (p.Ch + 1 + SM_COL_TILE - 1) / SM_COL_TILE; }

// iteration space of the element-wise / statistics kernels over the valid half spectrum
#define SM_EW_THREADS 256
#define SM_EW_COLS (SM_EW_THREADS * 4)

// internal (C++ linkage) variants with a device-side role pick: `sel` points at an int in device
// memory; if it is non-zero the two models swap roles (v0 = larger-norm model, fast_fourier.py:212-215)
int sm_slerp_reduce_sel(const sm_plan* plan, const float* reX, const float* reY, const int* sel,
                        const float* thr_cut, double* sums3, void* stream);
int sm_blend_sel(const sm_plan* plan, int mode, int agreement, const float* reX, const float* reY, const int* sel,
                 const float* thr_cut, const float* scal4, float t_sum, float* out_re, void* stream);
// forward column sweeps that skip the imaginary plane's final store when (*wsel != 0) == (wskip != 0)
int sm_fwd_cols_sel(const sm_plan* plan, const void* tables, float* re, float* im, const float* scale_dev, float scale_host,
                    int write_im, const int* wsel, int wskip, void* stream);
int sm_inv_cols_sel(const sm_plan* plan, const void* tables, float* re, float* im, float* im_alt, const int* sel,
                    const float* cull_thr, void* stream);
int sm_inv_rows_bf16_sel(const sm_plan* plan, const void* tables, const float* re, const float* im,
                         const float* im_alt, const int* sel, const float* cull_thr, const void* base_bf16,
                         void* out_bf16, const float* scale_dev, float scale_host, int check_ifft, uint32_t* flags4,
                         void* stream);
int sm_inv_rows_f32_sel(const sm_plan* plan, const void* tables, const float* re, const float* im, const float* im_alt,
                        const int* sel, const float* cull_thr, float* out, const float* scale_dev, float scale_host,
                        int check_ifft, uint32_t* flags4, void* stream);
