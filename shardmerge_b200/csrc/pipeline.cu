// pipeline.cu -- the fused, host-sync-free pair merge: the regular-layer body of
// FourierMerge._merge_layer (shard/merge/fast_fourier.py:147-276) for the common case of two
// bf16 finetunes, issued as one stream-ordered chain of kernels from a single C call.
//
// The reference decides three things on the host from the two delta norms: which model is "a"
// (the larger norm, :212-215), which branch runs (:223-244) and target_norm (:165).  Here a
// one-thread kernel (k_prepare) makes the same decisions on the device right after the row
// passes: it writes the per-model spectrum scales 1/||delta||, target_norm, the role flag
// `swap` and the branch code into the scalar block, and every later kernel reads what it needs
// from there.  When both finetunes share one base, one paired row pass transforms both (the base
// is read once) and its last CTA makes these decisions instead (sm_prepare_scalars, sm_internal.h).  The chain always continues down the SLERP branch (what the BASELINE configs
// take); if k_prepare found another branch, or an order-statistic window missed, the caller sees
// it in the scalar block afterwards and re-runs that tensor on the step-by-step path.
#include <vector>
#include "sm_internal.h"

namespace {

// use_host_sumsq: the row passes ran earlier and the host passes their sums of squares in (tree round 1)
__global__ void k_prepare(unsigned char* ctl, double target_norm_offset, double ext_tn, int use_host_sumsq, double hs0, double hs1) {
  sm_pdl_enter();
  double* sumsq = reinterpret_cast<double*>(ctl + SM_CTL_SUMSQ);
  if (use_host_sumsq) { sumsq[0] = hs0; sumsq[1] = hs1; }
  sm_prepare_scalars(ctl, sumsq[0], sumsq[1], target_norm_offset, ext_tn);
}

// ------------------------------------------------------------------ optional per-class timing
struct Rec { cudaEvent_t a, b; int cls; double bytes; int launches; };
bool g_prof = false;
std::vector<Rec> g_recs;

struct Scope {
  cudaStream_t st; Rec r; bool on;
  Scope(cudaStream_t s, int cls, double bytes, int launches) : st(s), on(g_prof) {
    if (!on) return;
    r.cls = cls; r.bytes = bytes; r.launches = launches;
    cudaEventCreate(&r.a); cudaEventCreate(&r.b);
    cudaEventRecord(r.a, st);
  }
  ~Scope() {
    if (!on) return;
    cudaEventRecord(r.b, st);
    g_recs.push_back(r);
  }
};

}  // namespace

extern "C" int sm_profile_enable(int on) {
  g_prof = on != 0;
  return 0;
}

extern "C" int sm_profile_collect(double* ms, double* bytes, int* launches, int n_classes) {
  for (int i = 0; i < n_classes; ++i) { ms[i] = 0.0; bytes[i] = 0.0; launches[i] = 0; }
  for (auto& r : g_recs) {
    cudaEventSynchronize(r.b);
    float t = 0.f;
    cudaEventElapsedTime(&t, r.a, r.b);
    if (r.cls >= 0 && r.cls < n_classes) { ms[r.cls] += t; bytes[r.cls] += r.bytes; launches[r.cls] += r.launches; }
    cudaEventDestroy(r.a); cudaEventDestroy(r.b);
  }
  g_recs.clear();
  return 0;
}

extern "C" int sm_pair_merge_async(const sm_plan* plan, const void* tables, const sm_pair_args* a, void* stream) {
  const SmPlan& p = plan->p;
  cudaStream_t st = (cudaStream_t)stream;
  const double N = (double)p.R * (double)p.C;
  unsigned char* ctl = reinterpret_cast<unsigned char*>(a->ctl);
  double* dbl = reinterpret_cast<double*>(ctl + SM_CTL_SUMSQ);
  float* flt = reinterpret_cast<float*>(ctl + SM_CTL_FLT);
  uint32_t* flags = reinterpret_cast<uint32_t*>(ctl + SM_CTL_FLAGS);
  const int* swap = reinterpret_cast<const int*>(ctl + SM_CTL_INT) + SM_I_SWAP;
  void* sel0 = ctl + SM_CTL_SEL;
  void* sel1 = ctl + SM_CTL_SEL + SM_SELECT_STATE_BYTES;
  const int sweeps = p.col_passes;
  const int col_launches = sm_plan_col_launches(plan);
  int rc;
  SM_CUDA_CHECK(cudaMemsetAsync(ctl, 0, SM_CTL_BYTES, st));
  const bool rows_done = a->rows_done != 0;
  const bool paired_rows = !rows_done && a->x32_0 == nullptr && a->x32_1 == nullptr && a->base0 == a->base1 &&
                           sm_fwd_rows_pair_supported(plan);
  if (paired_rows) {
    // one shared base: 2N + 2 x 2N read, 2 x 4N written; the pass's last CTA also does what k_prepare does
    Scope s(st, SM_CLS_ROW_FWD, 14.0 * N, 1);
    if ((rc = sm_fwd_rows_bf16_pair(plan, tables, a->base0, a->ft0, a->ft1, a->re[0], a->im[0], a->re[1], a->im[1], ctl,
                                    a->target_norm_offset, a->target_norm, st))) return rc;
  } else {
    if (!rows_done) {
      // bf16 (base, finetune) pairs: 2N + 2N read, 4N written; fp32 tree intermediates: 4N read, 4N written
      Scope s(st, SM_CLS_ROW_FWD, 16.0 * N, 2);
      if (a->x32_0 != nullptr) {
        if ((rc = sm_fwd_rows_f32(plan, tables, a->x32_0, 1.f, 1.f, a->re[0], a->im[0], dbl + 0, st))) return rc;
      } else if ((rc = sm_fwd_rows_bf16(plan, tables, a->base0, a->ft0, a->re[0], a->im[0], dbl + 0, st))) return rc;
      if (a->x32_1 != nullptr) {
        if ((rc = sm_fwd_rows_f32(plan, tables, a->x32_1, 1.f, 1.f, a->re[1], a->im[1], dbl + 1, st))) return rc;
      } else if ((rc = sm_fwd_rows_bf16(plan, tables, a->base1, a->ft1, a->re[1], a->im[1], dbl + 1, st))) return rc;
    }
    Scope s(st, SM_CLS_SCALARS, 0.0, 1);
    sm_launch(k_prepare, dim3(1), dim3(1), (size_t)(0), st, ctl, a->target_norm_offset, a->target_norm, rows_done ? 1 : 0,
                               rows_done ? a->sumsq[0] : 0.0, rows_done ? a->sumsq[1] : 0.0);
    SM_LAUNCH_CHECK();
  }
  {
    Scope s(st, SM_CLS_COL_FWD, 16.0 * N * (sweeps > 0 ? sweeps : 1) - 2.0 * N, 2 * col_launches);
    // only the model in role v0 (the larger norm, `swap` picks it) contributes its imaginary plane: the other one's
    // last sweep does not store it (2N bytes less)
    if ((rc = sm_fwd_cols_sel(plan, tables, a->re[0], a->im[0], flt + SM_F_SCALE_X, 1.f, 1, swap, 1, st))) return rc;
    if ((rc = sm_fwd_cols_sel(plan, tables, a->re[1], a->im[1], flt + SM_F_SCALE_Y, 1.f, 1, swap, 0, st))) return rc;
  }
  void* fs0 = ctl + SM_CTL_FS;
  void* fs1 = ctl + SM_CTL_FS + SM_FS_STATE_BYTES;
  const bool cull = a->cull_pct > 0;
  const bool fused_stats = sm_fstats_supported(plan) && a->select_mode == 0;
  // functions.py:113-120: sorted(cat(|re0|,|re1|))[int(2N*cutoff_pct)]  (Python float arithmetic); :140 for the cull
  const uint64_t rank_cut = (uint64_t)((2.0 * N) * a->cutoff_pct);
  const uint64_t rank_cull = (uint64_t)(N * a->cull_pct);
  if (fused_stats && a->cutoff_pct > 0) {
    // cutoff statistic + SLERP sums + scalars: one pass over Re X, Re Y (kernels_fstats.cu)
    Scope s(st, SM_CLS_SELECT2, 4.0 * N, 3);
    if ((rc = sm_fstats_cutoff(plan, a->re[0], a->re[1], swap, rank_cut, a->t, fs0, a->sel_ws, a->sel_ws_bytes,
                               flt + SM_F_THR_CUT, flt + SM_F_DOT, dbl + 2, st))) return rc;
  } else {
    if (a->cutoff_pct > 0) {
      Scope s(st, SM_CLS_SELECT2, 4.0 * N, 11);
      if ((rc = sm_select_kth_abs(plan, a->re[0], a->re[1], rank_cut, a->select_mode, sel0, a->sel_ws, a->sel_ws_bytes,
                                  flt + SM_F_THR_CUT, st))) return rc;
    }
    {
      Scope s(st, SM_CLS_REDUCE, 4.0 * N, 2);
      if ((rc = sm_slerp_reduce_sel(plan, a->re[0], a->re[1], swap, flt + SM_F_THR_CUT, dbl + 2, st))) return rc;
      if ((rc = sm_slerp_scalars(dbl + 2, a->t, flt + SM_F_DOT, st))) return rc;
    }
  }
  if (fused_stats && cull) {
    // blend + cull statistic of its output: one pass
    Scope s(st, SM_CLS_BLEND, 6.0 * N, 2);
    if ((rc = sm_fstats_blend_cull(plan, a->re[0], a->re[1], swap, flt + SM_F_THR_CUT, flt + SM_F_DOT, a->t_sum, a->re[2],
                                   rank_cull, fs1, a->sel_ws, a->sel_ws_bytes, flt + SM_F_THR_CULL, st))) return rc;
  } else {
    {
      Scope s(st, SM_CLS_BLEND, 6.0 * N, 1);
      if ((rc = sm_blend_sel(plan, 0, 1, a->re[0], a->re[1], swap, flt + SM_F_THR_CUT, flt + SM_F_DOT, a->t_sum, a->re[2], st)))
        return rc;
    }
    if (cull) {
      Scope s(st, SM_CLS_SELECT1, 2.0 * N, 11);
      if ((rc = sm_select_kth_abs(plan, a->re[2], nullptr, rank_cull, a->select_mode, sel1, a->sel_ws, a->sel_ws_bytes,
                                  flt + SM_F_THR_CULL, st))) return rc;
    }
  }
  if (sweeps > 0) {
    Scope s(st, SM_CLS_COL_INV, 8.0 * N * sweeps, col_launches);
    if ((rc = sm_inv_cols_sel(plan, tables, a->re[2], a->im[0], a->im[1], swap, cull ? flt + SM_F_THR_CULL : nullptr, st)))
      return rc;
  }
  {
    Scope s(st, SM_CLS_ROW_INV, 8.0 * N, 1);
    if (a->out_f32 != nullptr) {
      // an intermediate of the pair tree: merged * target_norm as fp32, the base is added after the last round only
      if ((rc = sm_inv_rows_f32_sel(plan, tables, a->re[2], a->im[0], a->im[1], swap, cull ? flt + SM_F_THR_CULL : nullptr,
                                    a->out_f32, flt + SM_F_OUT_SCALE, 1.f, 1, flags, st))) return rc;
    } else if ((rc = sm_inv_rows_bf16_sel(plan, tables, a->re[2], a->im[0], a->im[1], swap, cull ? flt + SM_F_THR_CULL : nullptr,
                                          a->base_out, a->out_bf16, flt + SM_F_OUT_SCALE, 1.f, 1, flags, st))) return rc;
  }
  return 0;
}
