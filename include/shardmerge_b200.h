/* shardmerge_b200.h -- C ABI of libshardmerge_b200.so (sm_100a CUDA kernels).
 *
 * This is the drop-in boundary for the per-tensor spectral ("SLERP-FFT") merge hot path
 * of 54rt1n/shardmerge.  The reference has no FFI of its own (it is pure Python over
 * torch); every entry point below replaces a span of torch library calls at a
 * reference call site, cited per function as `path:line` relative to the reference root.
 * The host side (shardmerge_b200/tensor/functions.py, shardmerge_b200/merge/fast_fourier.py)
 * binds these with ctypes and keeps the reference's Python signatures.
 *
 * Rules of the ABI
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless it is
 *     marked "host"; `stream` is a cudaStream_t passed as void*.
 *   - the library never allocates device memory: tables, spectra, workspaces and scalar
 *     blocks are caller-provided (sizes from the sm_*_bytes queries).
 *   - every call is asynchronous on `stream`; the only host synchronisation is whatever
 *     the caller does to read scalars back.
 *   - return value 0 = ok, negative = error; sm_last_error() gives the message.
 *
 * Spectrum layout ("half planar"): two fp32 planes re[R][P], im[R][P] holding the
 * Hermitian half spectrum, columns 0..C/2 valid, row pitch P = sm_plan_pitch().  Rows are
 * in *stored order*: stored row i holds frequency sm_plan_row_freq(plan, i) (identity
 * unless the column FFT needed two sweeps).  Global statistics count a stored bin once
 * for columns 0 and C/2 and twice otherwise (its mirror image is not stored).
 */
#ifndef SHARDMERGE_B200_H
#define SHARDMERGE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct sm_plan sm_plan;   /* opaque, host memory */

int sm_version(void);
const char* sm_last_error(void);

/* ---- plans ------------------------------------------------------------------------ */
/* Plan for tensors of shape [R][C] (R = 1 for 1-D tensors), C even.  Prime factors 2..13 of C/2 and R run as register
 * butterflies (the shapes of Llama-class models: specialised kernels); any larger prime factor up to 1021 (37 in 18944,
 * 167 in 128256 = a Llama-3 vocabulary) runs as a generic O(r)-per-point radix stage, so that torch.fft's "any length"
 * contract (shard/tensor/functions.py:55-58) holds for every weight shape in practice.  Returns NULL if the shape is
 * unsupported (odd C, a prime factor above 1021, or no four-step split of R that fits in shared memory). */
sm_plan* sm_plan_create(int R, int C);
void sm_plan_destroy(sm_plan* plan);
int sm_plan_pitch(const sm_plan* plan);                 /* P, in floats                       */
int sm_plan_row_freq(const sm_plan* plan, int stored);  /* stored row -> frequency index      */
int sm_plan_col_passes(const sm_plan* plan);            /* column sweeps per transform: 0, 1, 2 */
int sm_plan_col_launches(const sm_plan* plan);          /* kernel launches per column transform (one per sweep) */
int sm_plan_describe(const sm_plan* plan, char* buf, int buflen);   /* human-readable factorisation */
size_t sm_plan_table_bytes(const sm_plan* plan);        /* device bytes for the twiddle tables */
/* Fill the caller's table buffer (twiddles computed on the device in fp64, stored fp32). */
int sm_plan_init_tables(const sm_plan* plan, void* tables, void* stream);

/* ---- forward: delta + real 2-D FFT --------------------------------------------------
 * Replaces get_delta_for_models (shard/merge/base.py:121-137: fp32(ft) - fp32(base)), the
 * norm reduction of normalize_tensor (shard/tensor/functions.py:85) and the row half of
 * fft_transform (shard/tensor/functions.py:55-58).
 * sumsq (fp64, device) receives += sum(delta^2); the caller zeroes it beforehand. */
int sm_fwd_rows_bf16(const sm_plan* plan, const void* tables, const void* base_bf16, const void* ft_bf16,
                     float* re, float* im, double* sumsq, void* stream);
/* Same for an fp32 input tensor x (already a delta / any real tensor); the transform is
 * taken of (x*m1)*m2 (two fp32 roundings, as `a * norm_scale` / `b * weight_scale * norm_scale`
 * at shard/merge/fast_fourier.py:228-230), sumsq accumulates sum(x^2). */
int sm_fwd_rows_f32(const sm_plan* plan, const void* tables, const float* x, float m1, float m2,
                    float* re, float* im, double* sumsq, void* stream);
/* Column half of fft_transform, in place.  The spectrum is multiplied by *scale_dev (if
 * non-NULL) else by scale_host: this is where `tensor / norm` of normalize_tensor
 * (functions.py:88) is applied (the FFT is linear).  write_im = 0 skips storing the
 * imaginary plane (the blend never reads Im X1). */
int sm_fwd_cols(const sm_plan* plan, const void* tables, float* re, float* im,
                const float* scale_dev, float scale_host, int write_im, void* stream);
/* *out = 1/(float)sqrt(*sumsq), or 1 if the sum is 0 (normalize_tensor's `if norm != 0`). */
int sm_inv_norm(const double* sumsq, float* out, void* stream);

/* ---- order statistics ---------------------------------------------------------------
 * Replace the two full torch.sort calls of interpolate_fft_components
 * (shard/tensor/functions.py:113-122 cutoff, :138-148 cull): the element of 0-based rank
 * `rank` of |plane0| (and |plane1| concatenated, if non-NULL) over the FULL spectrum,
 * i.e. with the Hermitian multiplicities above.  Exact: the result is the bit pattern of
 * an actual element.
 *   mode 0 (fast): a random sample predicts a narrow window around the statistic, one
 *          streaming pass counts what lies below it and collects what lies inside, a
 *          radix select over the collected keys finishes.  If the window misses or the
 *          candidate buffer overflows, state->status != 0 and *thr_out = NaN.
 *   mode 1 (safe): window = everything; needs a workspace for all keys.
 * sel_state: >= SM_SELECT_STATE_BYTES device bytes.  ws: sm_select_ws_bytes() device bytes.
 * After completion (stream order) sel_state holds {u64 rank, u64 below, u32 prefix, u32 lo,
 * u32 hi, u32 ncand, u32 cap, u32 status, f32 value, u32 sticky}; `sticky` ORs the status of
 * every select that used this state since the caller last zeroed it. */
#define SM_SELECT_STATE_BYTES 64
size_t sm_select_ws_bytes(const sm_plan* plan, int n_planes, int mode);
int sm_select_kth_abs(const sm_plan* plan, const float* plane0, const float* plane1, uint64_t rank,
                      int mode, void* sel_state, void* ws, size_t ws_bytes, float* thr_out, void* stream);

/* ---- SLERP statistics and blend ------------------------------------------------------
 * Masked sums for slerp() (shard/tensor/functions.py:36-41) over
 * slerp_mask = sign(re0)==sign(re1) & ~(|re1| < thr_cut)  (functions.py:124-127; both
 * "small" masks test re1 in the reference): sums3 += {sum re0^2, sum re1^2, sum re0*re1},
 * fp64, Hermitian multiplicities applied.  *thr_cut is read on the device. */
int sm_slerp_reduce(const sm_plan* plan, const float* re0, const float* re1, const float* thr_cut,
                    double* sums3, void* stream);
/* scal4 = {dot, cos(theta), sin(theta), max(||v1 - v0*dot||, 1e-12)} as fp32
 * (functions.py:36-43; theta = acos(clamp(dot)) * t). */
int sm_slerp_scalars(const double* sums3, double t, float* scal4, void* stream);
/* Three-way masked blend of the real parts (functions.py:124-136); out may alias re0.
 * mode 0: SLERP blend with *thr_cut, scal4, t_sum.
 * mode 1: arithmetic blend of arithmetic_fft_components (functions.py:273-284):
 *         sign agreement -> re0 + t*re1, else re1 (the reference's "larger" mask is always
 *         False); agreement = 0 -> always re0 + t*re1.  t is passed in t_sum. */
int sm_blend(const sm_plan* plan, int mode, int agreement, const float* re0, const float* re1,
             const float* thr_cut, const float* scal4, float t_sum, float* out_re, void* stream);

/* ---- fused statistics (what the pair-merge chain uses for tensors of more than 2^20 elements) ----------
 * sm_fstats_cutoff = sm_select_kth_abs(re0, re1, rank) + sm_slerp_reduce + sm_slerp_scalars in ONE streaming
 * pass over the two real planes (functions.py:113-129, :36-43): thr_cut_out, scal4_out (and sums3_out, if
 * non-NULL) are written on the device.  `sel` (nullable, device int): non-zero swaps the roles, i.e.
 * (re0, re1) = (reY, reX).
 * sm_fstats_blend_cull = sm_blend(mode 0) + sm_select_kth_abs(out, rank) in one pass (functions.py:131-141).
 * Both use a sampled key window; fs_state (SM_FS_STATE_BYTES device bytes, zero before the first use) holds a
 * u32 at byte SM_FS_STATUS_OFF that is non-zero afterwards if the window missed / was too wide / a bucket
 * overflowed -- the thresholds are NaN then and the caller redoes the tensor with the step-by-step kernels
 * (sm_select_kth_abs mode 1).  ws: at least sm_fstats_ws_bytes() device bytes, zero-filled before the first use;
 * the kernels use the LAST sm_fstats_ws_bytes() of it and keep their histograms there from call to call (each call
 * clears what the previous one touched: nobody else may write to that part, and a buffer serves ONE plan), so one
 * buffer of sm_select_ws_bytes() + sm_fstats_ws_bytes() serves both families.  sm_fstats_supported() == 0: tensor
 * too small (launch bound; use the step-by-step kernels) or too large (>= 2^31 elements). */
#define SM_FS_STATE_BYTES 128
#define SM_FS_STATUS_OFF 28
#define SM_FS_STICKY_OFF 72      /* u32: OR of the status of every call that used this state since it was zeroed */
int sm_fstats_supported(const sm_plan* plan);
size_t sm_fstats_ws_bytes(const sm_plan* plan);
int sm_fstats_cutoff(const sm_plan* plan, const float* reX, const float* reY, const int* sel, uint64_t rank,
                     double t, void* fs_state, void* ws, size_t ws_bytes, float* thr_cut_out,
                     float* scal4_out, double* sums3_out, void* stream);
int sm_fstats_blend_cull(const sm_plan* plan, const float* reX, const float* reY, const int* sel,
                         const float* thr_cut, const float* scal4, float t_sum, float* out_re, uint64_t rank,
                         void* fs_state, void* ws, size_t ws_bytes, float* thr_cull_out, void* stream);

/* ---- inverse: cull + inverse 2-D FFT + epilogue ---------------------------------------
 * Column half of ifft_transform (functions.py:70-73), in place; values of the real plane
 * with |re| < *cull_thr are read as 0 (functions.py:146; cull_thr may be NULL). */
int sm_inv_cols(const sm_plan* plan, const void* tables, float* re, float* im, const float* cull_thr,
                void* stream);
/* Row half of ifft_transform + everything after it:
 *   x = ifft * 1/(R*C); NaN -> 0, count Inf            (functions.py:208-217)
 *   x = x * scale  (scale = *scale_dev or scale_host)  (fast_fourier.py:243, target_norm)
 *   y = fp32(base) + x; NaN -> 0, count Inf; bf16 RNE  (fast_fourier.py:269-276)
 * flags4 += {nan after ifft, inf after ifft, nan final, inf final} (u32 counters).
 * cull_thr is only honoured for 1-D plans (no column sweep).
 * check_ifft = 0 skips the first NaN->0 / Inf step: task_arithmetic_fft2 (functions.py:224-254)
 * returns the raw ifft, so a NaN there survives until the final check of _merge_layer. */
int sm_inv_rows_bf16(const sm_plan* plan, const void* tables, const float* re, const float* im,
                     const float* cull_thr, const void* base_bf16, void* out_bf16,
                     const float* scale_dev, float scale_host, int check_ifft, uint32_t* flags4, void* stream);
/* fp32 variant without the base add: out = ifft/(R*C) (NaN -> 0) * scale. */
int sm_inv_rows_f32(const sm_plan* plan, const void* tables, const float* re, const float* im,
                    const float* cull_thr, float* out, const float* scale_dev, float scale_host,
                    int check_ifft, uint32_t* flags4, void* stream);

/* ---- element-wise paths that need no FFT ------------------------------------------------
 * out_bf16 = bf16(fp32(base_out) + (ca*(ft0-base0) + cb*(ft1-base1)) * scale), NaN -> 0, Inf
 * counted in flags4[2..3].  Covers `merged = a + b` (fast_fourier.py:223-225), the
 * single-model case (:256-257) and the small-norm early returns of
 * merge_tensors_fft2_slerp (functions.py:184-190).  Any of ft1/base1 may be NULL (cb ignored). */
int sm_delta_axpby_bf16(size_t n, const void* base_out, const void* base0, const void* ft0, float ca,
                        const void* base1, const void* ft1, float cb, float scale, void* out_bf16,
                        uint32_t* flags4, void* stream);
/* pass-through copy with dtype cast to bf16 done by the writer: plain device copy of n bytes
 * (is_input / is_output tensors, fast_fourier.py:104-130). */
int sm_copy_bytes(void* dst, const void* src, size_t n, void* stream);

/* ---- API-level format conversion (not on the timed path) --------------------------------
 * Half planar (stored order) -> full complex64 [R][C] in natural order with the Hermitian
 * mirror filled in: what fft_transform returns (functions.py:55-58). */
int sm_expand_full(const sm_plan* plan, const float* re, const float* im, float* out_c64, void* stream);
/* Full complex64 [R][C] natural order -> half planar stored order, Hermitian-projected
 * ((Z[k] + conj(Z[-k]))/2), i.e. exactly the part `.real` of ifftn keeps (functions.py:73). */
int sm_pack_half(const sm_plan* plan, const float* in_c64, float* re, float* im, void* stream);


/* ---- fused pair merge (no host synchronisation) ---------------------------------------------
 * The regular-layer body of FourierMerge._merge_layer (shard/merge/fast_fourier.py:147-276) for two
 * bf16 finetunes, issued as ONE stream-ordered chain from a single call: row passes -> device-side
 * decisions (which model is `a`, :212-215; branch, :223-244; target_norm, :165) -> column sweeps ->
 * cutoff statistic -> SLERP sums -> blend -> cull statistic -> inverse sweeps -> epilogue.
 * The chain always runs the SLERP branch; afterwards the scalar block tells the caller whether that
 * was right: ints[SM_I_BRANCH] != SM_BRANCH_SLERP, a non-zero status in either fused-statistics state
 * (SM_CTL_FS + k * SM_FS_STATE_BYTES + SM_FS_STATUS_OFF) or a non-zero `sticky` in either select state
 * (small tensors), or flags[1] / flags[3] (Inf) mean "redo this tensor on the step-by-step path / raise".
 *
 * Scalar block layout (SM_CTL_BYTES device bytes, zeroed by the call): */
#define SM_CTL_BYTES   1024
#define SM_CTL_SUMSQ   0      /* double[2]  sum(delta^2) of model x, y                         */
#define SM_CTL_SUMS    16     /* double[3]  masked SLERP sums s00, s11, s01                    */
#define SM_CTL_FLT     64     /* float[16]  indexed by SM_F_*                                  */
#define SM_CTL_FLAGS   128    /* u32[4]     nan/inf after ifft, nan/inf final                  */
#define SM_CTL_INT     144    /* i32[4]     indexed by SM_I_*                                  */
#define SM_CTL_TN      160    /* double     target_norm                                        */
#define SM_CTL_SEL     192    /* 2 x SM_SELECT_STATE_BYTES: cutoff select, cull select (step-by-step path) */
#define SM_CTL_FS      512    /* 2 x SM_FS_STATE_BYTES: fused cutoff statistics, fused blend + cull   */
#define SM_F_THR_CUT 0
#define SM_F_THR_CULL 1
#define SM_F_DOT 2            /* dot, cos, sin, relnorm follow (scal4 of sm_slerp_scalars)     */
#define SM_F_SCALE_X 6
#define SM_F_SCALE_Y 7
#define SM_F_OUT_SCALE 8
#define SM_F_NORM_X 9
#define SM_F_NORM_Y 10
#define SM_I_SWAP 0
#define SM_I_BRANCH 1
#define SM_BRANCH_SLERP 0
#define SM_BRANCH_ADD 1
#define SM_BRANCH_ARITH 2
#define SM_BRANCH_EARLY 3
#define SM_BRANCH_LINEAR 4

typedef struct sm_pair_args {
  const void* base0; const void* ft0;      /* bf16 [R][C]: model x and the base it is a delta of */
  const void* base1; const void* ft1;      /* model y                                            */
  const void* base_out; void* out_bf16;    /* output base (added back) and the merged result      */
  float* re[3]; float* im[2];              /* planes: (re[0], im[0]) for x, (re[1], im[1]) for y, re[2] blend output */
  void* ctl;                               /* scalar block, SM_CTL_BYTES                          */
  void* sel_ws; size_t sel_ws_bytes;       /* statistics workspace: max(sm_fstats_ws_bytes, sm_select_ws_bytes for 2 planes) */
  double t;                                /* a_weight / (a_weight + b_weight), config order      */
  float t_sum;
  double cutoff_pct, cull_pct;
  double target_norm_offset;
  int select_mode;                         /* 0 fast (sampled window), 1 safe                     */
} sm_pair_args;

int sm_pair_merge_slerp_async(const sm_plan* plan, const void* tables, const sm_pair_args* args, void* stream);

/* The same chain as one pair merge INSIDE the pairwise tree that FourierMerge._merge_layer builds for more than two
 * finetunes (shard/merge/fast_fourier.py:171-254: round 1 merges pairs of deltas, later rounds merge the fp32 results,
 * cull_pct halves per round, target_norm is the mean over ALL models' norms, :165).  `ext` adds what the tree needs:
 *   x32_0 / x32_1  non-NULL: that input is an fp32 [R][C] tensor (an earlier round's result) instead of (base, ft);
 *   rows_done      1: the row passes of both inputs already ran into (re[k], im[k]) and `sumsq` holds their sums of
 *                  squares (round 1: the caller transforms every model once, reads the norms, pairs them on the host
 *                  like correlated_pairs does, :180-186);
 *   target_norm    > 0: use it instead of the mean of the two norms;
 *   out_f32        non-NULL: write merged * target_norm as fp32 (no base add, no bf16 cast): an intermediate of the tree.
 * Branch / role decisions stay on the device as in sm_pair_merge_slerp_async. */
typedef struct sm_pair_ext {
  const float* x32_0; const float* x32_1;
  int rows_done;
  double sumsq[2];
  double target_norm;
  float* out_f32;
} sm_pair_ext;
int sm_pair_merge_tree_async(const sm_plan* plan, const void* tables, const sm_pair_args* args, const sm_pair_ext* ext, void* stream);

/* Per-kernel-class CUDA-event timing of the fused chain (bench.py roofline).  Classes: */
#define SM_CLS_ROW_FWD 0
#define SM_CLS_COL_FWD 1
#define SM_CLS_SELECT2 2
#define SM_CLS_REDUCE 3
#define SM_CLS_SCALARS 4
#define SM_CLS_BLEND 5
#define SM_CLS_SELECT1 6
#define SM_CLS_COL_INV 7
#define SM_CLS_ROW_INV 8
#define SM_CLS_COUNT 9
int sm_profile_enable(int on);
/* Synchronises the recorded events; per class: milliseconds, algorithmic bytes, kernel launches
 * accumulated since the last collect (host arrays of n_classes entries). */
int sm_profile_collect(double* ms, double* bytes, int* launches, int n_classes);

/* ---- element-wise strategies (next to the spectral path: the reference's other MergeTensorsBase subclasses) ----------
 * mode 0: AdditionMerge._merge_layer (shard/merge/addition.py:44-83): out = sum_k (ft_k - base), every op rounded to
 *         the tensors' dtype like the reference's in-dtype arithmetic; the base is NOT added back.
 * mode 1: TaskAdditionMerge._merge_layer (shard/merge/taskaddition.py:44-83): deltas whose sign differs from the
 *         majority sign are zeroed, the rest summed (fp32 accumulation in model order, one rounding).
 * n elements, `fts` = HOST array of n_models device pointers; all 16-byte aligned.
 * sm_elem_merge: dtype 0 fp32, 1 bf16, 2 fp16 (every op in the tensors' own dtype, as torch does), 1..64 models; from 16
 * models on, mode 1 sums like torch.sum on the CPU (16-row groups folded into a second fp32 accumulator).  bf16 with <= 8
 * models runs kernels with a compile-time model count.  sm_elem_merge_bf16 = sm_elem_merge(dtype 1). */
int sm_elem_merge(int mode, int dtype, size_t n, const void* base, const void* const* fts, int n_models, void* out, void* stream);
int sm_elem_merge_bf16(int mode, size_t n, const void* base, const void* const* fts, int n_models, void* out, void* stream);

/* correlate_pairs (shard/tensor/functions.py:304-314), one pair: *out_sum = sum over the C columns of the cosine similarity
 * along dim 0 of two [R][C] device tensors (a 1-D tensor is [n][1]); the caller divides by C (torch's .mean()).
 * dtype 0: fp32, 1: bf16.  Both tensors are read once (HBM-bound). */
int sm_cosine_cols(int dtype, int R, int C, const void* a, const void* b, double* out_sum, void* stream);

/* ---- PEFT LoRA adapters: the finetuned weight formed from the base and the adapter's low-rank factors ------------------
 * ft_out[i][j] = round_to_dtype(base)( fp32(base[i][j]) + scaling * acc[i][j] ) with
 * acc[i][j] = sum_{k=0..r-1} fp32(lora_B[i][k]) * fp32(lora_A[k][j]): one fp32 FMA per term, ascending k, starting from 0;
 * the product with `scaling` and the add are rounded separately; the final rounding is round-to-nearest-even, and NaN and
 * Inf propagate as IEEE arithmetic does.  base and ft_out are [R][C] row-major in base_dtype, lora_A is [r][C] and lora_B
 * [R][r], both in ab_dtype (dtype codes of sm_elem_merge: 0 fp32, 1 bf16, 2 fp16).  Any R, C, r >= 1 (R <= 4,194,240);
 * ft_out must not alias base.  No allocation; asynchronous on `stream`. */
int sm_lora_materialize(int R, int C, int r, int base_dtype, const void* base, int ab_dtype, const void* lora_A,
                        const void* lora_B, float scaling, void* ft_out, void* stream);

/* ---- A checkpoint's difference from its base: the dense products of a randomized SVD of delta ---------------------------
 * delta[i][j] = fp32(M[i][j]) - fp32(W[i][j]) (one rounded fp32 subtraction) of two [R][C] row-major tensors W in w_dtype
 * and M in m_dtype (dtype codes 0 fp32, 1 bf16, 2 fp16); delta is formed on load and never stored.
 *   sm_lowrank_right:  Y[R][k] = delta . X[C][k];  if sumsq is non-null, *sumsq = sum of fp32(delta^2) in fp64
 *   sm_lowrank_left:   Z[k][C] = Q[R][k]^T . delta
 * X, Q, Y, Z are fp32 row-major.  Every output element is fp32 FMA chains over pieces of the reduction (C or R) added in a
 * fixed order: the result is bit-identical from run to run.  ws is a 16-byte aligned device workspace of at least
 * sm_lowrank_ws_bytes(R, C, k) bytes (one size serves both calls).  Any R, C, k >= 1 with R, C <= 8,388,480.
 * No allocation; asynchronous on `stream`. */
size_t sm_lowrank_ws_bytes(int R, int C, int k);
int sm_lowrank_right(int R, int C, int k, int w_dtype, const void* W, int m_dtype, const void* M, const float* X, float* Y,
                     double* sumsq, void* ws, size_t ws_bytes, void* stream);
int sm_lowrank_left(int R, int C, int k, int w_dtype, const void* W, int m_dtype, const void* M, const float* Q, float* Z,
                    void* ws, size_t ws_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SHARDMERGE_B200_H */
