// fft_bodies.cuh -- the per-CTA bodies of the four FFT sweeps, written against an
// "Exec" policy so that the very same code runs as a CUDA thread block
// (kernels_fft.cu: DeviceExec) and as a sequential loop over emulated threads
// (tests/hostemu: HostExec).  A body is a sequence of phases; every phase is executed
// by all threads of the CTA and is followed by a block barrier.
//
//   row_fwd_body : delta (ft - base) + real FFT of one row  [replaces get_delta_for_models
//                  shard/merge/base.py:121-137 + the row half of fft_transform
//                  shard/tensor/functions.py:55-58; sum of squares for normalize_tensor :85]
//   col_body     : one in-place sweep of the complex column FFT (forward or inverse)
//   row_inv_body : inverse real FFT of one row + epilogue (x 1/N, NaN->0, Inf flag,
//                  x target_norm, + base, NaN->0, Inf flag, bf16 RNE)
//                  [replaces ifft_transform functions.py:70-73, :208-217 and
//                  shard/merge/fast_fourier.py:243,269-276]
#pragma once
#include "fft_core.cuh"
#include "plan.h"

// A phase is a plain loop over the CTA's threads followed by a barrier.  On the device the loop
// runs exactly once (tid = threadIdx.x) and sync() is __syncthreads(); on the host it walks all
// emulated threads.  (No lambdas here: closures that capture by reference end up in local memory
// and turn every captured scalar into a generic load -- measured on k_row_inv, profiles/r01.)
#define SM_FOR_THREADS(ex, tid) for (int tid = (ex).tid_begin(), tid##_end = (ex).tid_end(); tid < tid##_end; ++tid)

namespace smfft {

// counter bump that works on both sides (device: a rare global atomic; host: plain increment)
SM_HD void sm_count(unsigned int* p) {
#if defined(__CUDA_ARCH__)
  atomicAdd(p, 1u);
#else
  *p += 1u;
#endif
}

// NaN -> 0 (counted in flags[which]), Inf kept (counted in flags[which+1]): the exceptional path of
// the epilogue, kept out of line so the hot loop stays small.
#if defined(__CUDACC__)
__host__ __device__ __noinline__
#else
inline
#endif
float sm_fix_nonfinite(float v, unsigned int* flags, int which) {
  const uint32_t u = f32_bits(v) & 0x7fffffffu;
  if (u > 0x7f800000u) { sm_count(flags + which); return 0.f; }
  if (u == 0x7f800000u) sm_count(flags + which + 1);
  return v;
}

// ------------------------------------------------------------------ smem accessors
struct RowSmem {               // one contiguous sequence, optional 1-in-16 padding
  cf* buf; int padmask;        // padmask = ~0 (padded) or 0
  SM_HD int phys(int i) const { return i + ((i >> 4) & padmask); }
  SM_HD void load(int i, float& re, float& im) const { cf v = buf[phys(i)]; re = v.x; im = v.y; }
  SM_HD void store(int i, float re, float im) const { cf v; v.x = re; v.y = im; buf[phys(i)] = v; }
};
struct ColSmem {               // [idx][32 columns], lane fastest: conflict free by construction
  cf* buf; int lane;
  SM_HD void load(int i, float& re, float& im) const { cf v = buf[i * SM_COL_TILE + lane]; re = v.x; im = v.y; }
  SM_HD void store(int i, float re, float im) const { cf v; v.x = re; v.y = im; buf[i * SM_COL_TILE + lane] = v; }
};

// ------------------------------------------------------------------ row forward
struct RowFwdArgs {
  int mode;                    // 0: bf16 base + bf16 finetune -> delta ; 1: fp32 input
  const uint16_t* base; const uint16_t* ft;
  const float* x32; float m1, m2;        // fp32 input is used as (x*m1)*m2
  float* re; float* im;        // output planes [R][P]
};

struct RowDeltaSrc {           // stage-1 source: element idx is the packed pair (x[2idx], x[2idx+1])
  int mode; const uint32_t* b32; const uint32_t* f32; const cf* x32; float m1, m2; float* acc;
  // *acc is a per-thread fp32 partial over the <= 64 values one thread loads for one row; the
  // caller widens it to fp64 per row, so the rounding of the partials averages out over rows.
  SM_HD void load(int i, float& re, float& im) const {
    float d0, d1;
    if (mode == 0) {
      const uint32_t bb = ldg_u32(b32 + i), ff = ldg_u32(f32 + i);
      d0 = bf16_bits_to_f32(ff & 0xffffu) - bf16_bits_to_f32(bb & 0xffffu);
      d1 = bits_f32(ff & 0xffff0000u) - bits_f32(bb & 0xffff0000u);
    } else {
      const cf v = ldg_cf(x32 + i);
      d0 = v.x; d1 = v.y;
    }
    *acc = fmaf(d0, d0, fmaf(d1, d1, *acc));
    if (mode != 0) { d0 = (d0 * m1) * m2; d1 = (d1 * m1) * m2; }
    re = d0; im = d1;
  }
};

template <class Exec>
SM_HD void row_fwd_body(Exec& ex, const SmPlan& pl, int row, const RowFwdArgs& a, const cf* twC, const cf* twQ,
                        cf* smem, float* acc) {
  const int Ch = pl.Ch, T = ex.nthreads();
  const int bufstride = pl.row_pad ? (Ch + (Ch >> 4) + 1) : Ch;
  const int padmask = pl.row_pad ? ~0 : 0;
  RowDeltaSrc gsrc;
  gsrc.mode = a.mode;
  gsrc.b32 = a.mode == 0 ? reinterpret_cast<const uint32_t*>(a.base + (size_t)row * pl.C) : nullptr;
  gsrc.f32 = a.mode == 0 ? reinterpret_cast<const uint32_t*>(a.ft + (size_t)row * pl.C) : nullptr;
  gsrc.x32 = a.mode != 0 ? reinterpret_cast<const cf*>(a.x32 + (size_t)row * pl.C) : nullptr;
  gsrc.m1 = a.m1; gsrc.m2 = a.m2; gsrc.acc = acc;
  int s = 1, cur = 0;
  for (int st = 0; st < pl.n_row; ++st) {
    const int r = pl.row_rad[st], nb = Ch / r;
    const bool last = (st == pl.n_row - 1);
    RowSmem sin{smem + (size_t)(cur ^ 1) * bufstride, padmask};   // written by the previous stage
    RowSmem sout{smem + (size_t)cur * bufstride, padmask};
    if (sm_radix_is_generic(r)) {             // never the first stage (sm_make_plan): the source is shared memory
      SM_FOR_THREADS(ex, tid) {
        for (int it = tid; it < Ch; it += T) {
          if (last) stockham_generic_output<true>(r, it, Ch, s, 2, twC, sin, sout);
          else      stockham_generic_output<false>(r, it, Ch, s, 2, twC, sin, sout);
        }
      }
      ex.sync();
      s *= r; cur ^= 1;
      continue;
    }
    SM_FOR_THREADS(ex, tid) {
      for (int b = tid; b < nb; b += T) {
        if (st == 0) {
          if (last) stockham_bfly_rt<true>(r, b, Ch, s, 2, twC, gsrc, sout);
          else      stockham_bfly_first_rt(r, b, Ch, twQ, gsrc, sout);
        } else {
          if (last) stockham_bfly_rt<true>(r, b, Ch, s, 2, twC, sin, sout);
          else      stockham_bfly_rt<false>(r, b, Ch, s, 2, twC, sin, sout);
        }
      }
    }
    ex.sync();
    s *= r; cur ^= 1;
  }
  // untangle the packed transform into the Hermitian half spectrum X[0..Ch]
  RowSmem z{smem + (size_t)(cur ^ 1) * bufstride, padmask};
  float* ore = a.re + (size_t)row * pl.P;
  float* oim = a.im + (size_t)row * pl.P;
  SM_FOR_THREADS(ex, tid) {
    for (int k = tid; k <= Ch; k += T) {
      const int k0 = (k == Ch) ? 0 : k;
      const int k1 = (k == 0 || k == Ch) ? 0 : Ch - k;
      float ar, ai, br, bi;
      z.load(k0, ar, ai);
      z.load(k1, br, bi);
      const float er = 0.5f * (ar + br), ei = 0.5f * (ai - bi);
      const float pr = 0.5f * (ai + bi), qi = -0.5f * (ar - br);
      const cf w = ldg_cf(twC + k);
      ore[k] = er + (pr * w.x - qi * w.y);
      oim[k] = ei + (pr * w.y + qi * w.x);
    }
  }
  ex.sync();
}

// ------------------------------------------------------------------ row inverse
struct RowInvArgs {
  const float* re; const float* im;      // spectrum planes [R][P] (after the inverse column sweeps)
  const float* im_alt; const int* sel;   // nullable: if *sel != 0 the imaginary plane is im_alt (device-side role pick)
  const float* cull_thr;                 // nullable; only used when R == 1 (no column sweep)
  int out_mode;                          // 0: bf16 = bf16(base + x*scale) ; 1: fp32 = x*scale
  const uint16_t* base; uint16_t* out_bf16; float* out_f32;
  float inv_n;                           // 1/(R*C)
  const float* scale_ptr; float scale_host;
  int check_ifft;                        // 1: NaN->0 / count Inf right after the ifft
  unsigned int* flags;                   // [0] nan after ifft [1] inf after ifft [2] nan final [3] inf final
};

struct RowTangleSrc {          // stage-1 source of the inverse: Z'[k] from X[k], X[Ch-k], already re/im swapped
  const float* re; const float* im; const cf* twC; int Ch; float thr;
  SM_HD float cull(float v) const { return (v < thr && -v < thr) ? 0.f : v; }   // |v| < thr, NaN kept
  SM_HD void load(int k, float& ore, float& oim) const {
    float xr = cull(ldg_f32(re + k)), xi = ldg_f32(im + k);
    float mr = cull(ldg_f32(re + Ch - k)), mi = ldg_f32(im + Ch - k);
    if (k == 0) { xi = 0.f; mi = 0.f; }    // .real semantics: bins 0 and Ch are real
    const float Ar = xr + mr, Ai = xi - mi;
    const float Br = xr - mr, Bi = xi + mi;
    const cf w = ldg_cf(twC + k);         // (cos, -sin); conj(w) = (cos, +sin)
    const float br = Br * w.x + Bi * w.y; // B * conj(w), conj(w) = (w.x, -w.y)
    const float bi = Bi * w.x - Br * w.y;
    // Z' = A + i*B' ; hand it to the forward engine swapped
    const float zr = Ar - bi, zi = Ai + br;
    ore = zi; oim = zr;
  }
};

struct RowEpilogueDst {        // last-stage sink of the inverse: element j is (x[2j], x[2j+1]) swapped
  int out_mode; const uint32_t* base32; uint32_t* out32; cf* outf; float inv_n, scale; int check;
  unsigned int* flags;         // global counters [4]; NaN / Inf are exceptional, so a direct atomic is fine
  SM_HD float fin(float v, int which) const { return sm_fix_nonfinite(v, flags, which); }
  SM_HD void store(int j, float a, float b) const {
    float x0 = b * inv_n, x1 = a * inv_n;
    if (check) { if (not_finite(x0)) x0 = fin(x0, 0); if (not_finite(x1)) x1 = fin(x1, 0); }
    x0 *= scale; x1 *= scale;
    if (out_mode == 0) {
      const uint32_t bb = ldg_u32(base32 + j);
      x0 = bf16_bits_to_f32(bb & 0xffffu) + x0;
      x1 = bits_f32(bb & 0xffff0000u) + x1;
      if (not_finite(x0)) x0 = fin(x0, 2);
      if (not_finite(x1)) x1 = fin(x1, 2);
      out32[j] = pack_bf16x2_rne(x0, x1);
    } else {
      cf v; v.x = x0; v.y = x1; outf[j] = v;
    }
  }
};

template <class Exec>
SM_HD void row_inv_body(Exec& ex, const SmPlan& pl, int row, const RowInvArgs& a, const cf* twC, const cf* twQ,
                        cf* smem) {
  const int Ch = pl.Ch, T = ex.nthreads();
  const int bufstride = pl.row_pad ? (Ch + (Ch >> 4) + 1) : Ch;
  const int padmask = pl.row_pad ? ~0 : 0;
  RowTangleSrc gsrc;
  gsrc.re = a.re + (size_t)row * pl.P;
  gsrc.im = ((a.sel != nullptr && *a.sel != 0) ? a.im_alt : a.im) + (size_t)row * pl.P;
  gsrc.twC = twC; gsrc.Ch = Ch;
  gsrc.thr = (a.cull_thr != nullptr) ? *a.cull_thr : 0.f;
  RowEpilogueDst gdst;
  gdst.out_mode = a.out_mode;
  gdst.base32 = a.out_mode == 0 ? reinterpret_cast<const uint32_t*>(a.base + (size_t)row * pl.C) : nullptr;
  gdst.out32 = a.out_mode == 0 ? reinterpret_cast<uint32_t*>(a.out_bf16 + (size_t)row * pl.C) : nullptr;
  gdst.outf = a.out_mode != 0 ? reinterpret_cast<cf*>(a.out_f32 + (size_t)row * pl.C) : nullptr;
  gdst.inv_n = a.inv_n; gdst.check = a.check_ifft;
  gdst.scale = a.scale_ptr ? *a.scale_ptr : a.scale_host;
  gdst.flags = a.flags;
  int s = 1, cur = 0;
  for (int st = 0; st < pl.n_row; ++st) {
    const int r = pl.row_rad[st], nb = Ch / r;
    const bool first = (st == 0), last = (st == pl.n_row - 1);
    RowSmem sin{smem + (size_t)(cur ^ 1) * bufstride, padmask};
    RowSmem sout{smem + (size_t)cur * bufstride, padmask};
    if (sm_radix_is_generic(r)) {             // never the first stage (sm_make_plan)
      SM_FOR_THREADS(ex, tid) {
        for (int it = tid; it < Ch; it += T) {
          if (last) stockham_generic_output<true>(r, it, Ch, s, 2, twC, sin, gdst);
          else      stockham_generic_output<false>(r, it, Ch, s, 2, twC, sin, sout);
        }
      }
      ex.sync();
      s *= r; cur ^= 1;
      continue;
    }
    SM_FOR_THREADS(ex, tid) {
      for (int b = tid; b < nb; b += T) {
        if (first && last)  stockham_bfly_rt<true>(r, b, Ch, s, 2, twC, gsrc, gdst);
        else if (first)     stockham_bfly_first_rt(r, b, Ch, twQ, gsrc, sout);
        else if (last)      stockham_bfly_rt<true>(r, b, Ch, s, 2, twC, sin, gdst);
        else                stockham_bfly_rt<false>(r, b, Ch, s, 2, twC, sin, sout);
      }
    }
    ex.sync();
    s *= r; cur ^= 1;
  }
}

// ------------------------------------------------------------------ column sweep
struct ColArgs {
  float* re; float* im;        // planes [R][P], transformed in place
  float* im_alt; const int* sel;   // nullable: if *sel != 0 the imaginary plane is im_alt
  int L; int n_rad; int rad[SM_MAX_STAGES];
  int inst_mul, elem_mul;      // stored row of element i of instance g: g*inst_mul + i*elem_mul
  int tw_mul;                  // W_L^e = twR[e * tw_mul], tw_mul = R / L
  int big_tw;                  // multiply output k of instance g by W_R^(g*k)
  int swap;                    // inverse sweep: swap re/im on load and on store
  const float* cull_thr;       // nullable: |re| < thr -> 0 on load (first inverse sweep)
  const float* scale_ptr; float scale_host; int use_scale;   // outputs *= scale (last forward sweep)
  int write_im;                // 0: do not store the imaginary plane
  const int* wsel; int wskip;  // nullable: forward, do not store the imaginary plane if (*wsel != 0) == (wskip != 0)
};

struct ColGlobalSrc {
  const float* re; const float* im; size_t row0; size_t estride; bool valid; int swap; float thr;
  SM_HD void load(int i, float& ore, float& oim) const {
    float xr = 0.f, xi = 0.f;
    if (valid) {
      const size_t off = row0 + (size_t)i * estride;
      xr = re[off]; xi = im[off];
      if (xr < thr && -xr < thr) xr = 0.f;
    }
    if (swap) { ore = xi; oim = xr; } else { ore = xr; oim = xi; }
  }
};
struct ColGlobalDst {
  float* re; float* im; size_t row0; size_t estride; bool valid; int swap;
  const cf* twR; int big_step;   // big_step = instance index (0 when no inter-sweep twiddle)
  float scale; int write_im;
  SM_HD void store(int k, float xr, float xi) const {
    if (big_step != 0) { const cf w = twR[(size_t)big_step * k]; cmul(xr, xi, w.x, w.y); }
    xr *= scale; xi *= scale;
    if (!valid) return;
    const size_t off = row0 + (size_t)k * estride;
    if (swap) { re[off] = xi; if (write_im) im[off] = xr; }
    else      { re[off] = xr; if (write_im) im[off] = xi; }
  }
};

// One CTA = one FFT instance x 32 adjacent columns.  tid -> (warp = butterfly slot, lane = column).
template <class Exec>
SM_HD void col_body(Exec& ex, const SmPlan& pl, int tile, int inst, const ColArgs& a, const cf* twR, cf* smem) {
  const int T = ex.nthreads(), nwarps = T / 32;
  const int L = a.L;
  const int col0 = tile * SM_COL_TILE;
  int s = 1, cur = 0;
  for (int st = 0; st < a.n_rad; ++st) {
    const int r = a.rad[st], nb = L / r;
    const bool first = (st == 0), last = (st == a.n_rad - 1);
    SM_FOR_THREADS(ex, tid) {
      const int lane = tid & 31, wid = tid >> 5;
      const int c = col0 + lane;
      const bool valid = (c <= pl.Ch);
      const size_t row0 = (size_t)inst * a.inst_mul * pl.P + c;
      const size_t estride = (size_t)a.elem_mul * pl.P;
      float* const imp = (a.sel != nullptr && *a.sel != 0) ? a.im_alt : a.im;
      ColGlobalSrc gsrc{a.re, imp, row0, estride, valid, a.swap, a.cull_thr ? *a.cull_thr : 0.f};
      ColGlobalDst gdst{a.re, imp, row0, estride, valid, a.swap, twR, a.big_tw ? inst : 0,
                        a.use_scale ? (a.scale_ptr ? *a.scale_ptr : a.scale_host) : 1.0f,
                        (a.write_im != 0 && !(a.wsel != nullptr && (*a.wsel != 0) == (a.wskip != 0))) ? 1 : 0};
      ColSmem sin{smem + (size_t)(cur ^ 1) * L * SM_COL_TILE, lane};
      ColSmem sout{smem + (size_t)cur * L * SM_COL_TILE, lane};
      if (sm_radix_is_generic(r)) {           // one output per (warp slot, lane = column) and iteration
        for (int it = wid; it < L; it += nwarps) {
          if (first && last)  stockham_generic_output<true>(r, it, L, s, a.tw_mul, twR, gsrc, gdst);
          else if (first)     stockham_generic_output<false>(r, it, L, s, a.tw_mul, twR, gsrc, sout);
          else if (last)      stockham_generic_output<true>(r, it, L, s, a.tw_mul, twR, sin, gdst);
          else                stockham_generic_output<false>(r, it, L, s, a.tw_mul, twR, sin, sout);
        }
      } else
      for (int b = wid; b < nb; b += nwarps) {
        if (first && last)  stockham_bfly_rt<true>(r, b, L, s, a.tw_mul, twR, gsrc, gdst);
        else if (first)     stockham_bfly_rt<false>(r, b, L, s, a.tw_mul, twR, gsrc, sout);
        else if (last)      stockham_bfly_rt<true>(r, b, L, s, a.tw_mul, twR, sin, gdst);
        else                stockham_bfly_rt<false>(r, b, L, s, a.tw_mul, twR, sin, sout);
      }
    }
    ex.sync();
    s *= r; cur ^= 1;
  }
}

// fill ColArgs for forward (dir=0) / inverse (dir=1) sweep `which` (0: A = strided, 1: B = contiguous)
static inline void sm_col_args(const SmPlan& pl, int which, int inverse, ColArgs* a, int* n_inst) {
  if (pl.col_passes == 1) {
    a->L = pl.R; a->n_rad = pl.nA; for (int i = 0; i < pl.nA; ++i) a->rad[i] = pl.radA[i];
    a->inst_mul = 0; a->elem_mul = 1; a->tw_mul = 1; a->big_tw = 0; *n_inst = 1;
  } else if (which == 0) {
    a->L = pl.Ra; a->n_rad = pl.nA; for (int i = 0; i < pl.nA; ++i) a->rad[i] = pl.radA[i];
    a->inst_mul = 1; a->elem_mul = pl.Rb; a->tw_mul = pl.Rb; *n_inst = pl.Rb;
    a->big_tw = inverse ? 0 : 1;
  } else {
    a->L = pl.Rb; a->n_rad = pl.nB; for (int i = 0; i < pl.nB; ++i) a->rad[i] = pl.radB[i];
    a->inst_mul = pl.Rb; a->elem_mul = 1; a->tw_mul = pl.Ra; *n_inst = pl.Ra;
    a->big_tw = inverse ? 1 : 0;
  }
  a->swap = inverse;
}

}  // namespace smfft

// =====================================================================================
// compile-time specialised sweeps (the hot shapes): all strides / trip counts fold to
// immediates, scalars arrive by value, inverse = plane pointers swapped at the call site.
// =====================================================================================
namespace smfft {

struct ColCtArgs {
  float* p0; float* p1;        // forward: (re, im); inverse: (im, re)  -- i.e. already swapped
  float* p0_alt; const int* sel;   // nullable: if *sel != 0 use p0_alt instead of p0 (inverse: role pick of Im)
  int P, Ch;                   // plane pitch / last valid column
  int inst_mul, elem_mul;      // stored row of element i of instance g: g*inst_mul + i*elem_mul
  int tw_mul;                  // W_L^e = twR[e * tw_mul]
  const float* thr_ptr;        // inverse only, nullable: |re| < *thr_ptr -> 0 on load
  const float* scale_ptr;      // nullable: outputs *= *scale_ptr, else *= scale
  float scale;
  int write_p1_fwd;            // forward: 0 -> do not store the imaginary plane
  const int* wsel; int wskip;  // nullable: forward, do not store the imaginary plane if (*wsel != 0) == (wskip != 0)
                               // (the fused chain: the model that ends up in role v1 only contributes Re, functions.py:108-136)
};
#define SM_COL_WRITE_P1(a) ((a).write_p1_fwd != 0 && !((a).wsel != nullptr && (*(a).wsel != 0) == ((a).wskip != 0)))

// ------------------------------------------------------------------ paired-column sweeps (pf: two adjacent columns per thread)
// Every thread carries two adjacent columns (c, c+1) through the butterflies as one packed value: half the FP /
// load-store / index instructions per element of one column per thread, 8-byte global accesses, 16-byte
// shared-memory accesses.  Lane mapping: 16 lanes x 2 columns = one 32-column tile row (128 B), two butterfly
// slots per warp.  The pair (Ch, Ch+1) touches one zero-filled padding column, whose transform is zero again.
SM_HD pf ldcg_pf(const float* p) {
#if defined(__CUDA_ARCH__)
  const float2 v = __ldcg(reinterpret_cast<const float2*>(p));
  return pf_make(v.x, v.y);
#else
  return pf_make(p[0], p[1]);
#endif
}
SM_HD void st_pf(float* p, pf v) {
#if defined(__CUDA_ARCH__)
  *reinterpret_cast<float2*>(p) = make_float2(pf_lo(v), pf_hi(v));
#else
  p[0] = pf_lo(v); p[1] = pf_hi(v);
#endif
}

struct pf4 { pf re, im; };     // one shared-memory element: (re_c, re_c+1, im_c, im_c+1), 16 bytes
struct ColSmemP {              // [idx][16 lane pairs]: a quarter warp covers all 32 banks, conflict free
  pf4* buf; int lane;
  SM_HD void load(int i, pf& re, pf& im) const { const pf4 v = buf[i * (SM_COL_TILE / 2) + lane]; re = v.re; im = v.im; }
  SM_HD void store(int i, pf re, pf im) const { pf4 v; v.re = re; v.im = im; buf[i * (SM_COL_TILE / 2) + lane] = v; }
};

template <bool kInverse>
struct ColCtSrcP {
  const float* p0; const float* p1; size_t row0; size_t estride; bool valid; float thr;
  SM_HD void load(int i, pf& a, pf& b) const {
    a = pf_make(0.f, 0.f); b = a;
    if (valid) {
      const size_t off = row0 + (size_t)i * estride;
      a = ldcg_pf(p0 + off); b = ldcg_pf(p1 + off);
      if (kInverse) {                                      // p1 is the real plane in the inverse: cull on load
        float b0 = pf_lo(b), b1 = pf_hi(b);
        if (b0 < thr && -b0 < thr) b0 = 0.f;
        if (b1 < thr && -b1 < thr) b1 = 0.f;
        b = pf_make(b0, b1);
      }
    }
  }
};
template <bool kBigTw>
struct ColCtDstP {
  float* p0; float* p1; size_t row0; size_t estride; bool valid; const cf* twR; int inst; float scale; bool write_p1;
  SM_HD void store(int k, pf a, pf b) const {
    if (kBigTw) { if (inst != 0) { const cf w = twR[(size_t)inst * k]; cmul(a, b, w.x, w.y); } }
    if (!valid) return;
    const size_t off = row0 + (size_t)k * estride;
    st_pf(p0 + off, mulc(a, scale));
    if (write_p1) st_pf(p1 + off, mulc(b, scale));
  }
};

// one CTA (NW warps = 2*NW butterfly slots) = one instance x 32 columns, L = R1*R2
template <int R1, int R2, int NW, bool kInverse, bool kBigTw, class Exec>
SM_HD void col_ct_body_p(Exec& ex, int tile, int inst, const ColCtArgs a, const cf* twR, pf4* smem) {
  constexpr int L = R1 * R2;
  constexpr int NS = 2 * NW;
  const size_t col0 = (size_t)tile * SM_COL_TILE;
  SM_FOR_THREADS(ex, tid) {
    const int lane = tid & 15, slot = tid >> 4;
    const size_t c = col0 + 2 * lane;
    const bool valid = (c <= (size_t)a.Ch);
    const size_t row0 = (size_t)(inst * a.inst_mul) * a.P + c;
    const size_t estride = (size_t)a.elem_mul * a.P;
    const float thr = (kInverse && a.thr_ptr) ? *a.thr_ptr : 0.f;
    const float scale = a.scale_ptr ? *a.scale_ptr : a.scale;
    float* const p0 = (a.sel != nullptr && *a.sel != 0) ? a.p0_alt : a.p0;
    ColCtSrcP<kInverse> gsrc{p0, a.p1, row0, estride, valid, thr};
    ColCtDstP<kBigTw> gdst{p0, a.p1, row0, estride, valid, twR, inst, scale, kInverse ? true : SM_COL_WRITE_P1(a)};
    if constexpr (R2 == 1) {
      for (int b = slot; b < 1; b += NS) stockham_bfly<R1, true, pf>(b, L, 1, a.tw_mul, twR, gsrc, gdst);
    } else {
      ColSmemP sout{smem, lane};
#pragma unroll
      for (int b = slot; b < R2; b += NS) stockham_bfly<R1, false, pf>(b, L, 1, a.tw_mul, twR, gsrc, sout);
    }
  }
  if constexpr (R2 > 1) {
    ex.sync();
    SM_FOR_THREADS(ex, tid) {
      const int lane = tid & 15, slot = tid >> 4;
      const size_t c = col0 + 2 * lane;
      const bool valid = (c <= (size_t)a.Ch);
      const size_t row0 = (size_t)(inst * a.inst_mul) * a.P + c;
      const size_t estride = (size_t)a.elem_mul * a.P;
      const float scale = a.scale_ptr ? *a.scale_ptr : a.scale;
      float* const p0 = (a.sel != nullptr && *a.sel != 0) ? a.p0_alt : a.p0;
      ColCtDstP<kBigTw> gdst{p0, a.p1, row0, estride, valid, twR, inst, scale, kInverse ? true : SM_COL_WRITE_P1(a)};
      ColSmemP sin{smem, lane};
#pragma unroll
      for (int b = slot; b < R1; b += NS) stockham_bfly<R2, true, pf>(b, L, R1, a.tw_mul, twR, sin, gdst);
    }
  }
}

// three register stages (radices <= 8) with the middle one in place: the two-stage sweeps of the long instances (L = 112 /
// 128) need a radix-16 butterfly of packed values, 80 registers, 6 CTAs per SM; radices <= 8 need ~56 (the L = 64 sweeps
// run at 6.0 TB/s with 9-10 CTAs per SM against 4.8 TB/s, profiles/r01).  L = R1*R2*R3, L / R1 <= 2 NW and L / R2 <= 2 NW.
template <int R1, int R2, int R3, int NW, bool kInverse, bool kBigTw, class Exec>
SM_HD void col_ct_body_p3(Exec& ex, int tile, int inst, const ColCtArgs a, const cf* twR, pf4* smem) {
  constexpr int L = R1 * R2 * R3;
  constexpr int NS = 2 * NW;
  static_assert(L / R2 <= NS, "col_ct_body_p3: at most one middle-stage butterfly per slot (it runs in place)");
  const size_t col0 = (size_t)tile * SM_COL_TILE;
  pf re2[R2], im2[R2];
  SM_FOR_THREADS(ex, tid) {
    const int lane = tid & 15, slot = tid >> 4;
    const size_t c = col0 + 2 * lane;
    const bool valid = (c <= (size_t)a.Ch);
    const size_t row0 = (size_t)(inst * a.inst_mul) * a.P + c;
    const size_t estride = (size_t)a.elem_mul * a.P;
    const float thr = (kInverse && a.thr_ptr) ? *a.thr_ptr : 0.f;
    float* const p0 = (a.sel != nullptr && *a.sel != 0) ? a.p0_alt : a.p0;
    ColCtSrcP<kInverse> gsrc{p0, a.p1, row0, estride, valid, thr};
    ColSmemP sm{smem, lane};
#pragma unroll
    for (int b = slot; b < L / R1; b += NS) stockham_bfly<R1, false, pf>(b, L, 1, a.tw_mul, twR, gsrc, sm);
  }
  ex.sync();
  SM_FOR_THREADS(ex, tid) {
    const int lane = tid & 15, slot = tid >> 4;
    ColSmemP sm{smem, lane};
    if (slot < L / R2) {
#pragma unroll
      for (int j = 0; j < R2; ++j) sm.load(slot + j * (L / R2), re2[j], im2[j]);
    }
  }
  ex.sync();
  SM_FOR_THREADS(ex, tid) {
    const int lane = tid & 15, slot = tid >> 4;
    ColSmemP sm{smem, lane};
    if (slot < L / R2) {
      Dft<R2>::run(re2, im2);
      const int p = slot / R1, q = slot - p * R1;
      const int obase = q + R1 * R2 * p, tstep = R1 * p * a.tw_mul;
      sm.store(obase, re2[0], im2[0]);
#pragma unroll
      for (int k = 1; k < R2; ++k) {
        const cf w = ldg_cf(twR + tstep * k);
        pf xr = re2[k], xi = im2[k];
        cmul(xr, xi, w.x, w.y);
        sm.store(obase + k * R1, xr, xi);
      }
    }
  }
  ex.sync();
  SM_FOR_THREADS(ex, tid) {
    const int lane = tid & 15, slot = tid >> 4;
    const size_t c = col0 + 2 * lane;
    const bool valid = (c <= (size_t)a.Ch);
    const size_t row0 = (size_t)(inst * a.inst_mul) * a.P + c;
    const size_t estride = (size_t)a.elem_mul * a.P;
    const float scale = a.scale_ptr ? *a.scale_ptr : a.scale;
    float* const p0 = (a.sel != nullptr && *a.sel != 0) ? a.p0_alt : a.p0;
    ColCtDstP<kBigTw> gdst{p0, a.p1, row0, estride, valid, twR, inst, scale, kInverse ? true : SM_COL_WRITE_P1(a)};
    ColSmemP sm{smem, lane};
#pragma unroll
    for (int b = slot; b < L / R3; b += NS) stockham_bfly<R3, true, pf>(b, L, R1 * R2, a.tw_mul, twR, sm, gdst);
  }
}

}  // namespace smfft

namespace smfft {

// ------------------------------------------------------------------ specialised row passes
// CH = R1*R2*R3*R4 (unused trailing radices = 1), T threads, padded smem when it fits.
template <int CH, int S, int R, bool kLast, int T, class Src, class Dst, class Exec>
SM_HD void row_ct_stage(Exec& ex, const cf* twC, const cf* twQ, const Src& src, const Dst& dst) {
  constexpr int nb = CH / R;
  SM_FOR_THREADS(ex, tid) {
#pragma unroll
    for (int b = tid; b < nb; b += T) {
      if constexpr (S == 1 && !kLast) stockham_bfly_first<R>(b, CH, twQ, src, dst);
      else stockham_bfly<R, kLast>(b, CH, S, 2, twC, src, dst);
    }
  }
  ex.sync();
}

// stage-1 sources that read a row staged in shared memory by a bulk async copy (kernels_fft.cu:
// k_row_fwd_tma / k_row_inv_tma); same arithmetic as RowDeltaSrc / RowTangleSrc, plain loads
struct RowDeltaStagedSrc {
  int mode; const uint32_t* b32; const uint32_t* f32; const cf* x32; float m1, m2; float* acc;
  SM_HD void load(int i, float& re, float& im) const {
    float d0, d1;
    if (mode == 0) {
      const uint32_t bb = b32[i], ff = f32[i];
      d0 = bf16_bits_to_f32(ff & 0xffffu) - bf16_bits_to_f32(bb & 0xffffu);
      d1 = bits_f32(ff & 0xffff0000u) - bits_f32(bb & 0xffff0000u);
    } else {
      const cf v = x32[i];
      d0 = v.x; d1 = v.y;
    }
    *acc = fmaf(d0, d0, fmaf(d1, d1, *acc));
    if (mode != 0) { d0 = (d0 * m1) * m2; d1 = (d1 * m1) * m2; }
    re = d0; im = d1;
  }
};

struct RowTangleStagedSrc {
  const float* re; const float* im; const cf* twC; int Ch; float thr;
  SM_HD float cull(float v) const { return (v < thr && -v < thr) ? 0.f : v; }
  SM_HD void load(int k, float& ore, float& oim) const {
    float xr = cull(re[k]), xi = im[k];
    float mr = cull(re[Ch - k]), mi = im[Ch - k];
    if (k == 0) { xi = 0.f; mi = 0.f; }
    const float Ar = xr + mr, Ai = xi - mi;
    const float Br = xr - mr, Bi = xi + mi;
    const cf w = ldg_cf(twC + k);
    const float br = Br * w.x + Bi * w.y;
    const float bi = Bi * w.x - Br * w.y;
    const float zr = Ar - bi, zi = Ai + br;
    ore = zi; oim = zr;
  }
};

struct RowEpilogueStagedDst {   // RowEpilogueDst with the base row read from shared memory
  int out_mode; const uint32_t* base32; uint32_t* out32; cf* outf; float inv_n, scale; int check;
  unsigned int* flags;
  SM_HD float fin(float v, int which) const { return sm_fix_nonfinite(v, flags, which); }
  SM_HD void store(int j, float a, float b) const {
    float x0 = b * inv_n, x1 = a * inv_n;
    if (check) { if (not_finite(x0)) x0 = fin(x0, 0); if (not_finite(x1)) x1 = fin(x1, 0); }
    x0 *= scale; x1 *= scale;
    if (out_mode == 0) {
      const uint32_t bb = base32[j];
      x0 = bf16_bits_to_f32(bb & 0xffffu) + x0;
      x1 = bits_f32(bb & 0xffff0000u) + x1;
      if (not_finite(x0)) x0 = fin(x0, 2);
      if (not_finite(x1)) x1 = fin(x1, 2);
      out32[j] = pack_bf16x2_rne(x0, x1);
    } else {
      cf v; v.x = x0; v.y = x1; outf[j] = v;
    }
  }
};

// forward row: stages + untangle, stage-1 source supplied by the caller
struct NoHook { SM_HD void after_first_stage() const {} };

// `hook.after_first_stage()` runs once the stage-1 barrier has passed, i.e. when the stage-1 source
// (a staging buffer in the bulk-copy kernels) may be refilled.
template <int R1, int R2, int R3, int R4, int T, bool kPad, class Src, class Hook, class Exec>
SM_HD void row_fwd_ct_stages(Exec& ex, const Src& gsrc, float* ore, float* oim, const cf* twC, const cf* twQ, cf* smem,
                             const Hook& hook) {
  constexpr int CH = R1 * R2 * R3 * R4;
  constexpr int bufstride = kPad ? (CH + (CH >> 4) + 1) : CH;
  constexpr int padmask = kPad ? ~0 : 0;
  RowSmem b0{smem, padmask}, b1{smem + bufstride, padmask};
  constexpr int nst = (R2 > 1) + (R3 > 1) + (R4 > 1) + 1;
  row_ct_stage<CH, 1, R1, nst == 1, T>(ex, twC, twQ, gsrc, b0);
  hook.after_first_stage();
  if constexpr (nst >= 2) row_ct_stage<CH, R1, R2, nst == 2, T>(ex, twC, twQ, b0, b1);
  if constexpr (nst >= 3) row_ct_stage<CH, R1 * R2, R3, nst == 3, T>(ex, twC, twQ, b1, b0);
  if constexpr (nst >= 4) row_ct_stage<CH, R1 * R2 * R3, R4, true, T>(ex, twC, twQ, b0, b1);
  const RowSmem z = (nst == 1 || nst == 3) ? b0 : b1;
  SM_FOR_THREADS(ex, tid) {
#pragma unroll 4
    for (int k = tid; k <= CH; k += T) {
      const int k0 = (k == CH) ? 0 : k;
      const int k1 = (k == 0 || k == CH) ? 0 : CH - k;
      float ar, ai, br, bi;
      z.load(k0, ar, ai);
      z.load(k1, br, bi);
      const float er = 0.5f * (ar + br), ei = 0.5f * (ai - bi);
      const float pr = 0.5f * (ai + bi), qi = -0.5f * (ar - br);
      const cf w = ldg_cf(twC + k);
      ore[k] = er + (pr * w.x - qi * w.y);
      oim[k] = ei + (pr * w.y + qi * w.x);
    }
  }
  ex.sync();
}

template <int R1, int R2, int R3, int R4, int T, bool kPad, class Exec>
SM_HD void row_fwd_ct_body(Exec& ex, int row, int C, int P, const RowFwdArgs a, const cf* twC, const cf* twQ, cf* smem, float* acc) {
  RowDeltaSrc gsrc;
  gsrc.mode = a.mode;
  gsrc.b32 = a.mode == 0 ? reinterpret_cast<const uint32_t*>(a.base + (size_t)row * C) : nullptr;
  gsrc.f32 = a.mode == 0 ? reinterpret_cast<const uint32_t*>(a.ft + (size_t)row * C) : nullptr;
  gsrc.x32 = a.mode != 0 ? reinterpret_cast<const cf*>(a.x32 + (size_t)row * C) : nullptr;
  gsrc.m1 = a.m1; gsrc.m2 = a.m2; gsrc.acc = acc;
  row_fwd_ct_stages<R1, R2, R3, R4, T, kPad>(ex, gsrc, a.re + (size_t)row * P, a.im + (size_t)row * P, twC, twQ, smem, NoHook{});
}

// inverse row: stages with caller-supplied stage-1 source and last-stage sink
template <int R1, int R2, int R3, int R4, int T, bool kPad, class Src, class Dst, class Hook, class Exec>
SM_HD void row_inv_ct_stages(Exec& ex, const Src& gsrc, const Dst& gdst, const cf* twC, const cf* twQ, cf* smem,
                             const Hook& hook) {
  constexpr int CH = R1 * R2 * R3 * R4;
  constexpr int bufstride = kPad ? (CH + (CH >> 4) + 1) : CH;
  constexpr int padmask = kPad ? ~0 : 0;
  RowSmem b0{smem, padmask}, b1{smem + bufstride, padmask};
  constexpr int nst = (R2 > 1) + (R3 > 1) + (R4 > 1) + 1;
  if constexpr (nst == 1) {
    row_ct_stage<CH, 1, R1, true, T>(ex, twC, twQ, gsrc, gdst);
    hook.after_first_stage();
  } else if constexpr (nst == 2) {
    row_ct_stage<CH, 1, R1, false, T>(ex, twC, twQ, gsrc, b0);
    hook.after_first_stage();
    row_ct_stage<CH, R1, R2, true, T>(ex, twC, twQ, b0, gdst);
  } else if constexpr (nst == 3) {
    row_ct_stage<CH, 1, R1, false, T>(ex, twC, twQ, gsrc, b0);
    hook.after_first_stage();
    row_ct_stage<CH, R1, R2, false, T>(ex, twC, twQ, b0, b1);
    row_ct_stage<CH, R1 * R2, R3, true, T>(ex, twC, twQ, b1, gdst);
  } else {
    row_ct_stage<CH, 1, R1, false, T>(ex, twC, twQ, gsrc, b0);
    hook.after_first_stage();
    row_ct_stage<CH, R1, R2, false, T>(ex, twC, twQ, b0, b1);
    row_ct_stage<CH, R1 * R2, R3, false, T>(ex, twC, twQ, b1, b0);
    row_ct_stage<CH, R1 * R2 * R3, R4, true, T>(ex, twC, twQ, b0, gdst);
  }
}

template <int R1, int R2, int R3, int R4, int T, bool kPad, class Exec>
SM_HD void row_inv_ct_body(Exec& ex, int row, int C, int P, const RowInvArgs a, const cf* twC, const cf* twQ, cf* smem) {
  constexpr int CH = R1 * R2 * R3 * R4;
  RowTangleSrc gsrc;
  gsrc.re = a.re + (size_t)row * P;
  gsrc.im = ((a.sel != nullptr && *a.sel != 0) ? a.im_alt : a.im) + (size_t)row * P;
  gsrc.twC = twC; gsrc.Ch = CH;
  gsrc.thr = (a.cull_thr != nullptr) ? *a.cull_thr : 0.f;
  RowEpilogueDst gdst;
  gdst.out_mode = a.out_mode;
  gdst.base32 = a.out_mode == 0 ? reinterpret_cast<const uint32_t*>(a.base + (size_t)row * C) : nullptr;
  gdst.out32 = a.out_mode == 0 ? reinterpret_cast<uint32_t*>(a.out_bf16 + (size_t)row * C) : nullptr;
  gdst.outf = a.out_mode != 0 ? reinterpret_cast<cf*>(a.out_f32 + (size_t)row * C) : nullptr;
  gdst.inv_n = a.inv_n; gdst.check = a.check_ifft;
  gdst.scale = a.scale_ptr ? *a.scale_ptr : a.scale_host;
  gdst.flags = a.flags;
  row_inv_ct_stages<R1, R2, R3, R4, T, kPad>(ex, gsrc, gdst, twC, twQ, smem, NoHook{});
}

}  // namespace smfft
