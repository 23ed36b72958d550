// kernels_fstats.cu -- fused statistics for the pair-merge chain (csrc/pipeline.cu).
//
// interpolate_fft_components (shard/tensor/functions.py:90-162) needs, between the forward and the
// inverse transform: the cutoff order statistic of cat(|Re X0|, |Re X1|) (:113-122), three masked
// sums for slerp() (:36-41 under the masks of :124-129), the blend (:134-136) and the cull order
// statistic of |Re R| (:138-148).  kernels_stats.cu does each of these as its own pass (that is
// the step-by-step API, 25 launches, 16N bytes); here they are folded into TWO streaming passes:
//
//   k_fs_sample<0>   256 K random keys of the full (mirrored) spectra; the last CTA to finish turns
//                    them into a key window [lo, hi] that brackets the cutoff statistic with ~6 sigma
//                    of sampling noise (<= 2^22 key bit patterns wide, else the status says so)
//   k_fs_pass<0>     ONE pass over Re X0, Re X1 (4N bytes).  Keys below the window are counted in
//                    registers.  The ~1 % inside it are histogrammed with fire-and-forget global
//                    reductions at two resolutions: `fine` has one bin per key BIT PATTERN of the
//                    window (2 M distinct addresses: no contention), `coarse` 2048 bins over it, kept
//                    per CTA in shared memory and added to the global copy once at the end (coalesced).
//                    SLERP sums are accumulated in registers for every element whose mask the window
//                    already decides; the few with lo <= |re1| <= hi and equal signs are appended to a
//                    per-CTA side list.  The last CTA picks the coarse bin of the statistic, then the
//                    exact key from that bin's <= 2048 fine counters.
//   k_fs_close       (cutoff pass only) all CTAs: add the side-list entries with |re1| >= key to the
//                    sums; the last CTA computes dot / cos / sin / ||rel||.
//   k_fs_sample<1>   the same sampling for |blend(re0, re1)| (the blend is cheap to evaluate at a
//                    sample position) -> window for the cull statistic
//   k_fs_pass<1>     the blend itself (read 4N, write 2N) with the count / histogram step folded into
//                    its epilogue; the last CTA produces the exact cull threshold.
//
// No thread waits on a returning global atomic or a block barrier inside the streaming loop, and no two
// CTAs reduce into the same cache line while streaming.  (The first version staged candidates in shared
// memory and flushed them under __syncthreads: barrier stalls were its largest stall reason and it moved
// 0.9 TB/s, profiles/r01_ncu_full_fs_pass_raw.csv.  A second one reduced straight into a global coarse
// histogram and per-bin partial sums: 64 + 384 contended cache lines made it 2x slower still.)
// Columns 1..Ch-1 all carry Hermitian multiplicity 2, so the interior of a row is processed
// unweighted and doubled at the end; the two edge column groups of each row (column 0, column Ch and
// the zero padding behind it) take a generic per-element path.
//
// Exactness: the thresholds are the bit patterns of actual elements at the exact rank (Hermitian
// multiplicities included), as in kernels_stats.cu; the masks therefore reproduce the reference's.
// A window that misses, is too wide, or overflows a side bucket (degenerate distributions) sets
// status bits and the thresholds become NaN; the caller re-runs the tensor on the step-by-step path.
// Only tensors with more than 2^20 elements come here (sm_fstats_supported); smaller ones are launch
// bound and use the step-by-step kernels.
#include <cstddef>
#include "sm_internal.h"

namespace {

constexpr int kBins = 2048;                    // coarse bins over the window
constexpr int kMaxLists = 4096;                // side lists (one per CTA of the streaming pass)
constexpr unsigned int kFineLog = 22;          // the window spans at most 2^22 key bit patterns
constexpr unsigned int kFineMax = 1u << kFineLog;
constexpr unsigned int kNS = 1u << 18;         // samples
constexpr int kSampleThreads = 1024, kSamplePer = 1;

struct FsState {                     // SM_FS_STATE_BYTES device bytes
  unsigned long long rank;           // rank of the statistic in the full key multiset
  unsigned long long below;          // keys below the window
  unsigned int lo, hi;               // window [lo, hi] (key bit patterns)
  unsigned int shift;                // coarse bin = (key - lo) >> shift
  unsigned int status;               // bit0 window missed, bit1 side bucket overflow, bit2 window too wide   (SM_FS_STATUS_OFF)
  unsigned int ticket;
  unsigned int key;
  float value;
  unsigned int bstar;
  double s_in[3];                    // decided part of the SLERP sums (s00, s11, s01)
  unsigned int sticky;               // OR of every status this state has ended with (kernels never clear it)   (SM_FS_STICKY_OFF)
  unsigned int dense;                // the sample found > 1.6 % of the keys inside the window: tied keys, combine per warp
  unsigned int pad[12];
};
static_assert(sizeof(FsState) == SM_FS_STATE_BYTES, "FsState layout");
static_assert(offsetof(FsState, status) == SM_FS_STATUS_OFF, "FsState status offset");
static_assert(offsetof(FsState, sticky) == SM_FS_STICKY_OFF, "FsState sticky offset");

constexpr int kSampleShift = 18;                         // sample histogram digit: key bits [30:18] (exponent + 5 mantissa bits)
constexpr int kSampleBins = 1 << (31 - kSampleShift);    // 8192

struct FsWs {                        // carved out of the caller's workspace
  // one contiguous block; the caller hands it over zero-filled once, afterwards k_fs_sample keeps it so (coarse and scnt
  // are cleared by every sample kernel; of `fine` only the counters the previous pass can have touched, meta[0] of them):
  unsigned int* shist;               // [kSampleBins] sample histogram
  unsigned int* coarse;              // [kBins]  keys (with multiplicity) per coarse bin
  unsigned int* scnt;                // [kMaxLists]  entries in the side list of pass CTA i
  unsigned int* fine;                // [kFineMax] keys (with multiplicity) per bit pattern of the window
  unsigned int* meta;                // [16]  [0]: how many leading `fine` counters the last pass may have left non-zero
  size_t zero_bytes;                 // size of that block
  // not zeroed (guarded by scnt):
  float2* sbkt;                      // [n_lists][scap]  (|re0| with "multiplicity 1" in the sign bit, |re1|)
  unsigned int scap, n_lists;
};

__device__ __forceinline__ unsigned int absbits(float v) { return __float_as_uint(v) & 0x7fffffffu; }
__device__ __forceinline__ int sgn(float v) { return (v > 0.f) - (v < 0.f); }

__device__ __forceinline__ unsigned long long mix64(unsigned long long x) {
  x += 0x9e3779b97f4a7c15ull;
  x = (x ^ (x >> 30)) * 0xbf58476d1ce4e5b9ull;
  x = (x ^ (x >> 27)) * 0x94d049bb133111ebull;
  return x ^ (x >> 31);
}

// the blend of one element (functions.py:124-136; one rounding per torch op)
struct BlendScal { float thr, dot, ct, sn, rn, t_sum; };
__device__ __forceinline__ float blend1(float a, float b, const BlendScal& s) {
  const bool same = (sgn(a) == sgn(b));
  if (same) {
    if (!(fabsf(b) < s.thr)) {
      const float rel = __fsub_rn(b, __fmul_rn(a, s.dot));
      return __fadd_rn(__fmul_rn(a, s.ct), __fmul_rn(__fdiv_rn(rel, s.rn), s.sn));
    }
    return __fadd_rn(a, __fmul_rn(s.t_sum, b));
  }
  return (fabsf(a) > fabsf(b)) ? a : b;
}

// ---------------------------------------------------------------------------------------------
// block-wide search of a histogram for the bin holding 0-based `rank` (NT threads).
// load(b) returns the count of bin b.
// ---------------------------------------------------------------------------------------------
struct Pick { int bin; unsigned long long rank_in_bin; };

template <int NT, class Load>
__device__ void block_pick(const Load& load, int nbins, unsigned long long rank, Pick* out /*shared*/) {
  __shared__ unsigned long long wtot[NT / 32];
  const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
  const int per = (nbins + NT - 1) / NT;
  if (t == 0) { out->bin = -1; out->rank_in_bin = 0ull; }
  unsigned long long v = 0ull;
  for (int j = 0; j < per; ++j) { const int b = t * per + j; if (b < nbins) v += load(b); }
  unsigned long long incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned long long n = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += n;
  }
  if (lane == 31) wtot[wid] = incl;
  __syncthreads();
  if (wid == 0) {
    const unsigned long long w = lane < NT / 32 ? wtot[lane] : 0ull;
    unsigned long long wi = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long n = __shfl_up_sync(0xffffffffu, wi, o);
      if (lane >= o) wi += n;
    }
    if (lane < NT / 32) wtot[lane] = wi - w;
  }
  __syncthreads();
  unsigned long long excl = wtot[wid] + incl - v;
  if (rank >= excl && rank < excl + v) {
    for (int j = 0; j < per; ++j) {
      const int b = t * per + j;
      if (b >= nbins) break;
      const unsigned long long h = load(b);
      if (rank < excl + h) { out->bin = b; out->rank_in_bin = rank - excl; break; }
      excl += h;
    }
  }
  __syncthreads();
}

struct LoadSmem32 { const unsigned int* h; __device__ unsigned long long operator()(int b) const { return h[b]; } };

__device__ __forceinline__ double block_sum_d(double v, double* sh /* >= 32 */) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  __syncthreads();
  if (lane == 0) sh[wid] = v;
  __syncthreads();
  double r = 0.0;
  if (wid == 0) {
    r = lane < nw ? sh[lane] : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) r += __shfl_xor_sync(0xffffffffu, r, o);
  }
  return r;                           // valid in warp 0
}

// scalars of slerp() from the three masked sums (functions.py:36-43); same arithmetic as k_slerp_scalars
__device__ void fs_scalars(const double* s, double t, float* scal4) {
  const double s00 = s[0], s11 = s[1], s01 = s[2];
  const float n0 = (float)sqrt(s00), n1 = (float)sqrt(s11);
  float dot = (float)s01 / (n0 * n1);
  dot = fminf(fmaxf(dot, -1.0f), 1.0f);
  if (!(dot == dot)) dot = __uint_as_float(0x7fc00000u);
  const float theta = (float)acos((double)dot) * (float)t;
  const float ct = (float)cos((double)theta), sn = (float)sin((double)theta);
  const double d = (double)dot;
  double rn2 = s11 - 2.0 * d * s01 + d * d * s00;
  if (rn2 < 0.0) rn2 = 0.0;
  float rn = (float)sqrt(rn2);
  if (rn < 1e-12f) rn = 1e-12f;
  if (!(d == d)) rn = __uint_as_float(0x7fc00000u);
  scal4[0] = dot; scal4[1] = ct; scal4[2] = sn; scal4[3] = rn;
}

// returns true in every thread of the last CTA to arrive
__device__ __forceinline__ bool fs_last_block(FsState* st) {
  __shared__ int s_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int n = gridDim.x * gridDim.y;
    s_last = (atomicAdd(&st->ticket, 1u) == n - 1u) ? 1 : 0;
  }
  __syncthreads();
  if (s_last) __threadfence();
  return s_last != 0;
}

// ---------------------------------------------------------------------------------------------
// sampling + window
// ---------------------------------------------------------------------------------------------
struct FsCommon {
  const float* reX; const float* reY; const int* sel;     // role pick: *sel != 0 -> (re0, re1) = (reY, reX)
  const float* thr_cut; const float* scal4; float t_sum;  // MODE 1 only
};

// 256 K random keys of the full (mirrored) spectrum are histogrammed by their top 13 key bits -- per CTA in
// shared memory first (same-address global reductions serialise in L2), then one global reduction per CTA and
// non-empty bin; the last CTA to finish copies the 8 K bins to shared memory (all loads in flight at once:
// single-CTA epilogues must not chain L2 round trips), finds the bins holding the sample ranks k_lo / k_hi and
// takes their outer edges as the key window: at most one bin (3 % of the key value) wider per side than the
// exact sample statistics would give.
template <int MODE>
__global__ void __launch_bounds__(kSampleThreads) k_fs_sample(const __grid_constant__ SmPlan pl, const __grid_constant__ FsCommon c,
                                                              FsState* st, const __grid_constant__ FsWs ws, unsigned long long rank,
                                                              long long k_lo, long long k_hi) {
  sm_pdl_enter();
  __shared__ Pick out_a, out_b;
  __shared__ unsigned int s_h[kSampleBins];
  const unsigned int ns = kNS;
  const unsigned long long per_plane = (unsigned long long)pl.R * (unsigned long long)pl.C;
  const unsigned long long total = per_plane * (MODE == 0 ? 2ull : 1ull);
  const bool sw = (c.sel != nullptr && *c.sel != 0);
  const float* re0 = sw ? c.reY : c.reX;
  const float* re1 = sw ? c.reX : c.reY;
  BlendScal bs{};
  if (MODE == 1) { bs.thr = *c.thr_cut; bs.dot = c.scal4[0]; bs.ct = c.scal4[1]; bs.sn = c.scal4[2]; bs.rn = c.scal4[3]; bs.t_sum = c.t_sum; }
#pragma unroll
  for (int j = 0; j < kSampleBins / kSampleThreads; ++j) s_h[threadIdx.x + kSampleThreads * j] = 0u;
  {  // this kernel also clears the histograms of the pass that follows (fire-and-forget stores, done long before it starts):
     // no memset node in the chain.  The sample histogram itself is left clean by the last CTA below.  Of the 16 MB of
     // `fine` only the first meta[0] counters can be non-zero: the window of the previous pass (usually 2 - 4 MB).
    uint4* const z = reinterpret_cast<uint4*>(ws.coarse);          // [coarse | scnt | fine] is one contiguous block
    unsigned int dirty = __ldcg(ws.meta);                          // read before this CTA's ticket: the last CTA rewrites it
    if (dirty > kFineMax) dirty = kFineMax;
    const size_t n16 = ((size_t)kBins + kMaxLists + dirty + 3) / 4;
    const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) z[i] = zero;
  }
  __syncthreads();
  {
    float va[kSamplePer], vb[kSamplePer];                // all gathers of a thread in flight together
#pragma unroll
    for (int q = 0; q < kSamplePer; ++q) {
      const unsigned int i = (blockIdx.x * kSamplePer + q) * kSampleThreads + threadIdx.x;
      unsigned long long j = __umul64hi(mix64(i + (MODE ? 0x51ed27ull : 0ull)), total);
      const float* pp = re0;
      if (MODE == 0 && j >= per_plane) { j -= per_plane; pp = re1; }
      const unsigned int row = (unsigned int)(j / (unsigned long long)pl.C);
      unsigned int col = (unsigned int)(j - (unsigned long long)row * pl.C);
      if (col > (unsigned int)pl.Ch) col = pl.C - col;
      const size_t off = (size_t)row * pl.P + col;
      if (MODE == 0) { va[q] = pp[off]; vb[q] = 0.f; }
      else { va[q] = re0[off]; vb[q] = re1[off]; }
    }
#pragma unroll
    for (int q = 0; q < kSamplePer; ++q) {
      const unsigned int i = (blockIdx.x * kSamplePer + q) * kSampleThreads + threadIdx.x;
      const unsigned int key = (MODE == 0) ? absbits(va[q]) : absbits(blend1(va[q], vb[q], bs));
      if (i < ns) atomicAdd(&s_h[key >> kSampleShift], 1u);
    }
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < kSampleBins / kSampleThreads; ++j) {
    const unsigned int v = s_h[threadIdx.x + kSampleThreads * j];
    if (v) atomicAdd(ws.shist + threadIdx.x + kSampleThreads * j, v);
  }
  const bool last = fs_last_block(st);
  if (!last) return;
  const bool want_a = (k_lo >= 0 && k_lo < (long long)ns), want_b = (k_hi >= 0 && k_hi < (long long)ns);
  {
    unsigned int v[kSampleBins / kSampleThreads];
#pragma unroll
    for (int j = 0; j < kSampleBins / kSampleThreads; ++j) v[j] = __ldcg(ws.shist + threadIdx.x + kSampleThreads * j);
#pragma unroll
    for (int j = 0; j < kSampleBins / kSampleThreads; ++j) s_h[threadIdx.x + kSampleThreads * j] = v[j];
#pragma unroll
    for (int j = 0; j < kSampleBins / kSampleThreads; ++j) ws.shist[threadIdx.x + kSampleThreads * j] = 0u;   // clean for the next call
  }
  __syncthreads();
  block_pick<kSampleThreads>(LoadSmem32{s_h}, kSampleBins, want_a ? (unsigned long long)k_lo : 0ull, &out_a);
  block_pick<kSampleThreads>(LoadSmem32{s_h}, kSampleBins, want_b ? (unsigned long long)k_hi : 0ull, &out_b);
  const int bin_a = out_a.bin, bin_b = out_b.bin;
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int lo = (want_a && bin_a >= 0) ? ((unsigned int)bin_a << kSampleShift) : 0u;
    unsigned int hi = (want_b && bin_b >= 0) ? ((((unsigned int)bin_b + 1u) << kSampleShift) - 1u) : 0x7f800000u;
    if (hi > 0x7f800000u) hi = 0x7f800000u;             // NaN keys stay above every window
    unsigned int status = 0u;
    const unsigned long long width = hi >= lo ? (unsigned long long)hi - lo + 1ull : 0ull;
    unsigned int l2 = 0;
    while ((1ull << l2) < width) ++l2;
    if (width == 0ull || l2 > kFineLog) status |= 4u;    // the fine histogram has one counter per bit pattern
    unsigned int in_window = 0u;                           // sample keys inside the window (at most 17 bins wide when it is usable)
    if (status == 0u)
      for (unsigned int b = lo >> kSampleShift; b <= (hi >> kSampleShift) && b < (unsigned int)kSampleBins; ++b) in_window += s_h[b];
    st->dense = (in_window > (ns >> 6)) ? 1u : 0u;         // > 1.6 % of the sample
    st->rank = rank; st->below = 0ull; st->lo = lo; st->hi = hi;
    st->shift = l2 > 11 ? l2 - 11 : 0;
    st->status = status; st->key = 0u; st->value = 0.f; st->bstar = 0u;
    st->s_in[0] = 0.0; st->s_in[1] = 0.0; st->s_in[2] = 0.0;
    st->ticket = 0u;
    ws.meta[0] = status == 0u ? (unsigned int)width : 0u;   // the counters the pass that follows may touch (a dead pass: none)
  }
}

// ---------------------------------------------------------------------------------------------
// the streaming pass
// ---------------------------------------------------------------------------------------------
// Straight-line fast path + per-warp deferral.  A float4 item is handled completely by branch-free code when it
// is an interior column group (every key has multiplicity 2), no product a_i * b_i is zero / NaN (the sign of
// the product then decides torch.sign(a) == torch.sign(b)) and none of its 8 keys lies inside the window.  Any
// other item (~10 % of them) is appended -- operands and all -- to a queue private to the warp in shared
// memory; whenever the queue holds 32 entries the warp drains it with ALL lanes busy, one entry per lane, through
// the generic per-element code (weights, exact signs, histogram reductions, side list).  The first two versions
// branched per key inside the loop: with 32 lanes x 8 keys some lane takes every branch, so the rare code ran
// at 1/32 efficiency and made up half of the executed instructions (88 per element pair; now ~25).
constexpr int kQCap = 96;            // entries per warp queue: < 32 left after a drain, <= 64 pushed per iteration (two items)

struct PassCtx {
  float lo_f, hi_f;                  // the window as floats: for non-NaN keys, float order == bit-pattern order
  unsigned int lo, shift, scap, dense;
  unsigned int* fine;
  float2* slist;                     // this CTA's side list
  unsigned int* status;
  float* out;                        // MODE 1
  int Ch;
};

// the out-of-line drain reads its parameters from shared memory (no pointer arguments, nothing forced into local memory)
__shared__ PassCtx g_fs_ctx;
__shared__ BlendScal g_fs_bs;
__shared__ unsigned int g_fs_coarse[kBins];             // streaming phase: this CTA's coarse histogram; last CTA: scratch
__shared__ unsigned int g_fs_nside;
// one CTA of 1024 threads per SM: a quarter of the CTAs means a quarter of the end-of-kernel reductions into the
// same 64 cache lines of the global coarse histogram (they serialise in L2: 3.5 us with 592 CTAs, measured)
constexpr int kPassThreads = 512, kPassCtasPerSm = 2, kPassWarps = kPassThreads / 32;
// the warp queues live in dynamic shared memory (60 KB): [kPassWarps][kQCap] of float4 a, float4 b, uint2 meta
extern __shared__ __align__(16) unsigned char g_fs_dyn[];
__device__ __forceinline__ float4* fs_qa(int wid) { return reinterpret_cast<float4*>(g_fs_dyn) + wid * kQCap; }
__device__ __forceinline__ float4* fs_qb(int wid) { return reinterpret_cast<float4*>(g_fs_dyn) + (kPassWarps + wid) * kQCap; }
__device__ __forceinline__ uint2* fs_qm(int wid) {      // x: element offset of the item, y: first column | generic << 31
  return reinterpret_cast<uint2*>(g_fs_dyn + (size_t)2 * kPassWarps * kQCap * sizeof(float4)) + wid * kQCap;
}
constexpr size_t kPassDynSmem = (size_t)kPassWarps * kQCap * (2 * sizeof(float4) + sizeof(uint2));
// work distribution: every CTA (= SM) owns an equal contiguous share of the items; inside it a warp takes chunks
// of kChunkIters x 64 consecutive float4 items, the first by its own number, further ones from a shared-memory
// counter (fetched one chunk ahead), so all warps of an SM finish together.  With a static split over 4 CTAs per
// SM the slowest CTA finished 40 % after the fastest (measured with per-CTA phase timestamps).
constexpr unsigned int kChunkIters = 2, kChunkItems = kChunkIters * 64;
__shared__ unsigned int g_fs_chunk;

// the three-way blend, predicated (functions.py:134-136, one rounding per torch op; same arithmetic as blend1 / k_blend)
__device__ __forceinline__ float fs_blend(const BlendScal& bs, float a, float b, bool same) {
  const float rel = __fsub_rn(b, __fmul_rn(a, bs.dot));
  const float o_slerp = __fadd_rn(__fmul_rn(a, bs.ct), __fmul_rn(__fdiv_rn(rel, bs.rn), bs.sn));
  const float o_sum = __fadd_rn(a, __fmul_rn(bs.t_sum, b));
  const float o_big = (fabsf(a) > fabsf(b)) ? a : b;
  return same ? ((fabsf(b) < bs.thr) ? o_sum : o_slerp) : o_big;
}

// NaN-propagating minimum (fminf would drop a NaN operand)
__device__ __forceinline__ float fmin_nan(float x, float y) { float r; asm("min.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(x), "f"(y)); return r; }

// The fast path decides torch.sign(a) == torch.sign(b) by a * b > 0.  That is wrong only if the product is NaN or if it
// underflowed to zero with both operands non-zero; an item with such a product (the NaN-propagating minimum of its four
// |products| is not > 0) is queued and the drain compares the signs exactly.  Exact zeros land there too -- spectra of later
// pair-tree rounds hold ~1 % of them, i.e. ~10 % of their items are queued -- which costs less than a test that tells the
// harmless zeros apart would: that test is a basic-block boundary per item, the drain handles 32 queued items in ~180
// instructions (measured both ways, profiles/r02_fs_pass_prefetch_variants.log).

struct Acc { unsigned int below, anyw; float p00, p11, p01; };

// Classify one key against the window in four instructions: |v| < lo -> ++below; else |v| <= hi -> anyw = 1.  (Written in PTX
// because the compiler, short of predicate registers for the 16 keys of an iteration, recomputed every compare where the
// count was consumed: 5.5 instructions per key.)  NaN keys compare false both times: above the window, like their bit
// patterns.
__device__ __forceinline__ void fs_key(float v, float lo, float hi, unsigned int& below, unsigned int& anyw) {
  asm("{\n\t.reg .pred p, q;\n\t.reg .f32 t;\n\t"
      "abs.f32 t, %2;\n\t"
      "setp.lt.f32 p, t, %3;\n\t"
      "@p add.u32 %0, %0, 1;\n\t"
      "setp.le.and.f32 q, t, %4, !p;\n\t"
      "@q mov.u32 %1, 1;\n\t}"
      : "+r"(below), "+r"(anyw) : "f"(v), "f"(lo), "f"(hi));
}

// interior element pair of a plain item, multiplicity 2 (the caller doubles counts and sums at the end); p = a * b.
// A key inside the window only raises a flag (the item is then queued as well).
template <int MODE>
__device__ __forceinline__ float fs_elem(const PassCtx& x, const BlendScal& bs, float a, float b, float p, Acc& c) {
  const bool same = p > 0.f;
  if (MODE == 0) {
    fs_key(a, x.lo_f, x.hi_f, c.below, c.anyw);
    fs_key(b, x.lo_f, x.hi_f, c.below, c.anyw);
    // |re1| >= thr for every thr in the window (NaN: never < thr) -> the element is in the SLERP sums; masked operands
    // instead of a branch (2 selects + 3 FMAs)
    const bool in = same && !(fabsf(b) <= x.hi_f);
    const float ma = in ? a : 0.f, mb = in ? b : 0.f;
    c.p00 = fmaf(ma, ma, c.p00); c.p11 = fmaf(mb, mb, c.p11); c.p01 = fmaf(ma, mb, c.p01);
    return 0.f;
  } else {
    const float o = fs_blend(bs, a, b, same);
    fs_key(o, x.lo_f, x.hi_f, c.below, c.anyw);
    return o;
  }
}

// one key inside the window, multiplicity w: a fire-and-forget global reduction into its own counter (the window spans
// ~2 M counters, so two keys rarely meet) and a shared-memory one into the CTA's coarse histogram
// Lanes of the warp that carry the SAME key (and multiplicity) combine first: rounding-noise keys -- the culled bins of an
// earlier pair-tree round, a few ulps of the transform's largest terms -- take a handful of distinct values, and 2 % of a
// tensor's keys reducing into ten counters serialise in L2 (the cutoff pass of a round-2 spectrum took 5x as long).
// The sample tells the two cases apart (FsState::dense): a smooth density puts ~1 % of the keys into the window, a tied one
// more; the match costs ~7 % of the pass when keys are distinct, so it is only done where it pays.
__device__ __forceinline__ void fs_red_key(const PassCtx& x, unsigned int key, unsigned int w) {
  const unsigned int d = key - x.lo;
  if (x.dense) {                                                             // uniform over the grid
    const unsigned int act = __activemask();
    const unsigned int peers = __match_any_sync(act, (d << 2) | w);          // d < 2^22, w in {1, 2}
    if ((int)(threadIdx.x & 31u) == __ffs((int)peers) - 1) {
      const unsigned int tot = w * (unsigned int)__popc(peers);
      atomicAdd(x.fine + d, tot);
      atomicAdd(&g_fs_coarse[d >> x.shift], tot);
    }
  } else {
    atomicAdd(x.fine + d, w);
    atomicAdd(&g_fs_coarse[d >> x.shift], w);
  }
}

// what the drain adds to the block totals (only touched out of line)
struct DrainAcc { unsigned long long below; double s00, s11, s01; };

// Drain the top `n` (<= 32) entries of this warp's queue, one entry per lane.  A queued item is either "generic"
// (edge column group: multiplicity 1 at columns 0 and Ch, 2 inside, 0 for the zero padding behind Ch; or an item
// with a zero / NaN product: exact sign comparison) -- then everything is done here -- or a plain interior item with
// a key inside the window: the fast path has done the counts, sums and (MODE 1) the output, only the window work is left.
template <int MODE>
__device__ __noinline__ void fs_drain(int wid, int first, int n, DrainAcc& acc) {
  const PassCtx& x = g_fs_ctx;
  const BlendScal& bs = g_fs_bs;
  const int lane = threadIdx.x & 31;
  __syncwarp();
  if (lane < n) {
    const float4 av = fs_qa(wid)[first + lane], bv = fs_qb(wid)[first + lane];
    const uint2 m = fs_qm(wid)[first + lane];
    const bool generic = (m.y >> 31) != 0u;
    const int c0 = (int)(m.y & 0x7fffffffu);
    const float a[4] = {av.x, av.y, av.z, av.w}, b[4] = {bv.x, bv.y, bv.z, bv.w};
    float o[4];
    unsigned int below = 0u;
    double s00 = 0.0, s11 = 0.0, s01 = 0.0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int col = c0 + i;
      const unsigned int w = col > x.Ch ? 0u : ((col == 0 || col == x.Ch) ? 1u : 2u);
      const bool same = (sgn(a[i]) == sgn(b[i]));         // torch.sign(a) == torch.sign(b) (sign(+-0) = sign(NaN) = 0)
      if (MODE == 0) {
        const float fa = fabsf(a[i]), fb = fabsf(b[i]);
        const bool wa = fa >= x.lo_f && fa <= x.hi_f, wb = fb >= x.lo_f && fb <= x.hi_f;
        if (wa && w) fs_red_key(x, __float_as_uint(fa), w);
        if (wb && w) {
          fs_red_key(x, __float_as_uint(fb), w);
          if (same) {                                     // in the SLERP sums or not: known once the exact threshold is (k_fs_close)
            const unsigned int pos = atomicAdd(&g_fs_nside, 1u);
            if (pos < x.scap) x.slist[pos] = make_float2(w == 1u ? -fa : fa, fb);
            else atomicOr(x.status, 2u);
          }
        }
        if (generic) {
          below += (fa < x.lo_f ? w : 0u) + (fb < x.lo_f ? w : 0u);
          if (same && !(fb <= x.hi_f) && w) {
            const double da = (double)a[i], db = (double)b[i], dw = (double)w;
            s00 += dw * da * da; s11 += dw * db * db; s01 += dw * da * db;
          }
        }
      } else {
        o[i] = fs_blend(bs, a[i], b[i], same);
        const float fo = fabsf(o[i]);
        if (fo >= x.lo_f && fo <= x.hi_f && w) fs_red_key(x, __float_as_uint(fo), w);
        if (generic) below += fo < x.lo_f ? w : 0u;
      }
    }
    if (MODE == 1 && generic) *reinterpret_cast<float4*>(x.out + m.x) = make_float4(o[0], o[1], o[2], o[3]);
    if (generic) { acc.below += below; acc.s00 += s00; acc.s11 += s11; acc.s01 += s01; }
  }
  __syncwarp();
}

template <int MODE>
__global__ void __launch_bounds__(kPassThreads, kPassCtasPerSm) k_fs_pass(const __grid_constant__ SmPlan pl, const __grid_constant__ FsCommon c,
                                                            FsState* st, const __grid_constant__ FsWs ws, float* out,
                                                            float* thr_out) {
  sm_pdl_enter();
  __shared__ unsigned long long s_below[kPassWarps];
  __shared__ double s_red[32];
  __shared__ Pick pick;
  __shared__ unsigned long long s_rank;
  __shared__ int s_ok;
  unsigned int* const s_hist = g_fs_coarse;
  constexpr int NT = kPassThreads;
  const bool sw = (c.sel != nullptr && *c.sel != 0);
  const float* __restrict__ re0 = sw ? c.reY : c.reX;
  const float* __restrict__ re1 = sw ? c.reX : c.reY;
  PassCtx x;
  x.lo = st->lo; x.shift = st->shift; x.scap = ws.scap; x.dense = st->dense;
  x.lo_f = __uint_as_float(x.lo); x.hi_f = __uint_as_float(st->hi);       // hi <= +inf (k_fs_sample)
  x.fine = ws.fine; x.slist = ws.sbkt + (size_t)blockIdx.x * ws.scap;
  x.status = &st->status; x.out = out; x.Ch = pl.Ch;
  const bool dead = st->status != 0u;
  BlendScal bs{};
  if (MODE == 1) { bs.thr = *c.thr_cut; bs.dot = c.scal4[0]; bs.ct = c.scal4[1]; bs.sn = c.scal4[2]; bs.rn = c.scal4[3]; bs.t_sum = c.t_sum; }
  if (threadIdx.x == 0) { g_fs_ctx = x; g_fs_bs = bs; g_fs_nside = 0u; g_fs_chunk = 0u; }
#pragma unroll
  for (int j = 0; j < kBins / NT; ++j) g_fs_coarse[threadIdx.x + NT * j] = 0u;
  __syncthreads();
  const int Ch = pl.Ch;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  unsigned int below_in = 0u;                            // keys below the window, fast path (unweighted)
  double d00 = 0.0, d11 = 0.0, d01 = 0.0;                // SLERP sums, fast path (unweighted)
  DrainAcc da{0ull, 0.0, 0.0, 0.0};                      // generic items (weighted)
  int qn = 0;                                            // entries in this warp's queue (warp-uniform)
  float4* const qa = fs_qa(wid); float4* const qb = fs_qb(wid); uint2* const qm = fs_qm(wid);
  // Work items are float4 column groups, numbered row-major over rows x G groups (G covers columns 0..Ch).
  const unsigned int G = (unsigned int)(Ch + 4) / 4u;
  const unsigned int total = (unsigned int)pl.R * G;
  const unsigned int nchunks = (total + kChunkItems - 1u) / kChunkItems;
  const unsigned int cpb = (nchunks + gridDim.x - 1u) / gridDim.x;               // chunks per CTA
  const unsigned int c0 = blockIdx.x * cpb, c_end = min(c0 + cpb, nchunks);
  if (!dead) {
    unsigned int chunk = c0 + wid, next = 0u;
    while (chunk < c_end) {                              // warp-uniform
      if (lane == 0) next = c0 + kPassWarps + atomicAdd(&g_fs_chunk, 1u);        // consumed after this chunk
      unsigned int idx = chunk * kChunkItems + lane;
      unsigned int row = idx / G, g = idx - row * G;
#pragma unroll 1
      for (unsigned int it = 0; it < kChunkIters; ++it, idx += 64u) {
        // two items per iteration: this lane's and the one 32 further (a warp reads 1 KB contiguous per plane)
        unsigned int row1 = row, g1 = g + 32u;
        while (g1 >= G) { g1 -= G; ++row1; }
        const bool v0 = idx < total, v1 = idx + 32u < total;
        const size_t off0 = v0 ? (size_t)row * pl.P + 4u * g : 0;
        const size_t off1 = v1 ? (size_t)row1 * pl.P + 4u * g1 : off0;
        float4 a0, b0, a1, b1;                           // both items in flight before the first is consumed
        a0 = *reinterpret_cast<const float4*>(re0 + off0); b0 = *reinterpret_cast<const float4*>(re1 + off0);
        a1 = *reinterpret_cast<const float4*>(re0 + off1); b1 = *reinterpret_cast<const float4*>(re1 + off1);
        bool want[2];
        unsigned int meta[2];
#pragma unroll
        for (int r = 0; r < 2; ++r) {
          const float4 av = r == 0 ? a0 : a1, bv = r == 0 ? b0 : b1;
          const bool valid = r == 0 ? v0 : v1;
          const unsigned int gg = r == 0 ? g : g1;
          const size_t off = r == 0 ? off0 : off1;
          const float4 pv = make_float4(av.x * bv.x, av.y * bv.y, av.z * bv.z, av.w * bv.w);
          const bool edge = (gg == 0u) | (gg == G - 1u);
          // branch-free: an item with a zero / NaN product is simply queued (the drain compares signs exactly); the relaxed
          // test for exact zeros (fs_item_plain) is not worth a basic-block boundary per item here
          const bool generic = edge | !(fmin_nan(fmin_nan(fabsf(pv.x), fabsf(pv.y)), fmin_nan(fabsf(pv.z), fabsf(pv.w))) > 0.f);
          Acc ac{0u, 0u, 0.f, 0.f, 0.f};                 // fp32 over one float4, fp64 across
          float4 o;
          o.x = fs_elem<MODE>(x, bs, av.x, bv.x, pv.x, ac); o.y = fs_elem<MODE>(x, bs, av.y, bv.y, pv.y, ac);
          o.z = fs_elem<MODE>(x, bs, av.z, bv.z, pv.z, ac); o.w = fs_elem<MODE>(x, bs, av.w, bv.w, pv.w, ac);
          const bool fast = valid && !generic;
          below_in += fast ? ac.below : 0u;              // selects, not a branch: the iteration stays one basic block
          if (MODE == 0) {
            d00 += (double)(fast ? ac.p00 : 0.f); d11 += (double)(fast ? ac.p11 : 0.f); d01 += (double)(fast ? ac.p01 : 0.f);
          } else if (fast) {
            *reinterpret_cast<float4*>(out + off) = o;   // a predicated store
          }
          want[r] = valid && (generic || ac.anyw != 0u);
          meta[r] = 4u * gg | (generic ? 0x80000000u : 0u);
        }
        {  // both items of the iteration join the queue in one step (some lane wants to in 9 iterations out of 10)
          const unsigned int m0 = __ballot_sync(0xffffffffu, want[0]), m1 = __ballot_sync(0xffffffffu, want[1]);
          if (m0 | m1) {                                 // warp-uniform
            const unsigned int lt = (1u << lane) - 1u;
            if (want[0]) {
              const int slot = qn + __popc(m0 & lt);
              qa[slot] = a0; qb[slot] = b0; qm[slot] = make_uint2((unsigned int)off0, meta[0]);
            }
            qn += __popc(m0);
            if (want[1]) {
              const int slot = qn + __popc(m1 & lt);
              qa[slot] = a1; qb[slot] = b1; qm[slot] = make_uint2((unsigned int)off1, meta[1]);
            }
            qn += __popc(m1);
            while (qn >= 32) { qn -= 32; fs_drain<MODE>(wid, qn, 32, da); }
          }
        }
        // advance by 64 items
        row = row1; g = g1 + 32u;
        while (g >= G) { g -= G; ++row; }
      }
      chunk = __shfl_sync(0xffffffffu, next, 0);
    }
    if (qn > 0) fs_drain<MODE>(wid, 0, qn, da);
  }
  {
    unsigned long long below = 2ull * below_in + da.below;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) below += __shfl_xor_sync(0xffffffffu, below, o);
    if ((threadIdx.x & 31) == 0) s_below[threadIdx.x >> 5] = below;
    __syncthreads();                                     // also: every shared-memory reduction of the loop has landed
    if (threadIdx.x == 0) {
      unsigned long long bsum = 0ull;
      for (int i = 0; i < kPassWarps; ++i) bsum += s_below[i];
      if (bsum) atomicAdd(&st->below, bsum);
      if (MODE == 0) ws.scnt[blockIdx.x] = g_fs_nside < ws.scap ? g_fs_nside : ws.scap;
    }
    // this CTA's coarse histogram -> the global one: one coalesced reduction per warp and 32 bins
#pragma unroll
    for (int j = 0; j < kBins / NT; ++j) {
      const unsigned int v = g_fs_coarse[threadIdx.x + NT * j];
      if (v) atomicAdd(ws.coarse + threadIdx.x + NT * j, v);
    }
  }
  if (MODE == 0) {
    const double r0 = block_sum_d(2.0 * d00 + da.s00, s_red), r1 = block_sum_d(2.0 * d11 + da.s11, s_red),
                 r2 = block_sum_d(2.0 * d01 + da.s01, s_red);
    if (threadIdx.x == 0 && (r0 != 0.0 || r1 != 0.0 || r2 != 0.0)) {
      atomicAdd(&st->s_in[0], r0); atomicAdd(&st->s_in[1], r1); atomicAdd(&st->s_in[2], r2);
    }
  }
  const bool last_cta = fs_last_block(st);
  if (!last_cta) return;

  // ---- last CTA: coarse bin of the statistic -> exact key from that bin's fine counters
  if (threadIdx.x == 0) {
    const unsigned long long r = st->rank, bl = *((volatile unsigned long long*)&st->below);
    unsigned int status = *((volatile unsigned int*)&st->status);
    if (r < bl) { status |= 1u; s_rank = 0ull; } else s_rank = r - bl;
    st->status = status;
    s_ok = status == 0u ? 1 : 0;
  }
  __syncthreads();
  bool ok = s_ok != 0;                                    // block-uniform from here on
  unsigned int key = 0u;
  int bstar = -1;
  if (ok) {
    {  // key counts per coarse bin -> shared memory, every load in flight at once
      unsigned int v[kBins / NT];
#pragma unroll
      for (int j = 0; j < kBins / NT; ++j) v[j] = __ldcg(ws.coarse + threadIdx.x + NT * j);
#pragma unroll
      for (int j = 0; j < kBins / NT; ++j) s_hist[threadIdx.x + NT * j] = v[j];
    }
    __syncthreads();
    block_pick<NT>(LoadSmem32{s_hist}, kBins, s_rank, &pick);
    bstar = pick.bin;
    if (bstar < 0) ok = false;                            // rank beyond the window: the sample window missed
  }
  if (ok) {
    // the bin covers 2^shift <= 2048 bit patterns, one fine counter each
    const unsigned long long rin = pick.rank_in_bin;
    const unsigned int nf = 1u << x.shift;
    const unsigned int f0 = (unsigned int)bstar << x.shift;
    __syncthreads();
    {
      unsigned int v[kBins / NT];
#pragma unroll
      for (int j = 0; j < kBins / NT; ++j) {
        const unsigned int i = threadIdx.x + NT * j;
        v[j] = i < nf ? __ldcg(ws.fine + f0 + i) : 0u;
      }
#pragma unroll
      for (int j = 0; j < kBins / NT; ++j) s_hist[threadIdx.x + NT * j] = v[j];
    }
    __syncthreads();
    block_pick<NT>(LoadSmem32{s_hist}, kBins, rin, &pick);
    if (pick.bin < 0) ok = false;
    else key = x.lo + f0 + (unsigned int)pick.bin;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    if (!ok && st->status == 0u) st->status = 1u;
    st->sticky |= st->status;
    st->ticket = 0u;
    if (st->status != 0u) {
      st->value = __uint_as_float(0x7fc00000u);
    } else {
      st->key = key; st->value = __uint_as_float(key); st->bstar = (unsigned int)bstar;
    }
    if (thr_out) *thr_out = st->value;
  }
}

// cutoff pass, second half: the side-list entries with |re1| >= key join the SLERP sums; the last CTA turns the sums
// into the scalars of slerp().
__global__ void __launch_bounds__(SM_EW_THREADS) k_fs_close(FsState* st, const __grid_constant__ FsWs ws, double t, float* scal4,
                                                            double* sums_out) {
  sm_pdl_enter();
  __shared__ double s_red[32];
  const bool ok = st->status == 0u;
  const unsigned int key = st->key;
  double acc[3] = {0.0, 0.0, 0.0};
  if (ok) {
    for (unsigned int l = blockIdx.x; l < ws.n_lists; l += gridDim.x) {
      const unsigned int n = __ldcg(ws.scnt + l);
      const float2* lst = ws.sbkt + (size_t)l * ws.scap;
      for (unsigned int i = threadIdx.x; i < n; i += blockDim.x) {
        const float2 e = __ldcg(lst + i);
        if (__float_as_uint(e.y) >= key) {
          const double a = (double)fabsf(e.x), b = (double)e.y, w = (__float_as_uint(e.x) >> 31) ? 1.0 : 2.0;
          acc[0] += w * a * a; acc[1] += w * b * b; acc[2] += w * a * b;
        }
      }
    }
  }
  for (int j = 0; j < 3; ++j) {
    const double r = block_sum_d(acc[j], s_red);
    if (threadIdx.x == 0 && r != 0.0) atomicAdd(&st->s_in[j], r);
  }
  if (!fs_last_block(st)) return;
  if (threadIdx.x == 0) {
    st->ticket = 0u;
    if (ok) {
      double s[3] = {*((volatile double*)&st->s_in[0]), *((volatile double*)&st->s_in[1]), *((volatile double*)&st->s_in[2])};
      if (sums_out) { sums_out[0] = s[0]; sums_out[1] = s[1]; sums_out[2] = s[2]; }
      if (scal4) fs_scalars(s, t, scal4);
    }
  }
}

inline dim3 fs_grid(const SmPlan& p) {
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) sms = 148;
  const long long items = (long long)p.R * ((p.Ch + 4) / 4);
  long long ctas = (long long)sms * kPassCtasPerSm;      // one resident wave
  const long long need = (items + 2 * kPassThreads - 1) / (2 * kPassThreads);
  if (ctas > need) ctas = need;
  if (ctas > kMaxLists) ctas = kMaxLists;
  if (ctas < 1) ctas = 1;
  return dim3((unsigned int)ctas, 1);
}

void fs_sample_ranks(unsigned long long rank, unsigned long long total, long long* k_lo, long long* k_hi) {
  const double pq = (double)rank / (double)total;
  const double ks = pq * (double)kNS;
  const double delta = 6.0 * sqrt((double)kNS * pq * (1.0 - pq)) + 16.0;
  *k_lo = (long long)floor(ks - delta); *k_hi = (long long)ceil(ks + delta);
}

// side list capacity per CTA: the window holds ~frac of the keys of one plane (widest window any rank can need,
// p = 0.5, plus the two sample-histogram bins of slack), the CTAs share them evenly; x4 headroom.
double fs_max_frac() { return 2.0 * (6.0 * sqrt((double)kNS * 0.25) + 16.0) / (double)kNS + 0.02; }
unsigned int fs_scap(const SmPlan& p, unsigned int n_lists) {
  const double entries = fs_max_frac() * (double)p.R * (double)(p.Ch + 1);
  return (unsigned int)(entries / (double)n_lists * 4.0) + 256u;
}

}  // namespace

// ================================================================== C ABI
extern "C" int sm_fstats_supported(const sm_plan* plan) {
  const SmPlan& p = plan->p;
  const unsigned long long n = (unsigned long long)p.R * p.C;
  return (n > (1ull << 20) && 2ull * n < 0xfffffff0ull) ? 1 : 0;
}

static size_t fs_zero_bytes() {
  return (size_t)kSampleBins * 4 + (size_t)kBins * 4 + (size_t)kMaxLists * 4 + (size_t)kFineMax * 4 + 64;
}

extern "C" size_t sm_fstats_ws_bytes(const sm_plan* plan) {
  const SmPlan& p = plan->p;
  if (!sm_fstats_supported(plan)) return 256;
  const unsigned int n_lists = fs_grid(p).x;
  size_t b = fs_zero_bytes();
  b += (size_t)n_lists * fs_scap(p, n_lists) * 8;
  return b + 512;                // + alignment
}

static int fs_carve(const sm_plan* plan, void* wsp, size_t ws_bytes, FsWs* w) {
  const SmPlan& p = plan->p;
  if (!sm_fstats_supported(plan)) { sm_set_error("fstats: tensor too small / too large for the fused statistics"); return -2; }
  if (ws_bytes < sm_fstats_ws_bytes(plan)) { sm_set_error("fstats: workspace too small"); return -3; }
  // the LAST sm_fstats_ws_bytes() of the caller's buffer: its histograms persist (zero) from call to call, and a
  // caller that shares one buffer with sm_select_kth_abs (which uses the front) must not have them overwritten
  char* b = reinterpret_cast<char*>(wsp) + (ws_bytes - sm_fstats_ws_bytes(plan));
  b = reinterpret_cast<char*>(((uintptr_t)b + 63) / 64 * 64);
  char* const z0 = b;
  w->shist = reinterpret_cast<unsigned int*>(b); b += (size_t)kSampleBins * 4;
  w->coarse = reinterpret_cast<unsigned int*>(b); b += (size_t)kBins * 4;
  w->scnt = reinterpret_cast<unsigned int*>(b); b += (size_t)kMaxLists * 4;
  w->fine = reinterpret_cast<unsigned int*>(b); b += (size_t)kFineMax * 4;
  w->meta = reinterpret_cast<unsigned int*>(b); b += 64;
  w->zero_bytes = (size_t)(b - z0);
  w->n_lists = fs_grid(p).x;
  w->scap = fs_scap(p, w->n_lists);
  w->sbkt = reinterpret_cast<float2*>(b);
  return 0;
}

static int fs_pass_attr() {          // opt in to the dynamic shared memory of k_fs_pass (the warp queues), once
  static int rc = 1;
  if (rc == 1) {
    cudaError_t e = cudaFuncSetAttribute((const void*)k_fs_pass<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPassDynSmem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute((const void*)k_fs_pass<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPassDynSmem);
    if (e != cudaSuccess) { sm_set_error("fstats: shared-memory opt-in failed: %s", cudaGetErrorString(e)); rc = -100; } else rc = 0;
  }
  return rc;
}

static inline int fs_sample_grid() { return (int)((kNS + kSampleThreads * kSamplePer - 1) / (kSampleThreads * kSamplePer)); }

// Cutoff statistic + SLERP sums + scalars in one streaming pass (see the header of this file).
extern "C" int sm_fstats_cutoff(const sm_plan* plan, const float* reX, const float* reY, const int* sel, uint64_t rank,
                                double t, void* fs_state, void* ws, size_t ws_bytes, float* thr_cut_out,
                                float* scal4_out, double* sums3_out, void* stream) {
  const SmPlan& p = plan->p;
  cudaStream_t s = (cudaStream_t)stream;
  FsWs w;
  int rc = fs_carve(plan, ws, ws_bytes, &w);
  if (rc) return rc;
  const unsigned long long total = 2ull * (unsigned long long)p.R * p.C;
  if (rank >= total) rank = total - 1;
  FsState* st = reinterpret_cast<FsState*>(fs_state);
  FsCommon c{reX, reY, sel, nullptr, nullptr, 1.f};
  long long k_lo = 0, k_hi = 0;
  fs_sample_ranks(rank, total, &k_lo, &k_hi);
  sm_launch(k_fs_sample<0>, dim3(fs_sample_grid()), dim3(kSampleThreads), (size_t)(0), s, p, c, st, w, rank, k_lo, k_hi);
  SM_LAUNCH_CHECK();
  if ((rc = fs_pass_attr())) return rc;
  sm_launch(k_fs_pass<0>, dim3(w.n_lists), dim3(kPassThreads), (size_t)(kPassDynSmem), s, p, c, st, w, nullptr, thr_cut_out);
  SM_LAUNCH_CHECK();
  const unsigned int close_grid = w.n_lists < 148u ? w.n_lists : 148u;
  sm_launch(k_fs_close, dim3(close_grid), dim3(SM_EW_THREADS), (size_t)(0), s, st, w, t, scal4_out, sums3_out);
  SM_LAUNCH_CHECK();
  return 0;
}

// Blend (SLERP mode) + cull statistic of its output in one streaming pass.
extern "C" int sm_fstats_blend_cull(const sm_plan* plan, const float* reX, const float* reY, const int* sel,
                                    const float* thr_cut, const float* scal4, float t_sum, float* out_re, uint64_t rank,
                                    void* fs_state, void* ws, size_t ws_bytes, float* thr_cull_out, void* stream) {
  const SmPlan& p = plan->p;
  cudaStream_t s = (cudaStream_t)stream;
  FsWs w;
  int rc = fs_carve(plan, ws, ws_bytes, &w);
  if (rc) return rc;
  const unsigned long long total = (unsigned long long)p.R * p.C;
  if (rank >= total) rank = total - 1;
  FsState* st = reinterpret_cast<FsState*>(fs_state);
  FsCommon c{reX, reY, sel, thr_cut, scal4, t_sum};
  long long k_lo = 0, k_hi = 0;
  fs_sample_ranks(rank, total, &k_lo, &k_hi);
  sm_launch(k_fs_sample<1>, dim3(fs_sample_grid()), dim3(kSampleThreads), (size_t)(0), s, p, c, st, w, rank, k_lo, k_hi);
  SM_LAUNCH_CHECK();
  if ((rc = fs_pass_attr())) return rc;
  sm_launch(k_fs_pass<1>, dim3(w.n_lists), dim3(kPassThreads), (size_t)(kPassDynSmem), s, p, c, st, w, out_re, thr_cull_out);
  SM_LAUNCH_CHECK();
  return 0;
}
