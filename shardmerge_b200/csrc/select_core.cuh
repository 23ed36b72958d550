// select_core.cuh -- the radix digit pick of the exact order-statistic selects, shared by kernels_stats.cu (one select over
// spectrum magnitudes) and kernels_sparse.cu (one select per model over delta magnitudes).  Keys are 31-bit; three digits
// of 11, 10 and 10 bits (shifts 20, 10, 0) resolve them.  A SelState carries one select from digit to digit.
#pragma once
#include <cstddef>
#include "../../include/shardmerge_b200.h"

namespace {

constexpr int kHistBins = 2048;

struct SelState {              // must match SM_SELECT_STATE_BYTES / the header comment
  unsigned long long rank;
  unsigned long long below;
  unsigned int prefix;
  unsigned int lo, hi;
  unsigned int ncand;
  unsigned int cap;
  unsigned int status;         // bit0: window missed the statistic, bit1: candidate overflow
  float value;
  unsigned int sticky;         // OR of every status this state has ended with (k_sel_init keeps it)
  unsigned int pad[4];
};
static_assert(sizeof(SelState) == SM_SELECT_STATE_BYTES, "SelState layout");
static_assert(offsetof(SelState, sticky) == SM_SELECT_STICKY_OFF, "SelState sticky offset");

enum { PICK_NONE = 0, PICK_ADJUST = 1, PICK_FINISH = 3 };

// block of 1024 threads: find the bin of a 2048-bin histogram (global or shared) that holds 0-based
// `rank`; returns through shared outputs.  The histogram is zeroed on the way.
struct PickOut { int bin; unsigned long long rank_in_bin; };
__device__ __forceinline__ void block_pick(unsigned int* hist, unsigned long long rank, PickOut* s_out /*shared*/,
                                           int nbins = kHistBins, bool zero = true) {
  __shared__ unsigned long long wtot[32];
  const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
  if (t == 0) { s_out->bin = -1; s_out->rank_in_bin = 0ull; }
  const bool live = (2 * t + 1) < nbins;
  const unsigned int h0 = live ? hist[2 * t] : 0u, h1 = live ? hist[2 * t + 1] : 0u;
  if (zero && live) { hist[2 * t] = 0u; hist[2 * t + 1] = 0u; }
  const unsigned long long v = (unsigned long long)h0 + h1;
  unsigned long long incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned long long n = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += n;
  }
  if (lane == 31) wtot[wid] = incl;
  __syncthreads();
  if (wid == 0) {
    const unsigned long long w = wtot[lane];
    unsigned long long wi = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long n = __shfl_up_sync(0xffffffffu, wi, o);
      if (lane >= o) wi += n;
    }
    wtot[lane] = wi - w;                             // exclusive warp offsets
  }
  __syncthreads();
  const unsigned long long excl = wtot[wid] + incl - v;
  if (rank >= excl && rank < excl + h0) { s_out->bin = 2 * t; s_out->rank_in_bin = rank - excl; }
  else if (rank >= excl + h0 && rank < excl + v) { s_out->bin = 2 * t + 1; s_out->rank_in_bin = rank - excl - h0; }
  __syncthreads();
}

// block of 1024 threads: extend the prefix of `st` by one radix digit from the histogram of digit `pass`; afterwards
// st->rank is the rank of the statistic among the keys that share the extended prefix
__device__ __forceinline__ void sel_pick_digit(unsigned int* __restrict__ hist, SelState* st, int pass, int action,
                                               float* thr_out) {
  __shared__ PickOut out;
  __shared__ unsigned long long s_rank;
  if (threadIdx.x == 0) {
    unsigned long long r = st->rank;
    if (action == PICK_ADJUST) {
      const unsigned long long below = st->below;
      const unsigned int nc = st->ncand;
      if (nc > st->cap) st->status |= 2u;
      if (r < below || r - below >= (unsigned long long)nc) { st->status |= 1u; r = 0ull; }
      else r -= below;
      st->rank = r;
    }
    s_rank = r;
  }
  __syncthreads();
  block_pick(hist, s_rank, &out);
  if (threadIdx.x == 0) {
    const int shift = pass == 0 ? 20 : (pass == 1 ? 10 : 0);
    if (st->status == 0u) {
      if (out.bin >= 0) { st->prefix |= (unsigned int)out.bin << shift; st->rank = out.rank_in_bin; }
      else st->status |= 1u;
    }
    if (action == PICK_FINISH) {
      const float val = (st->status == 0u) ? __uint_as_float(st->prefix) : __uint_as_float(0x7fc00000u);
      st->value = val;
      st->sticky |= st->status;
      if (thr_out) *thr_out = val;
    }
  }
}

}  // namespace
