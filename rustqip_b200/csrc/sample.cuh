// sample.cuh -- decision rules of inverse-CDF sampling (qipb200_state_sample), shared by the device kernels
// (kernels.cu: k_sample_resolve) and the CPU model of the whole algorithm (tests/native/sample_model.cpp).
//
// A draw r selects the first canonical index i whose inclusive cumulative probability is >= r
// (measurement_ops.rs:153-176: `r -= |a_i|^2; if r <= 0 { stop }`); no such index -> index 0 (the reference's
// `measured_indx = 0`).  The state is cut into chunks of 2^kSampleChunkLog2 amplitudes; P[c] is the inclusive
// prefix of the chunk sums of this rank's shard, and a rank's total is P[last].
//
// Resolving a draw on its owner: chunk search on P, then a scan of the chunk in 32-amplitude groups from base
// P[c-1] (warp inclusive scan, crossing test below).  The chunk-level and amplitude-level sums round differently,
// so the scan may leave the chunk without crossing: it then continues into the following chunks, and if it runs past
// the end of the shard it takes the last amplitude with non-zero probability it passed (the draw lies within
// rounding of the shard's total).
#pragma once

#include <cstdint>

#if defined(__CUDACC__)
#define QIP_SAMPLE_HD __host__ __device__ __forceinline__
#else
#define QIP_SAMPLE_HD inline
#endif

namespace qipb200 {

static const uint32_t kSampleChunkLog2 = 10;     // 1024 amplitudes: 16 KiB (f64) read per resolved draw at most
static const uint64_t kSampleBatch = 1ull << 20; // draws per device batch: 16 B of scratch each

// Owner of draw r among W ranks with totals T[0..W): the lowest rank t with r <= T[0] + ... + T[t] (summed in rank
// order, hence bit-identical on every rank).  Returns W when r exceeds the grand total (or is NaN): index 0.
// *local = the part of r left for the owner, clamped to its total so that the owner's chunk search always lands.
QIP_SAMPLE_HD int sample_owner(const double *T, int W, double r, double *local) {
  double below = 0.0;
  for (int t = 0; t < W; ++t) {
    const double upto = below + T[t];
    if (r <= upto) {
      const double l = r - below;
      *local = l < T[t] ? l : T[t];
      return t;
    }
    below = upto;
  }
  *local = 0.0;
  return W;
}

// First chunk c with P[c] >= t (lower bound).  The tree-ordered prefix may be non-monotone by a rounding step;
// the search still returns a c with P[c] >= t and (c == 0 or P[c-1] < t), and never `chunks` when P[chunks-1] >= t.
QIP_SAMPLE_HD uint64_t sample_chunk(const double *P, uint64_t chunks, double t) {
  uint64_t lo = 0, hi = chunks;
  while (lo < hi) {
    const uint64_t mid = lo + ((hi - lo) >> 1);
    if (P[mid] < t)
      lo = mid + 1;
    else
      hi = mid;
  }
  return lo;
}

// Inclusive scan of 32 values in the order of the device's warp scan (shuffle-up by 1, 2, 4, 8, 16): the CPU model
// runs this on arrays, the device on registers, with identical rounding.
QIP_SAMPLE_HD void sample_warp_scan(double *v) {
  for (int o = 1; o < 32; o <<= 1)
    for (int j = 31; j >= o; --j) v[j] = v[j] + v[j - o];
}

// The crossing test inside a chunk: amplitude i (inclusive running sum base + incl) is selected when it reaches t.
QIP_SAMPLE_HD bool sample_crosses(double base, double incl, double t) { return base + incl >= t; }

// extract_bits(i, [n-1-q for q in indices]) (measurement_ops.rs:174-175): bit j of the outcome from bitpos[j].
QIP_SAMPLE_HD uint64_t sample_outcome(uint64_t index, const uint8_t *bitpos, uint32_t n_bits) {
  uint64_t m = 0;
  for (uint32_t j = 0; j < n_bits; ++j) m |= ((index >> bitpos[j]) & 1ull) << j;
  return m;
}

}  // namespace qipb200
