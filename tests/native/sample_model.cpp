// sample_model.cpp -- CPU model of qipb200_state_sample (api.cu: sample_impl, kernels.cu: k_sample_*) on host arrays:
// the same chunk layout, the same decision rules (rustqip_b200/csrc/sample.cuh), W emulated ranks each holding a
// contiguous shard of the canonical vector.  Built by tests/test_sample_cpu.py.
#include <cstdint>
#include <vector>

#include "../../rustqip_b200/csrc/sample.cuh"

using namespace qipb200;

namespace {

// One rank's view: its chunk prefix and its resolve of a draw (k_sample_resolve's loop, a 32-lane group at a time).
struct Shard {
  const double *psi;  // interleaved (re, im) of this shard
  uint64_t len, base;
  uint32_t chunk_log2;
  std::vector<double> P;

  double prob(uint64_t i) const { return psi[2 * i] * psi[2 * i] + psi[2 * i + 1] * psi[2 * i + 1]; }

  void prefix() {
    const uint64_t chunks = len >> chunk_log2;
    P.assign(chunks, 0.0);
    for (uint64_t c = 0; c < chunks; ++c) {
      double s = 0.0;
      for (uint64_t i = c << chunk_log2; i < (c + 1) << chunk_log2; ++i) s += prob(i);
      P[c] = (c ? P[c - 1] : 0.0) + s;
    }
  }

  uint64_t resolve(double t) const {
    const uint64_t chunks = P.size();
    uint64_t c = sample_chunk(P.data(), chunks, t);
    double base_sum = c ? P[c - 1] : 0.0;
    uint64_t last_nonzero = c << chunk_log2;
    for (; c < chunks; ++c) {
      const uint64_t begin = c << chunk_log2, end = begin + (1ull << chunk_log2);
      for (uint64_t g = begin; g < end; g += 32) {
        double v[32];
        for (int l = 0; l < 32; ++l) v[l] = g + l < end ? prob(g + l) : 0.0;
        uint64_t nz = 0;
        for (int l = 0; l < 32; ++l) nz |= (uint64_t)(v[l] > 0.0) << l;
        sample_warp_scan(v);
        for (int l = 0; l < 32; ++l)
          if (g + l < end && sample_crosses(base_sum, v[l], t)) return base + g + l;
        for (int l = 31; l >= 0; --l)
          if ((nz >> l) & 1) {
            last_nonzero = g + l;
            break;
          }
        base_sum += v[31];
      }
    }
    return base + last_nonzero;
  }
};

}  // namespace

// out[j] = outcome of draw r[j] on the n-qubit state psi (2^n interleaved doubles) sharded over W ranks.
extern "C" int sample_model(uint32_t n, int W, const double *psi, const uint64_t *indices, uint32_t n_indices,
                            const double *r, uint64_t n_draws, uint64_t *out) {
  int g = 0;
  while ((1 << g) < W) ++g;
  if ((1 << g) != W || (uint32_t)g > n || n_indices > 64) return 1;
  const uint32_t n_local = n - (uint32_t)g;
  std::vector<Shard> shards(W);
  std::vector<double> T(W);
  for (int t = 0; t < W; ++t) {
    Shard &s = shards[t];
    s.len = 1ull << n_local;
    s.base = (uint64_t)t << n_local;
    s.psi = psi + 2 * s.base;
    s.chunk_log2 = n_local < kSampleChunkLog2 ? n_local : kSampleChunkLog2;
    s.prefix();
    T[t] = s.P.back();
  }
  uint8_t bitpos[64];
  for (uint32_t i = 0; i < n_indices; ++i) bitpos[i] = (uint8_t)(n - 1 - indices[i]);
  for (uint64_t j = 0; j < n_draws; ++j) {
    double t;
    const int owner = sample_owner(T.data(), W, r[j], &t);
    const uint64_t index = owner == W ? 0 : shards[owner].resolve(t);
    out[j] = sample_outcome(index, bitpos, n_indices);
  }
  return 0;
}
