// kernels.cuh -- launch interface of the sm_100a gate kernels (see kernels.cu).
#pragma once

#include <cuda_runtime.h>

#include <cstdint>

#include "opcompile.h"
#include "sample.cuh"

namespace qipb200 {

static const int kMaxIns = 12;      // max bit positions removed from the work-item counter
static const int kMaxRegK = 4;      // largest dense block handled in registers
static const int kMaxDiagParamK = 4; // largest diagonal table passed by kernel parameter

// Launch helpers.  `psi` is the device buffer of the (local) state with 2^n_local
// amplitudes, interleaved (re,im) of R.  All return cudaError_t of the launch and
// add the number of kernels launched to *launches.
cudaError_t launch_dense(qip_prec prec, void *psi, uint32_t n_local, const FlatOp &f, cudaStream_t s,
                         uint64_t *launches);
cudaError_t launch_diag(qip_prec prec, void *psi, uint32_t n_local, uint64_t ctrl_mask,
                        const std::vector<uint32_t> &bits, const std::vector<cplx> &d, cudaStream_t s,
                        uint64_t *launches);
// Dense blocks on 5..10 target bits, in place (k = 5: groups in registers, matrix in shared memory; k >= 6: staged
// through shared memory, matrix through L1/L2), and diagonals on 5..10 bits (table in shared memory).
cudaError_t launch_dense_wide(qip_prec prec, void *psi, uint32_t n_local, const FlatOp &f, cudaStream_t s,
                              uint64_t *launches);
cudaError_t launch_diag_wide(qip_prec prec, void *psi, uint32_t n_local, uint64_t ctrl_mask,
                             const std::vector<uint32_t> &bits, const std::vector<cplx> &d, cudaStream_t s,
                             uint64_t *launches);
cudaError_t launch_flip(qip_prec prec, void *psi, uint32_t n_local, uint64_t ctrl_mask, uint32_t tbit,
                        cudaStream_t s, uint64_t *launches);
cudaError_t launch_bitswap(qip_prec prec, void *psi, uint32_t n_local, uint64_t ctrl_mask, uint32_t p,
                           uint32_t q, cudaStream_t s, uint64_t *launches);

// Universal out-of-place row kernel with the reference's exact semantics
// (apply_op_row_indices, qip-iterators/src/matrix_ops.rs:62-94), offsets and
// accumulate mode included.  Device copies of the matrix / CSR are made with
// stream-ordered allocations.
cudaError_t launch_gather(qip_prec prec, const FlatOp &f, uint32_t n_qubits, const void *in,
                          uint64_t in_len, uint64_t in_off, void *out, uint64_t out_len,
                          uint64_t out_off, bool accumulate, cudaStream_t s, uint64_t *launches);
// apply_ops with several ops as the reference computes it (multi-op row iterator, accumulating; 2..8 ops).
cudaError_t launch_multi_gather(qip_prec prec, const std::vector<FlatOp> &fs, const void *in, uint64_t in_len, uint64_t in_off,
                                void *out, uint64_t out_len, uint64_t out_off, cudaStream_t s, uint64_t *launches);

// sum |a|^2 into *d_out (a device double, zeroed by the launcher).
cudaError_t launch_norm2(qip_prec prec, const void *psi, uint64_t len, double *d_out, cudaStream_t s,
                         uint64_t *launches);
// max over amplitudes of max(|re_a-re_b|, |im_a-im_b|) into *d_out (a device double).
cudaError_t launch_max_abs_diff(qip_prec prec, const void *a, const void *b, uint64_t len, double *d_out, cudaStream_t s,
                                uint64_t *launches);
cudaError_t launch_set_basis(qip_prec prec, void *psi, uint64_t len, uint64_t index, bool owns_index,
                             cudaStream_t s, uint64_t *launches);

// Measurement (qip/src/state_ops/measurement_ops.rs).
// hist[m] += sum of |a|^2 over amplitudes whose bits at bitpos[i] spell m (bit i of m <-> bitpos[i]).
cudaError_t launch_measure_probs(qip_prec prec, const void *psi, uint64_t len, uint64_t index_base,
                                 const uint32_t *bitpos, uint32_t n_bits, double *d_hist, cudaStream_t s,
                                 uint64_t *launches);
// per-chunk sums of |a|^2 (chunk = 2^chunk_log2 amplitudes): the one read sweep of inverse-CDF sampling.
cudaError_t launch_chunk_sums(qip_prec prec, const void *psi, uint64_t len, uint32_t chunk_log2,
                              double *d_sums, cudaStream_t s, uint64_t *launches);
// Inverse-CDF sampling (qipb200_state_sample; rules in sample.cuh).
// d[0..n) <- its inclusive prefix sum, in a fixed order (repeated calls give identical bits).
cudaError_t launch_sample_scan(double *d, uint64_t n, cudaStream_t s, uint64_t *launches);
struct SampleArgs {
  uint64_t n_draws;
  uint64_t chunks;      // of this shard, 2^chunk_log2 amplitudes each
  uint64_t index_base;  // global index of the shard's first amplitude
  uint32_t chunk_log2;
  int rank, world;      // totals[0..world) are the ranks' totals
};
// out[j] = global index drawn by draws[j] if this rank owns the draw, else 0 (P = inclusive prefix of the chunk sums).
cudaError_t launch_sample_resolve(qip_prec prec, const void *psi, const double *P, const double *totals,
                                  const double *draws, double *out, const SampleArgs &a, cudaStream_t s,
                                  uint64_t *launches);
// res[j] (a global index held as a double) <- its outcome bits as a uint64, bit i from bitpos[i].
cudaError_t launch_sample_outcomes(double *res, uint64_t n_draws, const uint8_t *bitpos, uint32_t n_bits,
                                   cudaStream_t s, uint64_t *launches);
// measure_state: zero where (index & row_mask) != measured_mask, else scale by p_mult.
cudaError_t launch_collapse(qip_prec prec, void *psi, uint64_t len, uint64_t index_base,
                            uint64_t row_mask, uint64_t measured_mask, double p_mult, cudaStream_t s,
                            uint64_t *launches);

}  // namespace qipb200
