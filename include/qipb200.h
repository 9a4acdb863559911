/*
 * qipb200.h -- C ABI of libqipb200: B200-native (sm_100a) state-vector gate
 * application behind RustQIP's operator API.
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  Every entry point names
 * the reference interface it replaces (paths relative to the RustQIP tree).
 * A Rust `extern "C"` block / bindgen run over this header is all a
 * maintainer needs (INTEGRATION.md shows the shim).
 *
 * Conventions
 *   - amplitudes: interleaved (re,im) of float (QIP_F32) or double (QIP_F64),
 *     i.e. the memory layout of `&[Complex<P>]`; lengths/offsets are counted
 *     in amplitudes, not bytes.
 *   - qubit q <-> index bit n-1-q; see include/qip_op.h for the op descriptor.
 *   - every function returns a qipb200_status (0 == OK) and never aborts the
 *     process; the message of the last failure is available through
 *     qipb200_last_error().  (The reference's constructors return
 *     CircuitResult<T>, qip/src/errors.rs:6-22; apply_op* itself panics on
 *     misuse -- here both surface as status codes.)
 *   - there is NO CPU fallback: without a CUDA device qipb200_init() fails
 *     with QIPB200_ERR_CUDA and nothing else can be called.
 *   - a ctx / state handle is not thread-safe (it is the `&mut` of the
 *     reference); distinct handles may be driven from distinct host threads.
 */
#ifndef QIPB200_H
#define QIPB200_H

#include "qip_op.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef enum qipb200_status {
  QIPB200_OK = 0,
  QIPB200_ERR_INVALID_ARG = 1,   /* null pointer, bad enum, malformed op tree            */
  QIPB200_ERR_SIZE_MISMATCH = 2, /* len(dense) != 4^k, swap halves differ, empty indices */
  QIPB200_ERR_BAD_INDEX = 3,     /* qubit index >= n, or repeated                        */
  QIPB200_ERR_CUDA = 4,          /* CUDA runtime/driver error (message has the details)  */
  QIPB200_ERR_COMM = 5,          /* multi-GPU exchange set-up or peer access failure     */
  QIPB200_ERR_OOM = 6,           /* device allocation failed                             */
  QIPB200_ERR_UNSUPPORTED = 7    /* valid request this build cannot serve (e.g. k too large) */
} qipb200_status;

typedef struct qipb200_ctx qipb200_ctx;     /* one CUDA device + stream + scratch         */
typedef struct qipb200_state qipb200_state; /* device-resident 2^n amplitudes (or a shard) */

/* Schedule flags for qipb200_state_apply_schedule / qipb200_calculate_state. */
enum {
  QIPB200_SCHED_DEFAULT = 0u,   /* fusion allowed: sequential PRODUCT of the ops        */
  QIPB200_SCHED_NO_FUSION = 1u  /* one kernel sweep per op, exactly as the reference's
                                   per-entry loop (qip/src/builder.rs:423-514)          */
};

/* ---- library / context ------------------------------------------------------- */

/* ABI version of this header (major*1000 + minor). */
int qipb200_abi_version(void);

/* Create a context bound to CUDA device `device_id` (one process per GPU).
 * Replaces nothing in the reference (it has no device); owns the stream the
 * gate kernels run on.  Fails with QIPB200_ERR_CUDA when no usable sm_100
 * device exists -- there is no CPU path. */
int qipb200_init(qipb200_ctx **ctx, int device_id);
/* One context over SEVERAL devices of this process (n_devices a power of two; device_ids == NULL means 0..n-1):
 * the drop-in for a single-process host such as LocalBuilder::calculate_state_with_init
 * (qip/src/builder.rs:400-519), which has no notion of ranks.  States created on it with qipb200_state_new are
 * sharded over the devices by their top log2(n_devices) index bits; every state call is served by one host thread
 * per device inside the library, the devices map each other with CUDA peer access (NVLink / NVSwitch) and run
 * the same exchange kernels as the one-process-per-GPU path.  upload/download address the whole 2^n vector. */
int qipb200_init_multi(qipb200_ctx **ctx, int n_devices, const int *device_ids);
void qipb200_shutdown(qipb200_ctx *ctx);

/* Message of the last failing call on `ctx` (or, with ctx == NULL, of the last
 * failing call on this thread that had no ctx yet).  Never NULL. */
const char *qipb200_last_error(const qipb200_ctx *ctx);

/* The CUDA stream (a `cudaStream_t`) every kernel of `ctx` is launched on, so that a
 * caller can bracket work with its own CUDA events. */
int qipb200_stream_handle(const qipb200_ctx *ctx, void **stream);

/* Number of this library's kernels launched through `ctx` so far. */
uint64_t qipb200_kernel_launches(const qipb200_ctx *ctx);
/* out4 = { all kernels, fused tile passes, NVLink exchange kernels, reference ops folded into tile passes }. */
int qipb200_launch_stats(const qipb200_ctx *ctx, uint64_t *out4);

/* Generated kernels (absent in the reference): fused tile passes of big states are compiled by NVRTC into
 * kernels specialised to the pass (rustqip_b200/csrc/jit_codegen.cpp); a pass whose kernel is still being compiled
 * in the background runs the generic kernel meanwhile.  With wait != 0 this call blocks until the background
 * compilations have finished.  out4 = { tile passes run by generated kernels, all tile passes (this context),
 * programs compiled so far (process, valid with wait), their total compile time in ms (valid with wait) };
 * `note` (may be NULL) receives the reason the generated path was last declined, if any.
 * Environment: QIPB200_JIT = off | async (default from 22 local qubits) | sync (compile before launching). */
int qipb200_jit_stats(qipb200_ctx *ctx, int wait, double *out4, char *note, size_t note_len);
/* Host-only (no GPU, ctx-free): plan the schedule for an n-qubit single-device state, generate and NVRTC-compile
 * the kernel of every fused pass into the process-wide cache (a later qipb200_state_apply_schedule of the same
 * schedule then starts on generated kernels at once).  out5 = { passes, passes covered by the generator, compiled
 * without error, wall ms, sum of per-program compile ms }; `log` (may be NULL) receives the last compiler message. */
int qipb200_jit_precompile(qip_prec prec, uint32_t n_qubits, const qip_op *ops, size_t n_ops, double *out5, char *log,
                           size_t log_len);

/* Optional device timing by category (absent in the reference): while enabled, every fused tile pass and every
 * NVLink exchange (kernel + its two flag barriers) is bracketed by a CUDA-event pair on the context's stream.
 * profile_read synchronises the stream and returns
 *   out4 = { tile-pass ms, tile passes, exchange ms, exchanges }  since the previous read, then resets. */
int qipb200_profile_enable(qipb200_ctx *ctx, int on);
int qipb200_profile_read(qipb200_ctx *ctx, double *out4);

/* Validate an op exactly as the reference's constructors do
 * (qip/src/state_ops/matrix_ops.rs:12-122: non-empty indices, len(dense)==4^k,
 * sparse row count 2^k and no empty row, equal swap halves, >=1 control) plus
 * index range / distinctness for an n-qubit state.  Needs no GPU (ctx may be NULL). */
int qipb200_validate_op(const qipb200_ctx *ctx, qip_prec prec, uint32_t n_qubits, const qip_op *op);

/* ---- stateless drop-ins for qip_iterators::matrix_ops (HOST buffers) ---------- */

/* qip_iterators::matrix_ops::apply_op (qip-iterators/src/matrix_ops.rs:98-123):
 * output[o] += row(output_offset+o) . input, partners outside
 * [input_offset, input_offset+input_len) read as zero.  Copies both buffers to
 * the device, runs the gate kernel, copies `output` back. */
int qipb200_apply_op(qipb200_ctx *ctx, qip_prec prec, uint32_t n_qubits, const qip_op *op,
                     const void *input, uint64_t input_len, void *output, uint64_t output_len,
                     uint64_t input_offset, uint64_t output_offset);

/* qip_iterators::matrix_ops::apply_op_overwrite (matrix_ops.rs:127-152):
 * same with `=` instead of `+=`; `output` is write-only. */
int qipb200_apply_op_overwrite(qipb200_ctx *ctx, qip_prec prec, uint32_t n_qubits, const qip_op *op,
                               const void *input, uint64_t input_len, void *output,
                               uint64_t output_len, uint64_t input_offset, uint64_t output_offset);

/* qip_iterators::matrix_ops::apply_ops (matrix_ops.rs:158-219).
 *   n_ops == 0 : copy of the overlapping index range (matrix_ops.rs:170-183);
 *   n_ops == 1 : apply_op;
 *   n_ops  > 1 : output += the reference's multi-op row sum (matrix_ops.rs:184-217 with
 *                sum_for_ops_cols, iterators/iterator_mapper.rs:8-31, and MultiOpIterator,
 *                qubit_multi_iterator.rs:38-78), restated AS IT IS: op i reads its row from
 *                the low bits left of the sub-row while columns are composed first-op-high
 *                (SURVEY.md section 8 quirk Q5), so for ops that are not all alike the
 *                result is not their tensor product -- exactly what the reference returns.
 *                Offsets and ragged windows as in apply_op.  2..8 ops, at most 40 indices
 *                in total (else QIPB200_ERR_UNSUPPORTED).  To apply gates one after the
 *                other use a state + qipb200_state_apply_schedule. */
int qipb200_apply_ops(qipb200_ctx *ctx, qip_prec prec, uint32_t n_qubits, const qip_op *ops,
                      size_t n_ops, const void *input, uint64_t input_len, void *output,
                      uint64_t output_len, uint64_t input_offset, uint64_t output_offset);

/* ---- device-resident state: the body of LocalBuilder::calculate_state_with_init
 *      (qip/src/builder.rs:400-519) ------------------------------------------------ */

/* `let mut state = vec![Complex::zero(); 1 << n]` (builder.rs:406); all zero. */
int qipb200_state_new(qipb200_ctx *ctx, qip_prec prec, uint32_t n_qubits, qipb200_state **state);
void qipb200_state_free(qipb200_state *state);

/* `state[initial_index] = Complex::one()` after clearing (builder.rs:421). */
int qipb200_state_set_basis(qipb200_state *state, uint64_t index);

/* Copy `len` amplitudes host<->device starting at amplitude `offset`
 * (the reference returns/accepts the Vec itself, builder.rs:518). */
int qipb200_state_upload(qipb200_state *state, const void *host, uint64_t offset, uint64_t len);
int qipb200_state_download(qipb200_state *state, void *host, uint64_t offset, uint64_t len);

/* One pipeline entry: `apply_op_overwrite(n,&uop,&state,&mut arena,0,0)` followed by
 * the buffer swap (builder.rs:499,514); logically state <- U state.  Stream-ordered. */
int qipb200_state_apply_op(qipb200_state *state, const qip_op *op);

/* The whole fold over the pipeline (builder.rs:423-514) for unitary entries:
 * state <- ops[n_ops-1] ... ops[0] state.  With QIPB200_SCHED_NO_FUSION every op
 * is one sweep; otherwise runs of ops are fused into shared-memory tile passes. */
int qipb200_state_apply_schedule(qipb200_state *state, const qip_op *ops, size_t n_ops,
                                 uint32_t flags);

/* sum |a|^2 over the WHOLE state: prob_magnitude, measurement_ops.rs:11-13.  On a sharded state the call is
 * COLLECTIVE (every rank calls it; the per-rank sums are added through the peers' reduction slots over NVLink)
 * and every rank receives the same total. */
int qipb200_state_norm2(qipb200_state *state, double *out);

/* max over the (local) amplitudes of max(|re_a - re_b|, |im_a - im_b|), computed on the device: the
 * comparison behind the fused-vs-unfused parity checks at sizes no host oracle reaches (two 16 GiB
 * states at N=30).  Both states must live on the same context and have the same shape and layout.
 * Replaces nothing in the reference (its tests compare Vecs on the host). */
int qipb200_state_max_abs_diff(qipb200_state *a, qipb200_state *b, double *out);

/* Block until everything queued on the state's stream has finished. */
int qipb200_state_sync(qipb200_state *state);

/* One call == LocalBuilder::calculate_state_with_init for a unitary pipeline:
 * allocate, set |init_index>, run the schedule, copy the 2^n amplitudes to
 * `host_out` (HOST memory, 2^n complex<prec>).  This is the end-to-end entry
 * bench.py's `e2e` times. */
int qipb200_calculate_state(qipb200_ctx *ctx, qip_prec prec, uint32_t n_qubits, uint64_t init_index,
                            const qip_op *ops, size_t n_ops, uint32_t flags, void *host_out);

/* ---- measurement on the device (qip/src/state_ops/measurement_ops.rs) ----------
 * On a sharded state all four calls are COLLECTIVE: every rank calls with the same arguments and every rank
 * receives the result for the whole 2^n vector (histograms / scalars are summed across the ranks in rank order
 * through peer-mapped reduction slots, so the values are bit-identical on all ranks and can be fed to
 * qipb200_state_collapse as they are).  measure_probs is limited to 16 measured qubits there. */

/* measure_probs (measurement_ops.rs:115-127): out[m] for m in 0..2^n_indices,
 * bit i of m <-> indices[i].  `out` is HOST memory of 2^n_indices doubles. */
int qipb200_state_measure_probs(qipb200_state *state, const uint64_t *indices, uint32_t n_indices,
                                double *out);
/* measure_prob (measurement_ops.rs:44-58). */
int qipb200_state_measure_prob(qipb200_state *state, uint64_t measured, const uint64_t *indices,
                               uint32_t n_indices, double *out);
/* soft_measure (measurement_ops.rs:153-176) with the uniform draw r in [0,1)
 * supplied by the caller (the reference calls rand::random). */
int qipb200_state_soft_measure(qipb200_state *state, const uint64_t *indices, uint32_t n_indices,
                               double r, uint64_t *measured);
/* K draws at once from the state, without changing it: out[j] is what qipb200_state_soft_measure(state, indices,
 * n_indices, r[j], &m) returns for the same state (measurement_ops.rs:153-176 applied K times).  r and out are HOST
 * arrays of n_draws entries; r[j] in [0, 1].  Cost: about one read sweep of the state plus O(n_draws) small gathers,
 * independent of the qubits measured (all n qubits allowed).  COLLECTIVE on a sharded state: every rank passes the
 * same indices and draws and receives the same out[]. */
int qipb200_state_sample(qipb200_state *state, const uint64_t *indices, uint32_t n_indices, const double *r, uint64_t n_draws, uint64_t *out);
/* measure_state (measurement_ops.rs:220-269): zero the amplitudes that
 * contradict `measured`, scale the rest by 1/sqrt(measured_prob); in place. */
int qipb200_state_collapse(qipb200_state *state, const uint64_t *indices, uint32_t n_indices,
                           uint64_t measured, double measured_prob);

/* ---- multi-GPU: the 2^n state sharded by its top log2(world) index bits,
 *      one process per GPU (absent in the reference; its only hook is the
 *      input_offset/output_offset slice model, matrix_ops.rs:74-89) -------------- */

#define QIPB200_IPC_HANDLE_BYTES 64

/* Create rank `rank`'s shard (2^(n - log2 world) amplitudes) of an n-qubit state.
 * world_size must be a power of two. */
int qipb200_state_new_sharded(qipb200_ctx *ctx, qip_prec prec, uint32_t n_qubits, int rank,
                              int world_size, qipb200_state **state);
/* Export this shard's CUDA-IPC handles (amplitude buffer + flag page), each
 * QIPB200_IPC_HANDLE_BYTES long, for the caller to all-gather. */
int qipb200_state_ipc_export(qipb200_state *state, void *amp_handle, void *flag_handle);
/* Import all peers' handles (world_size * QIPB200_IPC_HANDLE_BYTES each, rank order):
 * maps every peer shard over NVLink so exchange kernels can load/store it directly. */
int qipb200_state_ipc_import(qipb200_state *state, const void *amp_handles, const void *flag_handles);
/* Current logical-qubit -> physical-index-bit map of a sharded state (n entries):
 * the exchange pass migrates "hot" qubits to local bits instead of moving them back. */
int qipb200_state_qubit_map(qipb200_state *state, uint32_t *bit_of_qubit);
/* Bytes this rank has pulled/pushed over NVLink so far. */
int qipb200_state_exchange_bytes(qipb200_state *state, uint64_t *bytes);

/* Host-side plan only (no GPU, ctx may be NULL): for each op, report whether a
 * world_size-way sharded n-qubit state needs an exchange to apply it
 * (needs_exchange[i] = number of rank bits the op acts on non-diagonally). */
int qipb200_plan_exchanges(qip_prec prec, uint32_t n_qubits, int world_size, const qip_op *ops,
                           size_t n_ops, uint32_t *needs_exchange);

/* ---- N3: gate-schedule wire format "QIPS" -----------------------------------------
 * The reference's only export is OpenQASM 2.0 (qip/src/qasm.rs:112-184), which drops MAT
 * entries; QIPS carries exactly the `qip_op` records this ABI consumes (byte layout:
 * rustqip_b200/wire.py, rustqip_b200/csrc/wire.cpp).  Host-only: no GPU, no context.
 *
 * parse: builds an owned schedule from `len` bytes; on a malformed buffer returns
 * QIPB200_ERR_INVALID_ARG with a message in errbuf (may be NULL).  The returned records stay valid
 * until qipb200_schedule_free and can be passed to qipb200_state_apply_schedule /
 * qipb200_calculate_state as they are.
 * serialise: returns the number of bytes the schedule needs and writes them when cap suffices
 * (call with buf=NULL to size the buffer); 0 on a malformed op tree. */
typedef struct qipb200_schedule qipb200_schedule;
int qipb200_schedule_parse(const void *buf, size_t len, qipb200_schedule **out, char *errbuf, size_t errlen);
const qip_op *qipb200_schedule_ops(const qipb200_schedule *s, size_t *n_ops, uint32_t *n_qubits, qip_prec *prec);
void qipb200_schedule_free(qipb200_schedule *s);
size_t qipb200_schedule_serialise(qip_prec prec, uint32_t n_qubits, const qip_op *ops, size_t n_ops, void *buf,
                                  size_t cap);

/* State files "QIPA" (checkpoint / resume; the reference keeps its state in two Vecs for the duration of one call,
 * qip/src/builder.rs:406-407, and has no equivalent): one file per shard -- 40-byte header {magic "QIPA", version 1,
 * prec, n_qubits, rank, world, first_index, n_amplitudes} followed by the shard's amplitudes in canonical index
 * order, streamed through a 64 MiB bounce buffer.  load checks the header against the target state.  On a
 * multi-device state (qipb200_init_multi) the shards go to "<path>.<rank>".  Byte-compatible with
 * rustqip_b200.wire.dump_state / load_state. */
int qipb200_state_save(qipb200_state *state, const char *path);
int qipb200_state_load(qipb200_state *state, const char *path);

#ifdef __cplusplus
}
#endif
#endif /* QIPB200_H */
