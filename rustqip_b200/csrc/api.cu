// api.cu -- the extern "C" boundary of libqipb200 (include/qipb200.h).
//
// Host runtime above the kernels: owns the device amplitude buffer and the gate
// schedule, exactly the role of the fold in LocalBuilder::calculate_state_with_init
// (qip/src/builder.rs:400-519).  No CPU fallback: every compute entry needs a
// context, and a context needs a CUDA device.
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <exception>
#include <new>
#include <thread>
#include <string>
#include <vector>

#include "../../include/qipb200.h"
#include "dist.cuh"
#include "kernels.cuh"
#include "opcompile.h"
#include "schedule.h"
#include "tile.cuh"
#include "jit_codegen.h"
#include "state.h"

using namespace qipb200;

namespace {

thread_local std::string g_tls_err = "";

int set_err(const qipb200_ctx *ctx, int status, const std::string &msg) {
  if (ctx)
    const_cast<qipb200_ctx *>(ctx)->err = msg;
  else
    g_tls_err = msg;
  return status;
}

int cuda_fail(const qipb200_ctx *ctx, cudaError_t e, const char *what) {
  std::string m = std::string(what) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")";
  cudaGetLastError();  // clear sticky-free errors
  return set_err(ctx, e == cudaErrorMemoryAllocation ? QIPB200_ERR_OOM : QIPB200_ERR_CUDA, m);
}

#define CU(ctx, call)                                          \
  do {                                                         \
    cudaError_t e__ = (call);                                  \
    if (e__ != cudaSuccess) return cuda_fail(ctx, e__, #call); \
  } while (0)

int grow(qipb200_ctx *ctx, void **p, size_t *have, size_t need) {
  if (*have >= need) return QIPB200_OK;
  if (*p) {
    cudaStreamSynchronize(ctx->stream);
    cudaFree(*p);
    *p = nullptr;
    *have = 0;
  }
  cudaError_t e = cudaMalloc(p, need);
  if (e != cudaSuccess) return cuda_fail(ctx, e, "cudaMalloc(staging)");
  *have = need;
  return QIPB200_OK;
}

// No C++ exception may cross the C boundary (the library allocates through std::vector / std::string):
// an allocation failure becomes QIPB200_ERR_OOM, anything else QIPB200_ERR_INVALID_ARG with its message.
template <typename F>
int guarded(const qipb200_ctx *ctx, F f) {
  try {
    return f();
  } catch (const std::bad_alloc &) {
    return set_err(ctx, QIPB200_ERR_OOM, "out of host memory");
  } catch (const std::exception &e) {
    return set_err(ctx, QIPB200_ERR_INVALID_ARG, std::string("internal error: ") + e.what());
  }
}

// Run f(shard, rank) on every shard of a multi-device state, one host thread per device (the shards are
// ordinary sharded states: their exchange kernels wait for each other on the GPUs, so they must be driven
// concurrently, exactly as the one-process-per-GPU model drives them).  First failing status wins.
template <typename F>
int each_shard(qipb200_state *p, F f) {
  const size_t G = p->shards.size();
  std::vector<int> st(G, QIPB200_OK);
  auto run = [&](size_t r) {
    try {
      st[r] = f(p->shards[r], (int)r);
    } catch (const std::bad_alloc &) {
      st[r] = set_err(p->shards[r]->ctx, QIPB200_ERR_OOM, "out of host memory");
    } catch (const std::exception &e) {
      st[r] = set_err(p->shards[r]->ctx, QIPB200_ERR_INVALID_ARG, std::string("internal error: ") + e.what());
    }
  };
  std::vector<std::thread> th;
  bool spawn_failed = false;
  try {
    th.reserve(G);
    for (size_t r = 1; r < G; ++r) th.emplace_back(run, r);
  } catch (const std::exception &) {  // no thread for some device: the started ones run into the flag barriers' timeout
    spawn_failed = true;
  }
  if (!spawn_failed) run(0);
  for (std::thread &t : th) t.join();
  if (spawn_failed) return set_err(p->ctx, QIPB200_ERR_OOM, "could not start one host thread per device");
  for (size_t r = 0; r < G; ++r)
    if (st[r] != QIPB200_OK) return set_err(p->ctx, st[r], p->shards[r]->ctx->err);
  return QIPB200_OK;
}

bool is_pow2(int x) { return x > 0 && (x & (x - 1)) == 0; }
int ilog2(int x) {
  int l = 0;
  while ((1 << l) < x) ++l;
  return l;
}

}  // namespace

// ===================================================================================
// library / context
// ===================================================================================

extern "C" int qipb200_abi_version(void) { return 1000; }

static int init_device_ctx(qipb200_ctx **out, int device_id);

extern "C" int qipb200_init(qipb200_ctx **out, int device_id) {
  if (!out) return set_err(nullptr, QIPB200_ERR_INVALID_ARG, "qipb200_init: ctx out-pointer is NULL");
  *out = nullptr;
  return guarded(nullptr, [&]() { return init_device_ctx(out, device_id); });
}

extern "C" int qipb200_init_multi(qipb200_ctx **out, int n_devices, const int *device_ids) {
  if (!out) return set_err(nullptr, QIPB200_ERR_INVALID_ARG, "qipb200_init_multi: ctx out-pointer is NULL");
  *out = nullptr;
  if (!is_pow2(n_devices) || n_devices > kMaxWorld)
    return set_err(nullptr, QIPB200_ERR_INVALID_ARG, "qipb200_init_multi: n_devices must be a power of two <= 16");
  return guarded(nullptr, [&]() {
    qipb200_ctx *parent = new qipb200_ctx();
    for (int i = 0; i < n_devices; ++i) {
      const int dev = device_ids ? device_ids[i] : i;
      for (int j = 0; j < i; ++j)
        if (parent->children[j]->device == dev) {
          qipb200_shutdown(parent);
          return set_err(nullptr, QIPB200_ERR_INVALID_ARG, "qipb200_init_multi: a device is listed twice");
        }
      qipb200_ctx *c = nullptr;
      int st = init_device_ctx(&c, dev);
      if (st != QIPB200_OK) {
        qipb200_shutdown(parent);
        return st;  // message already in the thread-local slot
      }
      c->parent = parent;
      parent->children.push_back(c);
    }
    // every device maps every other one (NVLink / NVSwitch peer access: the exchange kernels load and store
    // the partner's shard directly)
    for (int i = 0; i < n_devices; ++i) {
      cudaSetDevice(parent->children[i]->device);
      for (int j = 0; j < n_devices; ++j) {
        if (i == j) continue;
        int can = 0;
        cudaDeviceCanAccessPeer(&can, parent->children[i]->device, parent->children[j]->device);
        cudaError_t e = can ? cudaDeviceEnablePeerAccess(parent->children[j]->device, 0) : cudaErrorPeerAccessUnsupported;
        if (e == cudaErrorPeerAccessAlreadyEnabled) {
          cudaGetLastError();
          e = cudaSuccess;
        }
        if (e != cudaSuccess) {
          int st = cuda_fail(nullptr, e, "cudaDeviceEnablePeerAccess");
          qipb200_shutdown(parent);
          return st == QIPB200_ERR_CUDA ? QIPB200_ERR_COMM : st;
        }
      }
    }
    parent->device = parent->children[0]->device;
    parent->sm_count = parent->children[0]->sm_count;
    *out = parent;
    return (int)QIPB200_OK;
  });
}

static int init_device_ctx(qipb200_ctx **out, int device_id) {
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    cudaGetLastError();
    return set_err(nullptr, QIPB200_ERR_CUDA,
                   std::string("qipb200_init: no CUDA device (") + cudaGetErrorString(e) +
                       "); libqipb200 has no CPU path");
  }
  if (device_id < 0 || device_id >= count)
    return set_err(nullptr, QIPB200_ERR_INVALID_ARG, "qipb200_init: device_id out of range");
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device_id);
  if (e != cudaSuccess) return cuda_fail(nullptr, e, "cudaGetDeviceProperties");
  if (prop.major != 10)
    return set_err(nullptr, QIPB200_ERR_CUDA,
                   std::string("qipb200_init: device '") + prop.name +
                       "' is not sm_100 (Blackwell B200); this library ships sm_100a code only");
  e = cudaSetDevice(device_id);
  if (e != cudaSuccess) return cuda_fail(nullptr, e, "cudaSetDevice");
  qipb200_ctx *ctx = new (std::nothrow) qipb200_ctx();
  if (!ctx) return set_err(nullptr, QIPB200_ERR_OOM, "qipb200_init: out of host memory");
  ctx->device = device_id;
  ctx->sm_count = prop.multiProcessorCount;
  e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaMalloc((void **)&ctx->d_scalar, 64);
  if (e != cudaSuccess) {
    int st = cuda_fail(nullptr, e, "qipb200_init");
    delete ctx;
    return st;
  }
  *out = ctx;
  return QIPB200_OK;
}

extern "C" void qipb200_shutdown(qipb200_ctx *ctx) {
  if (!ctx) return;
  if (!ctx->children.empty() || (!ctx->stream && !ctx->d_scalar)) {  // multi-device parent: owns its children
    for (size_t i = 0; i < ctx->children.size(); ++i) qipb200_shutdown(ctx->children[i]);
    delete ctx;
    return;
  }
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  if (ctx->d_in) cudaFree(ctx->d_in);
  if (ctx->d_out) cudaFree(ctx->d_out);
  if (ctx->d_scalar) cudaFree(ctx->d_scalar);
  if (ctx->pool_buf) cudaFree(ctx->pool_buf);
  if (ctx->h_pinned) cudaFreeHost(ctx->h_pinned);
  for (int cat = 0; cat < 2; ++cat)
    for (size_t i = 0; i < ctx->prof_events[cat].size(); ++i) {
      cudaEventDestroy(ctx->prof_events[cat][i].first);
      cudaEventDestroy(ctx->prof_events[cat][i].second);
    }
  for (size_t i = 0; i < ctx->prof_pool.size(); ++i) cudaEventDestroy(ctx->prof_pool[i]);
  jit_unload(&ctx->jit_loaded);
  for (int i = 0; i < 2; ++i) {
    if (ctx->ev_pass[i]) cudaEventDestroy(ctx->ev_pass[i]);
    if (ctx->ev_exch[i]) cudaEventDestroy(ctx->ev_exch[i]);
  }
  if (ctx->stream2) cudaStreamDestroy(ctx->stream2);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

extern "C" const char *qipb200_last_error(const qipb200_ctx *ctx) {
  return ctx ? ctx->err.c_str() : g_tls_err.c_str();
}

extern "C" int qipb200_stream_handle(const qipb200_ctx *ctx, void **stream) {
  if (!ctx || !stream) return set_err(ctx, QIPB200_ERR_INVALID_ARG, "stream_handle: NULL argument");
  *stream = (void *)(ctx->children.empty() ? ctx->stream : ctx->children[0]->stream);
  return QIPB200_OK;
}

extern "C" uint64_t qipb200_kernel_launches(const qipb200_ctx *ctx) {
  if (!ctx) return 0;
  uint64_t n = ctx->launches;
  for (size_t i = 0; i < ctx->children.size(); ++i) n += ctx->children[i]->launches;
  return n;
}

extern "C" int qipb200_launch_stats(const qipb200_ctx *ctx, uint64_t *out4) {
  if (!ctx || !out4) return set_err(ctx, QIPB200_ERR_INVALID_ARG, "launch_stats: NULL argument");
  out4[0] = ctx->launches;
  out4[1] = ctx->tile_launches;
  out4[2] = ctx->exchange_launches;
  out4[3] = ctx->fused_gates;
  for (size_t i = 0; i < ctx->children.size(); ++i) {  // multi-device context: summed over the devices
    const qipb200_ctx *c = ctx->children[i];
    out4[0] += c->launches;
    out4[1] += c->tile_launches;
    out4[2] += c->exchange_launches;
    out4[3] += i == 0 ? c->fused_gates : 0;  // every device folds the same gates: count them once
  }
  return QIPB200_OK;
}

// Host-only (no GPU, no context): plan `ops` for an n-qubit single-device state, generate the specialised source
// of every fused pass and compile it with NVRTC for sm_100a.  out[0] = passes planned, out[1] = passes the
// generator covered, out[2] = of those compiled without error, out[3] = total NVRTC wall time (ms, all passes in
// parallel on the worker pool), out[4] = sum of the per-program compile times (ms).
extern "C" int qipb200_jit_precompile(qip_prec prec, uint32_t n_qubits, const qip_op *ops, size_t n_ops, double *out5,
                                      char *log, size_t log_len) {
  if (!out5 || (!ops && n_ops)) return set_err(nullptr, QIPB200_ERR_INVALID_ARG, "jit_precompile: NULL argument");
  for (int i = 0; i < 5; ++i) out5[i] = 0.0;
  if (log && log_len) log[0] = 0;
  std::string why;
  if (!jit_available(&why) && why.find("driver") == std::string::npos) {  // the driver is only needed to LAUNCH
    if (log && log_len) snprintf(log, log_len, "%s", why.c_str());
    return set_err(nullptr, QIPB200_ERR_UNSUPPORTED, why);
  }
  std::vector<FlatOp> flat(n_ops);
  for (size_t i = 0; i < n_ops; ++i) {
    std::string err;
    int st = compile_op(&ops[i], prec, n_qubits, &flat[i], &err);
    if (st != QIPB200_OK) return set_err(nullptr, st, err);
  }
  const PlanConfig cfg = default_plan_config(prec, n_qubits);
  std::vector<PlanStep> steps;
  plan_passes(flat, n_qubits, prec, cfg, &steps);
  std::vector<std::string> sources;
  for (size_t i = 0; i < steps.size(); ++i) {
    if (!steps[i].is_pass) continue;
    out5[0] += 1;
    JitProgram prog;
    if (!jit_generate(steps[i].pass, prec, &prog, &why)) {
      if (log && log_len) snprintf(log, log_len, "declined: %s", why.c_str());
      continue;
    }
    out5[1] += 1;
    sources.push_back(prog.source);
  }
  const auto t0 = std::chrono::steady_clock::now();
  for (size_t i = 0; i < sources.size(); ++i) (void)jit_request(sources[i], false);
  for (size_t i = 0; i < sources.size(); ++i) {
    std::shared_ptr<const JitCubin> c = jit_request(sources[i], true);
    if (c && c->ok) {
      out5[2] += 1;
      out5[4] += c->compile_ms;
    } else if (log && log_len && c) {
      snprintf(log, log_len, "%s", c->log.c_str());
    }
  }
  out5[3] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  if (getenv("QIPB200_JIT_CACHE_DIR") && log && log_len && !log[0]) {
    uint64_t n_disk = 0;
    jit_wait_all(nullptr, nullptr, &n_disk);
    snprintf(log, log_len, "disk cache: %llu programs loaded from QIPB200_JIT_CACHE_DIR so far in this process", (unsigned long long)n_disk);
  }
  return QIPB200_OK;
}

extern "C" int qipb200_jit_stats(qipb200_ctx *ctx, int wait, double *out4, char *note, size_t note_len) {
  if (!ctx || !out4) return set_err(ctx, QIPB200_ERR_INVALID_ARG, "jit_stats: NULL argument");
  uint64_t n = 0;
  double ms = 0.0;
  if (wait) jit_wait_all(&n, &ms);
  out4[0] = (double)ctx->jit_launches;
  out4[1] = (double)ctx->tile_launches;
  for (size_t i = 0; i < ctx->children.size(); ++i) {
    out4[0] += (double)ctx->children[i]->jit_launches;
    out4[1] += (double)ctx->children[i]->tile_launches;
    if (!ctx->children[i]->jit_note.empty()) ctx->jit_note = ctx->children[i]->jit_note;
  }
  out4[2] = (double)n;
  out4[3] = ms;
  if (note && note_len) snprintf(note, note_len, "%s", ctx->jit_note.c_str());
  return QIPB200_OK;
}

extern "C" int qipb200_profile_enable(qipb200_ctx *ctx, int on) {
  if (!ctx) return set_err(nullptr, QIPB200_ERR_INVALID_ARG, "profile_enable: ctx is NULL");
  ctx->profile = on != 0;
  for (size_t i = 0; i < ctx->children.size(); ++i) ctx->children[i]->profile = on != 0;
  return QIPB200_OK;
}

extern "C" int qipb200_profile_read(qipb200_ctx *ctx, double *out4) {
  if (!ctx || !out4) return set_err(ctx, QIPB200_ERR_INVALID_ARG, "profile_read: NULL argument");
  if (!ctx->children.empty()) {  // multi-device context: the first device's timings (all devices run the same steps)
    for (size_t i = 1; i < ctx->children.size(); ++i) {
      double drop[4];
      qipb200_profile_read(ctx->children[i], drop);
    }
    return qipb200_profile_read(ctx->children[0], out4);
  }
  CU(ctx, cudaSetDevice(ctx->device));
  CU(ctx, cudaStreamSynchronize(ctx->stream));
  for (int cat = 0; cat < 2; ++cat) {
    double ms = 0.0;
    for (size_t i = 0; i < ctx->prof_events[cat].size(); ++i) {
      float t = 0.f;
      if (cudaEventElapsedTime(&t, ctx->prof_events[cat][i].first, ctx->prof_events[cat][i].second) == cudaSuccess) ms += t;
      ctx->prof_pool.push_back(ctx->prof_events[cat][i].first);
      ctx->prof_pool.push_back(ctx->prof_events[cat][i].second);
    }
    out4[2 * cat] = ms;
    double n = 0.0;
    for (size_t i = 0; i < ctx->prof_events[cat].size(); ++i) n += ctx->prof_events[cat][i].weight;
    out4[2 * cat + 1] = n;
    ctx->prof_events[cat].clear();
  }
  return QIPB200_OK;
}

extern "C" int qipb200_validate_op(const qipb200_ctx *ctx, qip_prec prec, uint32_t n_qubits, const qip_op *op) {
  return guarded(ctx, [&]() -> int {
    std::string err;
    int st = validate_op(op, prec, n_qubits, &err);
    if (st != QIPB200_OK) return set_err(ctx, st, err);
    return (int)QIPB200_OK;
  });
}

// ===================================================================================
// stateless drop-ins (host buffers)
// ===================================================================================

namespace {

int host_apply(qipb200_ctx *ctx, qip_prec prec, uint32_t n, const qip_op *op, const void *input,
               uint64_t input_len, void *output, uint64_t output_len, uint64_t input_offset,
               uint64_t output_offset, bool accumulate) {
  if (!ctx) return set_err(nullptr, QIPB200_ERR_INVALID_ARG, "ctx is NULL (call qipb200_init first; there is no CPU path)");
  if (!ctx->children.empty()) {  // a multi-device context serves the host-buffer drop-ins on its first device
    qipb200_ctx *parent = ctx;
    int st = host_apply(parent->children[0], prec, n, op, input, input_len, output, output_len, input_offset, output_offset, accumulate);
    if (st != QIPB200_OK) parent->err = parent->children[0]->err;
    return st;
  }
  if ((!input && input_len) || (!output && output_len))
    return set_err(ctx, QIPB200_ERR_INVALID_ARG, "apply_op: NULL amplitude buffer");
  if (n > 40 || input_len > (1ull << 40) || output_len > (1ull << 40))  // keeps len * amp_bytes far from wrapping
    return set_err(ctx, QIPB200_ERR_SIZE_MISMATCH, "apply_op: buffer length out of range");
  FlatOp f;
  std::string err;
  int st = compile_op(op, prec, n, &f, &err);
  if (st != QIPB200_OK) return set_err(ctx, st, err);
  CU(ctx, cudaSetDevice(ctx->device));
  const size_t ab = amp_bytes(prec);
  if ((st = grow(ctx, &ctx->d_in, &ctx->d_in_bytes, std::max<size_t>(input_len * ab, 16))) != QIPB200_OK) return st;
  if ((st = grow(ctx, &ctx->d_out, &ctx->d_out_bytes, std::max<size_t>(output_len * ab, 16))) != QIPB200_OK) return st;
  if (input_len) CU(ctx, cudaMemcpyAsync(ctx->d_in, input, input_len * ab, cudaMemcpyHostToDevice, ctx->stream));
  if (accumulate && output_len)
    CU(ctx, cudaMemcpyAsync(ctx->d_out, output, output_len * ab, cudaMemcpyHostToDevice, ctx->stream));
  CU(ctx, launch_gather(prec, f, n, ctx->d_in, input_len, input_offset, ctx->d_out, output_len, output_offset,
                        accumulate, ctx->stream, &ctx->launches));
  if (output_len) CU(ctx, cudaMemcpyAsync(output, ctx->d_out, output_len * ab, cudaMemcpyDeviceToHost, ctx->stream));
  CU(ctx, cudaStreamSynchronize(ctx->stream));
  return QIPB200_OK;
}

}  // namespace

extern "C" int qipb200_apply_op(qipb200_ctx *ctx, qip_prec prec, uint32_t n, const qip_op *op, const void *input,
                                uint64_t input_len, void *output, uint64_t output_len, uint64_t input_offset,
                                uint64_t output_offset) {
  return guarded(ctx, [&]() { return host_apply(ctx, prec, n, op, input, input_len, output, output_len, input_offset, output_offset, true); });
}

extern "C" int qipb200_apply_op_overwrite(qipb200_ctx *ctx, qip_prec prec, uint32_t n, const qip_op *op,
                                          const void *input, uint64_t input_len, void *output,
                                          uint64_t output_len, uint64_t input_offset, uint64_t output_offset) {
  return guarded(ctx, [&]() { return host_apply(ctx, prec, n, op, input, input_len, output, output_len, input_offset, output_offset, false); });
}

// ===================================================================================
// device-resident state
// ===================================================================================

namespace {

int state_alloc(qipb200_ctx *ctx, qip_prec prec, uint32_t n, int rank, int world, qipb200_state **out) {
  if (!ctx) return set_err(nullptr, QIPB200_ERR_INVALID_ARG, "ctx is NULL (call qipb200_init first; there is no CPU path)");
  if (!out) return set_err(ctx, QIPB200_ERR_INVALID_ARG, "state out-pointer is NULL");
  *out = nullptr;
  if (prec != QIP_F32 && prec != QIP_F64) return set_err(ctx, QIPB200_ERR_INVALID_ARG, "precision must be QIP_F32 or QIP_F64");
  if (!is_pow2(world) || world > kMaxWorld || rank < 0 || rank >= world)
    return set_err(ctx, QIPB200_ERR_INVALID_ARG, "world_size must be a power of two <= 16 and 0 <= rank < world_size");
  const int g = ilog2(world);
  if (n == 0 || n > 40 || (int)n - g < 2 * (world > 1))
    return set_err(ctx, QIPB200_ERR_INVALID_ARG, "n_qubits out of range for this world size");
  CU(ctx, cudaSetDevice(ctx->device));
  qipb200_state *s = new (std::nothrow) qipb200_state();
  if (!s) return set_err(ctx, QIPB200_ERR_OOM, "out of host memory");
  s->ctx = ctx;
  s->prec = prec;
  s->n = n;
  s->n_local = n - g;
  s->rank = rank;
  s->world = world;
  s->bytes = amp_bytes(prec) << s->n_local;
  s->phys_of_logical.resize(n);
  for (uint32_t b = 0; b < n; ++b) s->phys_of_logical[b] = b;
  cudaError_t e = cudaSuccess;
  if (world == 1 && ctx->pool_buf && ctx->pool_bytes == s->bytes) {  // the buffer a freed state of this size left behind
    s->buf = ctx->pool_buf;
    ctx->pool_buf = nullptr;
    ctx->pool_bytes = 0;
  } else {
    // a sharded state carries the staging area of the push exchange behind its amplitudes: one allocation, so the
    // one CUDA-IPC handle (or peer pointer) of the shard covers both
    // (opt-in, QIPB200_STAGED_EXCHANGE=1: measured r2h on 2 x B200 -- in-place pair exchange 16.1 ms per migration,
    // stand-alone push + copy 20.5 ms, push fused into the last pass +4.0 ms on that pass and a 14.3 ms tail: SM-issued
    // NVLink traffic tops out near 535-600 GB/s per direction whichever way it is issued, so the variant that moves
    // the fewest bytes locally wins)
    s->has_stage = world > 1 && getenv("QIPB200_STAGED_EXCHANGE") != nullptr;
    e = cudaMalloc(&s->buf, s->has_stage ? 2 * s->bytes : s->bytes);
  }
  if (e == cudaSuccess) e = cudaMemsetAsync(s->buf, 0, s->bytes, ctx->stream);
  if (e == cudaSuccess && world > 1) {
    e = cudaMalloc((void **)&s->flags, kFlagAllocBytes);  // flag page + reduction slot (dist.cuh)
    if (e == cudaSuccess) e = cudaMemsetAsync(s->flags, 0, kFlagAllocBytes, ctx->stream);
  }
  if (e != cudaSuccess) {
    int st = cuda_fail(ctx, e, "qipb200_state_new");
    if (s->buf) cudaFree(s->buf);
    if (s->flags) cudaFree(s->flags);
    delete s;
    return st;
  }
  *out = s;
  return QIPB200_OK;
}

bool layout_is_identity(const qipb200_state *s) {
  for (uint32_t b = 0; b < s->n; ++b)
    if (s->phys_of_logical[b] != b) return false;
  return true;
}

int check_barrier_error(qipb200_state *s) {
  uint32_t flag = 0;
  CU(s->ctx, cudaMemcpyAsync(&flag, s->flags + kFlagErrorSlot, sizeof(flag), cudaMemcpyDeviceToHost, s->ctx->stream));
  CU(s->ctx, cudaStreamSynchronize(s->ctx->stream));
  if (flag) return set_err(s->ctx, QIPB200_ERR_COMM, "multi-GPU flag barrier timed out (a peer rank is not participating)");
  return QIPB200_OK;
}

}  // namespace
namespace qipb200 {
int join_halves(qipb200_state *s);
bool overlap_exchange_enabled();
}
namespace {

// Swap physical rank bit R (>= n_local) with local bit l.
// Protocol (push through staging, dist.cu): [barrier] every rank pushes the half it gives away (bit l == !rb) into
// the partner's staging area [barrier] every rank copies its own staging half into the slots it gave away.  When the
// last tile pass before the exchange already pushed the half (s->send_stage == 2, schedule.cu) only the tail runs.
// Default (no staging area): the in-place pair exchange (k_pair_exchange), which measured fastest (see state_alloc).
int exchange_bits(qipb200_state *s, uint32_t R, uint32_t l) {
  qipb200_ctx *ctx = s->ctx;
  if (!s->ipc_ready)
    return set_err(ctx, QIPB200_ERR_COMM, "sharded state: peers not mapped (call qipb200_state_ipc_import)");
  if (s->halves_pending) {  // an overlapped migration is still in flight on the second stream
    int stj = join_halves(s);
    if (stj != QIPB200_OK) return stj;
  }
  const uint32_t r = R - s->n_local;
  const int partner = s->rank ^ (1 << r);
  const int rb = (s->rank >> r) & 1;
  {
    ProfileScope prof(ctx, 1);
    if (s->has_stage) {
      const int give = 1 - rb;
      char *my_stage = (char *)s->buf + s->bytes;
      char *peer_stage = (char *)s->peer_buf[partner] + s->bytes;
      if (s->send_stage && (s->send_R != R || s->send_l != l))
        return set_err(ctx, QIPB200_ERR_COMM, "internal: the tile pass pushed a different half than the exchange needs");
      if (s->send_stage < 1)
        CU(ctx, launch_flag_barrier(s->peer_flags.data(), s->flags, s->rank, s->world, ++s->epoch,
                                    s->flags + kFlagErrorSlot, ctx->stream, &ctx->launches));
      if (s->send_stage < 2) {
        static const bool use_ce = []() {
          const char *e = getenv("QIPB200_STAGED_EXCHANGE");
          return e && !strcmp(e, "ce");
        }();
        if (use_ce) {
          // the give-half as a strided copy on the copy engines: rows of 2^l amplitudes every 2^(l+1)
          const size_t ab = amp_bytes(s->prec);
          const size_t width = ab << l, pitch = ab << (l + 1);
          const size_t height = (size_t)1 << (s->n_local - 1 - l);
          const char *src = (const char *)s->buf + ((size_t)give << l) * ab;
          char *dst = peer_stage + ((size_t)(1 - give) << l) * ab;
          if (pitch <= ((size_t)1 << 30) && height > 1) {
            CU(ctx, cudaMemcpy2DAsync(dst, pitch, src, pitch, width, height, cudaMemcpyDeviceToDevice, ctx->stream));
          } else {
            for (size_t r = 0; r < height; ++r)
              CU(ctx, cudaMemcpyAsync(dst + r * pitch, src + r * pitch, width, cudaMemcpyDeviceToDevice, ctx->stream));
          }
        } else {
          CU(ctx, launch_copy_half(s->prec, s->buf, peer_stage, s->n_local, l, give, true, ctx->stream, &ctx->launches));
        }
      }
      s->send_stage = 0;
      CU(ctx, launch_flag_barrier(s->peer_flags.data(), s->flags, s->rank, s->world, ++s->epoch,
                                  s->flags + kFlagErrorSlot, ctx->stream, &ctx->launches));
      CU(ctx, launch_copy_half(s->prec, my_stage, s->buf, s->n_local, l, give, false, ctx->stream, &ctx->launches));
    } else {
      uint32_t s_bit = s->n_local - 1;
      if (s_bit == l) s_bit = s->n_local - 2;
      CU(ctx, launch_flag_barrier(s->peer_flags.data(), s->flags, s->rank, s->world, ++s->epoch,
                                  s->flags + kFlagErrorSlot, ctx->stream, &ctx->launches));
      CU(ctx, launch_pair_exchange(s->prec, s->buf, s->peer_buf[partner], s->n_local, l, s_bit, rb, ctx->stream,
                                   &ctx->launches));
      CU(ctx, launch_flag_barrier(s->peer_flags.data(), s->flags, s->rank, s->world, ++s->epoch,
                                  s->flags + kFlagErrorSlot, ctx->stream, &ctx->launches));
    }
    ++ctx->exchange_launches;
  }
  s->exchange_bytes += (uint64_t)amp_bytes(s->prec) << (s->n_local - 1);
  // update the map: the logical bits living at R and l trade places
  for (uint32_t b = 0; b < s->n; ++b) {
    if (s->phys_of_logical[b] == R)
      s->phys_of_logical[b] = l;
    else if (s->phys_of_logical[b] == l)
      s->phys_of_logical[b] = R;
  }
  return QIPB200_OK;
}

// Swap two physical bits (any kind) so that the layout can be restored.
int swap_physical_bits(qipb200_state *s, uint32_t p, uint32_t q) {
  qipb200_ctx *ctx = s->ctx;
  if (p == q) return QIPB200_OK;
  if (p < q) std::swap(p, q);  // p > q
  const uint32_t nl = s->n_local;
  if (p < nl) {
    CU(ctx, launch_bitswap(s->prec, s->buf, nl, 0, q, p, ctx->stream, &ctx->launches));
    for (uint32_t b = 0; b < s->n; ++b) {
      if (s->phys_of_logical[b] == p)
        s->phys_of_logical[b] = q;
      else if (s->phys_of_logical[b] == q)
        s->phys_of_logical[b] = p;
    }
    return QIPB200_OK;
  }
  if (q < nl) return exchange_bits(s, p, q);
  // both rank bits: route through a local bit
  const uint32_t l = nl - 1;
  int st;
  if ((st = exchange_bits(s, p, l)) != QIPB200_OK) return st;
  if ((st = exchange_bits(s, q, l)) != QIPB200_OK) return st;
  return exchange_bits(s, p, l);
}

int restore_layout(qipb200_state *s) {
  // an unsharded state whose qubits were rotated through the low positions (schedule.cu: run_rotating): many displaced
  // bits -- swap-only tile passes instead of one half-sweep per transposition
  if (s->world == 1 && s->n_local >= 6 && rotate_enabled()) return restore_layout_planned(s);
  for (int p = (int)s->n - 1; p >= 0; --p) {
    const uint32_t where = s->phys_of_logical[p];
    if (where == (uint32_t)p) continue;
    int st = swap_physical_bits(s, (uint32_t)p, where);
    if (st != QIPB200_OK) return st;
  }
  return QIPB200_OK;
}

}  // namespace

namespace qipb200 {

// Non-diagonal target bits of a compiled op (the ones that must be local).
static void nondiag_bits(const FlatOp &f, std::vector<uint32_t> *out) {
  out->clear();
  switch (f.cls) {
    case CLASS_DENSE:
    case CLASS_FLIP:
      *out = f.tgt_sorted;
      break;
    case CLASS_BITSWAP:
      for (size_t i = 0; i < f.swaps.size(); ++i) {
        out->push_back(f.swaps[i].first);
        out->push_back(f.swaps[i].second);
      }
      break;
    case CLASS_GENERAL:
      for (uint32_t j = f.nc; j < f.k; ++j) out->push_back(f.idx_bits[j]);
      break;
    default:
      break;
  }
}

// Restrict a compiled op (physical bits, non-diagonal targets all local) to this rank:
// controls held by the rank index either vanish or switch the op off; diagonal bits held
// by the rank index select a slice of the diagonal.  No communication.  *skip = true when
// the op is the identity on this rank.
int restrict_to_rank(const qipb200_state *s, const FlatOp &f_in, FlatOp *out, bool *skip) {
  return restrict_to_rank_as(s, s->rank, f_in, out, skip);
}

// ... as rank `rank` of this state's world would see the op (rank == world - 1: every rank-held bit is 1)
int restrict_to_rank_as(const qipb200_state *s, int rank, const FlatOp &f_in, FlatOp *out, bool *skip) {
  restrict_flat_op(f_in, s->n_local, rank, out, skip);  // opcompile.cpp
  return QIPB200_OK;
}

// Launch the per-gate kernel of an op whose bits are all local (after restrict_to_rank).
int launch_local_op(qipb200_state *s, const FlatOp &f) {
  qipb200_ctx *ctx = s->ctx;
  const uint32_t nl = s->n_local;
  const uint64_t cm = f.ctrl_mask;
  switch (f.cls) {
    case CLASS_IDENTITY:
      return QIPB200_OK;
    case CLASS_DIAGONAL:
      if (__builtin_popcountll(cm) > kMaxIns) break;
      if (f.diag_bits.size() <= (size_t)kMaxDiagParamK) {
        CU(ctx, launch_diag(s->prec, s->buf, nl, cm, f.diag_bits, f.diag, ctx->stream, &ctx->launches));
        return QIPB200_OK;
      }
      if (f.diag_bits.size() <= 10) {
        CU(ctx, launch_diag_wide(s->prec, s->buf, nl, cm, f.diag_bits, f.diag, ctx->stream, &ctx->launches));
        return QIPB200_OK;
      }
      break;
    case CLASS_FLIP:
      CU(ctx, launch_flip(s->prec, s->buf, nl, cm, f.tgt_sorted[0], ctx->stream, &ctx->launches));
      return QIPB200_OK;
    case CLASS_BITSWAP:
      for (size_t i = 0; i < f.swaps.size(); ++i)
        CU(ctx, launch_bitswap(s->prec, s->buf, nl, cm, f.swaps[i].first, f.swaps[i].second, ctx->stream,
                               &ctx->launches));
      return QIPB200_OK;
    case CLASS_DENSE:
      if (f.tgt_sorted.size() <= (size_t)kMaxRegK &&
          __builtin_popcountll(cm) + f.tgt_sorted.size() <= (size_t)kMaxIns) {
        CU(ctx, launch_dense(s->prec, s->buf, nl, f, ctx->stream, &ctx->launches));
        return QIPB200_OK;
      }
      // k = 5..10 in place (the reference applies any k through the same row loop, qubit_iterators.rs:23-55)
      if (f.tgt_sorted.size() >= 5 && f.tgt_sorted.size() <= 10 &&
          __builtin_popcountll(cm) + f.tgt_sorted.size() <= (size_t)kMaxIns && nl >= f.tgt_sorted.size() + __builtin_popcountll(cm) &&
          (f.tgt_sorted.size() == 5 || nl - (uint32_t)__builtin_popcountll(cm) >= 8)) {
        CU(ctx, launch_dense_wide(s->prec, s->buf, nl, f, ctx->stream, &ctx->launches));
        return QIPB200_OK;
      }
      break;
    default:
      break;
  }
  // Fallback: out-of-place row kernel with the reference's gather semantics.
  if (s->world > 1)
    return set_err(ctx, QIPB200_ERR_UNSUPPORTED,
                   "this op needs the out-of-place row kernel, which is not available on a sharded state");
  if (!s->scratch) {
    cudaError_t e = cudaMalloc(&s->scratch, s->bytes);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "cudaMalloc(scratch arena)");
  }
  const uint64_t len = 1ull << nl;
  CU(ctx, launch_gather(s->prec, f, s->n, s->buf, len, 0, s->scratch, len, 0, false, ctx->stream, &ctx->launches));
  std::swap(s->buf, s->scratch);  // `Ok((arena, state, ..))`, builder.rs:514
  return QIPB200_OK;
}

int apply_flat_local(qipb200_state *s, const FlatOp &f_in) {
  FlatOp f;
  bool skip = false;
  int st = restrict_to_rank(s, f_in, &f, &skip);
  if (st != QIPB200_OK || skip) return st;
  return launch_local_op(s, f);
}

int report_error(qipb200_state *s, int status, const std::string &msg) { return set_err(s->ctx, status, msg); }
int report_cuda_error(qipb200_state *s, cudaError_t e, const char *what) { return cuda_fail(s->ctx, e, what); }

// The local bit a migration evicts: not used by this op, next non-diagonal use furthest away.
static int choose_victim(const qipb200_state *s, const FlatOp &f, const uint64_t *next_use) {
  uint64_t used = f.ctrl_mask;
  for (uint32_t j = 0; j < f.k; ++j) used |= 1ull << f.idx_bits[j];
  int best = -1;
  uint64_t best_key = 0;
  // with overlapped migrations (opt-in) the top local bit is never evicted: it splits the shard into the two halves
  // an overlapped migration works on
  const uint32_t l_end = overlap_exchange_enabled() && s->n_local > 3 ? s->n_local - 1 : s->n_local;
  for (uint32_t l = 0; l < l_end; ++l) {
    if ((used >> l) & 1ull) continue;
    uint64_t key = 1;
    if (next_use) {
      uint32_t logical = 0;
      for (uint32_t b = 0; b < s->n; ++b)
        if (s->phys_of_logical[b] == l) logical = b;
      key = next_use[logical] + 1;
    }
    // prefer high bits on ties: low bits give the exchange its coalescing
    if (best < 0 || key > best_key || (key == best_key && l > (uint32_t)best)) {
      best = (int)l;
      best_key = key;
    }
  }
  return best;
}

// The first exchange compile_and_localize(op) would perform under the current layout (none: returns false).
bool peek_first_exchange(const qipb200_state *s, const qip_op *op, const uint64_t *next_use, uint32_t *R, uint32_t *l) {
  if (s->world == 1) return false;
  FlatOp f;
  std::string err;
  if (compile_op(op, s->prec, s->n, &f, &err, s->phys_of_logical.data()) != QIPB200_OK) return false;
  if (f.cls == CLASS_BITSWAP && f.ctrl_mask == 0) return false;  // a relabelling: nothing moves
  std::vector<uint32_t> nd;
  nondiag_bits(f, &nd);
  for (size_t i = 0; i < nd.size(); ++i) {
    if (nd[i] < s->n_local) continue;
    const int v = choose_victim(s, f, next_use);
    if (v < 0) return false;
    *R = nd[i];
    *l = (uint32_t)v;
    return true;
  }
  return false;
}

// The flag barrier that opens an exchange (every rank has emptied its staging area), for the tile pass that pushes
// the give-half itself; afterwards exchange_bits(R, l) only runs the tail of the protocol.
int exchange_open_for_send(qipb200_state *s, uint32_t R, uint32_t l, void **peer_stage, int *give) {
  qipb200_ctx *ctx = s->ctx;
  if (!s->ipc_ready || !s->has_stage) return QIPB200_ERR_UNSUPPORTED;
  const uint32_t r = R - s->n_local;
  const int partner = s->rank ^ (1 << r);
  *give = 1 - ((s->rank >> r) & 1);
  *peer_stage = (char *)s->peer_buf[partner] + s->bytes;
  CU(ctx, launch_flag_barrier(s->peer_flags.data(), s->flags, s->rank, s->world, ++s->epoch, s->flags + kFlagErrorSlot,
                              ctx->stream, &ctx->launches));
  s->send_stage = 1;  // the caller raises it to 2 once the pushing pass is launched
  s->send_R = R;
  s->send_l = l;
  return QIPB200_OK;
}

// Overlapped migrations (two half exchanges on a second stream, passes on either side run in halves): measured on
// 2 x B200 at N=31 (profiles/r2l_*, r2m_*): 229.6 ms vs 233.8 ms without -- the exchange and the pass contend for the
// same HBM and SM slots, the gain is ~2 %.  Parity-green (sharded worker incl. generated kernels), but opt-in.
bool overlap_exchange_enabled() {
  static const bool on = getenv("QIPB200_OVERLAP_EXCHANGE") != nullptr;
  return on;
}

int ensure_overlap_resources(qipb200_state *s) {
  qipb200_ctx *ctx = s->ctx;
  if (ctx->stream2) return QIPB200_OK;
  // highest priority: the exchange needs few resident warps but must not queue behind the pass's thousands of CTAs
  int prio_lo = 0, prio_hi = 0;
  CU(ctx, cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
  CU(ctx, cudaStreamCreateWithPriority(&ctx->stream2, cudaStreamNonBlocking, prio_hi));
  for (int i = 0; i < 2; ++i) {
    CU(ctx, cudaEventCreateWithFlags(&ctx->ev_pass[i], cudaEventDisableTiming));
    CU(ctx, cudaEventCreateWithFlags(&ctx->ev_exch[i], cudaEventDisableTiming));
  }
  return QIPB200_OK;
}

// The migration R <-> l as TWO half exchanges (lower / upper half of the shard = top local bit 0 / 1) on the context's
// second stream: half v starts when ctx->ev_pass[v] (recorded by the caller on the main stream: "this half is final")
// has fired, and ctx->ev_exch[v] fires when it is done -- the tile pass before the migration overlaps the exchange of
// the half it finished first, the pass after it starts on the half that arrived first.  Every rank runs exactly this
// protocol (two barrier-exchange-barrier groups); what a rank overlaps with it is its own business.
int exchange_bits_split(qipb200_state *s, uint32_t R, uint32_t l) {
  qipb200_ctx *ctx = s->ctx;
  if (!s->ipc_ready) return set_err(ctx, QIPB200_ERR_COMM, "sharded state: peers not mapped (call qipb200_state_ipc_import)");
  if (s->n_local < 4 || l >= s->n_local - 1) return set_err(ctx, QIPB200_ERR_UNSUPPORTED, "internal: split exchange on the top local bit");
  int st0 = ensure_overlap_resources(s);
  if (st0 != QIPB200_OK) return st0;
  const uint32_t r = R - s->n_local;
  const int partner = s->rank ^ (1 << r);
  const int rb = (s->rank >> r) & 1;
  const uint32_t nh = s->n_local - 1;  // bits of a half
  uint32_t s_bit = nh - 1;
  if (s_bit == l) s_bit = nh - 2;
  const size_t half_bytes = s->bytes >> 1;
  for (int v = 0; v < 2; ++v) {
    CU(ctx, cudaStreamWaitEvent(ctx->stream2, ctx->ev_pass[v], 0));
    cudaEvent_t t0 = nullptr, t1 = nullptr;
    if (ctx->profile) {
      auto take = [&]() {
        cudaEvent_t e = nullptr;
        if (!ctx->prof_pool.empty()) {
          e = ctx->prof_pool.back();
          ctx->prof_pool.pop_back();
        } else if (cudaEventCreate(&e) != cudaSuccess) {
          e = nullptr;
        }
        return e;
      };
      t0 = take();
      t1 = take();
      if (t0) cudaEventRecord(t0, ctx->stream2);
    }
    CU(ctx, launch_flag_barrier(s->peer_flags.data(), s->flags, s->rank, s->world, ++s->epoch, s->flags + kFlagErrorSlot,
                                ctx->stream2, &ctx->launches));
    static const unsigned split_ctas = []() {
      const char *e = getenv("QIPB200_EXCH_CTAS");
      return (unsigned)(e ? atoi(e) : 296);
    }();
    CU(ctx, launch_pair_exchange(s->prec, (char *)s->buf + v * half_bytes, (char *)s->peer_buf[partner] + v * half_bytes, nh, l, s_bit,
                                 rb, ctx->stream2, &ctx->launches, split_ctas));
    CU(ctx, launch_flag_barrier(s->peer_flags.data(), s->flags, s->rank, s->world, ++s->epoch, s->flags + kFlagErrorSlot,
                                ctx->stream2, &ctx->launches));
    if (t0 && t1) {
      cudaEventRecord(t1, ctx->stream2);
      qipb200_ctx::ProfEvent pe = {t0, t1, 0.5};
      ctx->prof_events[1].push_back(pe);
    }
    CU(ctx, cudaEventRecord(ctx->ev_exch[v], ctx->stream2));
  }
  ++ctx->exchange_launches;
  s->halves_pending = true;
  s->exchange_bytes += (uint64_t)amp_bytes(s->prec) << (s->n_local - 1);
  for (uint32_t b = 0; b < s->n; ++b) {
    if (s->phys_of_logical[b] == R)
      s->phys_of_logical[b] = l;
    else if (s->phys_of_logical[b] == l)
      s->phys_of_logical[b] = R;
  }
  return QIPB200_OK;
}

// ---- migration fused into a tile pass, in place (paired send) ----
void paired_partner(const qipb200_state *s, uint32_t R, int *partner, int *give) {
  const uint32_t r = R - s->n_local;
  *partner = s->rank ^ (1 << r);
  *give = 1 - ((s->rank >> r) & 1);
}

// The rank's part of the per-tile protocol by a stand-alone kernel (its last pass ran without the send).
int paired_send_standin(qipb200_state *s, uint32_t R, uint32_t l, uint32_t cbit, uint32_t seq, const PassHeader &hdr) {
  qipb200_ctx *ctx = s->ctx;
  int partner = 0, give = 0;
  paired_partner(s, R, &partner, &give);
  PairedSendArgs a;
  memset(&a, 0, sizeof(a));
  a.mine = s->buf;
  a.peer = s->peer_buf[partner];
  a.my_flags = reinterpret_cast<uint32_t *>(reinterpret_cast<char *>(s->flags) + kPairFlagOffsetBytes);
  a.peer_flags = reinterpret_cast<uint32_t *>(reinterpret_cast<char *>(s->peer_flags[partner]) + kPairFlagOffsetBytes);
  a.error_word = s->flags + kFlagErrorSlot;
  a.seq = seq;
  a.n_local = s->n_local;
  a.T = hdr.T;
  a.L = hdr.L;
  a.m = hdr.m;
  a.l = l;
  a.cbit = cbit;
  a.give = (uint32_t)give;
  for (uint32_t i = 0; i < 8; ++i) a.hi_pos[i] = hdr.hi_pos[i];
  ProfileScope prof(ctx, 1);
  CU(ctx, launch_paired_send(s->prec, a, ctx->stream, &ctx->launches));
  return QIPB200_OK;
}

int finish_paired_exchange(qipb200_state *s, uint32_t R, uint32_t l) {
  qipb200_ctx *ctx = s->ctx;
  {
    ProfileScope prof(ctx, 1);
    CU(ctx, launch_flag_barrier(s->peer_flags.data(), s->flags, s->rank, s->world, ++s->epoch, s->flags + kFlagErrorSlot,
                                ctx->stream, &ctx->launches));
  }
  ++ctx->exchange_launches;
  s->exchange_bytes += (uint64_t)amp_bytes(s->prec) << (s->n_local - 1);
  for (uint32_t b = 0; b < s->n; ++b) {
    if (s->phys_of_logical[b] == R)
      s->phys_of_logical[b] = l;
    else if (s->phys_of_logical[b] == l)
      s->phys_of_logical[b] = R;
  }
  return QIPB200_OK;
}

// Make the main stream wait for an overlapped migration (both halves).
int join_halves(qipb200_state *s) {
  if (!s->halves_pending) return QIPB200_OK;
  qipb200_ctx *ctx = s->ctx;
  CU(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_exch[0], 0));
  CU(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_exch[1], 0));
  s->halves_pending = false;
  return QIPB200_OK;
}

// Compile `op` against the current layout and migrate rank-held target bits to
// local bits if needed.  `next_use` (optional, n entries indexed by logical bit):
// position in the schedule of the next non-diagonal use, used to pick the victim.
int compile_and_localize(qipb200_state *s, const qip_op *op, FlatOp *f, const uint64_t *next_use) {
  qipb200_ctx *ctx = s->ctx;
  std::string err;
  int st = compile_op(op, s->prec, s->n, f, &err, s->phys_of_logical.data());
  if (st != QIPB200_OK) return set_err(ctx, st, err);
  if (s->world == 1) return QIPB200_OK;
  if (f->cls == CLASS_BITSWAP && f->ctrl_mask == 0) {
    // An uncontrolled Swap is a relabelling of index bits: update the map, move nothing.
    for (size_t i = 0; i < f->swaps.size(); ++i) {
      const uint32_t p = f->swaps[i].first, q = f->swaps[i].second;
      for (uint32_t b = 0; b < s->n; ++b) {
        if (s->phys_of_logical[b] == p)
          s->phys_of_logical[b] = q;
        else if (s->phys_of_logical[b] == q)
          s->phys_of_logical[b] = p;
      }
    }
    f->cls = CLASS_IDENTITY;
    return QIPB200_OK;
  }
  std::vector<uint32_t> nd;
  nondiag_bits(*f, &nd);
  for (size_t i = 0; i < nd.size(); ++i) {
    if (nd[i] < s->n_local) continue;
    const int best = choose_victim(s, *f, next_use);
    if (best < 0) return set_err(ctx, QIPB200_ERR_UNSUPPORTED, "op touches every local bit: cannot migrate a rank bit");
    if ((st = exchange_bits(s, nd[i], (uint32_t)best)) != QIPB200_OK) return st;
    // recompile after every move so later decisions see the new layout
    st = compile_op(op, s->prec, s->n, f, &err, s->phys_of_logical.data());
    if (st != QIPB200_OK) return set_err(ctx, st, err);
    nondiag_bits(*f, &nd);
    i = (size_t)-1;  // restart scan
  }
  return QIPB200_OK;
}

}  // namespace qipb200

// ---- multi-device (single process) states ---------------------------------------------------
namespace {

double *comm_of(uint32_t *flags) { return reinterpret_cast<double *>(reinterpret_cast<char *>(flags) + kCommOffsetBytes); }

int multi_state_new(qipb200_ctx *parent, qip_prec prec, uint32_t n, qipb200_state **out) {
  const int G = (int)parent->children.size();
  qipb200_state *p = new qipb200_state();
  p->ctx = parent;
  p->prec = prec;
  p->n = n;
  p->world = 1;
  p->n_local = n;
  for (int r = 0; r < G; ++r) {
    qipb200_state *sh = nullptr;
    int st = state_alloc(parent->children[r], prec, n, r, G, &sh);
    if (st != QIPB200_OK) {
      set_err(parent, st, parent->children[r]->err);
      for (size_t i = 0; i < p->shards.size(); ++i) qipb200_state_free(p->shards[i]);
      delete p;
      return st;
    }
    p->shards.push_back(sh);
  }
  for (int r = 0; r < G; ++r) {  // peers are plain device pointers here: peer access was enabled by init_multi
    qipb200_state *sh = p->shards[r];
    sh->peer_buf.assign(G, nullptr);
    sh->peer_flags.assign(G, nullptr);
    sh->peer_comm.assign(G, nullptr);
    for (int t = 0; t < G; ++t) {
      sh->peer_buf[t] = p->shards[t]->buf;
      sh->peer_flags[t] = p->shards[t]->flags;
      sh->peer_comm[t] = comm_of(p->shards[t]->flags);
    }
    sh->ipc_ready = true;
    cudaSetDevice(sh->ctx->device);
    cudaStreamSynchronize(sh->ctx->stream);  // the zero fill of buffer and flag page, before any peer touches them
  }
  *out = p;
  return QIPB200_OK;
}

// out[0..count) (device, on the rank's stream) <- sum over all ranks of their out[]; collective.
int allreduce_sum(qipb200_state *s, double *d_vec, uint32_t count) {
  qipb200_ctx *ctx = s->ctx;
  if (s->world == 1) return QIPB200_OK;
  if (!s->ipc_ready) return set_err(ctx, QIPB200_ERR_COMM, "sharded state: peers not mapped (call qipb200_state_ipc_import)");
  if (count > (uint32_t)kCommDoubles) return set_err(ctx, QIPB200_ERR_UNSUPPORTED, "cross-rank reduction larger than the reduction slot");
  CU(ctx, cudaMemcpyAsync(comm_of(s->flags), d_vec, count * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
  CU(ctx, launch_flag_barrier(s->peer_flags.data(), s->flags, s->rank, s->world, ++s->epoch, s->flags + kFlagErrorSlot,
                              ctx->stream, &ctx->launches));
  CU(ctx, launch_comm_sum(s->peer_comm.data(), s->world, d_vec, count, ctx->stream, &ctx->launches));
  CU(ctx, launch_flag_barrier(s->peer_flags.data(), s->flags, s->rank, s->world, ++s->epoch, s->flags + kFlagErrorSlot,
                              ctx->stream, &ctx->launches));
  return QIPB200_OK;
}

}  // namespace

extern "C" int qipb200_state_new(qipb200_ctx *ctx, qip_prec prec, uint32_t n_qubits, qipb200_state **state) {
  return guarded(ctx, [&]() -> int {
    if (ctx && !ctx->children.empty()) {
      if (!state) return set_err(ctx, QIPB200_ERR_INVALID_ARG, "state out-pointer is NULL");
      *state = nullptr;
      if (ctx->children.size() == 1) return state_alloc(ctx->children[0], prec, n_qubits, 0, 1, state);
      return multi_state_new(ctx, prec, n_qubits, state);
    }
    return state_alloc(ctx, prec, n_qubits, 0, 1, state);
  });
}

extern "C" int qipb200_state_new_sharded(qipb200_ctx *ctx, qip_prec prec, uint32_t n_qubits, int rank,
                                         int world_size, qipb200_state **state) {
  if (ctx && !ctx->children.empty())
    return set_err(ctx, QIPB200_ERR_INVALID_ARG, "state_new_sharded: a multi-device context shards its states itself (use qipb200_state_new)");
  return guarded(ctx, [&]() { return state_alloc(ctx, prec, n_qubits, rank, world_size, state); });
}

extern "C" void qipb200_state_free(qipb200_state *s) {
  if (!s) return;
  if (!s->shards.empty()) {
    for (size_t i = 0; i < s->shards.size(); ++i) {  // all work must have drained before any buffer goes away
      cudaSetDevice(s->shards[i]->ctx->device);
      cudaStreamSynchronize(s->shards[i]->ctx->stream);
    }
    for (size_t i = 0; i < s->shards.size(); ++i) qipb200_state_free(s->shards[i]);
    delete s;
    return;
  }
  qipb200_ctx *ctx = s->ctx;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  if (s->ipc_mapped)
    for (int t = 0; t < (int)s->peer_buf.size(); ++t) {
      if (t == s->rank) continue;
      if (s->peer_buf[t]) cudaIpcCloseMemHandle(s->peer_buf[t]);
      if (s->peer_flags[t]) cudaIpcCloseMemHandle(s->peer_flags[t]);
    }
  if (s->buf) {
    if (s->world == 1 && !ctx->pool_buf) {  // keep one buffer for the next state of this size
      ctx->pool_buf = s->buf;
      ctx->pool_bytes = s->bytes;
    } else {
      cudaFree(s->buf);
    }
  }
  if (s->scratch) cudaFree(s->scratch);
  if (s->flags) cudaFree(s->flags);
  delete s;
}

static int set_basis_impl(qipb200_state *s, uint64_t index) {
  qipb200_ctx *ctx = s->ctx;
  if (index >> s->n) return set_err(ctx, QIPB200_ERR_BAD_INDEX, "initial index out of range");
  CU(ctx, cudaSetDevice(ctx->device));
  for (uint32_t b = 0; b < s->n; ++b) s->phys_of_logical[b] = b;  // a fresh state has the canonical layout
  const uint64_t len = 1ull << s->n_local;
  const bool owns = (index >> s->n_local) == (uint64_t)s->rank;
  CU(ctx, launch_set_basis(s->prec, s->buf, len, index & (len - 1), owns, ctx->stream, &ctx->launches));
  return QIPB200_OK;
}

extern "C" int qipb200_state_set_basis(qipb200_state *s, uint64_t index) {
  if (!s) return set_err(nullptr, QIPB200_ERR_INVALID_ARG, "state is NULL");
  return guarded(s->ctx, [&]() -> int {
    if (!s->shards.empty()) {
      if (index >> s->n) return set_err(s->ctx, QIPB200_ERR_BAD_INDEX, "initial index out of range");
      return each_shard(s, [&](qipb200_state *sh, int) { return set_basis_impl(sh, index); });
    }
    return set_basis_impl(s, index);
  });
}

static int transfer_impl(qipb200_state *s, void *host, uint64_t offset, uint64_t len, bool upload) {
  qipb200_ctx *ctx = s->ctx;
  const char *what = upload ? "upload" : "download";
  if (!host && len) return set_err(ctx, QIPB200_ERR_INVALID_ARG, std::string(what) + ": host pointer is NULL");
  if (len > (1ull << s->n_local) || offset > (1ull << s->n_local) - len)
    return set_err(ctx, QIPB200_ERR_SIZE_MISMATCH, std::string(what) + ": range exceeds the local state");
  CU(ctx, cudaSetDevice(ctx->device));
  if (!layout_is_identity(s)) {
    int st = restore_layout(s);
    if (st != QIPB200_OK) return st;
  }
  const size_t ab = amp_bytes(s->prec);
  if (len) {
    if (upload)
      CU(ctx, cudaMemcpyAsync((char *)s->buf + offset * ab, host, len * ab, cudaMemcpyHostToDevice, ctx->stream));
    else
      CU(ctx, cudaMemcpyAsync(host, (const char *)s->buf + offset * ab, len * ab, cudaMemcpyDeviceToHost, ctx->stream));
  }
  CU(ctx, cudaStreamSynchronize(ctx->stream));
  if (s->world > 1 && s->ipc_ready) return check_barrier_error(s);
  return QIPB200_OK;
}

// A multi-device state is addressed as ONE 2^n vector: the range is cut at the shard boundaries.  Every shard
// takes part even when its piece is empty (restoring the canonical layout is a collective exchange).
static int multi_transfer(qipb200_state *p, void *host, uint64_t offset, uint64_t len, bool upload) {
  if (!host && len) return set_err(p->ctx, QIPB200_ERR_INVALID_ARG, "upload/download: host pointer is NULL");
  if (len > (1ull << p->n) || offset > (1ull << p->n) - len)
    return set_err(p->ctx, QIPB200_ERR_SIZE_MISMATCH, "upload/download: range exceeds the state");
  const size_t ab = amp_bytes(p->prec);
  return each_shard(p, [&](qipb200_state *sh, int r) {
    const uint64_t lo = (uint64_t)r << sh->n_local, hi = lo + (1ull << sh->n_local);
    const uint64_t a = std::max(lo, offset), b = std::min(hi, offset + len);
    if (b <= a) return transfer_impl(sh, host, 0, 0, upload);
    return transfer_impl(sh, (char *)host + (a - offset) * ab, a - lo, b - a, upload);
  });
}

extern "C" int qipb200_state_upload(qipb200_state *s, const void *host, uint64_t offset, uint64_t len) {
  if (!s) return set_err(nullptr, QIPB200_ERR_INVALID_ARG, "state is NULL");
  return guarded(s->ctx, [&]() -> int {
    if (!s->shards.empty()) return multi_transfer(s, const_cast<void *>(host), offset, len, true);
    return transfer_impl(s, const_cast<void *>(host), offset, len, true);
  });
}

extern "C" int qipb200_state_download(qipb200_state *s, void *host, uint64_t offset, uint64_t len) {
  if (!s) return set_err(nullptr, QIPB200_ERR_INVALID_ARG, "state is NULL");
  return guarded(s->ctx, [&]() -> int {
    if (!s->shards.empty()) return multi_transfer(s, host, offset, len, false);
    return transfer_impl(s, host, offset, len, false);
  });
}

static int apply_op_impl(qipb200_state *s, const qip_op *op) {
  CU(s->ctx, cudaSetDevice(s->ctx->device));
  FlatOp f;
  int st = compile_and_localize(s, op, &f, nullptr);
  if (st != QIPB200_OK) return st;
  return apply_flat_local(s, f);
}

extern "C" int qipb200_state_apply_op(qipb200_state *s, const qip_op *op) {
  if (!s) return set_err(nullptr, QIPB200_ERR_INVALID_ARG, "state is NULL");
  return guarded(s->ctx, [&]() -> int {
    if (!s->shards.empty()) return each_shard(s, [&](qipb200_state *sh, int) { return apply_op_impl(sh, op); });
    return apply_op_impl(s, op);
  });
}

extern "C" int qipb200_state_apply_schedule(qipb200_state *s, const qip_op *ops, size_t n_ops, uint32_t flags) {
  if (!s) return set_err(nullptr, QIPB200_ERR_INVALID_ARG, "state is NULL");
  if (!ops && n_ops) return set_err(s->ctx, QIPB200_ERR_INVALID_ARG, "schedule: ops is NULL");
  return guarded(s->ctx, [&]() -> int {
    auto one = [&](qipb200_state *sh, int) -> int {
      CU(sh->ctx, cudaSetDevice(sh->ctx->device));
      return run_schedule(sh, ops, n_ops, flags);
    };
    if (!s->shards.empty()) return each_shard(s, one);
    return one(s, 0);
  });
}

// sum |a|^2 of the WHOLE state: on a sharded state the per-rank sums are all-reduced (collective call).
static int norm2_impl(qipb200_state *s, double *out) {
  qipb200_ctx *ctx = s->ctx;
  CU(ctx, cudaSetDevice(ctx->device));
  CU(ctx, launch_norm2(s->prec, s->buf, 1ull << s->n_local, ctx->d_scalar, ctx->stream, &ctx->launches));
  int st = allreduce_sum(s, ctx->d_scalar, 1);
  if (st != QIPB200_OK) return st;
  CU(ctx, cudaMemcpyAsync(out, ctx->d_scalar, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CU(ctx, cudaStreamSynchronize(ctx->stream));
  return QIPB200_OK;
}

extern "C" int qipb200_state_norm2(qipb200_state *s, double *out) {
  if (!s || !out) return set_err(s ? s->ctx : nullptr, QIPB200_ERR_INVALID_ARG, "norm2: NULL argument");
  return guarded(s->ctx, [&]() -> int {
    if (!s->shards.empty()) {
      std::vector<double> v(s->shards.size(), 0.0);
      int st = each_shard(s, [&](qipb200_state *sh, int r) { return norm2_impl(sh, &v[r]); });
      *out = v[0];
      return st;
    }
    return norm2_impl(s, out);
  });
}

static int max_abs_diff_impl(qipb200_state *a, qipb200_state *b, double *out) {
  qipb200_ctx *ctx = a->ctx;
  if (a->ctx != b->ctx || a->prec != b->prec || a->n != b->n || a->world != b->world || a->rank != b->rank)
    return set_err(ctx, QIPB200_ERR_SIZE_MISMATCH, "max_abs_diff: the two states differ in context, precision or shape");
  if (a->phys_of_logical != b->phys_of_logical)
    return set_err(ctx, QIPB200_ERR_UNSUPPORTED, "max_abs_diff: the two sharded states hold different qubit layouts");
  CU(ctx, cudaSetDevice(ctx->device));
  CU(ctx, launch_max_abs_diff(a->prec, a->buf, b->buf, 1ull << a->n_local, ctx->d_scalar, ctx->stream, &ctx->launches));
  CU(ctx, cudaMemcpyAsync(out, ctx->d_scalar, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CU(ctx, cudaStreamSynchronize(ctx->stream));
  return QIPB200_OK;
}

extern "C" int qipb200_state_max_abs_diff(qipb200_state *a, qipb200_state *b, double *out) {
  if (!a || !b || !out) return set_err(a ? a->ctx : nullptr, QIPB200_ERR_INVALID_ARG, "max_abs_diff: NULL argument");
  return guarded(a->ctx, [&]() -> int {
    if (a->shards.size() != b->shards.size())
      return set_err(a->ctx, QIPB200_ERR_SIZE_MISMATCH, "max_abs_diff: the two states differ in context, precision or shape");
    if (!a->shards.empty()) {
      std::vector<double> v(a->shards.size(), 0.0);
      int st = each_shard(a, [&](qipb200_state *sh, int r) { return max_abs_diff_impl(sh, b->shards[r], &v[r]); });
      *out = *std::max_element(v.begin(), v.end());
      return st;
    }
    return max_abs_diff_impl(a, b, out);
  });
}

static int sync_impl(qipb200_state *s) {
  CU(s->ctx, cudaSetDevice(s->ctx->device));
  CU(s->ctx, cudaStreamSynchronize(s->ctx->stream));
  if (s->world > 1 && s->ipc_ready) return check_barrier_error(s);
  return QIPB200_OK;
}

extern "C" int qipb200_state_sync(qipb200_state *s) {
  if (!s) return set_err(nullptr, QIPB200_ERR_INVALID_ARG, "state is NULL");
  return guarded(s->ctx, [&]() -> int {
    if (!s->shards.empty()) return each_shard(s, [&](qipb200_state *sh, int) { return sync_impl(sh); });
    return sync_impl(s);
  });
}

extern "C" int qipb200_calculate_state(qipb200_ctx *ctx, qip_prec prec, uint32_t n_qubits, uint64_t init_index,
                                       const qip_op *ops, size_t n_ops, uint32_t flags, void *host_out) {
  if (!ctx) return set_err(nullptr, QIPB200_ERR_INVALID_ARG, "ctx is NULL (call qipb200_init first; there is no CPU path)");
  if (!host_out) return set_err(ctx, QIPB200_ERR_INVALID_ARG, "calculate_state: host_out is NULL");
  qipb200_state *s = nullptr;
  int st = qipb200_state_new(ctx, prec, n_qubits, &s);
  if (st != QIPB200_OK) return st;
  st = qipb200_state_set_basis(s, init_index);
  if (st == QIPB200_OK) st = qipb200_state_apply_schedule(s, ops, n_ops, flags);
  if (st == QIPB200_OK) st = qipb200_state_download(s, host_out, 0, 1ull << n_qubits);
  qipb200_state_free(s);
  return st;
}

extern "C" int qipb200_apply_ops(qipb200_ctx *ctx, qip_prec prec, uint32_t n, const qip_op *ops, size_t n_ops,
                                 const void *input, uint64_t input_len, void *output, uint64_t output_len,
                                 uint64_t input_offset, uint64_t output_offset) {
  if (!ctx) return set_err(nullptr, QIPB200_ERR_INVALID_ARG, "ctx is NULL (call qipb200_init first; there is no CPU path)");
  const size_t ab = amp_bytes(prec);
  if (n_ops == 0) {
    // matrix_ops.rs:170-183: copy of the overlapping index range
    const uint64_t lower = std::max(input_offset, output_offset);
    const uint64_t upper = std::min(input_offset + input_len, output_offset + output_len);
    if (upper > lower) {
      if (!input || !output) return set_err(ctx, QIPB200_ERR_INVALID_ARG, "apply_ops: NULL amplitude buffer");
      memcpy((char *)output + (lower - output_offset) * ab, (const char *)input + (lower - input_offset) * ab,
             (upper - lower) * ab);
    }
    return QIPB200_OK;
  }
  if (n_ops == 1)  // matrix_ops.rs:167
    return qipb200_apply_op(ctx, prec, n, ops, input, input_len, output, output_len, input_offset, output_offset);
  // Several ops: the reference's multi-op row iterator (matrix_ops.rs:184-217), restated as it is -- including
  // SURVEY.md quirk Q5 -- by k_multi_gather; accumulates into `output` like the reference (:212).
  return guarded(ctx, [&]() -> int {
    qipb200_ctx *c = ctx->children.empty() ? ctx : ctx->children[0];
    if ((!input && input_len) || (!output && output_len)) return set_err(ctx, QIPB200_ERR_INVALID_ARG, "apply_ops: NULL amplitude buffer");
    if (n > 40 || input_len > (1ull << 40) || output_len > (1ull << 40))
      return set_err(ctx, QIPB200_ERR_SIZE_MISMATCH, "apply_ops: buffer length out of range");
    if (n_ops > 8) return set_err(ctx, QIPB200_ERR_UNSUPPORTED, "apply_ops: more than 8 ops in one multi-op sweep");
    std::vector<FlatOp> fs(n_ops);
    uint32_t ktot = 0;
    for (size_t i = 0; i < n_ops; ++i) {
      std::string err;
      int st = compile_op(&ops[i], prec, n, &fs[i], &err);
      if (st != QIPB200_OK) return set_err(ctx, st, err);
      ktot += fs[i].k;
    }
    if (ktot > 40) return set_err(ctx, QIPB200_ERR_UNSUPPORTED, "apply_ops: more than 40 indices over all ops");
    if (cudaSetDevice(c->device) != cudaSuccess) return set_err(ctx, QIPB200_ERR_CUDA, "cudaSetDevice");
    int st;
    if ((st = grow(c, &c->d_in, &c->d_in_bytes, std::max<size_t>(input_len * ab, 16))) != QIPB200_OK ||
        (st = grow(c, &c->d_out, &c->d_out_bytes, std::max<size_t>(output_len * ab, 16))) != QIPB200_OK) {
      if (c != ctx) ctx->err = c->err;
      return st;
    }
    cudaError_t e = cudaSuccess;
    if (input_len) e = cudaMemcpyAsync(c->d_in, input, input_len * ab, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess && output_len) e = cudaMemcpyAsync(c->d_out, output, output_len * ab, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess)
      e = launch_multi_gather(prec, fs, c->d_in, input_len, input_offset, c->d_out, output_len, output_offset, c->stream, &c->launches);
    if (e == cudaSuccess && output_len) e = cudaMemcpyAsync(output, c->d_out, output_len * ab, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) return set_err(ctx, QIPB200_ERR_CUDA, std::string("apply_ops: ") + cudaGetErrorString(e));
    return (int)QIPB200_OK;
  });
}

// ===================================================================================
// N3: state files ("QIPA" v1, one file per shard; layout in rustqip_b200/wire.py) -- checkpoint / resume
// ===================================================================================

namespace {

struct QipaHeader {
  uint32_t magic, version, prec, n_qubits, rank, world;
  uint64_t first_index, n_amplitudes;
};
static_assert(sizeof(QipaHeader) == 40, "QIPA header is 40 bytes");
const uint32_t kQipaMagic = 0x41504951u;
const size_t kFileChunkBytes = 64u << 20;  // host bounce buffer: the shard never sits in host memory as a whole

int state_file_impl(qipb200_state *s, const char *path, bool save) {
  qipb200_ctx *ctx = s->ctx;
  CU(ctx, cudaSetDevice(ctx->device));
  if (!layout_is_identity(s)) {  // files hold the canonical layout (collective on a sharded state)
    int st = restore_layout(s);
    if (st != QIPB200_OK) return st;
  }
  const size_t ab = amp_bytes(s->prec);
  const uint64_t len = 1ull << s->n_local;
  FILE *f = fopen(path, save ? "wb" : "rb");
  if (!f) return set_err(ctx, QIPB200_ERR_INVALID_ARG, std::string("state file: cannot open ") + path);
  QipaHeader h;
  int st = QIPB200_OK;
  if (save) {
    h.magic = kQipaMagic, h.version = 1, h.prec = (uint32_t)s->prec, h.n_qubits = s->n, h.rank = (uint32_t)s->rank;
    h.world = (uint32_t)s->world, h.first_index = (uint64_t)s->rank << s->n_local, h.n_amplitudes = len;
    if (fwrite(&h, sizeof(h), 1, f) != 1) st = set_err(ctx, QIPB200_ERR_INVALID_ARG, "state file: write failed");
  } else {
    if (fread(&h, sizeof(h), 1, f) != 1 || h.magic != kQipaMagic || h.version != 1)
      st = set_err(ctx, QIPB200_ERR_INVALID_ARG, "not a QIPA version-1 state file");
    else if (h.prec != (uint32_t)s->prec || h.n_qubits != s->n || h.rank != (uint32_t)s->rank || h.world != (uint32_t)s->world ||
             h.n_amplitudes != len)
      st = set_err(ctx, QIPB200_ERR_SIZE_MISMATCH, "state file does not match the target state (prec/n/rank/world/length)");
  }
  std::vector<char> bounce;
  if (st == QIPB200_OK) bounce.resize((size_t)std::min<uint64_t>(kFileChunkBytes, len * ab));
  for (uint64_t done = 0; st == QIPB200_OK && done < len * ab;) {
    const size_t n = (size_t)std::min<uint64_t>(bounce.size(), len * ab - done);
    cudaError_t e;
    if (save) {
      e = cudaMemcpyAsync(bounce.data(), (const char *)s->buf + done, n, cudaMemcpyDeviceToHost, ctx->stream);
      if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
      if (e != cudaSuccess) st = cuda_fail(ctx, e, "state file: device -> host");
      else if (fwrite(bounce.data(), 1, n, f) != n) st = set_err(ctx, QIPB200_ERR_INVALID_ARG, "state file: write failed");
    } else {
      if (fread(bounce.data(), 1, n, f) != n) {
        st = set_err(ctx, QIPB200_ERR_INVALID_ARG, "state file truncated");
        break;
      }
      e = cudaMemcpyAsync((char *)s->buf + done, bounce.data(), n, cudaMemcpyHostToDevice, ctx->stream);
      if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
      if (e != cudaSuccess) st = cuda_fail(ctx, e, "state file: host -> device");
    }
    done += n;
  }
  if (st == QIPB200_OK && !save && fgetc(f) != EOF) st = set_err(ctx, QIPB200_ERR_INVALID_ARG, "state file: trailing bytes");
  if (fclose(f) != 0 && st == QIPB200_OK && save) st = set_err(ctx, QIPB200_ERR_INVALID_ARG, "state file: close failed");
  return st;
}

int state_file(qipb200_state *s, const char *path, bool save) {
  if (!s || !path) return set_err(s ? s->ctx : nullptr, QIPB200_ERR_INVALID_ARG, "state file: NULL argument");
  return guarded(s->ctx, [&]() -> int {
    if (!s->shards.empty())  // multi-device state: one file per shard, "<path>.<rank>"
      return each_shard(s, [&](qipb200_state *sh, int r) { return state_file_impl(sh, (std::string(path) + "." + std::to_string(r)).c_str(), save); });
    return state_file_impl(s, path, save);
  });
}

}  // namespace

extern "C" int qipb200_state_save(qipb200_state *s, const char *path) { return state_file(s, path, true); }
extern "C" int qipb200_state_load(qipb200_state *s, const char *path) { return state_file(s, path, false); }

// ===================================================================================
// measurement (collective on a sharded state: every rank calls, every rank gets the answer)
// ===================================================================================

namespace {

int check_indices(qipb200_state *s, const uint64_t *indices, uint32_t n_indices) {
  if (!indices || n_indices == 0 || n_indices > s->n)
    return set_err(s->ctx, QIPB200_ERR_INVALID_ARG, "measurement: bad index list");
  uint64_t seen = 0;
  for (uint32_t i = 0; i < n_indices; ++i) {
    if (indices[i] >= s->n) return set_err(s->ctx, QIPB200_ERR_BAD_INDEX, "measurement: qubit index out of range");
    if ((seen >> indices[i]) & 1) return set_err(s->ctx, QIPB200_ERR_BAD_INDEX, "measurement: repeated qubit index");
    seen |= 1ull << indices[i];
  }
  return QIPB200_OK;
}

int measure_probs_impl(qipb200_state *s, const uint64_t *indices, uint32_t n_indices, double *out) {
  qipb200_ctx *ctx = s->ctx;
  if (n_indices > 26) return set_err(ctx, QIPB200_ERR_UNSUPPORTED, "measure_probs: more than 26 measured qubits");
  if (s->world > 1 && (1u << n_indices) > (uint32_t)kCommDoubles)
    return set_err(ctx, QIPB200_ERR_UNSUPPORTED, "measure_probs on a sharded state: more than 16 measured qubits");
  CU(ctx, cudaSetDevice(ctx->device));
  uint32_t bitpos[32];
  for (uint32_t i = 0; i < n_indices; ++i) bitpos[i] = s->phys_of_logical[s->n - 1 - (uint32_t)indices[i]];
  double *d_hist = nullptr;
  CU(ctx, cudaMallocAsync((void **)&d_hist, sizeof(double) << n_indices, ctx->stream));
  CU(ctx, launch_measure_probs(s->prec, s->buf, 1ull << s->n_local, (uint64_t)s->rank << s->n_local, bitpos,
                               n_indices, d_hist, ctx->stream, &ctx->launches));
  // measurement_ops.rs:115-127 sums over the WHOLE vector: per-rank histograms are added across the ranks
  int st = allreduce_sum(s, d_hist, 1u << n_indices);
  if (st == QIPB200_OK)
    CU(ctx, cudaMemcpyAsync(out, d_hist, sizeof(double) << n_indices, cudaMemcpyDeviceToHost, ctx->stream));
  CU(ctx, cudaFreeAsync(d_hist, ctx->stream));
  CU(ctx, cudaStreamSynchronize(ctx->stream));
  return st;
}

// Inverse-CDF sampling of n_draws draws (measurement_ops.rs:153-176 applied to each; rules in sample.cuh): one read
// sweep for the chunk sums, their prefix, then one warp per draw.  The reference scans in canonical index order, so a
// permuted layout is restored first (collective on a sharded state: rank t then holds [t 2^nl, (t+1) 2^nl)).  The
// ranks' totals are all-reduced, the owner of each draw resolves it, and the indices are summed across the ranks.
int sample_impl(qipb200_state *s, const uint64_t *indices, uint32_t n_indices, const double *r, uint64_t n_draws,
                uint64_t *out) {
  qipb200_ctx *ctx = s->ctx;
  CU(ctx, cudaSetDevice(ctx->device));
  if (!layout_is_identity(s)) {
    int st = restore_layout(s);
    if (st != QIPB200_OK) return st;
  }
  const int W = s->world;
  SampleArgs a;
  a.n_draws = 0;
  a.chunk_log2 = std::min<uint32_t>(s->n_local, kSampleChunkLog2);
  a.chunks = 1ull << (s->n_local - a.chunk_log2);
  a.index_base = (uint64_t)s->rank << s->n_local;
  a.rank = s->rank;
  a.world = W;
  uint8_t bitpos[64];
  for (uint32_t i = 0; i < n_indices; ++i) bitpos[i] = (uint8_t)(s->n - 1 - indices[i]);
  const uint64_t batch = std::min<uint64_t>(n_draws, kSampleBatch);
  // [chunk prefix | rank totals | draws | results]
  double *d_P = nullptr;
  CU(ctx, cudaMallocAsync((void **)&d_P, (a.chunks + W + 2 * batch) * sizeof(double), ctx->stream));
  double *d_tot = d_P + a.chunks, *d_draw = d_tot + W, *d_res = d_draw + batch;
  auto run = [&]() -> int {
    CU(ctx, launch_chunk_sums(s->prec, s->buf, 1ull << s->n_local, a.chunk_log2, d_P, ctx->stream, &ctx->launches));
    CU(ctx, launch_sample_scan(d_P, a.chunks, ctx->stream, &ctx->launches));
    // a rank's total is the last prefix: the owner's chunk search always finds the chunk its share of the draw is in
    CU(ctx, cudaMemsetAsync(d_tot, 0, W * sizeof(double), ctx->stream));
    CU(ctx, cudaMemcpyAsync(d_tot + s->rank, d_P + a.chunks - 1, sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    int st = allreduce_sum(s, d_tot, (uint32_t)W);
    for (uint64_t done = 0; st == QIPB200_OK && done < n_draws; done += a.n_draws) {
      a.n_draws = std::min<uint64_t>(batch, n_draws - done);
      CU(ctx, cudaMemcpyAsync(d_draw, r + done, a.n_draws * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
      CU(ctx, launch_sample_resolve(s->prec, s->buf, d_P, d_tot, d_draw, d_res, a, ctx->stream, &ctx->launches));
      for (uint64_t o = 0; st == QIPB200_OK && W > 1 && o < a.n_draws; o += (uint64_t)kCommDoubles)
        st = allreduce_sum(s, d_res + o, (uint32_t)std::min<uint64_t>((uint64_t)kCommDoubles, a.n_draws - o));
      if (st != QIPB200_OK) break;
      CU(ctx, launch_sample_outcomes(d_res, a.n_draws, bitpos, n_indices, ctx->stream, &ctx->launches));
      CU(ctx, cudaMemcpyAsync(out + done, d_res, a.n_draws * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    }
    return st;
  };
  int st = run();
  cudaFreeAsync(d_P, ctx->stream);
  if (st != QIPB200_OK) return st;
  CU(ctx, cudaStreamSynchronize(ctx->stream));
  if (W > 1) return check_barrier_error(s);
  return QIPB200_OK;
}

int collapse_impl(qipb200_state *s, const uint64_t *indices, uint32_t n_indices, uint64_t measured, double measured_prob) {
  qipb200_ctx *ctx = s->ctx;
  if (measured_prob == 0.0) return QIPB200_OK;  // measurement_ops.rs:230: untouched
  CU(ctx, cudaSetDevice(ctx->device));
  uint64_t row_mask = 0, measured_mask = 0;
  for (uint32_t i = 0; i < n_indices; ++i) {
    const uint32_t bit = s->phys_of_logical[s->n - 1 - (uint32_t)indices[i]];
    row_mask |= 1ull << bit;
    measured_mask |= ((measured >> i) & 1ull) << bit;
  }
  // P::one() / measured_prob.sqrt() evaluated in the state's precision (measurement_ops.rs:231)
  double p_mult;
  if (s->prec == QIP_F32)
    p_mult = (double)(1.0f / sqrtf((float)measured_prob));
  else
    p_mult = 1.0 / sqrt(measured_prob);
  CU(ctx, launch_collapse(s->prec, s->buf, 1ull << s->n_local, (uint64_t)s->rank << s->n_local, row_mask,
                          measured_mask, p_mult, ctx->stream, &ctx->launches));
  return QIPB200_OK;
}

}  // namespace

extern "C" int qipb200_state_measure_probs(qipb200_state *s, const uint64_t *indices, uint32_t n_indices, double *out) {
  if (!s || !out) return set_err(s ? s->ctx : nullptr, QIPB200_ERR_INVALID_ARG, "measure_probs: NULL argument");
  return guarded(s->ctx, [&]() -> int {
    int st = check_indices(s, indices, n_indices);
    if (st != QIPB200_OK) return st;
    if (!s->shards.empty()) {
      if (n_indices > 16) return set_err(s->ctx, QIPB200_ERR_UNSUPPORTED, "measure_probs on a sharded state: more than 16 measured qubits");
      std::vector<std::vector<double>> v(s->shards.size(), std::vector<double>((size_t)1 << n_indices));
      st = each_shard(s, [&](qipb200_state *sh, int r) { return measure_probs_impl(sh, indices, n_indices, v[r].data()); });
      if (st == QIPB200_OK) memcpy(out, v[0].data(), sizeof(double) << n_indices);
      return st;
    }
    return measure_probs_impl(s, indices, n_indices, out);
  });
}

extern "C" int qipb200_state_measure_prob(qipb200_state *s, uint64_t measured, const uint64_t *indices,
                                          uint32_t n_indices, double *out) {
  if (!s || !out) return set_err(s ? s->ctx : nullptr, QIPB200_ERR_INVALID_ARG, "measure_prob: NULL argument");
  return guarded(s->ctx, [&]() -> int {
    int st = check_indices(s, indices, n_indices);
    if (st != QIPB200_OK) return st;
    if (n_indices > 26) return set_err(s->ctx, QIPB200_ERR_UNSUPPORTED, "measure_prob: more than 26 measured qubits");
    std::vector<double> probs(1ull << n_indices);
    st = qipb200_state_measure_probs(s, indices, n_indices, probs.data());
    if (st != QIPB200_OK) return st;
    *out = (measured >> n_indices) ? 0.0 : probs[measured];
    return (int)QIPB200_OK;
  });
}

// Every rank of a multi-device state computes the same answers; rank 0's are returned after the others are compared.
static int multi_sample(qipb200_state *s, const uint64_t *indices, uint32_t n_indices, const double *r, uint64_t n_draws,
                        uint64_t *out) {
  const size_t G = s->shards.size();
  std::vector<std::vector<uint64_t>> v(G);
  for (size_t k = 1; k < G; ++k) v[k].resize(n_draws);
  int st = each_shard(s, [&](qipb200_state *sh, int rk) {
    return sample_impl(sh, indices, n_indices, r, n_draws, rk == 0 ? out : v[rk].data());
  });
  if (st != QIPB200_OK) return st;
  for (size_t k = 1; k < G; ++k)
    if (n_draws && memcmp(v[k].data(), out, n_draws * sizeof(uint64_t)) != 0)
      return set_err(s->ctx, QIPB200_ERR_COMM, "sample: the shards disagree on the drawn outcomes");
  return QIPB200_OK;
}

extern "C" int qipb200_state_soft_measure(qipb200_state *s, const uint64_t *indices, uint32_t n_indices, double r,
                                          uint64_t *measured) {
  if (!s || !measured) return set_err(s ? s->ctx : nullptr, QIPB200_ERR_INVALID_ARG, "soft_measure: NULL argument");
  return guarded(s->ctx, [&]() -> int {
    int st = check_indices(s, indices, n_indices);
    if (st != QIPB200_OK) return st;
    if (!s->shards.empty()) return multi_sample(s, indices, n_indices, &r, 1, measured);
    return sample_impl(s, indices, n_indices, &r, 1, measured);
  });
}

extern "C" int qipb200_state_sample(qipb200_state *s, const uint64_t *indices, uint32_t n_indices, const double *r,
                                    uint64_t n_draws, uint64_t *out) {
  if (!s || !r || !out)
    return set_err(s ? s->ctx : nullptr, QIPB200_ERR_INVALID_ARG, "sample: NULL argument");
  return guarded(s->ctx, [&]() -> int {
    int st = check_indices(s, indices, n_indices);
    if (st != QIPB200_OK) return st;
    for (uint64_t j = 0; j < n_draws; ++j)
      if (!(r[j] >= 0.0 && r[j] <= 1.0))
        return set_err(s->ctx, QIPB200_ERR_INVALID_ARG, "sample: draw " + std::to_string(j) + " is not in [0, 1]");
    if (n_draws == 0) return (int)QIPB200_OK;
    if (!s->shards.empty()) return multi_sample(s, indices, n_indices, r, n_draws, out);
    return sample_impl(s, indices, n_indices, r, n_draws, out);
  });
}

extern "C" int qipb200_state_collapse(qipb200_state *s, const uint64_t *indices, uint32_t n_indices,
                                      uint64_t measured, double measured_prob) {
  if (!s) return set_err(nullptr, QIPB200_ERR_INVALID_ARG, "state is NULL");
  return guarded(s->ctx, [&]() -> int {
    int st = check_indices(s, indices, n_indices);
    if (st != QIPB200_OK) return st;
    if (!s->shards.empty())
      return each_shard(s, [&](qipb200_state *sh, int) { return collapse_impl(sh, indices, n_indices, measured, measured_prob); });
    return collapse_impl(s, indices, n_indices, measured, measured_prob);
  });
}

// ===================================================================================
// multi-GPU plumbing (one process per GPU: CUDA IPC)
// ===================================================================================

extern "C" int qipb200_state_ipc_export(qipb200_state *s, void *amp_handle, void *flag_handle) {
  if (!s || !amp_handle || !flag_handle) return set_err(s ? s->ctx : nullptr, QIPB200_ERR_INVALID_ARG, "ipc_export: NULL argument");
  qipb200_ctx *ctx = s->ctx;
  if (s->world == 1) return set_err(ctx, QIPB200_ERR_INVALID_ARG, "ipc_export: not a sharded state");
  static_assert(sizeof(cudaIpcMemHandle_t) == QIPB200_IPC_HANDLE_BYTES, "IPC handle size");
  CU(ctx, cudaSetDevice(ctx->device));
  CU(ctx, cudaStreamSynchronize(ctx->stream));
  cudaIpcMemHandle_t h;
  CU(ctx, cudaIpcGetMemHandle(&h, s->buf));
  memcpy(amp_handle, &h, sizeof(h));
  CU(ctx, cudaIpcGetMemHandle(&h, s->flags));
  memcpy(flag_handle, &h, sizeof(h));
  return QIPB200_OK;
}

extern "C" int qipb200_state_ipc_import(qipb200_state *s, const void *amp_handles, const void *flag_handles) {
  if (!s || !amp_handles || !flag_handles) return set_err(s ? s->ctx : nullptr, QIPB200_ERR_INVALID_ARG, "ipc_import: NULL argument");
  qipb200_ctx *ctx = s->ctx;
  if (s->world == 1) return set_err(ctx, QIPB200_ERR_INVALID_ARG, "ipc_import: not a sharded state");
  if (s->ipc_ready) return set_err(ctx, QIPB200_ERR_INVALID_ARG, "ipc_import: peers are already mapped");
  return guarded(ctx, [&]() -> int {
    CU(ctx, cudaSetDevice(ctx->device));
    s->peer_buf.assign(s->world, nullptr);
    s->peer_flags.assign(s->world, nullptr);
    s->peer_comm.assign(s->world, nullptr);
    s->ipc_mapped = true;
    for (int t = 0; t < s->world; ++t) {
      if (t == s->rank) {
        s->peer_buf[t] = s->buf;
        s->peer_flags[t] = s->flags;
        s->peer_comm[t] = comm_of(s->flags);
        continue;
      }
      cudaIpcMemHandle_t h;
      memcpy(&h, (const char *)amp_handles + (size_t)t * QIPB200_IPC_HANDLE_BYTES, sizeof(h));
      cudaError_t e = cudaIpcOpenMemHandle(&s->peer_buf[t], h, cudaIpcMemLazyEnablePeerAccess);
      if (e != cudaSuccess) {
        cuda_fail(ctx, e, "cudaIpcOpenMemHandle(amplitudes)");
        return (int)QIPB200_ERR_COMM;
      }
      memcpy(&h, (const char *)flag_handles + (size_t)t * QIPB200_IPC_HANDLE_BYTES, sizeof(h));
      void *fp = nullptr;
      e = cudaIpcOpenMemHandle(&fp, h, cudaIpcMemLazyEnablePeerAccess);
      if (e != cudaSuccess) {
        cuda_fail(ctx, e, "cudaIpcOpenMemHandle(flags)");
        return (int)QIPB200_ERR_COMM;
      }
      s->peer_flags[t] = (uint32_t *)fp;
      s->peer_comm[t] = comm_of((uint32_t *)fp);
    }
    s->ipc_ready = true;
    return (int)QIPB200_OK;
  });
}

extern "C" int qipb200_state_qubit_map(qipb200_state *s, uint32_t *bit_of_qubit) {
  if (!s || !bit_of_qubit) return set_err(s ? s->ctx : nullptr, QIPB200_ERR_INVALID_ARG, "qubit_map: NULL argument");
  const qipb200_state *src = s->shards.empty() ? s : s->shards[0];
  for (uint32_t q = 0; q < s->n; ++q) bit_of_qubit[q] = src->phys_of_logical[s->n - 1 - q];
  return QIPB200_OK;
}

extern "C" int qipb200_state_exchange_bytes(qipb200_state *s, uint64_t *bytes) {
  if (!s || !bytes) return set_err(s ? s->ctx : nullptr, QIPB200_ERR_INVALID_ARG, "exchange_bytes: NULL argument");
  *bytes = s->shards.empty() ? s->exchange_bytes : s->shards[0]->exchange_bytes;
  return QIPB200_OK;
}

extern "C" int qipb200_plan_exchanges(qip_prec prec, uint32_t n_qubits, int world_size, const qip_op *ops,
                                      size_t n_ops, uint32_t *needs_exchange) {
  if (!is_pow2(world_size) || (!ops && n_ops) || !needs_exchange)
    return set_err(nullptr, QIPB200_ERR_INVALID_ARG, "plan_exchanges: bad argument");
  return guarded(nullptr, [&]() -> int {
    const uint32_t n_local = n_qubits - (uint32_t)ilog2(world_size);
    for (size_t i = 0; i < n_ops; ++i) {
      FlatOp f;
      std::string err;
      int st = compile_op(&ops[i], prec, n_qubits, &f, &err);
      if (st != QIPB200_OK) return set_err(nullptr, st, err);
      std::vector<uint32_t> nd;
      nondiag_bits(f, &nd);
      uint32_t cnt = 0;
      for (size_t j = 0; j < nd.size(); ++j) cnt += nd[j] >= n_local;
      needs_exchange[i] = cnt;
    }
    return (int)QIPB200_OK;
  });
}
