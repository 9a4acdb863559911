// kernels.cu -- per-gate sm_100a kernels of libqipb200.
//
// Data layout: the (local) state is one HBM buffer of 2^n amplitudes, interleaved
// (re,im) of float or double == `&[Complex<P>]` of the reference.  Qubit q lives at
// index bit n-1-q (qip-iterators/src/matrix_ops.rs:12-21).
//
// All gate kernels except k_gather work IN PLACE: a k-qubit gate only couples the
// 2^k amplitudes that differ in its target bits, so one thread owns one such group
// (times VEC neighbouring groups that share a 16-byte access), reads it once and
// writes it once.  Algorithmic traffic per gate = 2 * 2^n * sizeof(amplitude)
// (SURVEY.md section 8d); controlled / diagonal gates touch only the amplitudes the
// reference would change (its identity rows multiply by exactly 1).
//
// Every kernel is HBM-bound (<= 2 flop/B for k<=2): the design rules are full
// 32-byte-sector utilisation on both streams, 16-byte accesses per lane, and
// enough independent loads in flight per SM.
#include "kernels.cuh"

#include <algorithm>
#include <cstdio>

namespace qipb200 {

// ---------------------------------------------------------------------------------
// helpers
// ---------------------------------------------------------------------------------

template <typename R>
struct Vec2;
template <>
struct Vec2<float> {
  typedef float2 type;
};
template <>
struct Vec2<double> {
  typedef double2 type;
};

// A lane's access: VEC consecutive amplitudes (16 bytes for <double,1> and <float,2>).
template <typename R, int VEC>
struct Pack {
  R re[VEC], im[VEC];
};

template <typename R, int VEC>
__device__ __forceinline__ Pack<R, VEC> ld_pack(const R *psi, uint64_t amp_index);
template <typename R, int VEC>
__device__ __forceinline__ void st_pack(R *psi, uint64_t amp_index, const Pack<R, VEC> &p);

template <>
__device__ __forceinline__ Pack<double, 1> ld_pack<double, 1>(const double *psi, uint64_t i) {
  double2 v = *reinterpret_cast<const double2 *>(psi + 2 * i);
  Pack<double, 1> p;
  p.re[0] = v.x;
  p.im[0] = v.y;
  return p;
}
template <>
__device__ __forceinline__ void st_pack<double, 1>(double *psi, uint64_t i, const Pack<double, 1> &p) {
  *reinterpret_cast<double2 *>(psi + 2 * i) = make_double2(p.re[0], p.im[0]);
}
template <>
__device__ __forceinline__ Pack<float, 1> ld_pack<float, 1>(const float *psi, uint64_t i) {
  float2 v = *reinterpret_cast<const float2 *>(psi + 2 * i);
  Pack<float, 1> p;
  p.re[0] = v.x;
  p.im[0] = v.y;
  return p;
}
template <>
__device__ __forceinline__ void st_pack<float, 1>(float *psi, uint64_t i, const Pack<float, 1> &p) {
  *reinterpret_cast<float2 *>(psi + 2 * i) = make_float2(p.re[0], p.im[0]);
}
template <>
__device__ __forceinline__ Pack<float, 2> ld_pack<float, 2>(const float *psi, uint64_t i) {
  float4 v = *reinterpret_cast<const float4 *>(psi + 2 * i);
  Pack<float, 2> p;
  p.re[0] = v.x;
  p.im[0] = v.y;
  p.re[1] = v.z;
  p.im[1] = v.w;
  return p;
}
template <>
__device__ __forceinline__ void st_pack<float, 2>(float *psi, uint64_t i, const Pack<float, 2> &p) {
  *reinterpret_cast<float4 *>(psi + 2 * i) = make_float4(p.re[0], p.im[0], p.re[1], p.im[1]);
}

// Work-item index -> amplitude index: re-insert a zero bit at each (ascending) position.
struct InsArgs {
  uint32_t n_ins;
  uint32_t pos[kMaxIns];
};

__device__ __forceinline__ uint64_t expand_index(uint64_t w, const InsArgs &ins) {
  uint64_t idx = w;
  for (uint32_t i = 0; i < ins.n_ins; ++i) {
    const uint32_t p = ins.pos[i];
    const uint64_t low = idx & ((1ull << p) - 1ull);
    idx = ((idx >> p) << (p + 1)) | low;
  }
  return idx;
}

static const int kThreads = 256;

static inline unsigned grid_for(uint64_t items) { return (unsigned)((items + kThreads - 1) / kThreads); }

// Collect the sorted insertion positions of a control mask plus extra bits.
static bool build_ins(uint64_t ctrl_mask, const uint32_t *extra, uint32_t n_extra, InsArgs *ins) {
  uint64_t all = ctrl_mask;
  for (uint32_t i = 0; i < n_extra; ++i) all |= 1ull << extra[i];
  ins->n_ins = 0;
  for (uint32_t b = 0; b < 64; ++b)
    if ((all >> b) & 1) {
      if (ins->n_ins >= (uint32_t)kMaxIns) return false;
      ins->pos[ins->n_ins++] = b;
    }
  return true;
}

// ---------------------------------------------------------------------------------
// K1/K2 dense block in registers (k <= 4), optional controls.
//   out_sub[u] = sum_v m[u][v] * in_sub[v]    (ops.rs:106 + qubit_iterators.rs:40-55)
// with the block already re-indexed on the host so that bit i of u is the i-th
// smallest target bit (opcompile.cpp: sort_block).
// ---------------------------------------------------------------------------------
template <typename R, int K>
struct DenseArgs {
  InsArgs ins;
  uint64_t ctrl_mask;
  uint64_t n_items;                 // work items (each VEC groups)
  uint64_t off[1 << K];             // amplitude offset of sub-index u
  R mre[1 << K][1 << K];
  R mim[1 << K][1 << K];
};

template <typename R, int K, int VEC>
__global__ void __launch_bounds__(kThreads)
    k_dense(R *__restrict__ psi, const __grid_constant__ DenseArgs<R, K> a) {
  const uint64_t w = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
  if (w >= a.n_items) return;
  const uint64_t base = expand_index(w * VEC, a.ins) | a.ctrl_mask;
  constexpr int S = 1 << K;
  Pack<R, VEC> in[S];
#pragma unroll
  for (int u = 0; u < S; ++u) in[u] = ld_pack<R, VEC>(psi, base + a.off[u]);
#pragma unroll
  for (int u = 0; u < S; ++u) {
    Pack<R, VEC> o;
#pragma unroll
    for (int l = 0; l < VEC; ++l) {
      R re = (R)0, im = (R)0;
#pragma unroll
      for (int v = 0; v < S; ++v) {
        const R mr = a.mre[u][v], mi = a.mim[u][v];
        re = fma(mr, in[v].re[l], re);
        re = fma(-mi, in[v].im[l], re);
        im = fma(mr, in[v].im[l], im);
        im = fma(mi, in[v].re[l], im);
      }
      o.re[l] = re;
      o.im[l] = im;
    }
    st_pack<R, VEC>(psi, base + a.off[u], o);
  }
}

template <typename R, int K>
static cudaError_t launch_dense_t(R *psi, uint32_t n_local, const FlatOp &f, cudaStream_t s,
                                  uint64_t *launches) {
  DenseArgs<R, K> a;
  if (!build_ins(f.ctrl_mask, f.tgt_sorted.data(), K, &a.ins)) return cudaErrorInvalidValue;
  a.ctrl_mask = f.ctrl_mask;
  constexpr int S = 1 << K;
  for (int u = 0; u < S; ++u) {
    uint64_t off = 0;
    for (int i = 0; i < K; ++i)
      if ((u >> i) & 1) off |= 1ull << f.tgt_sorted[i];
    a.off[u] = off;
    for (int v = 0; v < S; ++v) {
      a.mre[u][v] = (R)f.m_sorted[(size_t)u * S + v].real();
      a.mim[u][v] = (R)f.m_sorted[(size_t)u * S + v].imag();
    }
  }
  const uint64_t groups = 1ull << (n_local - a.ins.n_ins);
  // 16-byte lane accesses: two f32 amplitudes per access when no involved bit is bit 0.
  const bool vec2 = sizeof(R) == 4 && a.ins.pos[0] >= 1 && groups >= 2;
  if (vec2) {
    a.n_items = groups / 2;
    k_dense<R, K, (sizeof(R) == 4 ? 2 : 1)><<<grid_for(a.n_items), kThreads, 0, s>>>(psi, a);
  } else {
    a.n_items = groups;
    k_dense<R, K, 1><<<grid_for(a.n_items), kThreads, 0, s>>>(psi, a);
  }
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_dense(qip_prec prec, void *psi, uint32_t n_local, const FlatOp &f, cudaStream_t s,
                         uint64_t *launches) {
  const int K = (int)f.tgt_sorted.size();
#define DISPATCH(KK)                                                                              \
  case KK:                                                                                        \
    return prec == QIP_F32 ? launch_dense_t<float, KK>((float *)psi, n_local, f, s, launches)     \
                           : launch_dense_t<double, KK>((double *)psi, n_local, f, s, launches);
  switch (K) {
    DISPATCH(1)
    DISPATCH(2)
    DISPATCH(3)
    DISPATCH(4)
    default:
      return cudaErrorInvalidValue;
  }
#undef DISPATCH
}

// ---------------------------------------------------------------------------------
// K2 dense block on 5 target bits, in place: the 32 amplitudes of a group live in the registers of
// one thread (as for k <= 4), the 32 x 32 matrix in shared memory (16 KiB f64), read with broadcast
// 16-byte loads -- one LDS per four FMAs, every lane of a warp asks for the same entry.  Lanes run
// over neighbouring groups, so both the 32 loads and the 32 stores of a warp-instruction cover
// contiguous runs (the lowest non-target bits are the lane bits).  FP64: 128 FMA per amplitude, 4 flop/B
// beyond the HBM ridge of a B200 -- this kernel is FP64-pipe bound, not HBM bound (SURVEY.md section 7).
// Two output rows are accumulated at a time (four independent FMA chains).
// ---------------------------------------------------------------------------------
struct WideArgs {
  InsArgs ins;
  uint64_t ctrl_mask;
  uint64_t n_items;
  uint64_t off[32];  // amplitude offset of sub-index u (k = 5)
};

template <typename R>
__global__ void __launch_bounds__(128)
    k_dense5(R *__restrict__ psi, const R *__restrict__ mat, const __grid_constant__ WideArgs a) {
  typedef typename Vec2<R>::type V;
  __shared__ V m[32 * 32];
  for (int i = threadIdx.x; i < 32 * 32; i += 128) m[i] = reinterpret_cast<const V *>(mat)[i];
  __syncthreads();
  const uint64_t w = (uint64_t)blockIdx.x * 128 + threadIdx.x;
  if (w >= a.n_items) return;
  const uint64_t base = expand_index(w, a.ins) | a.ctrl_mask;
  V x[32];
#pragma unroll
  for (int v = 0; v < 32; ++v) x[v] = *reinterpret_cast<const V *>(psi + 2 * (base + a.off[v]));
#pragma unroll 1
  for (int u = 0; u < 32; u += 2) {
    R r0 = (R)0, i0 = (R)0, r1 = (R)0, i1 = (R)0;
    const V *row0 = m + u * 32, *row1 = row0 + 32;
#pragma unroll
    for (int v = 0; v < 32; ++v) {
      const V c0 = row0[v], c1 = row1[v];
      r0 = fma(c0.x, x[v].x, r0);
      r0 = fma(-c0.y, x[v].y, r0);
      i0 = fma(c0.x, x[v].y, i0);
      i0 = fma(c0.y, x[v].x, i0);
      r1 = fma(c1.x, x[v].x, r1);
      r1 = fma(-c1.y, x[v].y, r1);
      i1 = fma(c1.x, x[v].y, i1);
      i1 = fma(c1.y, x[v].x, i1);
    }
    V o0, o1;
    o0.x = r0, o0.y = i0, o1.x = r1, o1.y = i1;
    *reinterpret_cast<V *>(psi + 2 * (base + a.off[u])) = o0;  // the group is this thread's alone: its inputs are in x[]
    *reinterpret_cast<V *>(psi + 2 * (base + a.off[u + 1])) = o1;
  }
}

// Dense block on 6..10 target bits, in place: a CTA stages 2^k groups' worth of amplitudes (x 2^c
// neighbouring groups, k + c = 12: 4096 amplitudes) in shared memory, every thread accumulates 16 outputs
// from the staged inputs and the matrix (read through L1/L2: all lanes of a warp share the entry), the tile
// is written back after a barrier.  Compute bound by a wide margin (2^k complex MACs per amplitude):
// correctness and "never unsupported" rather than speed-of-light.
struct BigArgs {
  InsArgs ins;        // target + control positions (ascending)
  uint64_t ctrl_mask;
  uint64_t n_tiles;
  uint32_t k, c;      // c = companion groups per tile (log2)
  uint64_t off[10];   // amplitude offset of target bit i
};

template <typename R>
__global__ void __launch_bounds__(256)
    k_dense_big(R *__restrict__ psi, const R *__restrict__ mat, const __grid_constant__ BigArgs a) {
  typedef typename Vec2<R>::type V;
  extern __shared__ __align__(16) unsigned char smem_big[];
  V *x = reinterpret_cast<V *>(smem_big);  // x[v * C + cc]
  const uint32_t S = 1u << a.k, C = 1u << a.c;
  const uint64_t tile = blockIdx.x;
  if (tile >= a.n_tiles) return;
  for (uint32_t e = threadIdx.x; e < S * C; e += 256) {
    const uint32_t v = e >> a.c, cc = e & (C - 1u);
    uint64_t idx = expand_index(tile * C + cc, a.ins) | a.ctrl_mask;
    for (uint32_t i = 0; i < a.k; ++i)
      if ((v >> i) & 1u) idx += a.off[i];
    x[e] = *reinterpret_cast<const V *>(psi + 2 * idx);
  }
  __syncthreads();
  const uint32_t per = (S * C) / 256u;  // outputs per thread (16 for k + c = 12)
  V out[16];
  const uint32_t cc = threadIdx.x & (C - 1u), u0 = threadIdx.x >> a.c, ustep = 256u >> a.c;
  for (uint32_t q = 0; q < per; ++q) {
    const uint32_t u = u0 + q * ustep;
    const V *row = reinterpret_cast<const V *>(mat) + (size_t)u * S;
    R re = (R)0, im = (R)0;
    for (uint32_t v = 0; v < S; ++v) {
      const V cm = __ldg(row + v);
      const V xv = x[v * C + cc];
      re = fma(cm.x, xv.x, re);
      re = fma(-cm.y, xv.y, re);
      im = fma(cm.x, xv.y, im);
      im = fma(cm.y, xv.x, im);
    }
    out[q].x = re;
    out[q].y = im;
  }
  __syncthreads();
  for (uint32_t q = 0; q < per; ++q) {
    const uint32_t u = u0 + q * ustep;
    uint64_t idx = expand_index(tile * C + cc, a.ins) | a.ctrl_mask;
    for (uint32_t i = 0; i < a.k; ++i)
      if ((u >> i) & 1u) idx += a.off[i];
    *reinterpret_cast<V *>(psi + 2 * idx) = out[q];
  }
}

// ---------------------------------------------------------------------------------
// f64 dense blocks on 5 / 6 target bits on the FP64 TENSOR pipe (DMMA, mma.sync.m8n8k4.f64 -- the only tensor path
// for f64: tcgen05 has no f64 kind).  Y(S x G) = U(S x S) X(S x G) over G groups, complex as four real products:
//   Yr += Ur Xr;  Yr += (-Ui) Xi;  Yi += Ui Xr;  Yi += Ur Xi.
// A warp owns 8 * NT groups: it loads their amplitudes straight into B fragments (lane <-> sub-index v = 4 ks + lane % 4
// of group 8 nt + lane / 4: one 16-byte load yields the re and the im operand; neighbouring lanes cover neighbouring
// v, neighbouring quads neighbouring groups, so every 32-byte sector of a warp load is used whole), walks the matrix
// from shared memory (one conflict-free LDS.128 per 4 * NT DMMAs: rows padded by 4 entries) and stores the D fragments
// (rows 8 mt + lane / 4 of groups 8 nt + 2 (lane % 4) + {0, 1}) in place -- all its inputs are in registers by then.
// ---------------------------------------------------------------------------------
struct DmmaArgs {
  InsArgs ins;
  uint64_t ctrl_mask;
  uint64_t n_items;    // groups (a power of two >= 8 * NT)
  uint64_t off_lo[8];  // amplitude offset of sub-index v, v < 8
  uint64_t off_k[16];  // ... of v = 4 ks
  uint64_t off_m[8];   // ... of v = 8 mt
};

__device__ __forceinline__ void dmma_8x8x4(double &d0, double &d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

template <int K, int NT>
__global__ void __launch_bounds__(128)
    k_dense_dmma(double *__restrict__ psi, const double *__restrict__ mat, const __grid_constant__ DmmaArgs a) {
  constexpr int S = 1 << K, LD = S + 4, MT = S / 8, KS = S / 4;
  extern __shared__ __align__(16) unsigned char smem_dmma[];
  double2 *U = reinterpret_cast<double2 *>(smem_dmma);
  for (int i = threadIdx.x; i < S * S; i += 128) U[(i >> K) * LD + (i & (S - 1))] = reinterpret_cast<const double2 *>(mat)[i];
  __syncthreads();
  const int lane = threadIdx.x & 31, q = lane >> 2, r = lane & 3;
  const uint64_t w0 = ((uint64_t)blockIdx.x * 4 + (threadIdx.x >> 5)) * (8 * NT);
  if (w0 >= a.n_items) return;
  // B fragments: the warp's inputs
  double xr[KS][NT], xi[KS][NT];
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) {
    const uint64_t base = (expand_index(w0 + 8 * nt + q, a.ins) | a.ctrl_mask) + a.off_lo[r];
#pragma unroll
    for (int ks = 0; ks < KS; ++ks) {
      const double2 v = *reinterpret_cast<const double2 *>(psi + 2 * (base + a.off_k[ks]));
      xr[ks][nt] = v.x;
      xi[ks][nt] = v.y;
    }
  }
  uint64_t obase[NT][2];
#pragma unroll
  for (int nt = 0; nt < NT; ++nt)
#pragma unroll
    for (int j = 0; j < 2; ++j) obase[nt][j] = (expand_index(w0 + 8 * nt + 2 * r + j, a.ins) | a.ctrl_mask) + a.off_lo[q];
#pragma unroll
  for (int mt = 0; mt < MT; ++mt) {
    double yr[NT][2], yi[NT][2];
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) yr[nt][0] = yr[nt][1] = yi[nt][0] = yi[nt][1] = 0.0;
    const double2 *urow = U + (8 * mt + q) * LD + r;
#pragma unroll
    for (int ks = 0; ks < KS; ++ks) {
      const double2 u = urow[4 * ks];
      const double nui = -u.y;
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        dmma_8x8x4(yr[nt][0], yr[nt][1], u.x, xr[ks][nt]);
        dmma_8x8x4(yr[nt][0], yr[nt][1], nui, xi[ks][nt]);
        dmma_8x8x4(yi[nt][0], yi[nt][1], u.y, xr[ks][nt]);
        dmma_8x8x4(yi[nt][0], yi[nt][1], u.x, xi[ks][nt]);
      }
    }
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        double2 o;
        o.x = yr[nt][j];
        o.y = yi[nt][j];
        *reinterpret_cast<double2 *>(psi + 2 * (obase[nt][j] + a.off_m[mt])) = o;
      }
  }
}

template <int K, int NT>
static cudaError_t launch_dense_dmma(double *psi, uint32_t n_local, const FlatOp &f, const double *d_mat, cudaStream_t s) {
  constexpr int S = 1 << K;
  DmmaArgs a;
  memset(&a, 0, sizeof(a));
  if (!build_ins(f.ctrl_mask, f.tgt_sorted.data(), K, &a.ins)) return cudaErrorInvalidValue;
  a.ctrl_mask = f.ctrl_mask;
  a.n_items = 1ull << (n_local - a.ins.n_ins);
  auto off_of = [&](uint32_t v) {
    uint64_t off = 0;
    for (uint32_t i = 0; i < (uint32_t)K; ++i)
      if ((v >> i) & 1) off |= 1ull << f.tgt_sorted[i];
    return off;
  };
  for (uint32_t v = 0; v < 8; ++v) a.off_lo[v] = off_of(v);
  for (uint32_t ks = 0; ks < (uint32_t)S / 4; ++ks) a.off_k[ks] = off_of(4 * ks);
  for (uint32_t mt = 0; mt < (uint32_t)S / 8; ++mt) a.off_m[mt] = off_of(8 * mt);
  const size_t smem = (size_t)S * (S + 4) * sizeof(double2);
  if (smem > 48 * 1024) {  // a per-device opt-in: set it on the current device every time (cheap)
    cudaError_t e = cudaFuncSetAttribute((const void *)k_dense_dmma<K, NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  const uint64_t per_cta = 4ull * 8 * NT;
  k_dense_dmma<K, NT><<<(unsigned)((a.n_items + per_cta - 1) / per_cta), 128, smem, s>>>(psi, d_mat, a);
  return cudaGetLastError();
}

// QIPB200_DENSE_DMMA=0: f64 blocks on 5 / 6 bits on the FMA kernels (k_dense5 / k_dense_big) instead of the tensor pipe.
// (4-bit blocks stay on k_dense<4>: they are HBM-bound, and the fragment layout's half-sector stores cost more than the
// tensor pipe saves -- measured on B200, N=26, 200 blocks: 88.0 ms (8 * 2 groups per warp) / 105.9 ms (8 * 4) vs 73.9 ms,
// profiles/r2s_dense4_dmma_ab.txt.)
static bool dense_dmma_enabled() {
  static const bool on = []() {
    const char *e = getenv("QIPB200_DENSE_DMMA");
    return !e || atoi(e) != 0;
  }();
  return on;
}

template <typename R>
static cudaError_t launch_dense_wide_t(R *psi, uint32_t n_local, const FlatOp &f, cudaStream_t s, uint64_t *launches) {
  const uint32_t K = (uint32_t)f.tgt_sorted.size();
  const size_t S = (size_t)1 << K;
  // the matrix travels through a stream-ordered device allocation (16 KiB .. 16 MiB)
  std::vector<R> host(2 * S * S);
  for (size_t i = 0; i < S * S; ++i) {
    host[2 * i] = (R)f.m_sorted[i].real();
    host[2 * i + 1] = (R)f.m_sorted[i].imag();
  }
  R *d_mat = nullptr;
  cudaError_t e = cudaMallocAsync((void **)&d_mat, host.size() * sizeof(R), s);
  if (e != cudaSuccess) return e;
  e = cudaMemcpyAsync(d_mat, host.data(), host.size() * sizeof(R), cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);  // `host` is pageable and leaves scope
  if (e != cudaSuccess) {
    cudaFreeAsync(d_mat, s);
    return e;
  }
  const uint32_t n_ins = K + (uint32_t)__builtin_popcountll(f.ctrl_mask);
  if (sizeof(R) == 8 && (K == 5 || K == 6) && n_local >= n_ins + 4 && dense_dmma_enabled()) {
    e = K == 5 ? launch_dense_dmma<5, 2>((double *)psi, n_local, f, (const double *)d_mat, s)
               : launch_dense_dmma<6, 1>((double *)psi, n_local, f, (const double *)d_mat, s);
    ++*launches;
    cudaFreeAsync(d_mat, s);
    return e;
  }
  if (K == 5) {
    WideArgs a;
    if (!build_ins(f.ctrl_mask, f.tgt_sorted.data(), K, &a.ins)) return cudaFreeAsync(d_mat, s), cudaErrorInvalidValue;
    a.ctrl_mask = f.ctrl_mask;
    for (uint32_t u = 0; u < 32; ++u) {
      uint64_t off = 0;
      for (uint32_t i = 0; i < K; ++i)
        if ((u >> i) & 1) off |= 1ull << f.tgt_sorted[i];
      a.off[u] = off;
    }
    a.n_items = 1ull << (n_local - n_ins);
    k_dense5<R><<<(unsigned)((a.n_items + 127) / 128), 128, 0, s>>>(psi, d_mat, a);
  } else {
    BigArgs a;
    if (!build_ins(f.ctrl_mask, f.tgt_sorted.data(), K, &a.ins)) return cudaFreeAsync(d_mat, s), cudaErrorInvalidValue;
    a.ctrl_mask = f.ctrl_mask;
    a.k = K;
    const uint32_t groups_log2 = n_local - n_ins;
    a.c = std::min<uint32_t>(12u - std::min(12u, K), groups_log2);
    if (K + a.c < 8) a.c = std::min<uint32_t>(8u - K, groups_log2);  // at least one output per thread
    if ((1u << (K + a.c)) < 256u || ((1u << (K + a.c)) / 256u) > 16u) return cudaFreeAsync(d_mat, s), cudaErrorInvalidValue;
    for (uint32_t i = 0; i < K; ++i) a.off[i] = 1ull << f.tgt_sorted[i];
    a.n_tiles = 1ull << (groups_log2 - a.c);
    const size_t smem = ((size_t)2 * sizeof(R)) << (K + a.c);
    // > 48 KiB of dynamic shared memory is a per-device opt-in: set it on the current device every time (cheap)
    e = cudaFuncSetAttribute((const void *)k_dense_big<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
    if (e != cudaSuccess) return cudaFreeAsync(d_mat, s), e;
    k_dense_big<R><<<(unsigned)a.n_tiles, 256, smem, s>>>(psi, d_mat, a);
  }
  ++*launches;
  e = cudaGetLastError();
  cudaFreeAsync(d_mat, s);
  return e;
}

cudaError_t launch_dense_wide(qip_prec prec, void *psi, uint32_t n_local, const FlatOp &f, cudaStream_t s,
                              uint64_t *launches) {
  const size_t K = f.tgt_sorted.size();
  if (K < 5 || K > 10 || K + (size_t)__builtin_popcountll(f.ctrl_mask) > (size_t)kMaxIns) return cudaErrorInvalidValue;
  return prec == QIP_F32 ? launch_dense_wide_t<float>((float *)psi, n_local, f, s, launches)
                         : launch_dense_wide_t<double>((double *)psi, n_local, f, s, launches);
}

// ---------------------------------------------------------------------------------
// K5 diagonal: a[i] *= d[sub(i)] on the amplitudes whose control bits are all 1.
// After promotion (opcompile.cpp) T/S/Z/CZ/controlled-phase are a single scalar on
// a bit mask: only 1/2 .. 1/4 of the state is touched.
// ---------------------------------------------------------------------------------
template <typename R>
struct DiagArgs {
  InsArgs ins;  // control positions only
  uint64_t ctrl_mask;
  uint64_t n_items;
  uint32_t n_bits;
  uint32_t bits[kMaxDiagParamK];
  R dre[1 << kMaxDiagParamK];
  R dim[1 << kMaxDiagParamK];
};

template <typename R, int VEC>
__global__ void __launch_bounds__(kThreads)
    k_diag(R *__restrict__ psi, const __grid_constant__ DiagArgs<R> a) {
  const uint64_t w = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
  if (w >= a.n_items) return;
  const uint64_t base = expand_index(w * VEC, a.ins) | a.ctrl_mask;
  Pack<R, VEC> p = ld_pack<R, VEC>(psi, base);
#pragma unroll
  for (int l = 0; l < VEC; ++l) {
    const uint64_t i = base + l;
    uint32_t u = 0;
    for (uint32_t j = 0; j < a.n_bits; ++j) u |= (uint32_t)((i >> a.bits[j]) & 1ull) << j;
    const R dr = a.dre[u], di = a.dim[u];
    const R re = p.re[l], im = p.im[l];
    p.re[l] = fma(dr, re, -di * im);
    p.im[l] = fma(dr, im, di * re);
  }
  st_pack<R, VEC>(psi, base, p);
}

template <typename R>
static cudaError_t launch_diag_t(R *psi, uint32_t n_local, uint64_t ctrl_mask,
                                 const std::vector<uint32_t> &bits, const std::vector<cplx> &d,
                                 cudaStream_t s, uint64_t *launches) {
  DiagArgs<R> a;
  if (bits.size() > (size_t)kMaxDiagParamK) return cudaErrorInvalidValue;
  if (!build_ins(ctrl_mask, nullptr, 0, &a.ins)) return cudaErrorInvalidValue;
  a.ctrl_mask = ctrl_mask;
  a.n_bits = (uint32_t)bits.size();
  for (size_t j = 0; j < bits.size(); ++j) a.bits[j] = bits[j];
  for (size_t u = 0; u < d.size(); ++u) {
    a.dre[u] = (R)d[u].real();
    a.dim[u] = (R)d[u].imag();
  }
  const uint64_t groups = 1ull << (n_local - a.ins.n_ins);
  const bool vec2 = sizeof(R) == 4 && (a.ins.n_ins == 0 || a.ins.pos[0] >= 1) && groups >= 2;
  if (vec2) {
    a.n_items = groups / 2;
    k_diag<R, (sizeof(R) == 4 ? 2 : 1)><<<grid_for(a.n_items), kThreads, 0, s>>>(psi, a);
  } else {
    a.n_items = groups;
    k_diag<R, 1><<<grid_for(a.n_items), kThreads, 0, s>>>(psi, a);
  }
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_diag(qip_prec prec, void *psi, uint32_t n_local, uint64_t ctrl_mask,
                        const std::vector<uint32_t> &bits, const std::vector<cplx> &d, cudaStream_t s,
                        uint64_t *launches) {
  return prec == QIP_F32 ? launch_diag_t<float>((float *)psi, n_local, ctrl_mask, bits, d, s, launches)
                         : launch_diag_t<double>((double *)psi, n_local, ctrl_mask, bits, d, s, launches);
}

// Diagonal on 5..10 bits: the table (<= 1024 entries) is staged in shared memory per CTA; grid-stride over
// the touched amplitudes.  HBM bound like k_diag: one read + one write per touched amplitude.
struct DiagWideArgs {
  InsArgs ins;  // control positions only
  uint64_t ctrl_mask;
  uint64_t n_items;
  uint32_t n_bits;
  uint32_t bits[10];
};

template <typename R>
__global__ void __launch_bounds__(kThreads)
    k_diag_wide(R *__restrict__ psi, const R *__restrict__ table, const __grid_constant__ DiagWideArgs a) {
  typedef typename Vec2<R>::type V;
  __shared__ V tb[1024];
  const uint32_t entries = 1u << a.n_bits;
  for (uint32_t i = threadIdx.x; i < entries; i += kThreads) tb[i] = reinterpret_cast<const V *>(table)[i];
  __syncthreads();
  for (uint64_t w = (uint64_t)blockIdx.x * kThreads + threadIdx.x; w < a.n_items; w += (uint64_t)gridDim.x * kThreads) {
    const uint64_t i = expand_index(w, a.ins) | a.ctrl_mask;
    uint32_t u = 0;
    for (uint32_t j = 0; j < a.n_bits; ++j) u |= (uint32_t)((i >> a.bits[j]) & 1ull) << j;
    const V d = tb[u];
    V v = *reinterpret_cast<const V *>(psi + 2 * i);
    const R re = v.x, im = v.y;
    v.x = fma(d.x, re, -d.y * im);
    v.y = fma(d.x, im, d.y * re);
    *reinterpret_cast<V *>(psi + 2 * i) = v;
  }
}

template <typename R>
static cudaError_t launch_diag_wide_t(R *psi, uint32_t n_local, uint64_t ctrl_mask, const std::vector<uint32_t> &bits,
                                      const std::vector<cplx> &d, cudaStream_t s, uint64_t *launches) {
  DiagWideArgs a;
  if (bits.size() > 10 || d.size() != ((size_t)1 << bits.size())) return cudaErrorInvalidValue;
  if (!build_ins(ctrl_mask, nullptr, 0, &a.ins)) return cudaErrorInvalidValue;
  a.ctrl_mask = ctrl_mask;
  a.n_bits = (uint32_t)bits.size();
  for (size_t j = 0; j < bits.size(); ++j) a.bits[j] = bits[j];
  a.n_items = 1ull << (n_local - a.ins.n_ins);
  std::vector<R> host(2 * d.size());
  for (size_t u = 0; u < d.size(); ++u) {
    host[2 * u] = (R)d[u].real();
    host[2 * u + 1] = (R)d[u].imag();
  }
  R *d_tab = nullptr;
  cudaError_t e = cudaMallocAsync((void **)&d_tab, host.size() * sizeof(R), s);
  if (e != cudaSuccess) return e;
  e = cudaMemcpyAsync(d_tab, host.data(), host.size() * sizeof(R), cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  if (e == cudaSuccess) {
    const unsigned grid = (unsigned)std::min<uint64_t>((a.n_items + kThreads - 1) / kThreads, 148ull * 32);
    k_diag_wide<R><<<grid ? grid : 1, kThreads, 0, s>>>(psi, d_tab, a);
    ++*launches;
    e = cudaGetLastError();
  }
  cudaFreeAsync(d_tab, s);
  return e;
}

cudaError_t launch_diag_wide(qip_prec prec, void *psi, uint32_t n_local, uint64_t ctrl_mask,
                             const std::vector<uint32_t> &bits, const std::vector<cplx> &d, cudaStream_t s,
                             uint64_t *launches) {
  return prec == QIP_F32 ? launch_diag_wide_t<float>((float *)psi, n_local, ctrl_mask, bits, d, s, launches)
                         : launch_diag_wide_t<double>((double *)psi, n_local, ctrl_mask, bits, d, s, launches);
}

// ---------------------------------------------------------------------------------
// K4 permutations: X / CNOT / Toffoli-X (pair exchange on one bit) and Swap (exchange
// of two index bits), both under a control mask.  Pure moves: bit-exact.
// ---------------------------------------------------------------------------------
struct PermArgs {
  InsArgs ins;
  uint64_t ctrl_mask;
  uint64_t n_items;
  uint64_t off_a, off_b;  // the two amplitude offsets that trade places
};

template <typename R, int VEC>
__global__ void __launch_bounds__(kThreads)
    k_exchange(R *__restrict__ psi, const __grid_constant__ PermArgs a) {
  const uint64_t w = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
  if (w >= a.n_items) return;
  const uint64_t base = expand_index(w * VEC, a.ins) | a.ctrl_mask;
  const Pack<R, VEC> x = ld_pack<R, VEC>(psi, base + a.off_a);
  const Pack<R, VEC> y = ld_pack<R, VEC>(psi, base + a.off_b);
  st_pack<R, VEC>(psi, base + a.off_a, y);
  st_pack<R, VEC>(psi, base + a.off_b, x);
}

template <typename R>
static cudaError_t launch_exchange_t(R *psi, uint32_t n_local, PermArgs &a, cudaStream_t s,
                                     uint64_t *launches) {
  const uint64_t groups = 1ull << (n_local - a.ins.n_ins);
  const bool vec2 = sizeof(R) == 4 && a.ins.pos[0] >= 1 && groups >= 2;
  if (vec2) {
    a.n_items = groups / 2;
    k_exchange<R, (sizeof(R) == 4 ? 2 : 1)><<<grid_for(a.n_items), kThreads, 0, s>>>(psi, a);
  } else {
    a.n_items = groups;
    k_exchange<R, 1><<<grid_for(a.n_items), kThreads, 0, s>>>(psi, a);
  }
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_flip(qip_prec prec, void *psi, uint32_t n_local, uint64_t ctrl_mask, uint32_t tbit,
                        cudaStream_t s, uint64_t *launches) {
  PermArgs a;
  if (!build_ins(ctrl_mask, &tbit, 1, &a.ins)) return cudaErrorInvalidValue;
  a.ctrl_mask = ctrl_mask;
  a.off_a = 0;
  a.off_b = 1ull << tbit;
  return prec == QIP_F32 ? launch_exchange_t<float>((float *)psi, n_local, a, s, launches)
                         : launch_exchange_t<double>((double *)psi, n_local, a, s, launches);
}

cudaError_t launch_bitswap(qip_prec prec, void *psi, uint32_t n_local, uint64_t ctrl_mask, uint32_t p,
                           uint32_t q, cudaStream_t s, uint64_t *launches) {
  PermArgs a;
  uint32_t both[2] = {p, q};
  if (!build_ins(ctrl_mask, both, 2, &a.ins)) return cudaErrorInvalidValue;
  a.ctrl_mask = ctrl_mask;
  a.off_a = 1ull << p;  // (p=1,q=0) <-> (p=0,q=1); equal bits stay put
  a.off_b = 1ull << q;
  return prec == QIP_F32 ? launch_exchange_t<float>((float *)psi, n_local, a, s, launches)
                         : launch_exchange_t<double>((double *)psi, n_local, a, s, launches);
}

// ---------------------------------------------------------------------------------
// Universal row kernel: one thread == one evaluation of apply_op_row_indices
// (qip-iterators/src/matrix_ops.rs:62-94) for any op kind, with input/output
// offsets and the accumulate (`+=`, :110) / overwrite (`=`, :139) modes.
// Arithmetic is issued with the never-contracted __*_rn intrinsics in the
// reference's order (ascending non-zero columns from a zero accumulator,
// 4-mul/2-add complex product), so results are bit-identical to the CPU path.
// ---------------------------------------------------------------------------------
template <typename R>
struct Arith;
template <>
struct Arith<float> {
  static __device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
  static __device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
  static __device__ __forceinline__ float sub(float a, float b) { return __fsub_rn(a, b); }
};
template <>
struct Arith<double> {
  static __device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
  static __device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
  static __device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
};

struct GatherArgs {
  uint32_t k, kop;
  int base_kind;
  uint64_t thr;
  uint64_t all_mask;       // OR of all idx_bits
  uint32_t idx_bits[24];   // reference order: idx_bits[j] <-> sub-index bit k-1-j
  const void *dense;       // device, 4^kop complex<R>, reference order
  const uint64_t *sp_rowptr, *sp_col;
  const void *sp_val;
  uint64_t in_len, in_off, out_len, out_off;
  int accumulate;
};

template <typename R>
__global__ void __launch_bounds__(kThreads)
    k_gather(const R *__restrict__ in, R *__restrict__ out, const __grid_constant__ GatherArgs a) {
  const uint64_t o = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
  if (o >= a.out_len) return;
  const uint64_t row = a.out_off + o;
  uint64_t matrow = 0;  // full_to_sub, matrix_ops.rs:12-21
  for (uint32_t j = 0; j < a.k; ++j) matrow |= ((row >> a.idx_bits[j]) & 1ull) << (a.k - 1 - j);
  const uint64_t row_cleared = row & ~a.all_mask;
  R ar = (R)0, ai = (R)0;

  auto accum = [&](uint64_t col, R vr, R vi) {
    uint64_t colbits = row_cleared;  // sub_to_full, matrix_ops.rs:24-30
    for (uint32_t j = 0; j < a.k; ++j) colbits |= ((col >> (a.k - 1 - j)) & 1ull) << a.idx_bits[j];
    R tr = (R)0, ti = (R)0;
    if (colbits >= a.in_off) {
      const uint64_t vecrow = colbits - a.in_off;
      if (vecrow < a.in_len) {
        const R pr = in[2 * vecrow], pi = in[2 * vecrow + 1];
        tr = Arith<R>::sub(Arith<R>::mul(vr, pr), Arith<R>::mul(vi, pi));
        ti = Arith<R>::add(Arith<R>::mul(vr, pi), Arith<R>::mul(vi, pr));
      }
    }
    ar = Arith<R>::add(ar, tr);
    ai = Arith<R>::add(ai, ti);
  };

  if (matrow < a.thr) {
    accum(matrow, (R)1, (R)0);  // identity row of a control op, qubit_iterators.rs:160-169
  } else {
    const uint64_t r = matrow - a.thr;
    if (a.base_kind == QIP_OP_MATRIX) {
      const R *d = static_cast<const R *>(a.dense) + 2 * (r << a.kop);
      const uint64_t side = 1ull << a.kop;
      for (uint64_t c = 0; c < side; ++c) {
        const R vr = d[2 * c], vi = d[2 * c + 1];
        if (vr == (R)0 && vi == (R)0) continue;  // zero entries are skipped, qubit_iterators.rs:49
        accum(c + a.thr, vr, vi);
      }
    } else if (a.base_kind == QIP_OP_SPARSE) {
      const R *v = static_cast<const R *>(a.sp_val);
      for (uint64_t e = a.sp_rowptr[r]; e < a.sp_rowptr[r + 1]; ++e)
        accum(a.sp_col[e] + a.thr, v[2 * e], v[2 * e + 1]);
    } else {  // swap, qubit_iterators.rs:208-218
      const uint32_t half = a.kop >> 1;
      const uint64_t lower_mask = ~(~0ull << half);
      accum((((r & lower_mask) << half) + (r >> half)) + a.thr, (R)1, (R)0);
    }
  }
  if (a.accumulate) {
    out[2 * o] = Arith<R>::add(out[2 * o], ar);
    out[2 * o + 1] = Arith<R>::add(out[2 * o + 1], ai);
  } else {
    out[2 * o] = ar;
    out[2 * o + 1] = ai;
  }
}

template <typename R>
static cudaError_t launch_gather_t(const FlatOp &f, const R *in, uint64_t in_len, uint64_t in_off, R *out,
                                   uint64_t out_len, uint64_t out_off, bool accumulate, cudaStream_t s,
                                   uint64_t *launches) {
  if (out_len == 0) return cudaSuccess;
  GatherArgs a;
  a.k = f.k;
  a.kop = f.kop;
  a.base_kind = f.base_kind;
  a.thr = f.nc ? ((1ull << f.k) - (1ull << f.kop)) : 0;
  a.all_mask = 0;
  if (f.k > 24) return cudaErrorInvalidValue;
  for (uint32_t j = 0; j < f.k; ++j) {
    a.idx_bits[j] = f.idx_bits[j];
    a.all_mask |= 1ull << f.idx_bits[j];
  }
  a.dense = nullptr;
  a.sp_rowptr = a.sp_col = nullptr;
  a.sp_val = nullptr;
  a.in_len = in_len;
  a.in_off = in_off;
  a.out_len = out_len;
  a.out_off = out_off;
  a.accumulate = accumulate ? 1 : 0;

  void *d_a = nullptr, *d_b = nullptr, *d_c = nullptr;
  cudaError_t e = cudaSuccess;
  std::vector<R> tmp;
  if (f.base_kind == QIP_OP_MATRIX || (f.base_kind == QIP_OP_SPARSE && f.has_dense)) {
    // a densified sparse op is applied as a dense one (duplicates pre-summed)
    a.base_kind = QIP_OP_MATRIX;
    tmp.resize(2 * f.dense.size());
    for (size_t i = 0; i < f.dense.size(); ++i) {
      tmp[2 * i] = (R)f.dense[i].real();
      tmp[2 * i + 1] = (R)f.dense[i].imag();
    }
    if ((e = cudaMallocAsync(&d_a, tmp.size() * sizeof(R), s)) != cudaSuccess) return e;
    if ((e = cudaMemcpyAsync(d_a, tmp.data(), tmp.size() * sizeof(R), cudaMemcpyHostToDevice, s)) != cudaSuccess)
      return e;
    a.dense = d_a;
  } else if (f.base_kind == QIP_OP_SPARSE) {
    tmp.resize(2 * f.sp_val.size());
    for (size_t i = 0; i < f.sp_val.size(); ++i) {
      tmp[2 * i] = (R)f.sp_val[i].real();
      tmp[2 * i + 1] = (R)f.sp_val[i].imag();
    }
    if ((e = cudaMallocAsync(&d_a, tmp.size() * sizeof(R) + 16, s)) != cudaSuccess) return e;
    if ((e = cudaMallocAsync(&d_b, f.sp_rowptr.size() * 8, s)) != cudaSuccess) return e;
    if ((e = cudaMallocAsync(&d_c, f.sp_col.size() * 8 + 16, s)) != cudaSuccess) return e;
    cudaMemcpyAsync(d_a, tmp.data(), tmp.size() * sizeof(R), cudaMemcpyHostToDevice, s);
    cudaMemcpyAsync(d_b, f.sp_rowptr.data(), f.sp_rowptr.size() * 8, cudaMemcpyHostToDevice, s);
    cudaMemcpyAsync(d_c, f.sp_col.data(), f.sp_col.size() * 8, cudaMemcpyHostToDevice, s);
    a.sp_val = d_a;
    a.sp_rowptr = (const uint64_t *)d_b;
    a.sp_col = (const uint64_t *)d_c;
  }
  // the staging vectors are pageable: the async copies above have completed their
  // host read when they return, so `tmp` may go out of scope.
  k_gather<R><<<grid_for(out_len), kThreads, 0, s>>>(in, out, a);
  ++*launches;
  e = cudaGetLastError();
  if (d_a) cudaFreeAsync(d_a, s);
  if (d_b) cudaFreeAsync(d_b, s);
  if (d_c) cudaFreeAsync(d_c, s);
  return e;
}

// ---------------------------------------------------------------------------------
// apply_ops with several ops (qip-iterators/src/matrix_ops.rs:184-217): one thread == one output row of
// sum_for_ops_cols (iterators/iterator_mapper.rs:8-31) over the MultiOpIterator (qubit_multi_iterator.rs:38-78),
// restated as the reference computes it -- op i reads its row from the LOW bits of what is left of matrow
// (iterator_mapper.rs:17-18,24), the column is composed first-op-high (qubit_multi_iterator.rs:48-52), the value is
// ((one * v0) * v1) ..., the cursor of the last op moves fastest and the items are summed from zero in that order
// (SURVEY.md quirk Q5 included: for ops that are not all alike this is not their tensor product).  Same never-
// contracted arithmetic as k_gather, so results are bit-identical to the oracle's restatement.
// ---------------------------------------------------------------------------------
constexpr uint32_t kMultiMaxOps = 8;

struct MultiOpDesc {
  uint32_t k, kop;
  int base_kind;
  uint64_t thr;
  const void *dense;
  const uint64_t *sp_rowptr, *sp_col;
  const void *sp_val;
};

struct MultiGatherArgs {
  uint32_t n_ops, ktot;
  uint64_t all_mask;
  uint32_t idx_bits[40];  // concatenated, reference order: idx_bits[j] <-> sub-index bit ktot-1-j
  MultiOpDesc op[kMultiMaxOps];
  uint64_t in_len, in_off, out_len, out_off;
};

template <typename R>
__global__ void __launch_bounds__(kThreads)
    k_multi_gather(const R *__restrict__ in, R *__restrict__ out, const __grid_constant__ MultiGatherArgs a) {
  const uint64_t o = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
  if (o >= a.out_len) return;
  const uint64_t row = a.out_off + o;
  uint64_t matrow = 0;
  for (uint32_t j = 0; j < a.ktot; ++j) matrow |= ((row >> a.idx_bits[j]) & 1ull) << (a.ktot - 1 - j);
  const uint64_t row_cleared = row & ~a.all_mask;

  uint64_t op_row[kMultiMaxOps], cur[kMultiMaxOps], pcol[kMultiMaxOps + 1];
  R pr[kMultiMaxOps + 1], pi[kMultiMaxOps + 1];
  {
    uint64_t acc_row = matrow;
    for (uint32_t i = 0; i < a.n_ops; ++i) {
      op_row[i] = acc_row & ((1ull << a.op[i].k) - 1ull);
      acc_row >>= a.op[i].k;
    }
  }
  // next entry of op i's row at or after cursor cur[i] (cursor semantics per kind); false when the row is exhausted
  auto next_entry = [&](uint32_t i, uint64_t *col, R *vr, R *vi) -> bool {
    const MultiOpDesc &d = a.op[i];
    if (op_row[i] < d.thr) {  // identity row of a control op: the single entry (row, 1)
      if (cur[i]) return false;
      cur[i] = 1;
      *col = op_row[i];
      *vr = (R)1;
      *vi = (R)0;
      return true;
    }
    const uint64_t r = op_row[i] - d.thr;
    if (d.base_kind == QIP_OP_MATRIX) {
      const R *m = static_cast<const R *>(d.dense) + 2 * (r << d.kop);
      const uint64_t side = 1ull << d.kop;
      for (uint64_t c = cur[i]; c < side; ++c) {
        const R x = m[2 * c], y = m[2 * c + 1];
        if (x == (R)0 && y == (R)0) continue;
        cur[i] = c + 1;
        *col = c + d.thr;
        *vr = x;
        *vi = y;
        return true;
      }
      return false;
    }
    if (d.base_kind == QIP_OP_SPARSE) {
      const uint64_t e = d.sp_rowptr[r] + cur[i];
      if (e >= d.sp_rowptr[r + 1]) return false;
      const R *v = static_cast<const R *>(d.sp_val);
      cur[i] += 1;
      *col = d.sp_col[e] + d.thr;
      *vr = v[2 * e];
      *vi = v[2 * e + 1];
      return true;
    }
    if (cur[i]) return false;  // swap
    cur[i] = 1;
    const uint32_t half = d.kop >> 1;
    const uint64_t lower_mask = ~(~0ull << half);
    *col = (((r & lower_mask) << half) + (r >> half)) + d.thr;
    *vr = (R)1;
    *vi = (R)0;
    return true;
  };

  R ar = (R)0, ai = (R)0;
  pcol[0] = 0;
  pr[0] = (R)1;  // P::one()
  pi[0] = (R)0;
  int lvl = 0;
  cur[0] = 0;
  while (lvl >= 0) {
    uint64_t col;
    R vr, vi;
    if (!next_entry((uint32_t)lvl, &col, &vr, &vi)) {
      --lvl;
      continue;
    }
    pcol[lvl + 1] = (pcol[lvl] << a.op[lvl].k) | col;
    pr[lvl + 1] = Arith<R>::sub(Arith<R>::mul(pr[lvl], vr), Arith<R>::mul(pi[lvl], vi));  // acc_val * val
    pi[lvl + 1] = Arith<R>::add(Arith<R>::mul(pr[lvl], vi), Arith<R>::mul(pi[lvl], vr));
    if ((uint32_t)lvl + 1 < a.n_ops) {
      ++lvl;
      cur[lvl] = 0;
      continue;
    }
    const uint64_t c = pcol[lvl + 1];
    uint64_t colbits = row_cleared;
    for (uint32_t j = 0; j < a.ktot; ++j) colbits |= ((c >> (a.ktot - 1 - j)) & 1ull) << a.idx_bits[j];
    R tr = (R)0, ti = (R)0;
    if (colbits >= a.in_off && colbits - a.in_off < a.in_len) {
      const R xr = in[2 * (colbits - a.in_off)], xi = in[2 * (colbits - a.in_off) + 1];
      tr = Arith<R>::sub(Arith<R>::mul(pr[lvl + 1], xr), Arith<R>::mul(pi[lvl + 1], xi));
      ti = Arith<R>::add(Arith<R>::mul(pr[lvl + 1], xi), Arith<R>::mul(pi[lvl + 1], xr));
    }
    ar = Arith<R>::add(ar, tr);
    ai = Arith<R>::add(ai, ti);
  }
  out[2 * o] = Arith<R>::add(out[2 * o], ar);  // *outputloc += ... (matrix_ops.rs:212)
  out[2 * o + 1] = Arith<R>::add(out[2 * o + 1], ai);
}

template <typename R>
static cudaError_t launch_multi_gather_t(const std::vector<FlatOp> &fs, const R *in, uint64_t in_len, uint64_t in_off, R *out,
                                         uint64_t out_len, uint64_t out_off, cudaStream_t s, uint64_t *launches) {
  if (out_len == 0) return cudaSuccess;
  if (fs.size() < 2 || fs.size() > kMultiMaxOps) return cudaErrorInvalidValue;
  MultiGatherArgs a;
  memset(&a, 0, sizeof(a));
  a.n_ops = (uint32_t)fs.size();
  a.in_len = in_len;
  a.in_off = in_off;
  a.out_len = out_len;
  a.out_off = out_off;
  std::vector<void *> owned;
  cudaError_t e = cudaSuccess;
  auto dev_copy = [&](const void *src, size_t bytes, const void **dst) {
    void *d = nullptr;
    if (e != cudaSuccess) return;
    if ((e = cudaMallocAsync(&d, bytes + 16, s)) != cudaSuccess) return;
    owned.push_back(d);
    if (bytes) e = cudaMemcpyAsync(d, src, bytes, cudaMemcpyHostToDevice, s);
    *dst = d;
  };
  for (size_t i = 0; i < fs.size() && e == cudaSuccess; ++i) {
    const FlatOp &f = fs[i];
    if (a.ktot + f.k > 40) {
      e = cudaErrorInvalidValue;
      break;
    }
    for (uint32_t j = 0; j < f.k; ++j) {
      a.idx_bits[a.ktot++] = f.idx_bits[j];
      a.all_mask |= 1ull << f.idx_bits[j];
    }
    MultiOpDesc &d = a.op[i];
    d.k = f.k;
    d.kop = f.kop;
    d.base_kind = f.base_kind;
    d.thr = f.nc ? ((1ull << f.k) - (1ull << f.kop)) : 0;
    std::vector<R> tmp;
    if (f.base_kind == QIP_OP_MATRIX || (f.base_kind == QIP_OP_SPARSE && f.has_dense)) {
      d.base_kind = QIP_OP_MATRIX;
      tmp.resize(2 * f.dense.size());
      for (size_t t = 0; t < f.dense.size(); ++t) {
        tmp[2 * t] = (R)f.dense[t].real();
        tmp[2 * t + 1] = (R)f.dense[t].imag();
      }
      dev_copy(tmp.data(), tmp.size() * sizeof(R), &d.dense);
    } else if (f.base_kind == QIP_OP_SPARSE) {
      tmp.resize(2 * f.sp_val.size());
      for (size_t t = 0; t < f.sp_val.size(); ++t) {
        tmp[2 * t] = (R)f.sp_val[t].real();
        tmp[2 * t + 1] = (R)f.sp_val[t].imag();
      }
      dev_copy(tmp.data(), tmp.size() * sizeof(R), &d.sp_val);
      dev_copy(f.sp_rowptr.data(), f.sp_rowptr.size() * 8, (const void **)&d.sp_rowptr);
      dev_copy(f.sp_col.data(), f.sp_col.size() * 8, (const void **)&d.sp_col);
    }
  }
  if (e == cudaSuccess) {
    k_multi_gather<R><<<grid_for(out_len), kThreads, 0, s>>>(in, out, a);
    ++*launches;
    e = cudaGetLastError();
  }
  for (size_t i = 0; i < owned.size(); ++i) cudaFreeAsync(owned[i], s);
  return e;
}

cudaError_t launch_multi_gather(qip_prec prec, const std::vector<FlatOp> &fs, const void *in, uint64_t in_len, uint64_t in_off,
                                void *out, uint64_t out_len, uint64_t out_off, cudaStream_t s, uint64_t *launches) {
  return prec == QIP_F32 ? launch_multi_gather_t<float>(fs, (const float *)in, in_len, in_off, (float *)out, out_len, out_off, s, launches)
                         : launch_multi_gather_t<double>(fs, (const double *)in, in_len, in_off, (double *)out, out_len, out_off, s,
                                                         launches);
}

cudaError_t launch_gather(qip_prec prec, const FlatOp &f, uint32_t, const void *in, uint64_t in_len,
                          uint64_t in_off, void *out, uint64_t out_len, uint64_t out_off, bool accumulate,
                          cudaStream_t s, uint64_t *launches) {
  return prec == QIP_F32
             ? launch_gather_t<float>(f, (const float *)in, in_len, in_off, (float *)out, out_len, out_off,
                                      accumulate, s, launches)
             : launch_gather_t<double>(f, (const double *)in, in_len, in_off, (double *)out, out_len,
                                       out_off, accumulate, s, launches);
}

// ---------------------------------------------------------------------------------
// reductions / state set-up / measurement
// ---------------------------------------------------------------------------------
__device__ __forceinline__ double block_sum(double v) {
  __shared__ double sh[kThreads / 32];
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x < 32) {
    v = threadIdx.x < kThreads / 32 ? sh[threadIdx.x] : 0.0;
    for (int o = 4; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  }
  return v;  // valid in thread 0
}

template <typename R>
__global__ void __launch_bounds__(kThreads) k_norm2(const R *__restrict__ psi, uint64_t len, double *out) {
  double acc = 0.0;
  for (uint64_t i = (uint64_t)blockIdx.x * kThreads + threadIdx.x; i < len; i += (uint64_t)gridDim.x * kThreads) {
    typename Vec2<R>::type v = *reinterpret_cast<const typename Vec2<R>::type *>(psi + 2 * i);
    acc += (double)v.x * (double)v.x + (double)v.y * (double)v.y;
  }
  acc = block_sum(acc);
  if (threadIdx.x == 0) atomicAdd(out, acc);
}

cudaError_t launch_norm2(qip_prec prec, const void *psi, uint64_t len, double *d_out, cudaStream_t s,
                         uint64_t *launches) {
  cudaError_t e = cudaMemsetAsync(d_out, 0, sizeof(double), s);
  if (e != cudaSuccess) return e;
  unsigned grid = (unsigned)std::min<uint64_t>((len + kThreads - 1) / kThreads, 148ull * 16);
  if (grid == 0) grid = 1;
  if (prec == QIP_F32)
    k_norm2<float><<<grid, kThreads, 0, s>>>((const float *)psi, len, d_out);
  else
    k_norm2<double><<<grid, kThreads, 0, s>>>((const double *)psi, len, d_out);
  ++*launches;
  return cudaGetLastError();
}

// max over the amplitudes of max(|re_a - re_b|, |im_a - im_b|): the device-side comparison behind
// qipb200_state_max_abs_diff (fused-vs-unfused parity checks at sizes no host oracle reaches).
// Non-negative doubles order like their bit patterns, so the reduction is an atomicMax on u64;
// a NaN difference is reported as +inf.
template <typename R>
__global__ void __launch_bounds__(kThreads) k_maxdiff(const R *__restrict__ a, const R *__restrict__ b, uint64_t len,
                                                      unsigned long long *out) {
  double acc = 0.0;
  for (uint64_t i = (uint64_t)blockIdx.x * kThreads + threadIdx.x; i < len; i += (uint64_t)gridDim.x * kThreads) {
    typename Vec2<R>::type x = *reinterpret_cast<const typename Vec2<R>::type *>(a + 2 * i);
    typename Vec2<R>::type y = *reinterpret_cast<const typename Vec2<R>::type *>(b + 2 * i);
    double d0 = fabs((double)x.x - (double)y.x), d1 = fabs((double)x.y - (double)y.y);
    if (d0 != d0 || d1 != d1) d0 = __longlong_as_double(0x7ff0000000000000ll);
    acc = fmax(acc, fmax(d0, d1));
  }
  for (int o = 16; o > 0; o >>= 1) acc = fmax(acc, __shfl_down_sync(0xffffffffu, acc, o));
  if ((threadIdx.x & 31) == 0) atomicMax(out, (unsigned long long)__double_as_longlong(acc));
}

cudaError_t launch_max_abs_diff(qip_prec prec, const void *a, const void *b, uint64_t len, double *d_out, cudaStream_t s,
                                uint64_t *launches) {
  cudaError_t e = cudaMemsetAsync(d_out, 0, sizeof(double), s);
  if (e != cudaSuccess) return e;
  unsigned grid = (unsigned)std::min<uint64_t>((len + kThreads - 1) / kThreads, 148ull * 16);
  if (grid == 0) grid = 1;
  if (prec == QIP_F32)
    k_maxdiff<float><<<grid, kThreads, 0, s>>>((const float *)a, (const float *)b, len, (unsigned long long *)d_out);
  else
    k_maxdiff<double><<<grid, kThreads, 0, s>>>((const double *)a, (const double *)b, len, (unsigned long long *)d_out);
  ++*launches;
  return cudaGetLastError();
}

template <typename R>
__global__ void k_set_one(R *psi, uint64_t index) {
  psi[2 * index] = (R)1;
  psi[2 * index + 1] = (R)0;
}

cudaError_t launch_set_basis(qip_prec prec, void *psi, uint64_t len, uint64_t index, bool owns_index,
                             cudaStream_t s, uint64_t *launches) {
  const size_t amp = prec == QIP_F32 ? 8 : 16;
  cudaError_t e = cudaMemsetAsync(psi, 0, len * amp, s);
  if (e != cudaSuccess || !owns_index) return e;
  if (prec == QIP_F32)
    k_set_one<float><<<1, 1, 0, s>>>((float *)psi, index);
  else
    k_set_one<double><<<1, 1, 0, s>>>((double *)psi, index);
  ++*launches;
  return cudaGetLastError();
}

// measure_probs (measurement_ops.rs:115-127) as one histogram sweep: every amplitude
// adds |a|^2 to the bin spelled by its measured bits.  Small histograms live in
// shared memory per CTA and are flushed with one atomicAdd per bin.
static const uint32_t kHistSmemBits = 10;

struct HistArgs {
  uint32_t n_bits;
  uint32_t bitpos[32];
  uint64_t len, index_base;
};

template <typename R>
__global__ void __launch_bounds__(kThreads)
    k_hist(const R *__restrict__ psi, double *hist, const __grid_constant__ HistArgs a) {
  __shared__ double sh[1 << kHistSmemBits];
  const bool use_smem = a.n_bits <= kHistSmemBits;
  const uint32_t bins = 1u << a.n_bits;
  if (use_smem) {
    for (uint32_t b = threadIdx.x; b < bins; b += kThreads) sh[b] = 0.0;
    __syncthreads();
  }
  for (uint64_t i = (uint64_t)blockIdx.x * kThreads + threadIdx.x; i < a.len; i += (uint64_t)gridDim.x * kThreads) {
    typename Vec2<R>::type v = *reinterpret_cast<const typename Vec2<R>::type *>(psi + 2 * i);
    const double p = (double)v.x * (double)v.x + (double)v.y * (double)v.y;
    if (p == 0.0) continue;
    const uint64_t g = a.index_base + i;
    uint32_t m = 0;
    for (uint32_t j = 0; j < a.n_bits; ++j) m |= (uint32_t)((g >> a.bitpos[j]) & 1ull) << j;
    if (use_smem)
      atomicAdd(&sh[m], p);
    else
      atomicAdd(&hist[m], p);
  }
  if (use_smem) {
    __syncthreads();
    for (uint32_t b = threadIdx.x; b < bins; b += kThreads)
      if (sh[b] != 0.0) atomicAdd(&hist[b], sh[b]);
  }
}

cudaError_t launch_measure_probs(qip_prec prec, const void *psi, uint64_t len, uint64_t index_base,
                                 const uint32_t *bitpos, uint32_t n_bits, double *d_hist, cudaStream_t s,
                                 uint64_t *launches) {
  if (n_bits > 26) return cudaErrorInvalidValue;
  HistArgs a;
  a.n_bits = n_bits;
  for (uint32_t j = 0; j < n_bits; ++j) a.bitpos[j] = bitpos[j];
  a.len = len;
  a.index_base = index_base;
  cudaError_t e = cudaMemsetAsync(d_hist, 0, sizeof(double) << n_bits, s);
  if (e != cudaSuccess) return e;
  unsigned grid = (unsigned)std::min<uint64_t>((len + kThreads - 1) / kThreads, 148ull * 8);
  if (grid == 0) grid = 1;
  if (prec == QIP_F32)
    k_hist<float><<<grid, kThreads, 0, s>>>((const float *)psi, d_hist, a);
  else
    k_hist<double><<<grid, kThreads, 0, s>>>((const double *)psi, d_hist, a);
  ++*launches;
  return cudaGetLastError();
}

template <typename R>
__global__ void __launch_bounds__(kThreads)
    k_chunk_sums(const R *__restrict__ psi, uint64_t len, uint32_t chunk_log2, double *sums) {
  const uint64_t begin = (uint64_t)blockIdx.x << chunk_log2;
  uint64_t end = begin + (1ull << chunk_log2);
  if (end > len) end = len;
  double acc = 0.0;
  for (uint64_t i = begin + threadIdx.x; i < end; i += kThreads) {
    typename Vec2<R>::type v = *reinterpret_cast<const typename Vec2<R>::type *>(psi + 2 * i);
    acc += (double)v.x * (double)v.x + (double)v.y * (double)v.y;
  }
  acc = block_sum(acc);
  if (threadIdx.x == 0) sums[blockIdx.x] = acc;
}

cudaError_t launch_chunk_sums(qip_prec prec, const void *psi, uint64_t len, uint32_t chunk_log2,
                              double *d_sums, cudaStream_t s, uint64_t *launches) {
  const uint64_t chunks = (len + (1ull << chunk_log2) - 1) >> chunk_log2;
  if (prec == QIP_F32)
    k_chunk_sums<float><<<(unsigned)chunks, kThreads, 0, s>>>((const float *)psi, len, chunk_log2, d_sums);
  else
    k_chunk_sums<double><<<(unsigned)chunks, kThreads, 0, s>>>((const double *)psi, len, chunk_log2, d_sums);
  ++*launches;
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------
// inverse-CDF sampling (qipb200_state_sample; decision rules in sample.cuh)
// ---------------------------------------------------------------------------------
static const int kScanThreads = 1024;

// Inclusive scan over the warp; the same additions in the same order as sample_warp_scan.
__device__ __forceinline__ double warp_incl_scan(double v) {
  const int lane = threadIdx.x & 31;
  for (int o = 1; o < 32; o <<= 1) {
    const double x = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v = v + x;
  }
  return v;
}

// In-place inclusive scan of a[] in blocks of kScanThreads; block_tot[b] = total of block b (when non-NULL).
__global__ void __launch_bounds__(kScanThreads) k_sample_scan(double *a, uint64_t n, double *block_tot) {
  __shared__ double w[kScanThreads / 32];
  const uint64_t i = (uint64_t)blockIdx.x * kScanThreads + threadIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double v = warp_incl_scan(i < n ? a[i] : 0.0);
  if (lane == 31) w[warp] = v;
  __syncthreads();
  if (warp == 0) w[lane] = warp_incl_scan(w[lane]);
  __syncthreads();
  if (warp > 0) v += w[warp - 1];
  if (i < n) a[i] = v;
  if (block_tot && threadIdx.x == kScanThreads - 1) block_tot[blockIdx.x] = v;
}

// a[i] += prefix[b - 1] for every element of block b >= 1 (prefix = the scanned block totals).
__global__ void __launch_bounds__(kScanThreads) k_sample_add(double *a, uint64_t n, const double *prefix) {
  const uint64_t i = (uint64_t)(blockIdx.x + 1) * kScanThreads + threadIdx.x;
  if (i < n) a[i] += prefix[blockIdx.x];
}

cudaError_t launch_sample_scan(double *d, uint64_t n, cudaStream_t s, uint64_t *launches) {
  const uint64_t blocks = (n + kScanThreads - 1) / kScanThreads;
  if (blocks <= 1) {
    k_sample_scan<<<1, kScanThreads, 0, s>>>(d, n, nullptr);
    ++*launches;
    return cudaGetLastError();
  }
  double *tot = nullptr;
  cudaError_t e = cudaMallocAsync((void **)&tot, blocks * sizeof(double), s);
  if (e != cudaSuccess) return e;
  k_sample_scan<<<(unsigned)blocks, kScanThreads, 0, s>>>(d, n, tot);
  ++*launches;
  e = cudaGetLastError();
  if (e == cudaSuccess) e = launch_sample_scan(tot, blocks, s, launches);
  if (e == cudaSuccess) {
    k_sample_add<<<(unsigned)(blocks - 1), kScanThreads, 0, s>>>(d, n, tot);
    ++*launches;
    e = cudaGetLastError();
  }
  cudaError_t f = cudaFreeAsync(tot, s);
  return e != cudaSuccess ? e : f;
}

// One warp per draw: owner rank, chunk search, scan of the chunk in 32-amplitude groups (sample.cuh).
// out[j] = global index (as a double: < 2^53, exact) on the owner, 0 on every other rank.
template <typename R>
__global__ void __launch_bounds__(kThreads)
    k_sample_resolve(const R *__restrict__ psi, const double *__restrict__ P, const double *__restrict__ totals,
                     const double *__restrict__ draws, double *__restrict__ out, const SampleArgs a) {
  const uint64_t j = ((uint64_t)blockIdx.x * kThreads + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (j >= a.n_draws) return;  // uniform over the warp
  double t;
  if (sample_owner(totals, a.world, draws[j], &t) != a.rank) {
    if (lane == 0) out[j] = 0.0;
    return;
  }
  uint64_t c = sample_chunk(P, a.chunks, t);
  double base = c ? P[c - 1] : 0.0;
  uint64_t last_nonzero = c << a.chunk_log2;
  for (; c < a.chunks; ++c) {
    const uint64_t begin = c << a.chunk_log2, end = begin + (1ull << a.chunk_log2);
    for (uint64_t g = begin; g < end; g += 32) {
      const uint64_t i = g + lane;
      double p = 0.0;
      if (i < end) {
        const typename Vec2<R>::type v = *reinterpret_cast<const typename Vec2<R>::type *>(psi + 2 * i);
        p = (double)v.x * (double)v.x + (double)v.y * (double)v.y;
      }
      const double incl = warp_incl_scan(p);
      const unsigned hit = __ballot_sync(0xffffffffu, i < end && sample_crosses(base, incl, t));
      if (hit) {
        if (lane == 0) out[j] = (double)(a.index_base + g + (uint64_t)(__ffs(hit) - 1));
        return;
      }
      const unsigned nz = __ballot_sync(0xffffffffu, p > 0.0);
      if (nz) last_nonzero = g + (uint64_t)(31 - __clz(nz));
      base += __shfl_sync(0xffffffffu, incl, 31);
    }
  }
  if (lane == 0) out[j] = (double)(a.index_base + last_nonzero);
}

cudaError_t launch_sample_resolve(qip_prec prec, const void *psi, const double *P, const double *totals,
                                  const double *draws, double *out, const SampleArgs &a, cudaStream_t s,
                                  uint64_t *launches) {
  const uint64_t warps_per_block = kThreads / 32;
  const unsigned grid = (unsigned)((a.n_draws + warps_per_block - 1) / warps_per_block);
  if (grid == 0) return cudaSuccess;
  if (prec == QIP_F32)
    k_sample_resolve<float><<<grid, kThreads, 0, s>>>((const float *)psi, P, totals, draws, out, a);
  else
    k_sample_resolve<double><<<grid, kThreads, 0, s>>>((const double *)psi, P, totals, draws, out, a);
  ++*launches;
  return cudaGetLastError();
}

struct OutcomeArgs {
  uint64_t n_draws;
  uint32_t n_bits;
  uint8_t bitpos[64];
};

// res[j]: global index as a double -> outcome bits as a uint64, in place.
__global__ void __launch_bounds__(kThreads) k_sample_outcomes(double *res, const __grid_constant__ OutcomeArgs a) {
  const uint64_t j = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
  if (j >= a.n_draws) return;
  const uint64_t index = (uint64_t)res[j];
  reinterpret_cast<uint64_t *>(res)[j] = sample_outcome(index, a.bitpos, a.n_bits);
}

cudaError_t launch_sample_outcomes(double *res, uint64_t n_draws, const uint8_t *bitpos, uint32_t n_bits,
                                   cudaStream_t s, uint64_t *launches) {
  if (n_bits > 64) return cudaErrorInvalidValue;
  if (n_draws == 0) return cudaSuccess;
  OutcomeArgs a;
  a.n_draws = n_draws;
  a.n_bits = n_bits;
  for (uint32_t j = 0; j < n_bits; ++j) a.bitpos[j] = bitpos[j];
  k_sample_outcomes<<<grid_for(n_draws), kThreads, 0, s>>>(res, a);
  ++*launches;
  return cudaGetLastError();
}

template <typename R>
__global__ void __launch_bounds__(kThreads)
    k_collapse(R *__restrict__ psi, uint64_t len, uint64_t index_base, uint64_t row_mask,
               uint64_t measured_mask, R p_mult) {
  const uint64_t i = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
  if (i >= len) return;
  typedef typename Vec2<R>::type V;
  V *p = reinterpret_cast<V *>(psi + 2 * i);
  if ((((index_base + i) & row_mask) ^ measured_mask) != 0) {
    V z;
    z.x = (R)0;
    z.y = (R)0;
    *p = z;  // measurement_ops.rs:255-257
  } else {
    V v = *p;
    v.x *= p_mult;  // measurement_ops.rs:258-260
    v.y *= p_mult;
    *p = v;
  }
}

cudaError_t launch_collapse(qip_prec prec, void *psi, uint64_t len, uint64_t index_base, uint64_t row_mask,
                            uint64_t measured_mask, double p_mult, cudaStream_t s, uint64_t *launches) {
  if (prec == QIP_F32)
    k_collapse<float><<<grid_for(len), kThreads, 0, s>>>((float *)psi, len, index_base, row_mask,
                                                         measured_mask, (float)p_mult);
  else
    k_collapse<double><<<grid_for(len), kThreads, 0, s>>>((double *)psi, len, index_base, row_mask,
                                                          measured_mask, p_mult);
  ++*launches;
  return cudaGetLastError();
}

}  // namespace qipb200
