// sync_device.cuh -- building blocks shared by the five variants of the fused
// sync kernel (fused_sync_sgd.cu: LDG/STG pull, _tma.cu: cp.async.bulk pull,
// _push.cu: stores only, _ll.cu: flag-in-data words, _nvls.cu: multimem):
// PTX wrappers, bf16 pack / unpack / round, the ring order of the peers (peer)
// and the scale-then-sum step of the reduction (scaled / add_scaled, and
// reduce_scalar over every rank's diff_ or bf16 wire), the per-CTA cross-GPU
// barrier, the shard bounds (chunk), the shard/vector partition and its scalar
// head / tail, zeroing of diff_, the blob (segment) cursor and its shared-memory
// copy, the SGD update of a vector and of a scalar element in the reference's
// operation order and the same for the Nesterov, AdaGrad, RMSProp and AdaDelta
// solvers (update_vec / update_scalar), the all-gather of a scalar weight, and
// the host side of the launchers (argument check, SM count, world-size and
// solver dispatch).  Every kernel
// uses these except in the few places listed in DESIGN.md §3, where the helper
// changed the kernel's spills or static instruction counts.
#ifndef COS_SYNC_DEVICE_CUH_
#define COS_SYNC_DEVICE_CUH_

#include <cuda_bf16.h>
#include <stdint.h>

#include <type_traits>

#include "fused_sync_sgd.hpp"

namespace cosb {
namespace {

// ------------------------------------------------------------ PTX helpers

__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// streaming 128-bit load that does not allocate in L1 (each element is read once)
__device__ __forceinline__ float4 ld_stream(const float* p) {
  float4 v;
  asm volatile("ld.global.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p));
  return v;
}

__device__ __forceinline__ uint2 ld_stream_u2(const uint16_t* p) {
  uint2 v;
  asm volatile("ld.global.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p));
  return v;
}

__device__ __forceinline__ void st_vec(float* p, const float4& v) {
  asm volatile("st.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
               : "memory");
}

// NVLS (NVLink SHARP): one load on a multicast address returns the fp32 sum of the
// word on every rank, reduced inside the NVSwitch (SASS LDGMC.E.ADD.F32x4); one
// store on it lands on every rank.
__device__ __forceinline__ float4 mc_ld_reduce(const float* p) {
  float4 v;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p)
               : "memory");
  return v;
}

__device__ __forceinline__ void mc_st(float* p, const float4& v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
               "f"(v.w)
               : "memory");
}

__device__ __forceinline__ float bf16_bits_to_float(uint32_t bits16) { return __uint_as_float(bits16 << 16); }

__device__ __forceinline__ uint16_t float_to_bf16_bits(float f) {
  return __bfloat16_as_ushort(__float2bfloat16_rn(f));
}

// the value a gradient element has after crossing the bf16 wire
__device__ __forceinline__ float round_bf16(float x) { return bf16_bits_to_float(float_to_bf16_bits(x)); }

__device__ __forceinline__ float4 round_bf16x4(const float4& v) {
  return make_float4(round_bf16(v.x), round_bf16(v.y), round_bf16(v.z), round_bf16(v.w));
}

__device__ __forceinline__ uint2 pack_bf16x4(const float4& v) {
  uint2 o;
  o.x = static_cast<uint32_t>(float_to_bf16_bits(v.x)) | (static_cast<uint32_t>(float_to_bf16_bits(v.y)) << 16);
  o.y = static_cast<uint32_t>(float_to_bf16_bits(v.z)) | (static_cast<uint32_t>(float_to_bf16_bits(v.w)) << 16);
  return o;
}

__device__ __forceinline__ float4 unpack_bf16x4(const uint2& u) {
  return make_float4(bf16_bits_to_float(u.x & 0xffffu), bf16_bits_to_float(u.x >> 16),
                     bf16_bits_to_float(u.y & 0xffffu), bf16_bits_to_float(u.y >> 16));
}

// ------------------------------------------------------- reduction order

// The rank k places after `rank` on the ring (0 <= k < world).  Owner s sums the sources s, s+1, ... (mod N)
// in that order (socket_sync_cpu.cpp:108-133); pushes go to rank+1, rank+2, ... so that at any moment the
// ranks target different peers.
__device__ __forceinline__ int peer(int rank, int k, int world) {
  int x = rank + k;
  if (x >= world) x -= world;
  return x;
}

// Every gradient is scaled by 1/N BEFORE the sum (parallel_cpu.cpp:120-122 runs before
// socket_sync_cpu.cpp:112-132): acc = inv*x for the first source, acc = inv*x + acc for each later one.
__device__ __forceinline__ float scaled(float inv, float x) { return __fmul_rn(inv, x); }

__device__ __forceinline__ float4 scaled(float inv, const float4& x) {
  return make_float4(__fmul_rn(inv, x.x), __fmul_rn(inv, x.y), __fmul_rn(inv, x.z), __fmul_rn(inv, x.w));
}

__device__ __forceinline__ void add_scaled(float& acc, float inv, float x) { acc = __fadd_rn(__fmul_rn(inv, x), acc); }

__device__ __forceinline__ void add_scaled(float4& acc, float inv, const float4& x) {
  acc.x = __fadd_rn(__fmul_rn(inv, x.x), acc.x);
  acc.y = __fadd_rn(__fmul_rn(inv, x.y), acc.y);
  acc.z = __fadd_rn(__fmul_rn(inv, x.z), acc.z);
  acc.w = __fadd_rn(__fmul_rn(inv, x.w), acc.w);
}

// f(k) for k = 1 .. world-1, unrolled when the world size N is known at compile time (N = 0: run time)
template <int N, class F>
__device__ __forceinline__ void for_peers(int world, F&& f) {
  if (N > 0) {
#pragma unroll
    for (int k = 1; k < (N > 0 ? N : 1); ++k) f(k);
  } else {
    for (int k = 1; k < world; ++k) f(k);
  }
}

// ------------------------------------------------------ cross-GPU barrier

__device__ __forceinline__ uint32_t* flag_slot(uint32_t* base, int which, int cta, int src) {
  return base + (static_cast<size_t>(which) * kMaxCtas + cta) * kMaxRanks + src;
}

// Barrier between CTA blockIdx.x of every rank, split into its two halves.
// Thread t < world handles peer t.  cta_signal publishes this launch's epoch
// into the peer's flag slot [cta][rank]: the leading __syncthreads orders every
// store of the CTA (e.g. pushes into peer memory) before the releasing thread,
// and st.release.sys (= fence.acq_rel.sys + store, cumulative over the bar.sync)
// makes them visible before the flag is.  cta_wait spins on the LOCAL slot
// [cta][t] (peers store into it, so spinning costs no NVLink bandwidth) with
// relaxed loads and issues ONE acquire fence after the flag arrived.
// cta_wait returns false if a peer did not arrive within timeout_ns (status is set).
__device__ __forceinline__ uint32_t ld_relaxed_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// Optional diagnostics (option "trace"): the first participating thread of CTA 0 stamps %globaltimer into
// trace[5 + 4*which ...]: barrier entered (after __syncthreads), release fence done, flag arrived, acquire done.
__device__ __forceinline__ bool barrier_tracer(const SyncParams& p) {
  return p.trace != nullptr && blockIdx.x == 0 && static_cast<int>(threadIdx.x) == (p.rank == 0 ? 1 : 0);
}

__device__ __forceinline__ void cta_signal(const SyncParams& p, int which) {
  __syncthreads();
  const int t = threadIdx.x;
  if (t < p.world && t != p.rank) {
    const bool tr = barrier_tracer(p);
    if (tr) p.trace[5 + 4 * which] = globaltimer_ns();
    asm volatile("fence.acq_rel.sys;" ::: "memory");  // release: cumulative over the bar.sync above
    if (tr) p.trace[6 + 4 * which] = globaltimer_ns();
    asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(flag_slot(p.flags[t], which, blockIdx.x, p.rank)),
                 "r"(p.epoch)
                 : "memory");
  }
}

__device__ __forceinline__ bool cta_wait(const SyncParams& p, int which, int* s_abort) {
  const int t = threadIdx.x;
  if (t < p.world && t != p.rank) {
    const bool tr = barrier_tracer(p);
    const uint32_t* mine = flag_slot(p.flags[p.rank], which, blockIdx.x, t);
    const unsigned long long t0 = globaltimer_ns();
    unsigned spins = 0;
    for (;;) {
      uint32_t v = ld_relaxed_sys(mine);
      if (static_cast<int32_t>(v - p.epoch) >= 0) break;
      if ((++spins & 0x3ffu) == 0) {
        if (*reinterpret_cast<volatile int*>(s_abort)) break;
        if (globaltimer_ns() - t0 > p.timeout_ns) {
          atomicExch(p.status, 100 + which * 32 + t);  // which barrier, which peer
          *reinterpret_cast<volatile int*>(s_abort) = 1;
          break;
        }
      }
    }
    if (tr) p.trace[7 + 4 * which] = globaltimer_ns();
    asm volatile("fence.acq_rel.sys;" ::: "memory");  // acquire: later loads see what the peer released
    if (tr) p.trace[8 + 4 * which] = globaltimer_ns();
  }
  __syncthreads();
  return *reinterpret_cast<volatile int*>(s_abort) == 0;
}

__device__ __forceinline__ bool cta_barrier(const SyncParams& p, int which, int* s_abort) {
  cta_signal(p, which);
  return cta_wait(p, which, s_abort);
}

// ------------------------------------------------------------- partition

struct ShardRange {
  uint64_t lo, hi;        // element range
  uint64_t vec_lo;        // first float4 index fully inside
  uint64_t nvec;          // number of float4 vectors fully inside
  uint64_t head_end;      // [lo, head_end) scalar head
  uint64_t tail_begin;    // [tail_begin, hi) scalar tail
  // 512-byte aligned iteration space (push / NVLS kernels): thread index a = tid + k*stride addresses vector
  // vec_base + a, valid for off <= a < off + nvec.  vec_base is a multiple of 32 vectors, so every warp's 32 float4
  // cover exactly four 128-byte lines of data_ / diff_ / the receive slot -- with the plain j = tid + k*stride walk
  // a shard that starts mid-line (CaffeNet: every shard but one) makes EVERY warp access straddle lines: partial
  // sectors over NVLink (+3 % payload counted by NVML) and 7 % more time at N = 2 (422 vs 395 us).
  uint64_t vec_base;      // (lo / 4) rounded down to a multiple of 32
  uint64_t off;           // vec_lo - vec_base, 0..32
};

// aligned index a -> element index of its vector in shard r, or ~0 when a is outside the shard's vector body
__device__ __forceinline__ uint64_t vec_elem(const ShardRange& r, uint64_t a) {
  return (a >= r.off && a - r.off < r.nvec) ? ((r.vec_base + a) << 2) : ~0ull;
}

// First element of shard s; shard s is [chunk(count, world, s), chunk(count, world, s + 1)).
// socket_sync_cpu.cpp:46-54 chunk(): multiply first, then divide, in 64 bit.
__device__ __forceinline__ uint64_t chunk(uint64_t count, int world, uint64_t s) {
  return s * count / static_cast<uint64_t>(world);
}

__device__ __forceinline__ ShardRange shard_range(uint64_t count, int world, int s) {
  ShardRange r;
  r.lo = chunk(count, world, s);
  r.hi = chunk(count, world, s + 1ull);
  uint64_t vlo = (r.lo + 3) >> 2, vhi = r.hi >> 2;
  if (vhi > vlo) {
    r.vec_lo = vlo;
    r.nvec = vhi - vlo;
    r.head_end = vlo << 2;
    r.tail_begin = vhi << 2;
  } else {
    r.vec_lo = vlo;
    r.nvec = 0;
    r.head_end = r.hi;  // everything scalar
    r.tail_begin = r.hi;
  }
  r.vec_base = (r.lo >> 2) & ~31ull;
  r.off = r.vec_lo - r.vec_base;
  return r;
}

// Scalar head / tail element of range r handled by thread t of CTA 0, or ~0.  R is ShardRange or any range with
// the same lo / head_end / tail_begin / hi fields.
template <class R>
__device__ __forceinline__ uint64_t edge_element(const R& r, unsigned t) {
  const uint64_t nhead = r.head_end - r.lo, ntail = r.hi - r.tail_begin;
  if (t < nhead) return r.lo + t;
  if (t - nhead < ntail) return r.tail_begin + (t - nhead);
  return ~0ull;
}

// diff_ := 0 over the scalar head / tail of range r (CTA 0)
template <class R>
__device__ __forceinline__ void zero_edges(float* g, const R& r) {
  if (blockIdx.x == 0) {
    const uint64_t i = edge_element(r, threadIdx.x);
    if (i != ~0ull) g[i] = 0.f;
  }
}

// diff_ := 0 over shard range r with st_vec, which stays ordered behind the asm loads of the same words before it:
// the float4 body in the plain j = tid + k*stride walk (kAligned = false) or the 512-byte aligned vec_elem walk,
// then the scalar head / tail.
template <bool kAligned>
__device__ __forceinline__ void zero_range(float* g, const ShardRange& r, uint64_t tid, uint64_t stride) {
  const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
  if (kAligned) {
    for (uint64_t j = tid; j < r.off + r.nvec; j += stride) {
      const uint64_t i = vec_elem(r, j);
      if (i != ~0ull) st_vec(g + i, z);
    }
  } else {
    for (uint64_t j = tid; j < r.nvec; j += stride) st_vec(g + ((r.vec_lo + j) << 2), z);
  }
  zero_edges(g, r);
}

// ----------------------------------------------------------- SGD element

struct SegCursor {
  const uint64_t* end;
  const float* lr_mult;
  const float* decay_mult;
  int nseg;
  int k;
  __device__ __forceinline__ void seek(uint64_t i) {  // binary search: first k with end[k] > i
    int lo = 0, hi = nseg - 1;
    while (lo < hi) {
      int mid = (lo + hi) >> 1;
      if (end[mid] > i) hi = mid; else lo = mid + 1;
    }
    k = lo;
  }
  __device__ __forceinline__ void advance(uint64_t i) {
    while (k < nseg - 1 && i >= end[k]) ++k;
  }
};

// The segment table lives in shared memory at smem when it has at most max_seg entries; otherwise the cursor reads
// global memory.  copy_seg_table copies it there; the CTA must __syncthreads() before the first seek of a cursor
// from seg_cursor.  A kernel short of registers builds the cursor where it first needs it, not at kernel entry.
__device__ __forceinline__ void copy_seg_table(const SyncParams& p, unsigned char* smem, int max_seg) {
  uint64_t* s_end = reinterpret_cast<uint64_t*>(smem);
  float* s_lr = reinterpret_cast<float*>(s_end + p.nseg);
  float* s_dm = s_lr + p.nseg;
  if (p.nseg <= max_seg) {
    for (int k = threadIdx.x; k < p.nseg; k += blockDim.x) {
      s_end[k] = p.seg_end[k];
      s_lr[k] = p.seg_lr_mult[k];
      s_dm[k] = p.seg_decay_mult[k];
    }
  }
}

__device__ __forceinline__ SegCursor seg_cursor(const SyncParams& p, unsigned char* smem, int max_seg) {
  uint64_t* s_end = reinterpret_cast<uint64_t*>(smem);
  float* s_lr = reinterpret_cast<float*>(s_end + p.nseg);
  float* s_dm = s_lr + p.nseg;
  const bool in_smem = p.nseg <= max_seg;
  SegCursor c;
  c.end = in_smem ? s_end : p.seg_end;
  c.lr_mult = in_smem ? s_lr : p.seg_lr_mult;
  c.decay_mult = in_smem ? s_dm : p.seg_decay_mult;
  c.nseg = p.nseg;
  c.k = 0;
  return c;
}

__device__ __forceinline__ SegCursor load_seg_table(const SyncParams& p, unsigned char* smem, int max_seg) {
  copy_seg_table(p, smem, max_seg);
  return seg_cursor(p, smem, max_seg);
}

// Regularize + ComputeUpdateValue + Blob::Update for one element, in the
// reference's operation order with one rounding per operation:
//   L2: g = ld*w + g          (sgd_solver.cpp:155-160 caffe_axpy(local_decay, data, diff))
//   L1: g = ld*sign(w) + g    (sgd_solver.cpp:161-168 caffe_cpu_sign into temp_, then caffe_axpy; sign is
//                              (0 < w) - (w < 0): 0 for +-0 and NaN, math_functions.hpp caffe_sign)
//   h = m*h ; h = lr*g + h ; w = (-1*h) + w
template <bool L1>
__device__ __forceinline__ void sgd_element_t(float g, float& w, float& h, float lr, float ld, float m) {
  if (ld != 0.f) {
    const float x = L1 ? static_cast<float>((0.f < w) - (w < 0.f)) : w;
    g = __fadd_rn(__fmul_rn(ld, x), g);
  }
  h = __fmul_rn(m, h);
  h = __fadd_rn(__fmul_rn(lr, g), h);
  w = __fadd_rn(__fmul_rn(-1.0f, h), w);
}

// l1 is a launch-wide constant: ONE uniform branch selects the instantiation, so the (rare) L1 path adds no
// instructions to the L2 path (the TMA kernel's 8 consumer warps per SM are issue-bound: +18 % instructions from a
// branch-free select cost +25 % time at N = 1).
__device__ __forceinline__ void sgd_element(float g, float& w, float& h, float lr, float ld, float m, int l1 = 0) {
  if (l1) sgd_element_t<true>(g, w, h, lr, ld, m);
  else sgd_element_t<false>(g, w, h, lr, ld, m);
}

__device__ __forceinline__ void sgd_vec(const SyncParams& p, SegCursor& c, uint64_t i, const float4& g, float4& w,
                                        float4& h) {
  c.advance(i);
  if (i + 3 < c.end[c.k]) {
    const float lr = __fmul_rn(p.rate, c.lr_mult[c.k]);
    const float ld = __fmul_rn(p.weight_decay, c.decay_mult[c.k]);
    if (p.l1) {
      sgd_element_t<true>(g.x, w.x, h.x, lr, ld, p.momentum);
      sgd_element_t<true>(g.y, w.y, h.y, lr, ld, p.momentum);
      sgd_element_t<true>(g.z, w.z, h.z, lr, ld, p.momentum);
      sgd_element_t<true>(g.w, w.w, h.w, lr, ld, p.momentum);
    } else {
      sgd_element_t<false>(g.x, w.x, h.x, lr, ld, p.momentum);
      sgd_element_t<false>(g.y, w.y, h.y, lr, ld, p.momentum);
      sgd_element_t<false>(g.z, w.z, h.z, lr, ld, p.momentum);
      sgd_element_t<false>(g.w, w.w, h.w, lr, ld, p.momentum);
    }
  } else {  // the vector straddles one or more blob boundaries
    const float gg[4] = {g.x, g.y, g.z, g.w};
    float ww[4] = {w.x, w.y, w.z, w.w};
    float hh[4] = {h.x, h.y, h.z, h.w};
    int k = c.k;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      while (k < c.nseg - 1 && i + e >= c.end[k]) ++k;
      sgd_element(gg[e], ww[e], hh[e], __fmul_rn(p.rate, c.lr_mult[k]), __fmul_rn(p.weight_decay, c.decay_mult[k]),
                  p.momentum, p.l1);
    }
    w = make_float4(ww[0], ww[1], ww[2], ww[3]);
    h = make_float4(hh[0], hh[1], hh[2], hh[3]);
  }
}

// Scalar (head / tail) element i with reduced gradient g: update with its blob's multipliers (c is sought from
// scratch), store h and w locally, return the new weight.
__device__ __forceinline__ float sgd_scalar(const SyncParams& p, SegCursor c, uint64_t i, float g, float* wl,
                                            float* hl) {
  c.seek(i);
  float w = wl[i], h = hl[i];
  sgd_element(g, w, h, __fmul_rn(p.rate, c.lr_mult[c.k]), __fmul_rn(p.weight_decay, c.decay_mult[c.k]), p.momentum,
              p.l1);
  hl[i] = h;
  wl[i] = w;
  return w;
}

// ------------------------------------------------ the other solvers' element

// Regularize (as sgd_element_t), then ComputeUpdateValue of solver S, then Blob::Update w = (-1*g) + w, for one
// element.  The CPU branch of each solver, one rounding per operation in the BLAS order of mkl_alternate.hpp
// (axpby(a,x,b,y): y = b*y then y = a*x + y; add_scalar: y = y + d; scale: y = a*x; powx(x, 2) = x*x, powx(x, 0.5)
// taken as the correctly rounded square root, DESIGN.md §7):
//   Nesterov (nesterov_solver.cpp:21-41):  u = h; h = m*h; h = lr*g + h; u = (-m)*u; u = (1+m)*h + u; g = u
//   AdaGrad  (adagrad_solver.cpp:21-50):   u = g*g; h = u + h; u = sqrt(h); u = u + d; u = g / u;
//                                          g = 0*g; g = lr*u + g
//   RMSProp  (rmsprop_solver.cpp:24-51):   u = g*g; h = rho*h; h = (1-rho)*u + h; then as AdaGrad from u = sqrt(h)
//   AdaDelta (adadelta_solver.cpp:34-89):  u = g*g; h = m*h; h = (1-m)*u + h; u = d + h2; t = d + h; u = u / t;
//                                          u = sqrt(u); g = g*u; u = g*g; h2 = m*h2; h2 = (1-m)*u + h2; g = lr*g
// p.momentum is rho for RMSProp.  h2 is only read and written by AdaDelta.
template <int S, bool L1>
__device__ __forceinline__ void solver_element_t(const SyncParams& p, float g, float& w, float& h, float& h2, float lr,
                                                 float ld) {
  if (ld != 0.f) {
    const float x = L1 ? static_cast<float>((0.f < w) - (w < 0.f)) : w;
    g = __fadd_rn(__fmul_rn(ld, x), g);
  }
  if constexpr (S == kSolverNesterov) {
    float u = h;
    h = __fmul_rn(p.momentum, h);
    h = __fadd_rn(__fmul_rn(lr, g), h);
    u = __fmul_rn(p.neg_m, u);
    u = __fadd_rn(__fmul_rn(p.one_plus_m, h), u);
    g = u;
  } else if constexpr (S == kSolverAdaGrad || S == kSolverRMSProp) {
    float u = __fmul_rn(g, g);
    if constexpr (S == kSolverAdaGrad) {
      h = __fadd_rn(u, h);
    } else {
      h = __fmul_rn(p.momentum, h);
      h = __fadd_rn(__fmul_rn(p.one_minus, u), h);
    }
    u = __fsqrt_rn(h);
    u = __fadd_rn(u, p.delta);
    u = __fdiv_rn(g, u);
    g = __fmul_rn(0.f, g);
    g = __fadd_rn(__fmul_rn(lr, u), g);
  } else if constexpr (S == kSolverAdaDelta) {
    float u = __fmul_rn(g, g);
    h = __fmul_rn(p.momentum, h);
    h = __fadd_rn(__fmul_rn(p.one_minus, u), h);
    u = __fadd_rn(p.delta, h2);
    const float t = __fadd_rn(p.delta, h);
    u = __fdiv_rn(u, t);
    u = __fsqrt_rn(u);
    g = __fmul_rn(g, u);
    u = __fmul_rn(g, g);
    h2 = __fmul_rn(p.momentum, h2);
    h2 = __fadd_rn(__fmul_rn(p.one_minus, u), h2);
    g = __fmul_rn(lr, g);
  }
  w = __fadd_rn(__fmul_rn(-1.0f, g), w);
}

template <int S>
__device__ __forceinline__ void solver_element(const SyncParams& p, float g, float& w, float& h, float& h2, float lr,
                                               float ld) {
  if (p.l1) solver_element_t<S, true>(p, g, w, h, h2, lr, ld);
  else solver_element_t<S, false>(p, g, w, h, h2, lr, ld);
}

// sgd_vec for solver S != SGD: same blob-boundary split; AdaDelta reads and writes h2 at p.hist2 + i here
template <int S>
__device__ __forceinline__ void solver_vec(const SyncParams& p, SegCursor& c, uint64_t i, const float4& g, float4& w,
                                           float4& h) {
  float4 h2 = make_float4(0.f, 0.f, 0.f, 0.f);
  if constexpr (S == kSolverAdaDelta) h2 = *reinterpret_cast<const float4*>(p.hist2 + i);
  c.advance(i);
  if (i + 3 < c.end[c.k]) {
    const float lr = __fmul_rn(p.rate, c.lr_mult[c.k]);
    const float ld = __fmul_rn(p.weight_decay, c.decay_mult[c.k]);
    if (p.l1) {
      solver_element_t<S, true>(p, g.x, w.x, h.x, h2.x, lr, ld);
      solver_element_t<S, true>(p, g.y, w.y, h.y, h2.y, lr, ld);
      solver_element_t<S, true>(p, g.z, w.z, h.z, h2.z, lr, ld);
      solver_element_t<S, true>(p, g.w, w.w, h.w, h2.w, lr, ld);
    } else {
      solver_element_t<S, false>(p, g.x, w.x, h.x, h2.x, lr, ld);
      solver_element_t<S, false>(p, g.y, w.y, h.y, h2.y, lr, ld);
      solver_element_t<S, false>(p, g.z, w.z, h.z, h2.z, lr, ld);
      solver_element_t<S, false>(p, g.w, w.w, h.w, h2.w, lr, ld);
    }
  } else {  // the vector straddles one or more blob boundaries
    const float gg[4] = {g.x, g.y, g.z, g.w};
    float ww[4] = {w.x, w.y, w.z, w.w};
    float hh[4] = {h.x, h.y, h.z, h.w};
    float h2h[4] = {h2.x, h2.y, h2.z, h2.w};
    int k = c.k;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      while (k < c.nseg - 1 && i + e >= c.end[k]) ++k;
      solver_element<S>(p, gg[e], ww[e], hh[e], h2h[e], __fmul_rn(p.rate, c.lr_mult[k]),
                        __fmul_rn(p.weight_decay, c.decay_mult[k]));
    }
    w = make_float4(ww[0], ww[1], ww[2], ww[3]);
    h = make_float4(hh[0], hh[1], hh[2], hh[3]);
    h2 = make_float4(h2h[0], h2h[1], h2h[2], h2h[3]);
  }
  if constexpr (S == kSolverAdaDelta) *reinterpret_cast<float4*>(p.hist2 + i) = h2;
}

template <int S>
__device__ __forceinline__ float solver_scalar(const SyncParams& p, SegCursor c, uint64_t i, float g, float* wl,
                                               float* hl) {
  c.seek(i);
  float w = wl[i], h = hl[i], h2 = 0.f;
  if constexpr (S == kSolverAdaDelta) h2 = p.hist2[i];
  solver_element<S>(p, g, w, h, h2, __fmul_rn(p.rate, c.lr_mult[c.k]), __fmul_rn(p.weight_decay, c.decay_mult[c.k]));
  if constexpr (S == kSolverAdaDelta) p.hist2[i] = h2;
  hl[i] = h;
  wl[i] = w;
  return w;
}

// What the kernels call: SGD goes through sgd_vec / sgd_scalar unchanged, so its instantiations compile as before.
template <int S>
__device__ __forceinline__ void update_vec(const SyncParams& p, SegCursor& c, uint64_t i, const float4& g, float4& w,
                                           float4& h) {
  if constexpr (S == kSolverSGD) sgd_vec(p, c, i, g, w, h);
  else solver_vec<S>(p, c, i, g, w, h);
}

template <int S>
__device__ __forceinline__ float update_scalar(const SyncParams& p, const SegCursor& c, uint64_t i, float g, float* wl,
                                               float* hl) {
  if constexpr (S == kSolverSGD) return sgd_scalar(p, c, i, g, wl, hl);
  else return solver_scalar<S>(p, c, i, g, wl, hl);
}

// Scalar element i of shard s summed over every rank's diff_ (or bf16 wire) in the reference's order s, s+1, ...
// (mod N), each term scaled by 1/N first: the scalar head / tail of the pull kernels, and every element when the
// world size is known at run time only.
template <bool BF16>
__device__ __forceinline__ float reduce_scalar(const SyncParams& p, int s, uint64_t i) {
  float acc = 0.f;
  for (int j = 0; j < p.world; ++j) {
    const int src = peer(s, j, p.world);
    const float x = BF16 ? bf16_bits_to_float(p.wire[src][i]) : p.diff[src][i];
    if (j == 0) acc = scaled(p.inv_scale, x);
    else add_scaled(acc, p.inv_scale, x);
  }
  return acc;
}

// the all-gather of one scalar weight: element i of every peer's data_
__device__ __forceinline__ void store_peers(const SyncParams& p, int world, uint64_t i, float w) {
  for (int k = 1; k < world; ++k) p.data[peer(p.rank, k, world)][i] = w;
}

// -------------------------------------------------------------- host side

// world / rank of a launch; kernels that exchange data with peers ask for min_world = 2
inline bool check_world(const SyncParams& p, int min_world) {
  return p.world >= min_world && p.world <= kMaxRanks && p.rank >= 0 && p.rank < p.world;
}

// SMs of `device` (-1: the current device); 148 (B200) if the query fails
inline int sm_count(int device) {
  int sms = 0;
  if ((device < 0 && cudaGetDevice(&device) != cudaSuccess) ||
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || sms <= 0) {
    cudaGetLastError();
    sms = 148;
  }
  return sms;
}

// dynamic shared memory of a segment table the kernel copies into shared memory when nseg <= max_seg
inline size_t seg_smem_bytes(const SyncParams& p, int max_seg) {
  return p.nseg <= max_seg ? static_cast<size_t>(p.nseg) * (sizeof(uint64_t) + 2 * sizeof(float)) : 0;
}

// f(std::integral_constant<int, N>()) with N = world for the world sizes 2..8 the kernels are compiled for,
// N = 0 (world size known at run time only) for every other value
template <class F>
cudaError_t dispatch_world(int world, F&& f) {
  switch (world) {
    case 2: return f(std::integral_constant<int, 2>());
    case 3: return f(std::integral_constant<int, 3>());
    case 4: return f(std::integral_constant<int, 4>());
    case 5: return f(std::integral_constant<int, 5>());
    case 6: return f(std::integral_constant<int, 6>());
    case 7: return f(std::integral_constant<int, 7>());
    case 8: return f(std::integral_constant<int, 8>());
    default: return f(std::integral_constant<int, 0>());
  }
}

// f(std::integral_constant<int, S>()) with S = the SolverType p.solver; cudaErrorInvalidValue for any other value
template <class F>
cudaError_t dispatch_solver(int solver, F&& f) {
  switch (solver) {
    case kSolverSGD: return f(std::integral_constant<int, kSolverSGD>());
    case kSolverNesterov: return f(std::integral_constant<int, kSolverNesterov>());
    case kSolverAdaGrad: return f(std::integral_constant<int, kSolverAdaGrad>());
    case kSolverRMSProp: return f(std::integral_constant<int, kSolverRMSProp>());
    case kSolverAdaDelta: return f(std::integral_constant<int, kSolverAdaDelta>());
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace
}  // namespace cosb
#endif
