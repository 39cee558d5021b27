// fused_sync_sgd_push.cu -- the PUSH variant of the fused sync kernel: the
// latency-optimised path for small and medium messages, and the bf16-wire path
// (same reference mapping and same results as fused_sync_sgd.cu, two-shot only).
//
// The pull kernels (fused_sync_sgd.cu / _tma.cu) have the shard owner LOAD its
// shard from every peer: each load is a full NVLink round trip (2-4 us), the
// bf16 wire needs a whole-buffer cast pass before barrier A, and diff_ can only
// be zeroed after barrier B because peers read it.  Here every transfer is a
// fire-and-forget STORE and nobody ever reads remote memory:
//   phase 1  rank r stores shard q of its gradient into rank q's receive slot
//            [r] (fp32 -> bf16 cast in registers: no wire buffer, no extra pass);
//   barrier A  "my contributions have landed in your slots"; BETWEEN signalling
//            and waiting, the CTA zeroes what it has just pushed (ClearParamDiffs:
//            nobody else reads diff_ in this scheme, so it needs no barrier and
//            hides in the flag flight; pure streaming stores -- a store right
//            behind the load of the same line measured 3x slower on B200);
//   phase 2  the owner reduces its own gradient + the N-1 slots out of LOCAL
//            memory in the reference's order s, s+1, ... (mod N) with the 1/N
//            scale applied before the sum (parallel_cpu.cpp:120-122,
//            socket_sync_cpu.cpp:108-133), applies Regularize /
//            ComputeUpdateValue / Blob::Update (sgd_solver.cpp:145-243,
//            blob.cpp:162-179) and stores the new weights locally and into every
//            peer's data_ (the next on_start(), socket_sync_cpu.cpp:102-105);
//   barrier B  "my weight stores have landed" (own-shard diff_ zeroed between
//            signal and wait).
// The receive slots are the device-resident analogue of the reference's
// diff_recv_ scratch buffers (socket_sync_cpu.cpp:14-44, one per peer, own_size_
// elements).  They are safe to reuse every step without double buffering: a
// peer can only push step t+1 after passing barrier B of step t, which this
// rank signals after its last read of the slots.
// Critical path: 2 x (store round trip + flag flight) instead of the pull
// kernels' flag flight + load round trip + store round trip + flag flight +
// zero pass.  Same per-CTA partition as the other kernels (vector j of a shard
// belongs to CTA (j / blockDim) % gridDim on the sender AND the owner), so the
// per-CTA flags of sync_device.cuh are sufficient.
#include "fused_sync_sgd.hpp"
#include "sync_device.cuh"

namespace cosb {
namespace {

constexpr int kPushThreads = 512;
constexpr int kPushMaxSeg = 1024;

__device__ __forceinline__ void st_vec_u2(uint16_t* p, const uint2& v) {
  asm volatile("st.global.v2.u32 [%0], {%1,%2};" ::"l"(p), "r"(v.x), "r"(v.y) : "memory");
}

// Receive slot `src` (the gradient rank src sends) in rank q's receive buffer.  Slot element 0 stands for global
// element vec_base * 4 of q's shard.  T = float, or uint16_t (bf16 bits) on the bf16 wire.
template <class T>
__device__ __forceinline__ T* recv_slot(const SyncParams& p, int q, int src) {
  return static_cast<T*>(p.recv[q]) + static_cast<uint64_t>(src) * p.recv_stride;
}

// N = compile-time world size (2..8), 0 = run-time world (<= kMaxRanks); S = SolverType
template <int N, bool BF16, int S = kSolverSGD>
__global__ void __launch_bounds__(kPushThreads, 2) fused_sync_sgd_push_kernel(const SyncParams p) {
  extern __shared__ unsigned char smem_raw[];
  __shared__ int s_abort;
  uint64_t* s_end = reinterpret_cast<uint64_t*>(smem_raw);
  float* s_lr = reinterpret_cast<float*>(s_end + p.nseg);
  float* s_dm = s_lr + p.nseg;
  const bool seg_in_smem = p.nseg <= kPushMaxSeg;
  if (seg_in_smem) {
    for (int k = threadIdx.x; k < p.nseg; k += blockDim.x) {
      s_end[k] = p.seg_end[k];
      s_lr[k] = p.seg_lr_mult[k];
      s_dm[k] = p.seg_decay_mult[k];
    }
  }
  if (threadIdx.x == 0) s_abort = 0;
  const bool tracer = p.trace != nullptr && blockIdx.x == 0 && threadIdx.x == 0;
  if (tracer) p.trace[0] = globaltimer_ns();

  const int world = (N > 0) ? N : p.world;
  const int rank = p.rank;
  const uint64_t tid = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  float* g = const_cast<float*>(p.diff[rank]);
  const bool zero = p.zero_diff != 0;

  // ---- phase 1: scatter my gradient into the owners' receive slots ----------
  // Destinations are staggered (rank+1, rank+2, ...), so at any moment the ranks target different peers.  For a
  // compile-time world size the loads for ALL N-1 destinations (x kU vectors) are issued before the first store:
  // one local-memory latency per iteration instead of N-1 (what a small message is made of at N = 8).
  if (N > 0) {
    constexpr int D = N > 0 ? N - 1 : 1;
    constexpr int kU = D >= 4 ? 1 : (D >= 2 ? 2 : 4);
    constexpr int NN = N > 0 ? N : 1;  // (this branch is dead for N == 0)
    const uint64_t max_nvec = (((p.count + NN - 1) / NN + 3) >> 2) + 32;  // >= off + nvec of every shard
    for (uint64_t j0 = tid; j0 < max_nvec; j0 += stride * kU) {
      float4 v[kU][D];
#pragma unroll
      for (int u = 0; u < kU; ++u) {
        const uint64_t j = j0 + static_cast<uint64_t>(u) * stride;
#pragma unroll
        for (int d = 0; d < D; ++d) {
          const ShardRange r = shard_range(p.count, N, peer(rank, 1 + d, N));
          const uint64_t i = vec_elem(r, j);
          if (i != ~0ull) v[u][d] = ld_stream(g + i);
        }
      }
#pragma unroll
      for (int u = 0; u < kU; ++u) {
        const uint64_t j = j0 + static_cast<uint64_t>(u) * stride;
#pragma unroll
        for (int d = 0; d < D; ++d) {
          const int q = peer(rank, 1 + d, N);
          const ShardRange r = shard_range(p.count, N, q);
          const uint64_t i = vec_elem(r, j), base = r.vec_base << 2;
          if (i != ~0ull) {
            if (BF16) st_vec_u2(recv_slot<uint16_t>(p, q, rank) + (i - base), pack_bf16x4(v[u][d]));
            else st_vec(recv_slot<float>(p, q, rank) + (i - base), v[u][d]);
          }
        }
      }
    }
  } else {
    for (int d = 1; d < world; ++d) {
      const int q = peer(rank, d, world);
      const ShardRange r = shard_range(p.count, world, q);
      const uint64_t base = r.vec_base << 2;
      for (uint64_t j = tid; j < r.off + r.nvec; j += stride) {
        const uint64_t i = vec_elem(r, j);
        if (i == ~0ull) continue;
        const float4 v = ld_stream(g + i);
        if (BF16) st_vec_u2(recv_slot<uint16_t>(p, q, rank) + (i - base), pack_bf16x4(v));
        else st_vec(recv_slot<float>(p, q, rank) + (i - base), v);
      }
    }
  }
  if (blockIdx.x == 0) {  // scalar head / tail elements of every foreign shard
    for (int d = 1; d < world; ++d) {
      const int q = peer(rank, d, world);
      const ShardRange r = shard_range(p.count, world, q);
      const uint64_t base = r.vec_base << 2;
      const uint64_t i = edge_element(r, threadIdx.x);
      if (i != ~0ull) {
        if (BF16) recv_slot<uint16_t>(p, q, rank)[i - base] = float_to_bf16_bits(g[i]);
        else recv_slot<float>(p, q, rank)[i - base] = g[i];
      }
    }
  }
  if (tracer) p.trace[1] = globaltimer_ns();

  // ---- barrier A: every contribution to my shard has landed -----------------
  cta_signal(p, 0);
  if (zero) {  // ClearParamDiffs of what this CTA pushed, hidden in the flag flight
    for (int d = 1; d < world; ++d) zero_range<true>(g, shard_range(p.count, world, peer(rank, d, world)), tid, stride);
  }
  if (!cta_wait(p, 0, &s_abort)) return;
  if (tracer) p.trace[2] = globaltimer_ns();

  // ---- phase 2: reduce (local), update, push the new weights ----------------
  // inline, not seg_cursor(): rebuilding the pointers here costs spills, e.g. <3,true> 0 -> 12 B, <6,false> 68 -> 84 B
  SegCursor cur;
  cur.end = seg_in_smem ? s_end : p.seg_end;
  cur.lr_mult = seg_in_smem ? s_lr : p.seg_lr_mult;
  cur.decay_mult = seg_in_smem ? s_dm : p.seg_decay_mult;
  cur.nseg = p.nseg;
  cur.k = 0;
  {
    const ShardRange r = shard_range(p.count, world, rank);
    const uint64_t base = r.vec_base << 2;
    float* wl = p.data[rank];
    float* hl = p.hist;
    const float inv = p.inv_scale;
    bool sought = false;
    for (uint64_t j = tid; j < r.off + r.nvec; j += stride) {
      const uint64_t i = vec_elem(r, j);
      if (i == ~0ull) continue;
      if (!sought) {
        cur.seek(i);
        sought = true;
      }
      constexpr int M = N > 0 ? N : 1;
      float4 x[M];
      x[0] = ld_stream(g + i);
      if (N > 0) {
#pragma unroll
        for (int k = 1; k < M; ++k) {  // all N-1 slot loads in flight together (local memory)
          const int src = peer(rank, k, M);
          if (BF16) x[k] = unpack_bf16x4(ld_stream_u2(recv_slot<const uint16_t>(p, rank, src) + (i - base)));
          else x[k] = ld_stream(recv_slot<const float>(p, rank, src) + (i - base));
        }
      }
      float4 w = *reinterpret_cast<const float4*>(wl + i);
      float4 h = *reinterpret_cast<const float4*>(hl + i);
      if (BF16) x[0] = round_bf16x4(x[0]);
      float4 acc = scaled(inv, x[0]);
      if (N > 0) {
#pragma unroll
        for (int k = 1; k < M; ++k) add_scaled(acc, inv, x[k]);
      } else {
        for (int k = 1; k < world; ++k) {
          const int src = peer(rank, k, world);
          float4 y;
          if (BF16) y = unpack_bf16x4(ld_stream_u2(recv_slot<const uint16_t>(p, rank, src) + (i - base)));
          else y = ld_stream(recv_slot<const float>(p, rank, src) + (i - base));
          add_scaled(acc, inv, y);
        }
      }
      update_vec<S>(p, cur, i, acc, w, h);
      *reinterpret_cast<float4*>(hl + i) = h;
      *reinterpret_cast<float4*>(wl + i) = w;
      for_peers<N>(world, [&](int k) { st_vec(p.data[peer(rank, k, world)] + i, w); });
    }
    if (blockIdx.x == 0) {  // scalar head / tail of my shard
      const uint64_t i = edge_element(r, threadIdx.x);
      if (i != ~0ull) {
        float acc = scaled(inv, BF16 ? round_bf16(g[i]) : g[i]);
        for (int k = 1; k < world; ++k) {
          const int src = peer(rank, k, world);
          const float y = BF16 ? bf16_bits_to_float(recv_slot<const uint16_t>(p, rank, src)[i - base])
                               : recv_slot<const float>(p, rank, src)[i - base];
          add_scaled(acc, inv, y);
        }
        store_peers(p, world, i, update_scalar<S>(p, cur, i, acc, wl, hl));
      }
    }
  }
  if (tracer) p.trace[3] = globaltimer_ns();

  // ---- barrier B: every peer's weight shard has landed in my data_ ----------
  cta_signal(p, 1);
  if (zero) {  // own shard of diff_: read by this CTA in phase 2 only
    zero_range<true>(g, shard_range(p.count, world, rank), tid, stride);
  }
  if (!cta_wait(p, 1, &s_abort)) return;
  if (tracer) p.trace[4] = globaltimer_ns();
}

}  // namespace

uint64_t push_recv_stride(uint64_t count, int world) {
  const uint64_t max_shard = (count + world - 1) / world;  // shard sizes differ by at most one element
  return (max_shard + 4 * 32 + 8 + 31) / 32 * 32;          // + up to 32 vectors of 512-byte alignment slack in front
}

cudaError_t launch_fused_sync_sgd_push(const SyncParams& p, int grid, int block, int vecs_per_thread,
                                       cudaStream_t stream) {
  if (!check_world(p, 2)) return cudaErrorInvalidValue;
  if (p.mode != kModeTwoShot || p.recv_stride == 0) return cudaErrorInvalidValue;
  if (block <= 0) block = kPushThreads;
  if (block > kPushThreads || block < kMaxRanks || (block & 31)) return cudaErrorInvalidValue;
  if (vecs_per_thread <= 0) vecs_per_thread = 2;
  const int cap = 2 * 148 < kMaxCtas ? 2 * 148 : kMaxCtas;
  if (grid <= 0) {
    // sized by the scatter phase, which moves (N-1)/N of the buffer: vecs_per_thread of those vectors per thread
    // (the owner phase then has 1/(N-1) of that per thread).  Few CTAs = few flags, many CTAs = bandwidth.
    // Depends only on (P, N): identical on every rank, as the per-CTA barriers need.
    const uint64_t vecs = (p.count - p.count / p.world) >> 2;
    const uint64_t per_cta = static_cast<uint64_t>(block) * vecs_per_thread;
    uint64_t need = (vecs + per_cta - 1) / per_cta;
    if (need < 1) need = 1;
    grid = static_cast<int>(need > static_cast<uint64_t>(cap) ? cap : need);
  }
  if (grid > kMaxCtas) grid = kMaxCtas;
  const size_t smem = seg_smem_bytes(p, kPushMaxSeg);
  return dispatch_solver(p.solver, [&](auto S) {
    return dispatch_world(p.world, [&](auto N) {
      if (p.grad_bf16) fused_sync_sgd_push_kernel<N, true, S><<<grid, block, smem, stream>>>(p);
      else fused_sync_sgd_push_kernel<N, false, S><<<grid, block, smem, stream>>>(p);
      return cudaGetLastError();
    });
  });
}

}  // namespace cosb
