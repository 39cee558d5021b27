// fused_sync_sgd.cu -- the inter-executor gradient sync + SGD update as ONE
// sm_100a kernel over NVLink peer memory.
//
// Reference behaviour being replaced (paths relative to the reference repo):
//   parallel_cpu.cpp:120-122 / parallel.cpp:377   diff *= 1/solver_count
//   socket_sync_cpu.cpp:108-133 (socket_sync.cpp:125-154, rdma_sync.cpp:127-158)
//        reduce-scatter: owner r adds the shards of peers r+1, r+2, ... (mod N)
//        IN THAT ORDER:  diff[own] = recv_p + diff[own]
//   sgd_solver.cpp:145-204 Regularize (L2), :213-243 ComputeUpdateValue,
//   sgd_solver.cu:7-12 SGDUpdate, blob.cpp:162-179 Blob::Update  (w -= h)
//   socket_sync_cpu.cpp:102-105,135-163 on_start(): all-gather of weight shards
//   net.cpp:931-948 ClearParamDiffs (optional fold: diff := 0)
// The reference moves every shard GPU->host->TCP/verbs->host->GPU and runs
// N-1 add kernels, a scal, two axpy and the SGDUpdate kernel per iteration;
// here every rank launches this kernel once and
//   phase 0  (bf16 wire only) casts its fp32 gradient to bf16 for the peers,
//   barrier A  per-CTA flag exchange in peer memory: "my gradients are ready",
//   phase 1  the shard owner loads its shard of every peer's gradient straight
//            over NVLink, sums in the reference's order with fp32 accumulation,
//            applies decay + momentum + update, stores the new weights locally
//            AND into every peer's data_ (the all-gather as remote stores),
//   barrier B  "my reads of your diff_ are done, my weight stores have landed",
//   phase 2  (optional) zeroes the local diff_ for the next iteration.
// Every fp32 operation uses an explicitly rounded intrinsic (__fmul_rn /
// __fadd_rn), so nothing is contracted into FMA and the result is bit-identical
// to the un-fused CPU arithmetic of the reference (oracle/sync_oracle.c).
//
// Work partition: element ranges are cut into float4 vectors aligned to the
// buffer base; vector j of a shard belongs to CTA (j / blockDim) % gridDim on
// EVERY rank.  So CTA b of rank p only ever touches data that CTA b of the
// shard owner reads or writes, and per-CTA (not grid-wide) cross-GPU barriers
// are sufficient for all three phases.
#include "fused_sync_sgd.hpp"
#include "sync_device.cuh"

namespace cosb {
namespace {

constexpr int kDefaultThreads = 512;
constexpr int kMaxSegSmem = 1024;

// --------------------------------------------------------- reduce (phase 1)

// Sum of the world's gradients for vector/element i of shard s in the
// reference's order s, s+1, ..., s+N-1 (mod N), each scaled by 1/N BEFORE the
// sum (parallel_cpu.cpp:120-122 runs before socket_sync_cpu.cpp:112-132).
template <int N, bool BF16>
__device__ __forceinline__ float4 reduce_vec(const SyncParams& p, int s, uint64_t i) {
  float4 x[N];
#pragma unroll
  for (int j = 0; j < N; ++j) {  // all loads first: N independent 128-bit requests in flight
    const int src = peer(s, j, N);
    x[j] = BF16 ? unpack_bf16x4(ld_stream_u2(p.wire[src] + i)) : ld_stream(p.diff[src] + i);
  }
  float4 acc = scaled(p.inv_scale, x[0]);
#pragma unroll
  for (int j = 1; j < N; ++j) add_scaled(acc, p.inv_scale, x[j]);
  return acc;
}

template <int N, bool BF16>
__device__ __forceinline__ float4 reduce_vec_any(const SyncParams& p, int s, uint64_t i) {
  if (N > 0) return reduce_vec<(N > 0 ? N : 1), BF16>(p, s, i);
  return make_float4(reduce_scalar<BF16>(p, s, i), reduce_scalar<BF16>(p, s, i + 1),
                     reduce_scalar<BF16>(p, s, i + 2), reduce_scalar<BF16>(p, s, i + 3));
}

// ------------------------------------------------------------- the kernel

// N = compile-time world size (0 = runtime world, any size up to kMaxRanks).
// (The in-switch NVLS variant lives in fused_sync_sgd_nvls.cu.)
template <int N, bool BF16>
__global__ void __launch_bounds__(kDefaultThreads, 2) fused_sync_sgd_kernel(const SyncParams p) {
  extern __shared__ unsigned char smem_raw[];
  __shared__ int s_abort;
  SegCursor cur = load_seg_table(p, smem_raw, kMaxSegSmem);  // segment (= learnable blob) table
  if (threadIdx.x == 0) s_abort = 0;
  __syncthreads();

  const bool tracer = p.trace != nullptr && blockIdx.x == 0 && threadIdx.x == 0;
  if (tracer) p.trace[0] = globaltimer_ns();
  const int world = (N > 0) ? N : p.world;
  const int rank = p.rank;
  const uint64_t tid = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  const bool multi = p.mode != kModeLocal;

  // ---- phase 0: fp32 -> bf16 wire cast of the whole local gradient --------
  if (BF16 && (p.mode == kModeTwoShot || p.mode == kModeOneShot)) {
    const float* g = p.diff[rank];
    uint16_t* wv = p.wire[rank];
    for (int s = 0; s < world; ++s) {
      const ShardRange r = shard_range(p.count, world, s);
      for (uint64_t j = tid; j < r.nvec; j += stride) {
        const uint64_t i = (r.vec_lo + j) << 2;
        *reinterpret_cast<uint2*>(wv + i) = pack_bf16x4(ld_stream(g + i));
      }
      if (blockIdx.x == 0) {
        const uint64_t i = edge_element(r, threadIdx.x);
        if (i != ~0ull) wv[i] = float_to_bf16_bits(g[i]);
      }
    }
  }

  // ---- barrier A: every rank's gradients (and wire casts) are complete ----
  if (multi) {
    if (!cta_barrier(p, 0, &s_abort)) return;
  }
  if (tracer) p.trace[1] = globaltimer_ns();

  // ---- phase 1 ------------------------------------------------------------
  if (p.mode == kModeAllGather) {
    // on_start(): owned weight shard -> every peer's data_
    const ShardRange r = shard_range(p.count, world, rank);
    const float* w = p.data[rank];
    for (uint64_t j = tid; j < r.nvec; j += stride) {
      const uint64_t i = (r.vec_lo + j) << 2;
      const float4 v = ld_stream(w + i);
      for (int q = 1; q < world; ++q) st_vec(p.data[peer(rank, q, world)] + i, v);
    }
    if (blockIdx.x == 0) {
      const uint64_t i = edge_element(r, threadIdx.x);
      if (i != ~0ull) store_peers(p, world, i, w[i]);
    }
  } else {
    // shards this rank updates: its own (two-shot), all (one-shot), [0,P) (local)
    const int s_first = (p.mode == kModeOneShot) ? 0 : rank;
    const int s_last = (p.mode == kModeOneShot) ? world - 1 : rank;
    const bool push = p.mode == kModeTwoShot;
    float* wl = p.data[rank];
    float* hl = p.hist;
    for (int s = s_first; s <= s_last; ++s) {
      const ShardRange r = p.mode == kModeLocal ? shard_range(p.count, 1, 0) : shard_range(p.count, world, s);
      if (tid < r.nvec) cur.seek((r.vec_lo + tid) << 2);
      for (uint64_t j = tid; j < r.nvec; j += stride) {
        const uint64_t i = (r.vec_lo + j) << 2;
        float4 w = *reinterpret_cast<const float4*>(wl + i);
        float4 h = *reinterpret_cast<const float4*>(hl + i);
        float4 g;
        if (p.mode == kModeLocal) {
          g = ld_stream(p.diff[rank] + i);  // no scale at N == 1 (CaffeNet.cpp:206-216: no sync object)
          if (BF16) g = round_bf16x4(g);  // bf16 gradient inputs: same rounding the wire applies at N > 1
        } else {
          g = reduce_vec_any<N, BF16>(p, s, i);
        }
        sgd_vec(p, cur, i, g, w, h);
        *reinterpret_cast<float4*>(hl + i) = h;
        *reinterpret_cast<float4*>(wl + i) = w;
        if (push) for_peers<N>(world, [&](int q) { st_vec(p.data[peer(rank, q, world)] + i, w); });
      }
      if (blockIdx.x == 0) {  // scalar head / tail of the range (<= 3 elements each)
        const uint64_t i = edge_element(r, threadIdx.x);
        if (i != ~0ull) {
          float g = (p.mode == kModeLocal) ? p.diff[rank][i] : reduce_scalar<BF16>(p, s, i);
          if (BF16 && p.mode == kModeLocal) g = round_bf16(g);
          const float w = sgd_scalar(p, cur, i, g, wl, hl);
          if (push) store_peers(p, world, i, w);
        }
      }
    }
  }

  // ---- barrier B: peers finished reading my diff_, their pushes landed ----
  if (tracer) p.trace[2] = globaltimer_ns();
  if (multi) {
    if (!cta_barrier(p, 1, &s_abort)) return;
  }
  if (tracer) p.trace[3] = globaltimer_ns();

  // ---- phase 2: ClearParamDiffs of the next Step --------------------------
  if (p.zero_diff && p.mode != kModeAllGather) {
    // inline, not zero_range<false>: its asm stores are not unrolled (<5,false>: STG.E.128 36 -> 27 static)
    float* g = const_cast<float*>(p.diff[rank]);
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    if (p.mode == kModeLocal) {
      const uint64_t nvec = p.count >> 2;
      for (uint64_t j = tid; j < nvec; j += stride) *reinterpret_cast<float4*>(g + (j << 2)) = z;
      if (blockIdx.x == 0 && threadIdx.x < (p.count & 3)) g[(nvec << 2) + threadIdx.x] = 0.f;
    } else {
      for (int s = 0; s < world; ++s) {
        const ShardRange r = shard_range(p.count, world, s);
        for (uint64_t j = tid; j < r.nvec; j += stride) *reinterpret_cast<float4*>(g + ((r.vec_lo + j) << 2)) = z;
        zero_edges(g, r);
      }
    }
  }
  if (tracer) p.trace[4] = globaltimer_ns();
}

__device__ __forceinline__ uint64_t mix64(uint64_t z) {
  z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ULL;
  z = (z ^ (z >> 27)) * 0x94d049bb133111ebULL;
  return z ^ (z >> 31);
}

__global__ void fill_kernel(float* out, uint64_t n, uint64_t key, float amp) {
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
    uint64_t z = mix64(key + i * 0x9e3779b97f4a7c15ULL);
    int32_t v = static_cast<int32_t>(z >> 40) - (1 << 23);
    out[i] = __fmul_rn(amp, __fmul_rn(static_cast<float>(v), 1.0f / 8388608.0f));
  }
}

uint64_t host_mix64(uint64_t z) {
  z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ULL;
  z = (z ^ (z >> 27)) * 0x94d049bb133111ebULL;
  return z ^ (z >> 31);
}

}  // namespace

int default_sync_grid(int device) {
  return 2 * sm_count(device);  // __launch_bounds__(512, 2): two resident CTAs per SM
}

cudaError_t launch_fused_sync_sgd(const SyncParams& p, int grid, int block, cudaStream_t stream) {
  if (!check_world(p, 1)) return cudaErrorInvalidValue;
  if (block <= 0) block = kDefaultThreads;
  if (block > kDefaultThreads || block < kMaxRanks || (block & 31)) return cudaErrorInvalidValue;
  if (grid <= 0) grid = default_sync_grid(-1);
  if (grid > kMaxCtas) grid = kMaxCtas;
  // do not launch more CTAs than there is work for (tiny nets): one vector per thread
  uint64_t work_vecs = (p.mode == kModeOneShot || p.mode == kModeLocal) ? (p.count >> 2)
                                                                       : (p.count / p.world) >> 2;
  if (p.zero_diff || p.grad_bf16) work_vecs = p.count >> 2;
  uint64_t need = (work_vecs + block - 1) / block;
  if (need < 1) need = 1;
  if (static_cast<uint64_t>(grid) > need) grid = static_cast<int>(need);
  const size_t smem = seg_smem_bytes(p, kMaxSegSmem);
  const int n = (p.mode == kModeLocal || p.mode == kModeAllGather) ? 0 : p.world;
  return dispatch_world(n, [&](auto N) {
    if (p.grad_bf16) fused_sync_sgd_kernel<N, true><<<grid, block, smem, stream>>>(p);
    else fused_sync_sgd_kernel<N, false><<<grid, block, smem, stream>>>(p);
    return cudaGetLastError();
  });
}

// TMA (cp.async.bulk) pipelined variant: see fused_sync_sgd_tma.cu.

cudaError_t launch_fill(float* out, uint64_t n, uint64_t seed, uint64_t stream_id, float amp, cudaStream_t stream) {
  const uint64_t key = host_mix64(seed * 0x9e3779b97f4a7c15ULL + stream_id);
  int grid = static_cast<int>((n + 255) / 256);
  if (grid > 148 * 16) grid = 148 * 16;
  if (grid < 1) grid = 1;
  fill_kernel<<<grid, 256, 0, stream>>>(out, n, key, amp);
  return cudaGetLastError();
}

}  // namespace cosb
