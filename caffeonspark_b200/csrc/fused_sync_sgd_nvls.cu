// fused_sync_sgd_nvls.cu -- the fused sync kernel with the reduction and the
// weight broadcast done INSIDE the NVSwitch (NVLS / NVLink SHARP), optionally
// sharing the work with plain P2P loads/stores so that both the switch's
// reduction engines and the remaining link bandwidth are used.
//
// Same reference mapping as fused_sync_sgd.cu (two-shot, fp32 wire only):
//   parallel_cpu.cpp:120-122 scale, socket_sync_cpu.cpp:108-133 reduce-scatter,
//   sgd_solver.cpp:145-243 + blob.cpp:162-179 update, socket_sync_cpu.cpp:102-105
//   all-gather of the updated weight shards, net.cpp:931-948 ClearParamDiffs.
// Per float4 of the owned shard:
//   NVLS vector : ONE multimem.ld_reduce.add.v4.f32 on the multicast address of
//                 diff_ (SASS LDGMC.E.ADD.F32x4: the switch reads the word on
//                 every rank and returns the fp32 sum), 1/N scale, update, ONE
//                 multimem.st of the new weights on the multicast address of
//                 data_ (lands on every rank, this one included).
//   P2P vector  : N loads from the peers' diff_, summed in the reference's order
//                 with the scale before the sum (bit-exact), update, N-1 stores.
// NVLink bytes per direction per GPU: NVLS ~ 4P(1 + 1/N), P2P 8P(N-1)/N.  The
// switch chooses the order of the NVLS sum, so results match the reference to
// rounding (north star: 1e-5 relative), not bit for bit; every rank still ends
// up with IDENTICAL weights because only the owner computes a shard.
// Each thread keeps UN switch loads + UP x N peer loads + the local w/h loads in
// flight (all issued before the first use).
//
// ClearParamDiffs overlapped with the reduction.  The path is NVLink-bound, HBM
// is almost idle, yet zeroing diff_ (4P bytes) after barrier B was a serial
// ~30-70 us tail (profiles/r02_matrix_large_n8.json).  Now 15 of the 16 warps
// of a CTA reduce; vector j of a shard belongs to CTA (j / 480) % gridDim on
// every rank.  After each grid-stride iteration the owner's CTA publishes its
// iteration count into flag array C of every rank (one relaxed store per peer,
// no fence: it only says "my switch loads of these vectors have RETURNED", i.e.
// your diff_ has been read).  The 16th warp of the same-numbered CTA on every
// rank polls those counters in its LOCAL flag memory and zeroes, behind the
// readers, exactly the vectors that CTA of that owner has consumed.  When the
// reduction ends, diff_ is already zero; barrier B only waits for the weights.
#include "fused_sync_sgd.hpp"
#include "sync_device.cuh"

namespace cosb {
namespace {

constexpr int kNvlsThreads = 512;
constexpr int kNvlsMaxSeg = 1024;

constexpr int kWorkThreads = kNvlsThreads - 32;  // warps 0..14 reduce, warp 15 zeroes diff_ behind them
constexpr uint32_t kIterBits = 16;               // progress word = (epoch << 16) | iterations done (< 65536)

__device__ __forceinline__ void work_bar() { asm volatile("bar.sync 1, %0;" ::"n"(kWorkThreads) : "memory"); }

template <int UN, int UP, int N>
__global__ void __launch_bounds__(kNvlsThreads, 1) fused_sync_sgd_nvls_kernel(const SyncParams p) {
  extern __shared__ unsigned char smem_raw[];
  __shared__ int s_abort;
  SegCursor cur = load_seg_table(p, smem_raw, kNvlsMaxSeg);
  if (threadIdx.x == 0) s_abort = 0;
  const bool tracer = p.trace != nullptr && blockIdx.x == 0 && threadIdx.x == 0;
  if (tracer) p.trace[0] = globaltimer_ns();
  const int world = p.world;
  const int rank = p.rank;
  constexpr int U = UN + UP;
  constexpr int NP = N > 0 ? N : 1;
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * kWorkThreads;  // vectors per grid-wide round
  const uint64_t cta_first = static_cast<uint64_t>(blockIdx.x) * kWorkThreads;
  const uint32_t tag = p.epoch << kIterBits;

  // ---- barrier A: every rank has entered the kernel, i.e. its gradients are complete
  if (!cta_barrier(p, 0, &s_abort)) return;
  if (tracer) p.trace[1] = globaltimer_ns();

  if (threadIdx.x < kWorkThreads) {
    // =================== warps 0..14: reduce + update + broadcast ===================
    const ShardRange r = shard_range(p.count, world, rank);
    float* wl = p.data[rank];
    float* hl = p.hist;
    const float inv = p.inv_scale;
    const uint64_t tid = cta_first + threadIdx.x;
    // every work thread of the grid runs the same number of iterations, so the CTA-wide bar.sync below is safe
    const uint64_t iters = (r.off + r.nvec + stride * U - 1) / (stride * U);  // over the 512-byte aligned index space
    for (uint64_t it = 0; it < iters; ++it) {
      const uint64_t j0 = tid + it * stride * U;
      float4 s[UN > 0 ? UN : 1];
      float4 x[UP > 0 ? UP : 1][NP];
      float4 w[U], h[U];
      // -- issue every load of this iteration
#pragma unroll
      for (int u = 0; u < UN; ++u) {
        const uint64_t i = vec_elem(r, j0 + static_cast<uint64_t>(u) * stride);
        if (i != ~0ull) s[u] = mc_ld_reduce(p.mc_diff + i);
      }
#pragma unroll
      for (int u = 0; u < UP; ++u) {
        const uint64_t i = vec_elem(r, j0 + static_cast<uint64_t>(UN + u) * stride);
        if (i != ~0ull) {
#pragma unroll
          for (int k = 0; k < NP; ++k) x[u][k] = ld_stream(p.diff[peer(rank, k, NP)] + i);
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const uint64_t i = vec_elem(r, j0 + static_cast<uint64_t>(u) * stride);
        if (i != ~0ull) {
          w[u] = ld_stream(wl + i);
          h[u] = ld_stream(hl + i);
        }
      }
      // -- consume
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const uint64_t i = vec_elem(r, j0 + static_cast<uint64_t>(u) * stride);
        if (i != ~0ull) {
          float4 g;
          if (u < UN) {  // in-switch sum over all ranks, then the 1/N scale
            g = scaled(inv, s[u]);
          } else {       // reference order: scale first, then r, r+1, ... (mod N)
            const int q = u - UN;
            g = scaled(inv, x[q][0]);
#pragma unroll
            for (int k = 1; k < NP; ++k) add_scaled(g, inv, x[q][k]);
          }
          cur.seek(i);
          sgd_vec(p, cur, i, g, w[u], h[u]);
          st_vec(hl + i, h[u]);
          if (u < UN) {
            mc_st(p.mc_data + i, w[u]);  // one store: own data_ and every peer's data_
          } else {
            st_vec(wl + i, w[u]);
#pragma unroll
            for (int k = 1; k < NP; ++k) st_vec(p.data[peer(rank, k, NP)] + i, w[u]);
          }
        }
      }
      // -- every gradient load of this CTA's iteration has returned: tell the zeroing warps of all ranks
      if (p.zero_diff) {
        work_bar();
        if (static_cast<int>(threadIdx.x) < world)
          asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(flag_slot(p.flags[threadIdx.x], 2, blockIdx.x, rank)),
                       "r"(tag | static_cast<uint32_t>(it + 1))
                       : "memory");
      }
    }
    if (blockIdx.x == 0) {  // scalar head / tail of my shard (<= 3 elements each): plain P2P, reference order
      const uint64_t i = edge_element(r, threadIdx.x);
      if (i != ~0ull) {
        // inline, not reduce_scalar<false>: that changes the static FMUL count of <4,1,4> (515 -> 491)
        float acc = 0.f;
        for (int k = 0; k < world; ++k) {
          const float y = __fmul_rn(inv, p.diff[peer(rank, k, world)][i]);
          acc = (k == 0) ? y : __fadd_rn(y, acc);
        }
        store_peers(p, world, i, sgd_scalar(p, cur, i, acc, wl, hl));
      }
    }
  } else if (p.zero_diff) {
    // =================== warp 15: ClearParamDiffs behind the readers ===================
    const int lane = threadIdx.x - kWorkThreads;
    float* g = const_cast<float*>(p.diff[rank]);
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    uint32_t done[kMaxRanks];  // iterations of owner q (same CTA index) already zeroed here
    for (int q = 0; q < world; ++q) done[q] = 0;
    const unsigned long long t0 = globaltimer_ns();
    unsigned spins = 0;
    for (;;) {
      bool all = true, moved = false;
      for (int q = 0; q < world; ++q) {
        const ShardRange rq = shard_range(p.count, world, q);
        const uint32_t total = static_cast<uint32_t>((rq.off + rq.nvec + stride * U - 1) / (stride * U));
        if (done[q] >= total) continue;
        const uint32_t v = ld_relaxed_sys(flag_slot(p.flags[rank], 2, blockIdx.x, q));
        const uint32_t upto = (v >> kIterBits) == (tag >> kIterBits) ? (v & ((1u << kIterBits) - 1u)) : 0u;
        for (uint32_t it = done[q]; it < upto; ++it) {  // this CTA's vectors of iteration `it` of shard q
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const uint64_t first = cta_first + (static_cast<uint64_t>(it) * U + u) * stride;  // kWorkThreads vectors
            for (int t = lane; t < kWorkThreads; t += 32) {
              const uint64_t i = vec_elem(rq, first + t);
              if (i != ~0ull) st_vec(g + i, z);
            }
          }
        }
        if (upto > done[q]) {
          done[q] = upto;
          moved = true;
        }
        if (done[q] < total) all = false;
      }
      if (all) break;
      if (!moved) __nanosleep(256);  // leave the load/store unit to the 15 reducing warps
      if ((++spins & 0xffu) == 0) {
        if (*reinterpret_cast<volatile int*>(&s_abort)) break;
        if (globaltimer_ns() - t0 > p.timeout_ns) {  // an owner never finished its reduce phase
          if (lane == 0) {
            atomicExch(p.status, 400);
            *reinterpret_cast<volatile int*>(&s_abort) = 1;
          }
          break;
        }
      }
    }
  }
  if (tracer) p.trace[2] = globaltimer_ns();

  // ---- barrier B: the switch has read my diff_ for every owner, all weights have landed
  if (!cta_barrier(p, 1, &s_abort)) return;
  if (tracer) p.trace[3] = globaltimer_ns();

  // ---- the scalar head / tail elements of every shard (<= 3 each) were read with plain loads by CTA 0 of the
  // owners: zero them after barrier B
  if (p.zero_diff && blockIdx.x == 0) {
    float* g = const_cast<float*>(p.diff[rank]);
    for (int s = 0; s < world; ++s) zero_edges(g, shard_range(p.count, world, s));
  }
  if (tracer) p.trace[4] = globaltimer_ns();
}

template <int UN, int UP, int N>
cudaError_t launch_cfg(const SyncParams& p, int grid, size_t smem, cudaStream_t stream) {
  fused_sync_sgd_nvls_kernel<UN, UP, N><<<grid, kNvlsThreads, smem, stream>>>(p);
  return cudaGetLastError();
}

template <int UN>
cudaError_t launch_share(const SyncParams& p, int grid, size_t smem, cudaStream_t stream) {
  switch (p.world) {  // the P2P share needs the world size at compile time (register arrays)
    case 2: return launch_cfg<UN, 1, 2>(p, grid, smem, stream);
    case 4: return launch_cfg<UN, 1, 4>(p, grid, smem, stream);
    case 8: return launch_cfg<UN, 1, 8>(p, grid, smem, stream);
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace

cudaError_t launch_fused_sync_sgd_nvls(const SyncParams& p, int grid, cudaStream_t stream) {
  if (!check_world(p, 2)) return cudaErrorInvalidValue;
  if (p.solver != kSolverSGD) return cudaErrorInvalidValue;  // SGD only: the routing never sends another solver here
  if (p.mode != kModeTwoShot || p.grad_bf16 || !p.mc_data || !p.mc_diff) return cudaErrorInvalidValue;
  if (grid <= 0) grid = sm_count(-1);  // __launch_bounds__(512, 1): one resident CTA per SM
  if (grid > kMaxCtas) grid = kMaxCtas;
  uint64_t need = (((p.count / p.world) >> 2) + kWorkThreads - 1) / kWorkThreads;  // one vector per work thread
  if (need < 1) need = 1;
  if (static_cast<uint64_t>(grid) > need) grid = static_cast<int>(need);
  const size_t smem = seg_smem_bytes(p, kNvlsMaxSeg);
  {  // the per-CTA progress counter has kIterBits bits
    const uint64_t u = static_cast<uint64_t>((p.nvls_unroll > 0 ? p.nvls_unroll : 1) + (p.nvls_p2p > 0 ? 1 : 0));
    const uint64_t per_round = static_cast<uint64_t>(grid) * kWorkThreads * u;
    if ((((p.count / p.world) >> 2) + 64 + per_round) / per_round >= (1ull << kIterBits)) return cudaErrorInvalidValue;
  }
  const int un = p.nvls_unroll > 0 ? p.nvls_unroll : 1;
  if (p.nvls_p2p <= 0) {
    switch (un) {
      case 2: return launch_cfg<2, 0, 0>(p, grid, smem, stream);
      case 4: return launch_cfg<4, 0, 0>(p, grid, smem, stream);
      case 8: return launch_cfg<8, 0, 0>(p, grid, smem, stream);
      default: return launch_cfg<1, 0, 0>(p, grid, smem, stream);
    }
  }
  switch (un) {  // one P2P vector per `un` switch vectors
    case 1: return launch_share<1>(p, grid, smem, stream);
    case 2: return launch_share<2>(p, grid, smem, stream);
    case 3: return launch_share<3>(p, grid, smem, stream);
    default: return launch_share<4>(p, grid, smem, stream);
  }
}

}  // namespace cosb
