// fused_sync_sgd_tma.cu -- the fused sync kernel with ALL bulk data movement on
// the TMA engine (cp.async.bulk, SASS UBLKCP) and a multi-stage shared-memory
// pipeline; same arithmetic, same barriers and same results as the vector
// kernel in fused_sync_sgd.cu (see that file for the reference mapping).
//
// Why: over NVLink a peer load has ~2-4 us latency, so the achieved bandwidth of
// the LDG path is bounded by how many bytes each SM keeps in flight
// (threads x registers).  Here one elected thread per CTA keeps kStages-1 tiles
// per source in flight with bulk copies that need no registers at all:
//   per tile  : N gradient tiles (one per rank, read straight from the peers'
//               diff_ / bf16 wire buffer), the weight tile and the history tile
//               are bulk-loaded into one pipeline stage and complete on an
//               mbarrier (complete_tx::bytes);
//   consumers : 256 threads reduce the N tiles in the reference's order out of
//               shared memory, apply decay + momentum + update in place;
//   write-back: the elected thread bulk-stores the new weight tile to the local
//               data_ AND to every peer's data_ (the all-gather), and the
//               history tile locally.
// Work partition: tile t of a shard belongs to CTA t % gridDim on every rank, so
// the per-CTA cross-GPU barriers of sync_device.cuh remain sufficient.
#include "fused_sync_sgd.hpp"
#include "sync_device.cuh"

namespace cosb {
namespace {

constexpr int kTmaThreads = 256;
constexpr int kStages = 4;
constexpr int kMaxSegSmemTma = 512;

// ------------------------------------------------------------ PTX wrappers

__device__ __forceinline__ uint32_t smem_addr(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
}

__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes)
               : "memory");
}

__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_addr(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}

// global -> shared bulk copy completing on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void tma_load(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_addr(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_addr(bar))
               : "memory");
}

// shared -> global bulk copy, tracked by bulk async-groups
__device__ __forceinline__ void tma_store(void* dst_gmem, const void* src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem),
               "r"(smem_addr(src_smem)), "r"(bytes)
               : "memory");
}

__device__ __forceinline__ void tma_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void tma_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// make generic-proxy writes to shared memory visible to the async proxy (TMA)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// order generic-proxy accesses to GLOBAL memory (the bf16 wire cast of phase 0, the peers' gradients acquired
// through the generic-proxy flag loads of barrier A) against the async-proxy bulk copies that follow, and the
// completed bulk stores against the generic-proxy release of barrier B (PTX memory model: cross-proxy fence)
__device__ __forceinline__ void fence_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }

// ------------------------------------------------------------- job iterator

// Element range of a shard cut into an A-element-aligned body (bulk copies need
// 16-byte aligned addresses and sizes: A = 4 for fp32 sources, 8 for the bf16
// wire) and scalar head / tail pieces of at most A-1 elements each.
struct BodyRange {
  uint64_t lo, hi;      // shard element range
  uint64_t b0, b1;      // aligned body [b0, b1)
  uint64_t head_end;    // [lo, head_end) scalar head
  uint64_t tail_begin;  // [tail_begin, hi) scalar tail
};

__device__ __forceinline__ BodyRange body_range(const SyncParams& p, int s, uint64_t A) {
  BodyRange r;
  if (p.mode == kModeLocal) {
    r.lo = 0;
    r.hi = p.count;
  } else {
    r.lo = chunk(p.count, p.world, s);
    r.hi = chunk(p.count, p.world, s + 1ull);
  }
  const uint64_t b0 = (r.lo + A - 1) / A * A, b1 = r.hi / A * A;
  if (b1 > b0) {
    r.b0 = b0; r.b1 = b1; r.head_end = b0; r.tail_begin = b1;
  } else {
    r.b0 = r.b1 = b0; r.head_end = r.hi; r.tail_begin = r.hi;  // everything scalar
  }
  return r;
}

// The sequence of (shard, tile) jobs of this CTA: tile t of shard s belongs to
// CTA t % gridDim.  Identical on every thread and, run kStages-1 ahead, on the
// elected producer thread.
struct JobIter {
  int s, s_last;
  uint64_t tile_elems, t, A;
  BodyRange r;
  bool valid;

  __device__ void init(const SyncParams& p, uint64_t tile, uint64_t align) {
    tile_elems = tile;
    A = align;
    const bool all = p.mode == kModeOneShot;
    s = (all || p.mode == kModeLocal) ? 0 : p.rank;
    s_last = all ? p.world - 1 : s;
    r = body_range(p, s, A);
    t = blockIdx.x;
    settle(p);
  }
  __device__ uint64_t ntiles() const { return (r.b1 - r.b0 + tile_elems - 1) / tile_elems; }
  __device__ void settle(const SyncParams& p) {
    valid = true;
    while (t >= ntiles()) {
      if (s >= s_last) { valid = false; return; }
      ++s;
      r = body_range(p, s, A);
      t = blockIdx.x;
    }
  }
  __device__ void next(const SyncParams& p) {
    t += gridDim.x;
    settle(p);
  }
  __device__ uint64_t elem0() const { return r.b0 + t * tile_elems; }
  __device__ uint32_t elems() const {
    const uint64_t rem = r.b1 - elem0();
    return static_cast<uint32_t>(rem < tile_elems ? rem : tile_elems);
  }
};

// ------------------------------------------------------------------ kernel

struct StageView {
  unsigned char* src;   // world (or 1) gradient tiles, gsz bytes per element, back to back
  float* w;             // weight tile
  float* h;             // history tile
};

template <bool BF16>
__global__ void __launch_bounds__(kTmaThreads, 1)
fused_sync_sgd_tma_kernel(const SyncParams p, const int tile_elems) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ int s_abort;
  const int tid = threadIdx.x;
  const int world = p.world;
  const int rank = p.rank;
  const bool local = p.mode == kModeLocal;
  const bool multi = !local;
  const int nsrc = local ? 1 : world;
  const uint32_t gsz = (BF16 && !local) ? 2u : 4u;
  const uint64_t A = (BF16 && !local) ? 8 : 4;  // body alignment in elements (16-byte bulk copies)

  // smem carve-up: [full mbarriers][segment table][stages]
  uint64_t* full = reinterpret_cast<uint64_t*>(smem);
  size_t off = 128 + (p.nseg <= kMaxSegSmemTma ? static_cast<size_t>(p.nseg) * 16 : 0);
  off = (off + 127) & ~static_cast<size_t>(127);
  const size_t src_bytes = static_cast<size_t>(nsrc) * tile_elems * gsz;
  const size_t stage_bytes = src_bytes + 2ull * tile_elems * sizeof(float);
  auto stage = [&](int k) {
    StageView v;
    v.src = smem + off + static_cast<size_t>(k) * stage_bytes;
    v.w = reinterpret_cast<float*>(v.src + src_bytes);
    v.h = v.w + tile_elems;
    return v;
  };

  if (tid == 0) {
    s_abort = 0;
    for (int k = 0; k < kStages; ++k) mbar_init(&full[k], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  SegCursor cur = load_seg_table(p, smem + 128, kMaxSegSmemTma);
  __syncthreads();
  bool cur_seeked = false;

  // f(i) for the first element i of every float4 of this thread in the aligned body of r, with phase 1's tile -> CTA
  // partition (phases 0 and 2)
  auto for_body_vecs = [&](const BodyRange& r, auto&& f) {
    for (uint64_t t0 = r.b0 + static_cast<uint64_t>(blockIdx.x) * tile_elems; t0 < r.b1;
         t0 += static_cast<uint64_t>(gridDim.x) * tile_elems) {
      const uint64_t t1 = (t0 + tile_elems < r.b1) ? t0 + tile_elems : r.b1;
      for (uint64_t i = t0 + 4ull * tid; i < t1; i += 4ull * kTmaThreads) f(i);
    }
  };

  // ---- phase 0: fp32 -> bf16 wire cast, same tile -> CTA partition ----------
  if (BF16 && multi) {
    const float* g = p.diff[rank];
    uint16_t* wv = p.wire[rank];
    for (int s = 0; s < world; ++s) {
      const BodyRange r = body_range(p, s, A);
      for_body_vecs(r, [&](uint64_t i) { *reinterpret_cast<uint2*>(wv + i) = pack_bf16x4(ld_stream(g + i)); });
      if (blockIdx.x == 0) {
        const uint64_t i = edge_element(r, tid);
        if (i != ~0ull) wv[i] = float_to_bf16_bits(g[i]);
      }
    }
  }

  // ---- barrier A -----------------------------------------------------------
  if (multi) {
    if (!cta_barrier(p, 0, &s_abort)) return;
  }

  // ---- phase 1: pipelined reduce + SGD + write-back -------------------------
  const bool push = p.mode == kModeTwoShot;
  float* wl = p.data[rank];
  float* hl = p.hist;

  auto issue_loads = [&](const JobIter& j, int k) {  // elected thread only
    const StageView v = stage(k);
    const uint32_t n = j.elems();
    const uint64_t i0 = j.elem0();
    mbar_expect_tx(&full[k], n * (static_cast<uint32_t>(nsrc) * gsz + 8u));
    for (int q = 0; q < nsrc; ++q) {
      const int src = peer(j.s, q, world);
      const void* g = local ? static_cast<const void*>(p.diff[rank] + i0)
                            : (BF16 ? static_cast<const void*>(p.wire[src] + i0)
                                    : static_cast<const void*>(p.diff[src] + i0));
      tma_load(v.src + static_cast<size_t>(q) * tile_elems * gsz, g, n * gsz, &full[k]);
    }
    tma_load(v.w, wl + i0, n * 4u, &full[k]);
    tma_load(v.h, hl + i0, n * 4u, &full[k]);
  };

  JobIter cons, prod;
  cons.init(p, tile_elems, A);
  prod = cons;
  if (tid == 0) {  // prologue: kStages-1 tiles in flight
    fence_async_all();
    for (int k = 0; k < kStages - 1 && prod.valid; ++k) {
      issue_loads(prod, k);
      prod.next(p);
    }
  }
  uint32_t it = 0;
  for (; cons.valid; cons.next(p), ++it) {
    const int k = it % kStages;
    const uint32_t parity = (it / kStages) & 1u;
    {  // wait for the tile (bounded spin: a lost bulk copy must not hang the GPU)
      unsigned spins = 0;
      const unsigned long long t0 = globaltimer_ns();
      while (!mbar_try_wait(&full[k], parity)) {
        if ((++spins & 0xfffu) == 0 && globaltimer_ns() - t0 > p.timeout_ns) {
          atomicExch(p.status, 300);
          *reinterpret_cast<volatile int*>(&s_abort) = 1;
          break;
        }
      }
    }
    const StageView v = stage(k);
    const uint32_t n = cons.elems();
    const uint64_t i0 = cons.elem0();
    for (uint32_t e = 4u * tid; e < n; e += 4u * kTmaThreads) {
      float4 acc;
      if (local) {
        acc = *reinterpret_cast<const float4*>(v.src + static_cast<size_t>(e) * 4);
        if (BF16) acc = round_bf16x4(acc);
      } else {
        const float inv = p.inv_scale;
        for (int q = 0; q < nsrc; ++q) {  // order s, s+1, ... (mod N): tile q holds rank (s+q)%N
          float4 x;
          const unsigned char* base = v.src + static_cast<size_t>(q) * tile_elems * gsz;
          if (BF16) x = unpack_bf16x4(*reinterpret_cast<const uint2*>(base + static_cast<size_t>(e) * 2));
          else x = *reinterpret_cast<const float4*>(base + static_cast<size_t>(e) * 4);
          if (q == 0) acc = scaled(inv, x);
          else add_scaled(acc, inv, x);
        }
      }
      float4 w = *reinterpret_cast<const float4*>(v.w + e);
      float4 h = *reinterpret_cast<const float4*>(v.h + e);
      if (!cur_seeked) {
        cur.seek(i0 + e);
        cur_seeked = true;
      }
      sgd_vec(p, cur, i0 + e, acc, w, h);
      *reinterpret_cast<float4*>(v.w + e) = w;
      *reinterpret_cast<float4*>(v.h + e) = h;
    }
    fence_async_smem();
    __syncthreads();
    if (*reinterpret_cast<volatile int*>(&s_abort)) return;
    if (tid == 0) {
      tma_store(wl + i0, v.w, n * 4u);
      tma_store(hl + i0, v.h, n * 4u);
      if (push) {
        for (int q = 1; q < world; ++q) tma_store(p.data[peer(rank, q, world)] + i0, v.w, n * 4u);
      }
      tma_commit();
      // the stage used by the PREVIOUS iteration is free once its stores have
      // read shared memory: refill it with the tile kStages-1 ahead
      tma_wait_read<1>();
      if (prod.valid) {
        issue_loads(prod, (it + kStages - 1) % kStages);
        prod.next(p);
      }
    }
  }
  if (tid == 0) {
    tma_wait_all();  // every weight / history tile has landed (incl. peer memory)
    fence_async_all();
  }

  // scalar head / tail of each range (<= 3 elements each), plain loads/stores by CTA 0
  if (blockIdx.x == 0) {
    const int s_first = (p.mode == kModeOneShot || local) ? 0 : rank;
    const int s_last = (p.mode == kModeOneShot) ? world - 1 : (local ? 0 : rank);
    for (int s = s_first; s <= s_last; ++s) {
      const BodyRange r = body_range(p, s, A);
      const uint64_t i = edge_element(r, tid);
      if (i != ~0ull) {
        float g;
        if (local) {
          g = p.diff[rank][i];
          if (BF16) g = round_bf16(g);
        } else {
          g = reduce_scalar<BF16>(p, s, i);
        }
        const float w = sgd_scalar(p, cur, i, g, wl, hl);
        if (push) store_peers(p, world, i, w);
      }
    }
  }

  // ---- barrier B -----------------------------------------------------------
  if (multi) {
    if (!cta_barrier(p, 1, &s_abort)) return;
  }

  // ---- phase 2: diff := 0, same tile -> CTA partition ------------------------
  if (p.zero_diff) {
    float* g = const_cast<float*>(p.diff[rank]);
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    const int ns = local ? 1 : world;
    for (int s = 0; s < ns; ++s) {
      const BodyRange r = body_range(p, s, A);
      for_body_vecs(r, [&](uint64_t i) { *reinterpret_cast<float4*>(g + i) = z; });
      zero_edges(g, r);
    }
  }
}

}  // namespace

cudaError_t launch_fused_sync_sgd_tma(const SyncParams& p, int grid, cudaStream_t stream) {
  if (!check_world(p, 1) || p.mode == kModeAllGather) return cudaErrorInvalidValue;
  if (p.solver != kSolverSGD) return cudaErrorInvalidValue;  // SGD only: the routing never sends another solver here
  if (grid <= 0) grid = sm_count(-1);  // persistent: one CTA per SM
  if (grid > kMaxCtas) grid = kMaxCtas;
  const int nsrc = p.mode == kModeLocal ? 1 : p.world;
  const uint32_t gsz = (p.grad_bf16 && p.mode != kModeLocal) ? 2 : 4;
  // tile size: ~48 KB per stage, a multiple of 1024 elements, at least 1024
  const size_t per_elem = static_cast<size_t>(nsrc) * gsz + 8;
  int tile = static_cast<int>((48u << 10) / per_elem) / 1024 * 1024;
  if (tile < 1024) tile = 1024;
  if (tile > 8192) tile = 8192;
  while (static_cast<size_t>(kStages) * per_elem * tile > (200u << 10) && tile > 256) tile /= 2;
  // tiny nets: do not launch more CTAs than tiles
  const uint64_t work = (p.mode == kModeTwoShot) ? p.count / p.world : p.count;
  uint64_t tiles = (work + tile - 1) / tile;
  if (p.zero_diff || p.grad_bf16) tiles = (p.count / (p.mode == kModeLocal ? 1 : p.world) + tile - 1) / tile;
  if (tiles < 1) tiles = 1;
  if (static_cast<uint64_t>(grid) > tiles) grid = static_cast<int>(tiles);
  size_t smem = 128 + seg_smem_bytes(p, kMaxSegSmemTma);
  smem = (smem + 127) & ~static_cast<size_t>(127);
  smem += static_cast<size_t>(kStages) * (per_elem * tile);
  smem += 128;
  cudaError_t e;
  if (p.grad_bf16) {
    e = cudaFuncSetAttribute(fused_sync_sgd_tma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    fused_sync_sgd_tma_kernel<true><<<grid, kTmaThreads, smem, stream>>>(p, tile);
  } else {
    e = cudaFuncSetAttribute(fused_sync_sgd_tma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    fused_sync_sgd_tma_kernel<false><<<grid, kTmaThreads, smem, stream>>>(p, tile);
  }
  return cudaGetLastError();
}

}  // namespace cosb
