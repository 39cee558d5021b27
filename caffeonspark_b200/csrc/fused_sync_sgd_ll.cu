// fused_sync_sgd_ll.cu -- the LOW-LATENCY variant of the fused sync kernel for
// small nets (LeNet, CIFAR-10-quick): no barriers and no memory fences at all.
//
// Measured on B200 (profiles/r02_matrix_small_n2.json): in the barrier-based
// kernels one cross-GPU barrier costs 5-6 us, of which the two system-scope
// fences (release before the flag store, acquire after the poll) are ~2-3 us
// EACH and the flag flight ~1 us; a 64 KiB..2 MiB sync is two barriers plus a
// few microseconds of real work.  Here every 8-byte word that crosses NVLink
// carries its own flag (the launch epoch) next to 4 bytes of payload, written
// and read with single 64-bit accesses, which are single-copy atomic: a reader
// that sees the flag sees the payload, so no fence and no separate barrier is
// needed (the scheme NCCL calls "LL").  Twice the wire bytes -- irrelevant while
// the message is latency-bound; AUTO uses this kernel below ll_max_bytes only.
//
// Same arithmetic and the same results, bit for bit, as the other P2P kernels
// (reference mapping in fused_sync_sgd.cu / fused_sync_sgd_push.cu):
//   phase 1  store shard q of my gradient into rank q's LL gradient slot [me]
//            (bf16 wire: two bf16 per word, cast in registers), then zero what I
//            pushed (ClearParamDiffs; nobody else reads diff_);
//   phase 2  owner: poll the N-1 slots word by word, reduce with my own gradient
//            in the reference's order s, s+1, ... (mod N) with the 1/N scale before
//            the sum, apply decay + momentum + update, store w / h locally and w
//            into every peer's LL weight slot [me];
//   phase 3  poll the N-1 weight slots and copy the peers' shards into data_ (the
//            next on_start(), socket_sync_cpu.cpp:102-105).
// Slot reuse needs no barrier: a peer can only push step t+1 after it finished
// step t, which includes receiving MY step-t weights, which I send after my last
// read of the gradient slots; and it can only push step-t+1 weights after it has
// my step-t+1 gradient, which I send after my phase 3 of step t.  Epochs grow
// monotonically, so a stale word can never carry the current flag.
#include "fused_sync_sgd.hpp"
#include "sync_device.cuh"

namespace cosb {
namespace {

constexpr int kLLThreads = 512;
constexpr int kLLMaxSeg = 1024;
constexpr int kEdgeWords = 8;  // scalar head/tail elements of a shard travel in 8 extra words behind the body

__device__ __forceinline__ void st_ll2(uint64_t* p, uint64_t a, uint64_t b) {  // two atomic 8-byte words
  asm volatile("st.relaxed.sys.global.v2.u64 [%0], {%1,%2};" ::"l"(p), "l"(a), "l"(b) : "memory");
}
__device__ __forceinline__ void st_ll1(uint64_t* p, uint64_t a) {
  asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(a) : "memory");
}
__device__ __forceinline__ void ld_ll2(const uint64_t* p, uint64_t& a, uint64_t& b) {
  asm volatile("ld.relaxed.sys.global.v2.u64 {%0,%1}, [%2];" : "=l"(a), "=l"(b) : "l"(p) : "memory");
}
__device__ __forceinline__ uint64_t ld_ll1(const uint64_t* p) {
  uint64_t a;
  asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(a) : "l"(p) : "memory");
  return a;
}
__device__ __forceinline__ uint64_t ll_word(uint32_t payload, uint32_t flag) {
  return static_cast<uint64_t>(payload) | (static_cast<uint64_t>(flag) << 32);
}
__device__ __forceinline__ bool ll_ok(uint64_t w, uint32_t flag) { return static_cast<uint32_t>(w >> 32) == flag; }

struct Poll {  // bounded spinning shared by all polls of a thread
  const SyncParams& p;
  int* s_abort;
  unsigned spins = 0;
  unsigned long long t0 = 0;
  __device__ Poll(const SyncParams& pp, int* a) : p(pp), s_abort(a) {}
  __device__ __forceinline__ bool give_up(int src) {  // call once per failed try
    if ((++spins & 0x3ffu) != 0) return false;
    if (*reinterpret_cast<volatile int*>(s_abort)) return true;
    const unsigned long long now = globaltimer_ns();
    if (t0 == 0) t0 = now;
    if (now - t0 > p.timeout_ns) {
      atomicExch(p.status, 200 + src);
      *reinterpret_cast<volatile int*>(s_abort) = 1;
      return true;
    }
    return false;
  }
  __device__ __forceinline__ void progress() { t0 = 0; }
};

// K independent groups of W consecutive LL words (W = 4: one float4 of fp32 payload, W = 2: four bf16).  All
// loads of a round are issued before the first flag is looked at, so K x W/2 16-byte loads are in flight per
// thread; groups whose flags are not all current are re-read.  `live` masks the groups that exist.  Returns false
// on abort (peer never arrived).
template <int K, int W>
__device__ __forceinline__ bool poll_groups(const uint64_t* const (&ptr)[K], uint32_t live, uint32_t flag, Poll& poll,
                                            int src_for_status, uint64_t (&out)[K][W]) {
  uint32_t pending = live;
  while (pending) {
#pragma unroll
    for (int k = 0; k < K; ++k) {
      if (pending & (1u << k)) {
#pragma unroll
        for (int w = 0; w < W; w += 2) ld_ll2(ptr[k] + w, out[k][w], out[k][w + 1]);
      }
    }
#pragma unroll
    for (int k = 0; k < K; ++k) {
      if (pending & (1u << k)) {
        bool ok = true;
#pragma unroll
        for (int w = 0; w < W; ++w) ok = ok && ll_ok(out[k][w], flag);
        if (ok) pending &= ~(1u << k);
      }
    }
    if (pending && poll.give_up(src_for_status)) return false;
  }
  poll.progress();
  return true;
}
__device__ __forceinline__ bool poll1(const uint64_t* w, uint32_t flag, Poll& poll, int src, uint32_t& out) {
  uint64_t a;
  for (;;) {
    a = ld_ll1(w);
    if (ll_ok(a, flag)) break;
    if (poll.give_up(src)) return false;
  }
  poll.progress();
  out = static_cast<uint32_t>(a);
  return true;
}

// edge (scalar head / tail) element e of shard range r -> index into the kEdgeWords edge words of a slot
__device__ __forceinline__ uint64_t edge_index(const ShardRange& r, uint64_t e) {
  return e < r.head_end ? e - r.lo : 4 + (e - r.tail_begin);
}

// N = compile-time world size, 2..8 (the N-1 polled slots live in registers); S = SolverType
template <int N, bool BF16, int S = kSolverSGD>
__global__ void __launch_bounds__(kLLThreads, 1) fused_sync_sgd_ll_kernel(const SyncParams p) {
  extern __shared__ unsigned char smem_raw[];
  __shared__ int s_abort;
  copy_seg_table(p, smem_raw, kLLMaxSeg);
  if (threadIdx.x == 0) s_abort = 0;
  __syncthreads();
  const bool tracer = p.trace != nullptr && blockIdx.x == 0 && threadIdx.x == 0;
  if (tracer) p.trace[0] = globaltimer_ns();

  const int world = N;
  const int rank = p.rank;
  const uint32_t flag = p.epoch;
  const uint64_t tid = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  const uint64_t gslot = p.ll_grad_stride;   // 8-byte words per gradient slot (body + edge words)
  const uint64_t wslot = p.ll_weight_stride; // 8-byte words per weight slot
  float* g = const_cast<float*>(p.diff[rank]);
  const bool zero = p.zero_diff != 0;
  // body word index of element i in a slot of shard range r: fp32 wire / weights 1 element per word,
  // bf16 wire 2 elements per word; base = r.lo rounded down to a multiple of 4
  const uint64_t gedge = gslot - kEdgeWords, wedge = wslot - kEdgeWords;

  // ---- phase 1: my gradient -> the owners' LL gradient slots [rank] ---------
  // The loads for all N-1 destinations are issued before the first store: one local-memory latency per
  // iteration instead of N-1.
  constexpr int D = N - 1;
  const uint64_t max_nvec = ((p.count + N - 1) / N + 3) >> 2;  // >= nvec of every shard
  for (uint64_t j = tid; j < max_nvec; j += stride) {
    float4 v[D];
#pragma unroll
    for (int d = 0; d < D; ++d) {
      const int q = peer(rank, 1 + d, N);
      const ShardRange r = shard_range(p.count, N, q);
      if (j < r.nvec) v[d] = ld_stream(g + ((r.vec_lo + j) << 2));
    }
#pragma unroll
    for (int d = 0; d < D; ++d) {
      const int q = peer(rank, 1 + d, N);
      const ShardRange r = shard_range(p.count, N, q);
      if (j < r.nvec) {
        const uint64_t i = (r.vec_lo + j) << 2, base = r.lo & ~3ull;
        uint64_t* dst = p.ll_grad[q] + static_cast<uint64_t>(rank) * gslot;
        if (BF16) {
          const uint2 o = pack_bf16x4(v[d]);
          st_ll2(dst + ((i - base) >> 1), ll_word(o.x, flag), ll_word(o.y, flag));
        } else {
          uint64_t* w = dst + (i - base);
          st_ll2(w, ll_word(__float_as_uint(v[d].x), flag), ll_word(__float_as_uint(v[d].y), flag));
          st_ll2(w + 2, ll_word(__float_as_uint(v[d].z), flag), ll_word(__float_as_uint(v[d].w), flag));
        }
      }
    }
  }
  if (blockIdx.x == 0) {
    for (int d = 1; d < world; ++d) {
      const int q = peer(rank, d, world);
      const ShardRange r = shard_range(p.count, world, q);
      const uint64_t e = edge_element(r, threadIdx.x);
      if (e != ~0ull) {
        const float x = BF16 ? round_bf16(g[e]) : g[e];
        st_ll1(p.ll_grad[q] + static_cast<uint64_t>(rank) * gslot + gedge + edge_index(r, e), ll_word(__float_as_uint(x), flag));
      }
    }
  }
  if (tracer) p.trace[1] = globaltimer_ns();
  if (zero) {  // ClearParamDiffs of what I pushed: plain streaming stores behind the pushes, hidden in the flight time
    for (int d = 1; d < world; ++d) zero_range<false>(g, shard_range(p.count, world, peer(rank, d, world)), tid, stride);
  }
  if (tracer) p.trace[2] = globaltimer_ns();

  // ---- phase 2: poll + reduce + update + push the new weights ----------------
  SegCursor cur = seg_cursor(p, smem_raw, kLLMaxSeg);
  Poll poll(p, &s_abort);
  bool alive = true;
  {
    const ShardRange r = shard_range(p.count, world, rank);
    const uint64_t base = r.lo & ~3ull;
    float* wl = p.data[rank];
    float* hl = p.hist;
    const float inv = p.inv_scale;
    const uint64_t* mine = p.ll_grad[rank];
    if (tid < r.nvec) cur.seek((r.vec_lo + tid) << 2);
    for (uint64_t j = tid; alive && j < r.nvec; j += stride) {
      const uint64_t i = (r.vec_lo + j) << 2;
      float4 x = ld_stream(g + i);
      float4 w = *reinterpret_cast<const float4*>(wl + i);
      float4 h = *reinterpret_cast<const float4*>(hl + i);
      if (BF16) x = round_bf16x4(x);
      float4 acc = scaled(inv, x);
      constexpr int K = N - 1;  // the N-1 slots, polled together
      constexpr int W = BF16 ? 2 : 4;
      const uint64_t* ptr[K];
      uint64_t words[K][W];
#pragma unroll
      for (int k = 0; k < K; ++k) {
        const int src = peer(rank, 1 + k, world);
        ptr[k] = mine + src * gslot + (BF16 ? ((i - base) >> 1) : (i - base));
      }
      alive = poll_groups<K, W>(ptr, (1u << K) - 1u, flag, poll, rank, words);
      if (!alive) break;
#pragma unroll
      for (int k = 0; k < K; ++k) {  // reference order: rank+1, rank+2, ... (mod N)
        float4 y;
        if (BF16) {
          y = unpack_bf16x4(make_uint2(static_cast<uint32_t>(words[k][0]), static_cast<uint32_t>(words[k][1])));
        } else {
          y = make_float4(__uint_as_float(static_cast<uint32_t>(words[k][0])),
                          __uint_as_float(static_cast<uint32_t>(words[k][1])),
                          __uint_as_float(static_cast<uint32_t>(words[k][W - 2])),
                          __uint_as_float(static_cast<uint32_t>(words[k][W - 1])));
        }
        add_scaled(acc, inv, y);
      }
      if (!alive) break;
      update_vec<S>(p, cur, i, acc, w, h);
      *reinterpret_cast<float4*>(hl + i) = h;
      *reinterpret_cast<float4*>(wl + i) = w;
      const uint64_t wa = ll_word(__float_as_uint(w.x), flag), wb = ll_word(__float_as_uint(w.y), flag);
      const uint64_t wc = ll_word(__float_as_uint(w.z), flag), wd = ll_word(__float_as_uint(w.w), flag);
      for (int k = 1; k < world; ++k) {
        const int dst = peer(rank, k, world);
        uint64_t* o = p.ll_weight[dst] + static_cast<uint64_t>(rank) * wslot + (i - base);
        st_ll2(o, wa, wb);
        st_ll2(o + 2, wc, wd);
      }
    }
    if (alive && blockIdx.x == 0) {  // scalar head / tail of my shard
      const uint64_t e = edge_element(r, threadIdx.x);
      if (e != ~0ull) {
        float acc = scaled(inv, BF16 ? round_bf16(g[e]) : g[e]);
        for (int k = 1; alive && k < world; ++k) {
          const int src = peer(rank, k, world);
          uint32_t u;
          alive = poll1(mine + src * gslot + gedge + edge_index(r, e), flag, poll, src, u);
          if (alive) add_scaled(acc, inv, __uint_as_float(u));
        }
        if (alive) {
          const float w = update_scalar<S>(p, cur, e, acc, wl, hl);
          for (int k = 1; k < world; ++k) {
            const int dst = peer(rank, k, world);
            st_ll1(p.ll_weight[dst] + static_cast<uint64_t>(rank) * wslot + wedge + edge_index(r, e),
                   ll_word(__float_as_uint(w), flag));
          }
        }
      }
    }
    if (zero) {  // my own shard of diff_ (read above by exactly these threads)
      zero_range<false>(g, r, tid, stride);
    }
  }
  if (tracer) p.trace[3] = globaltimer_ns();

  // ---- phase 3: the peers' updated shards -> my data_ ------------------------
  // One vector of EVERY peer's shard per round: the 2(N-1) polling loads are in flight together.
  if (alive) {
    float* wl = p.data[rank];
    for (uint64_t j = tid; alive && j < max_nvec; j += stride) {
      const uint64_t* ptr[D];
      uint64_t words[D][4];
      uint64_t idx[D];
      uint32_t live = 0;
#pragma unroll
      for (int d = 0; d < D; ++d) {
        const int q = peer(rank, 1 + d, N);
        const ShardRange r = shard_range(p.count, N, q);
        const bool in = j < r.nvec;
        idx[d] = (r.vec_lo + j) << 2;
        ptr[d] = p.ll_weight[rank] + static_cast<uint64_t>(q) * wslot + (in ? idx[d] - (r.lo & ~3ull) : 0);
        if (in) live |= 1u << d;
      }
      alive = poll_groups<D, 4>(ptr, live, flag, poll, rank, words);
      if (!alive) break;
#pragma unroll
      for (int d = 0; d < D; ++d) {
        if (live & (1u << d))
          st_vec(wl + idx[d], make_float4(__uint_as_float(static_cast<uint32_t>(words[d][0])),
                                          __uint_as_float(static_cast<uint32_t>(words[d][1])),
                                          __uint_as_float(static_cast<uint32_t>(words[d][2])),
                                          __uint_as_float(static_cast<uint32_t>(words[d][3]))));
      }
    }
    if (alive && blockIdx.x == 0) {
      for (int d = 1; alive && d < world; ++d) {
        const int q = peer(rank, d, world);
        const ShardRange r = shard_range(p.count, world, q);
        const uint64_t e = edge_element(r, threadIdx.x);
        if (e != ~0ull) {
          uint32_t u;
          alive = poll1(p.ll_weight[rank] + static_cast<uint64_t>(q) * wslot + wedge + edge_index(r, e), flag, poll, q, u);
          if (alive) wl[e] = __uint_as_float(u);
        }
      }
    }
  }
  if (tracer) p.trace[4] = globaltimer_ns();
}

}  // namespace

// 8-byte words per LL slot (body + kEdgeWords): gradient slots hold one (fp32) or two (bf16) elements per word,
// weight slots one.
void ll_slot_words(uint64_t count, int world, bool bf16, uint64_t* grad_words, uint64_t* weight_words) {
  const uint64_t max_shard = (count + world - 1) / world;
  const uint64_t body = (max_shard + 4 + 3) / 4 * 4;  // + up to 3 elements of alignment slack in front
  *weight_words = body + kEdgeWords;
  *grad_words = (bf16 ? body / 2 : body) + kEdgeWords;
}

cudaError_t launch_fused_sync_sgd_ll(const SyncParams& p, int grid, int block, int vecs_per_thread,
                                     cudaStream_t stream) {
  if (!check_world(p, 2)) return cudaErrorInvalidValue;
  if (p.mode != kModeTwoShot || p.ll_grad_stride == 0 || p.ll_weight_stride == 0) return cudaErrorInvalidValue;
  if (block <= 0) block = kLLThreads;
  if (block > kLLThreads || block < kMaxRanks || (block & 31)) return cudaErrorInvalidValue;
  if (vecs_per_thread <= 0) vecs_per_thread = 2;
  // Every CTA spins on peer data in phases 2 and 3 after feeding the peers in phase 1: the whole grid must be
  // co-resident (__launch_bounds__(512, 1): one CTA per SM).
  const int sms = sm_count(-1);
  const int cap = sms < kMaxCtas ? sms : kMaxCtas;
  if (grid <= 0) {  // sized by the larger phases (1 and 3 move (N-1)/N of the buffer)
    const uint64_t vecs = (p.count - p.count / p.world) >> 2;
    const uint64_t per_cta = static_cast<uint64_t>(block) * vecs_per_thread;
    uint64_t need = (vecs + per_cta - 1) / per_cta;
    if (need < 1) need = 1;
    grid = static_cast<int>(need > static_cast<uint64_t>(cap) ? cap : need);
  }
  if (grid > cap) grid = cap;
  const size_t smem = seg_smem_bytes(p, kLLMaxSeg);
  return dispatch_solver(p.solver, [&](auto S) {
    return dispatch_world(p.world, [&](auto N) {
      if constexpr (decltype(N)::value == 0) {
        return cudaErrorInvalidValue;  // world sizes 9..16 use the barrier-based kernels
      } else {
        if (p.grad_bf16) fused_sync_sgd_ll_kernel<N, true, S><<<grid, block, smem, stream>>>(p);
        else fused_sync_sgd_ll_kernel<N, false, S><<<grid, block, smem, stream>>>(p);
        return cudaGetLastError();
      }
    });
  });
}

}  // namespace cosb
