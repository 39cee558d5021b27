// fused_sync_sgd.hpp -- launch interface of the hot-path kernels.
//
// One launch performs what the reference spreads over on_gradients_ready()
// (parallel_cpu.cpp:120-122 scale, socket_sync_cpu.cpp:108-133 reduce-scatter),
// SGDSolver::ApplyUpdate (sgd_solver.cpp:102-116) and the next Step's
// on_start() (socket_sync_cpu.cpp:102-105 all-gather), see fused_sync_sgd.cu.
#ifndef COS_FUSED_SYNC_SGD_HPP_
#define COS_FUSED_SYNC_SGD_HPP_

#include <cuda_runtime_api.h>
#include <stdint.h>

namespace cosb {

constexpr int kMaxRanks = 16;
constexpr int kMaxCtas = 2048;
// Flag region at the start of every rank's arena: three arrays [kMaxCtas][kMaxRanks]
// of 32-bit words: epochs A = "gradients ready" and B = "reads done + weights landed", and C = per-CTA
// progress of an owner's reduce phase (NVLS kernel: lets the peers zero diff_ behind the owner's reads).
constexpr size_t kFlagBytes = 3ull * kMaxCtas * kMaxRanks * sizeof(uint32_t);

enum SyncMode : int {
  kModeLocal = 0,      // world == 1: fused SGD only
  kModeTwoShot = 1,    // reduce-scatter -> SGD on owned shard -> weight push
  kModeOneShot = 2,    // every rank reduces and updates everything, no push
  kModeAllGather = 3,  // on_start() alone: push owned weight shard to peers
};

// Solver of the update half (SolverParameter.type).  The kernels are templates on it; TMA and NVLS run SGD only.
enum SolverType : int {
  kSolverSGD = 0,
  kSolverNesterov = 1,
  kSolverAdaGrad = 2,
  kSolverRMSProp = 3,
  kSolverAdaDelta = 4,
};

struct SyncParams {
  int world;
  int rank;
  int mode;
  int grad_bf16;   // reduce over the bf16 wire buffers (cast fused in phase 0)
  int zero_diff;   // fold the next Step's ClearParamDiffs into the kernel
  int l1;          // regularization_type: 0 = L2 (g += ld*w), 1 = L1 (g += ld*sign(w))
  int nseg;
  uint64_t count;  // P: fp32 elements in data_/diff_/history
  float* data[kMaxRanks];           // data_ of every rank ([rank] is local)
  const float* diff[kMaxRanks];     // diff_ of every rank (fp32)
  uint16_t* wire[kMaxRanks];        // bf16 gradient wire buffer of every rank
  uint32_t* flags[kMaxRanks];       // flag region of every rank
  void* recv[kMaxRanks];            // push kernel: receive slots of every rank ([src][recv_stride] fp32 or bf16)
  uint64_t recv_stride;             // elements per receive slot
  uint64_t* ll_grad[kMaxRanks];     // LL kernel: gradient slots of every rank ([src][ll_grad_stride] 8-byte words)
  uint64_t* ll_weight[kMaxRanks];   // LL kernel: weight slots of every rank ([src][ll_weight_stride] words)
  uint64_t ll_grad_stride;          // words per LL gradient slot (0: no LL region)
  uint64_t ll_weight_stride;        // words per LL weight slot
  float* mc_data;                   // NVLS: multicast address of data_ (a store lands on every rank)
  const float* mc_diff;             // NVLS: multicast address of diff_ (a load returns the in-switch sum)
  int nvls_unroll;                  // NVLS kernel: switch loads in flight per thread (1, 2, 4, 8)
  int nvls_p2p;                     // NVLS kernel: of every (nvls_unroll + nvls_p2p) vectors this many go over plain P2P
  float* hist;                      // local SGD history (momentum buffer)
  const uint64_t* seg_end;          // [nseg] cumulative blob ends (exclusive)
  const float* seg_lr_mult;         // [nseg]
  const float* seg_decay_mult;      // [nseg]
  float rate;                       // GetLearningRate() of this iteration
  float momentum;                   // the factor h is scaled by: momentum, or rms_decay for RMSProp
  float weight_decay;
  float inv_scale;                  // (float)(1.0 / solver_count)
  uint32_t epoch;                   // barrier epoch of this launch
  unsigned long long timeout_ns;    // barrier time-out
  int* status;                      // local device word: 0 ok, else error code
  unsigned long long* trace;        // optional: 13 x %globaltimer of CTA 0: [0..4] phase boundaries, [5..8] / [9..12]
                                    // inside barrier A / B (entered, release fence done, flag arrived, acquire done)
  // Solver fields, appended so that every field above keeps its offset in the kernel parameter block.  The host
  // derives the constants in float, as the reference's Dtype arithmetic does; the device never re-derives them.
  int solver;                       // SolverType
  float* hist2;                     // AdaDelta: local history of updates (history_[n + i]); null otherwise
  float delta;                      // SolverParameter.delta (AdaGrad, RMSProp, AdaDelta)
  float one_minus;                  // 1 - momentum (AdaDelta) or 1 - rms_decay (RMSProp)
  float one_plus_m;                 // 1 + momentum (Nesterov)
  float neg_m;                      // -momentum (Nesterov)
};

// The LDG, push and LL launchers run every SolverType; TMA and NVLS return cudaErrorInvalidValue for p.solver != SGD.
// Launches the vector (LDG/STG) kernel.  grid/block 0 = defaults.
cudaError_t launch_fused_sync_sgd(const SyncParams& p, int grid, int block, cudaStream_t stream);
// Launches the TMA (cp.async.bulk) pipelined variant of the same computation.
cudaError_t launch_fused_sync_sgd_tma(const SyncParams& p, int grid, cudaStream_t stream);
// Launches the push variant (two-shot only): gradient shards are STORED into the owners' receive slots
// (fp32 -> bf16 cast in registers), reduced from local memory, weights pushed back.  vecs_per_thread sizes
// the grid (0 = default).
cudaError_t launch_fused_sync_sgd_push(const SyncParams& p, int grid, int block, int vecs_per_thread,
                                       cudaStream_t stream);
// Launches the NVLS (multimem) variant with optional P2P share (fused_sync_sgd_nvls.cu).
cudaError_t launch_fused_sync_sgd_nvls(const SyncParams& p, int grid, cudaStream_t stream);
// Launches the low-latency (flag-in-data, fence-free) variant for small nets; world sizes 2..8.
cudaError_t launch_fused_sync_sgd_ll(const SyncParams& p, int grid, int block, int vecs_per_thread,
                                     cudaStream_t stream);
// 8-byte words per LL gradient / weight slot for (count, world, wire dtype).
void ll_slot_words(uint64_t count, int world, bool bf16, uint64_t* grad_words, uint64_t* weight_words);
// Largest message (4P bytes) an LL region is allocated for.
constexpr uint64_t kLLRegionMaxBytes = 8ull << 20;
// Elements per receive slot of the push kernel for (count, world).
uint64_t push_recv_stride(uint64_t count, int world);
// Occupancy-derived default grid (co-resident CTAs) for the vector kernel; device < 0: the current device.
int default_sync_grid(int device);
// Device-side synthetic fill, identical to cos_oracle_fill (tests/bench).
cudaError_t launch_fill(float* out, uint64_t n, uint64_t seed, uint64_t stream_id, float amp,
                        cudaStream_t stream);

}  // namespace cosb
#endif
