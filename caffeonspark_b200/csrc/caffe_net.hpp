// caffe_net.hpp -- object model behind the C ABI.
//
// Mirrors caffe-distri/include/CaffeNet.hpp:18-350 for the sync path:
//   CaffeNet        (base: solver spec, flat Params buffers, iteration state)
//   LocalCaffeNet   (cluster_size == 1: fused SGD only)            CaffeNet.hpp:163-203
//   NvlinkCaffeNet  (cluster_size  > 1: stands in for BOTH SocketCaffeNet
//                    CaffeNet.hpp:263-313 and RDMACaffeNet :206-260 -- the
//                    transport is NVLink peer memory instead of TCP / verbs)
// Method names follow the reference (localAddresses, connect, sync, deviceID,
// init, train, snapshot, getInitIter, getMaxIter, getTestIter,
// getTestInterval).
#ifndef COS_CAFFE_NET_HPP_
#define COS_CAFFE_NET_HPP_

#include <cuda_runtime_api.h>

#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/caffedistri_b200.h"
#include "caffe_proto_io.hpp"
#include "fused_sync_sgd.hpp"
#include "peer_adapter.hpp"
#include "peer_memory.hpp"
#include "solver_spec.hpp"

namespace cosb {

// AUTO uses the NVLS kernel from this world size on.  NVLink bytes per direction: NVLS 4P(1+1/N), P2P 8P(N-1)/N, but
// multimem traffic carries ~30 % protocol overhead vs ~13 % for plain stores (NVML raw vs payload counters): measured
// at CaffeNet size NVLS wins by 15-20 % at N = 8 and loses at N = 2; the N = 4 point of round 1 was a tie / small loss.
constexpr int kNvlsAutoMinWorld = 6;

class CaffeNet {
 public:
  // JniCaffeNet.cpp:41-64 dispatch.  Returns nullptr and sets *err on failure.
  static CaffeNet* create(const SolverSpec& spec, int num_local_devices, int cluster_size, int node_rank,
                          bool is_training, int connection_type, int start_device_id, std::string* err);
  virtual ~CaffeNet();

  virtual void localAddresses(std::vector<std::string>* vec) = 0;
  virtual bool connect(const std::vector<std::string>& addresses, std::string* err) = 0;
  virtual bool sync(std::string* err) { (void)err; return true; }  // CaffeNet.hpp:91

  // The object that serves local solver `solver_index` (one per local device, CaffeNet.hpp syncs_[i]);
  // a single-device net serves index 0 itself.
  virtual CaffeNet* rank_net(int solver_index) { return solver_index == 0 ? this : nullptr; }
  virtual int num_local_devices() const { return 1; }

  int deviceID(int solver_index) const;
  bool init(int solver_index, bool enable_nn, std::string* err);
  bool train(int solver_index, const cos_blob* data, int ndata, std::string* err);
  virtual int snapshot(std::string* err);
  std::string snapshot_filename(int iter, bool is_state) const;  // Solver::SnapshotFilename
  std::vector<BlobView> blob_views(const float* flat) const;
  // resume from snapshot files, ours or stock Caffe's (CaffeNet.cpp:198-205 restore path)
  virtual bool restore(const std::string& model_file, const std::string& state_file, std::string* err);
  int getInitIter(int solver_index) const { return solver_index == 0 ? spec_.init_iter : -1; }
  int getMaxIter(int solver_index) const { return solver_index == 0 ? spec_.max_iter : -1; }
  int getTestIter(int solver_index) const { return solver_index == 0 ? spec_.test_iter : -1; }
  int getTestInterval() const { return spec_.test_interval; }

  // hot path
  bool sync_step(int solver_index, cudaStream_t stream, bool use_own_stream, std::string* err);
  bool all_gather_weights(cudaStream_t stream, bool use_own_stream, std::string* err);
  virtual bool synchronize(std::string* err);
  // seeded device-side fill of data_ (0) / diff_ (1) / history (2), see cos_net_fill
  bool fill(int which, uint64_t seed, uint64_t stream_id, float amp, std::string* err);

  virtual void set_forward_backward(cos_forward_backward_fn fn, void* user) { fb_fn_ = fn; fb_user_ = user; }
  void set_solver_index(int i) { solver_index_ = i; }
  float* data() const { return data_; }
  float* diff() const { return diff_; }
  float* history() const { return hist_; }
  float* update_history() const { return hist2_; }  // AdaDelta's h2, nullptr for the other solvers
  uint64_t param_count() const { return count_; }
  int cluster_size() const { return world_; }
  int rank() const { return rank_; }
  int iter() const { return iter_; }
  float current_rate();
  float last_loss() const { return last_loss_; }
  float last_kernel_ms();
  virtual int64_t launch_count() const { return launches_; }
  virtual bool set_option(const std::string& name, int64_t v, std::string* err);
  virtual int64_t get_option(const std::string& name) const;
  int device() const { return device_; }
  const SolverSpec& spec() const { return spec_; }
  const std::vector<const char*>& address_cstrs() { return addr_cstrs_; }
  std::vector<std::string>& address_store() { return addr_store_; }

 protected:
  CaffeNet(const SolverSpec& spec, int cluster_size, int node_rank, bool is_training);
  bool allocate_device(int start_device_id, bool peer_mappable, std::string* err);
  bool launch(int mode, cudaStream_t stream, std::string* err);
  bool check_status(std::string* err);
  int resolved_algo() const;
  int resolved_kernel() const;

  SolverSpec spec_;
  const int world_;
  const int rank_;
  const bool is_training_;
  int device_ = -1;
  uint64_t count_ = 0;

  // Params<Dtype> (parallel.hpp:22-45): flat buffers, inside the peer-mappable arena
  DeviceArena arena_;
  size_t off_data_ = 0, off_diff_ = 0, off_hist_ = 0, off_wire_ = 0, off_recv_ = 0;
  size_t off_hist2_ = 0;           // AdaDelta only: second history region right after history
  uint64_t recv_stride_ = 0;       // elements per receive slot of the push kernel (0: no receive region)
  void* recv_ = nullptr;           // [world][recv_stride_] fp32 or bf16: the reference's diff_recv_ scratch, on device
  size_t off_llg_ = 0, off_llw_ = 0;  // LL kernel slots (small nets only): [world][ll_*_stride_] 8-byte words
  uint64_t ll_grad_stride_ = 0, ll_weight_stride_ = 0;
  float* data_ = nullptr;
  float* diff_ = nullptr;
  uint16_t* wire_ = nullptr;
  float* hist_ = nullptr;          // SGDSolver::history_ (sgd_solver.cpp:66-78); in the arena so that a
                                   // snapshot on rank 0 can read the owners' shards
  float* hist2_ = nullptr;         // AdaDelta's history of updates (history_[n + i]), nullptr for the other solvers
  int solver_ = kSolverSGD;        // SolverType of spec_.type
  uint64_t* seg_end_ = nullptr;    // device copies of the blob table
  float* seg_lr_ = nullptr;
  float* seg_dm_ = nullptr;
  int nseg_ = 0;
  int* status_ = nullptr;          // pinned + mapped: device-side error word
  float* loss_dev_ = nullptr;
  float* loss_host_ = nullptr;     // pinned

  // pointer tables for the kernel ([rank_] = local)
  float* peer_data_[kMaxRanks] = {};
  const float* peer_diff_[kMaxRanks] = {};
  uint16_t* peer_wire_[kMaxRanks] = {};
  const float* peer_hist_[kMaxRanks] = {};
  const float* peer_hist2_[kMaxRanks] = {};
  uint32_t* peer_flags_[kMaxRanks] = {};
  void* peer_recv_[kMaxRanks] = {};
  uint64_t* peer_llg_[kMaxRanks] = {};
  uint64_t* peer_llw_[kMaxRanks] = {};
  bool connected_ = false;
  bool nvls_active_ = false;        // multicast object bound on every rank (NvlinkCaffeNet::setup_nvls)
  char* mc_base_ = nullptr;         // multicast VA of the arena

  cudaStream_t stream_ = nullptr;
  cudaEvent_t ev_start_ = nullptr, ev_stop_ = nullptr, ev_done_ = nullptr;
  bool ev_valid_ = false, done_valid_ = false;
  int iter_ = 0;
  int current_step_ = 0;  // SGDSolver::current_step_
  uint32_t epoch_ = 0;
  int64_t launches_ = 0;
  float last_loss_ = 0.f;

  // options
  int opt_algo_ = COS_ALGO_AUTO;
  int opt_zero_diff_ = 1;
  int opt_grid_ = 0, opt_block_ = 0;
  int opt_kernel_ = -1;  // -1 auto, 0 LDG/STG pull, 1 TMA bulk-copy pull, 2 push, 3 NVLS (multimem), 4 LL (fence-free)
  int opt_timing_ = 0;   // CUDA events around every launch (cos_net_last_kernel_ms); benchmarks turn it on
  int opt_nvls_ = -1;    // -1 auto (multicast team when world >= kNvlsAutoMinWorld and 4P >= nvls_min_bytes), 0 off, 1 on
  int opt_nvls_unroll_ = 1;     // switch loads in flight per thread (1 measured best at N = 2 and N = 8: more only
                                // unbalances the CTAs, profiles/r02_matrix_large_n8.json)
  int opt_nvls_p2p_ = 0;        // 1: one plain-P2P vector per nvls_unroll switch vectors (link + switch both busy)
  int opt_push_vecs_ = 2;       // push kernel: float4 vectors per thread of the owner phase (sizes the grid)
  int64_t opt_push_max_bytes_ = int64_t(1) << 40;  // AUTO: push kernel below this message size (4P bytes), fp32 wire
  int64_t opt_ll_max_bytes_ = 2 << 20;     // AUTO: LL kernel below this message size (and <= kLLRegionMaxBytes)
  int64_t opt_nvls_min_bytes_ = 32 << 20;  // AUTO: NVLS kernel at or above this message size when world >= 6 (N = 8:
                                           // equal to push at 4-16 MiB, 13-15 % faster from 64 MiB; below, P2P is
                                           // as fast AND bit-exact)
  int opt_trace_ = 0;           // record %globaltimer at the phase boundaries of CTA 0 (diagnostics)
  int opt_initial_gather_ = 1;  // connect() runs the first on_start() (all-gather of weight shards)
  int64_t opt_timeout_ms_ = 20000;
  // AUTO picks one-shot only below this size.  0: never -- on B200 two-shot was at least as fast at every
  // measured size and world (profiles/r01_sweep_n2.json, r01_sweep_n8.json); one-shot stays selectable.
  int64_t opt_one_shot_max_bytes_ = 0;

  cos_forward_backward_fn fb_fn_ = nullptr;
  void* fb_user_ = nullptr;
  int solver_index_ = 0;  // index the gradient producer sees (local device number inside the executor)
  // Input path (row f3): the reference keeps a 2-deep Free/Full queue of host blobs between the transformer
  // threads and the solver thread (CaffeProcessor.scala:32-35,442-452) and MemoryInputAdapter::feed points the
  // data layer at the host blob (MemoryInputAdapter.cpp:24-32).  Here: two device-side staging sets; the H2D
  // copy of batch t runs on its own copy stream while the compute stream still works on batch t-1; train()
  // returns as soon as ITS batch has left host memory (the caller recycles the blobs after train() returns).
  struct InputStage {
    std::vector<void*> dev;
    std::vector<size_t> bytes;
    cudaEvent_t copied = nullptr;    // H2D of this stage finished
    cudaEvent_t consumed = nullptr;  // the step that read this stage finished
    bool consumed_valid = false;
  };
  InputStage stage_[2];
  int stage_idx_ = 0;
  cudaStream_t copy_stream_ = nullptr;
  cudaEvent_t loss_ev_[2] = {nullptr, nullptr};
  bool loss_pending_[2] = {false, false};
  int loss_idx_ = 0;
  int opt_train_pipeline_ = 1;      // 0: train() returns only after the whole Step finished (reference behaviour)
  void harvest_losses(bool wait);
  std::vector<std::string> addr_store_;
  std::vector<const char*> addr_cstrs_;
  std::mutex mu_;
};

class LocalCaffeNet : public CaffeNet {
 public:
  LocalCaffeNet(const SolverSpec& spec, bool is_training) : CaffeNet(spec, 1, 0, is_training) {}
  bool setup(int start_device_id, std::string* err) { return allocate_device(start_device_id, false, err); }
  void localAddresses(std::vector<std::string>* vec) override { vec->clear(); }  // CaffeNet.cpp:376-378
  bool connect(const std::vector<std::string>&, std::string*) override { connected_ = true; return true; }
};

class NvlinkCaffeNet : public CaffeNet {
 public:
  NvlinkCaffeNet(const SolverSpec& spec, int cluster_size, int node_rank, bool is_training);
  ~NvlinkCaffeNet() override;
  bool setup(int start_device_id, std::string* err);
  void localAddresses(std::vector<std::string>* vec) override;  // CaffeNet.cpp:394-404
  bool connect(const std::vector<std::string>& addresses, std::string* err) override;  // :456-480
  bool sync(std::string* err) override;  // :497-504

 private:
  // NVLS: cuMulticastCreate on rank 0, fd through the adapter, every rank adds its device, binds its
  // arena and maps the multicast VA.  Non-fatal: stays off unless EVERY rank succeeded.
  void setup_nvls(int timeout_ms);

  std::unique_ptr<PeerAdapter> adapter_;
  std::vector<std::unique_ptr<PeerMapping>> mappings_;
  MulticastMapping mcast_;
  std::string nvls_note_;
};

// `-devices k` inside one executor (SURVEY section 8 row f2).  The reference reduces the k local GPUs with a
// P2PSync tree and lets only the root GPU talk to other executors (parallel.cpp:202-418, CaffeNet.cpp:456-480);
// here every local GPU is a first-class rank of ONE collective of cluster_size*k ranks (rank = node_rank*k + i),
// so the tree, its extra D2D copies and the root bottleneck disappear.  Executor-level address strings carry
// the k per-device endpoints joined with ';'.
class MultiDeviceCaffeNet : public CaffeNet {
 public:
  MultiDeviceCaffeNet(const SolverSpec& spec, int num_local_devices, int cluster_size, int node_rank,
                      bool is_training);
  ~MultiDeviceCaffeNet() override;
  bool setup(int start_device_id, std::string* err);
  void localAddresses(std::vector<std::string>* vec) override;
  bool connect(const std::vector<std::string>& addresses, std::string* err) override;
  bool sync(std::string* err) override;
  CaffeNet* rank_net(int solver_index) override {
    return (solver_index >= 0 && solver_index < static_cast<int>(ranks_.size())) ? ranks_[solver_index].get() : nullptr;
  }
  int num_local_devices() const override { return static_cast<int>(ranks_.size()); }
  int snapshot(std::string* err) override { return ranks_[0]->snapshot(err); }
  // every local solver restores the same files (CaffeNet.cpp:196-205 runs per solver): weights, history,
  // iter_ and current_step_ on each local rank
  bool restore(const std::string& model_file, const std::string& state_file, std::string* err) override {
    for (auto& r : ranks_)
      if (!r->restore(model_file, state_file, err)) return false;
    return true;
  }
  bool synchronize(std::string* err) override;
  void set_forward_backward(cos_forward_backward_fn fn, void* user) override;
  int64_t launch_count() const override;
  bool set_option(const std::string& name, int64_t v, std::string* err) override;
  int64_t get_option(const std::string& name) const override { return ranks_[0]->get_option(name); }

 private:
  const int executors_;
  const int node_rank_;
  std::vector<std::unique_ptr<NvlinkCaffeNet>> ranks_;
};

}  // namespace cosb
#endif
