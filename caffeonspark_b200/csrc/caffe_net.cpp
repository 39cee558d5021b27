// caffe_net.cpp -- see caffe_net.hpp.
#include "caffe_net.hpp"

#include "caffe_proto_io.hpp"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

#include <sstream>

namespace cosb {
namespace {

std::string rt_err(const char* what, cudaError_t e) {
  std::ostringstream os;
  os << what << " failed: " << cudaGetErrorString(e);
  cudaGetLastError();
  return os.str();
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

#define COS_RT(call)                      \
  do {                                    \
    cudaError_t e__ = (call);             \
    if (e__ != cudaSuccess) {             \
      *err = rt_err(#call, e__);          \
      return false;                       \
    }                                     \
  } while (0)

}  // namespace

// ------------------------------------------------------------------ create

CaffeNet* CaffeNet::create(const SolverSpec& spec, int num_local_devices, int cluster_size, int node_rank,
                           bool is_training, int connection_type, int start_device_id, std::string* err) {
  // CaffeNet.cpp:123-124 CHECK_GE(num_local_devices_, 1), CHECK_GE(cluster_size_, 0)
  if (num_local_devices < 1) {
    *err = "number of local Devices must be greater than or equal to 1";
    return nullptr;
  }
  if (cluster_size < 1 || num_local_devices > kMaxRanks || cluster_size * num_local_devices > kMaxRanks) {
    *err = "cluster_size x num_local_devices must be in [1, " + std::to_string(kMaxRanks) + "]";
    return nullptr;
  }
  if (num_local_devices > 1) {  // -devices k: every local GPU is a rank of one collective (row f2)
    if (node_rank < 0 || node_rank >= cluster_size) {
      *err = "node_rank out of range";
      return nullptr;
    }
    if (cluster_size > 1 && connection_type != COS_CONNECTION_RDMA && connection_type != COS_CONNECTION_SOCKET) {
      *err = "unable to create CaffeNet object";
      return nullptr;
    }
    std::unique_ptr<MultiDeviceCaffeNet> n(
        new MultiDeviceCaffeNet(spec, num_local_devices, cluster_size, node_rank, is_training));
    if (!n->setup(start_device_id, err)) return nullptr;
    return n.release();
  }
  if (cluster_size == 1) {  // JniCaffeNet.cpp:42-46
    std::unique_ptr<LocalCaffeNet> n(new LocalCaffeNet(spec, is_training));
    if (!n->setup(start_device_id, err)) return nullptr;
    return n.release();
  }
  if (node_rank < 0 || node_rank >= cluster_size) {
    *err = "node_rank out of range";
    return nullptr;
  }
  if (connection_type != COS_CONNECTION_RDMA && connection_type != COS_CONNECTION_SOCKET) {
    *err = "unable to create CaffeNet object";  // JniCaffeNet.cpp:72-75 (no matching switch case)
    return nullptr;
  }
  std::unique_ptr<NvlinkCaffeNet> n(new NvlinkCaffeNet(spec, cluster_size, node_rank, is_training));
  if (!n->setup(start_device_id, err)) return nullptr;
  return n.release();
}

CaffeNet::CaffeNet(const SolverSpec& spec, int cluster_size, int node_rank, bool is_training)
    : spec_(spec), world_(cluster_size), rank_(node_rank), is_training_(is_training) {
  count_ = spec_.param_count();
  iter_ = spec_.init_iter;
  if (const char* t = getenv("COS_BARRIER_TIMEOUT_MS")) opt_timeout_ms_ = atoll(t);
}

CaffeNet::~CaffeNet() {
  if (device_ >= 0) {
    cudaSetDevice(device_);
    if (stream_) cudaStreamSynchronize(stream_);
    cudaDeviceSynchronize();
    for (InputStage& st : stage_) {
      for (void* p : st.dev)
        if (p) cudaFree(p);
      if (st.copied) cudaEventDestroy(st.copied);
      if (st.consumed) cudaEventDestroy(st.consumed);
    }
    for (cudaEvent_t e : loss_ev_)
      if (e) cudaEventDestroy(e);
    if (copy_stream_) cudaStreamDestroy(copy_stream_);
    if (seg_end_) cudaFree(seg_end_);
    if (seg_lr_) cudaFree(seg_lr_);
    if (seg_dm_) cudaFree(seg_dm_);
    if (loss_dev_) cudaFree(loss_dev_);
    if (loss_host_) cudaFreeHost(loss_host_);
    if (status_) cudaFreeHost(status_);
    if (ev_start_) cudaEventDestroy(ev_start_);
    if (ev_stop_) cudaEventDestroy(ev_stop_);
    if (ev_done_) cudaEventDestroy(ev_done_);
    if (stream_) cudaStreamDestroy(stream_);
    arena_.destroy();
    cudaGetLastError();
  }
}

// CaffeNet.cpp:130-142: devices are grabbed starting after start_device_id
// (Caffe::FindDevice picks the first usable one).
bool CaffeNet::allocate_device(int start_device_id, bool peer_mappable, std::string* err) {
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev <= 0) {
    *err = "cannot grab GPU device: " + std::string(e != cudaSuccess ? cudaGetErrorString(e) : "no CUDA device") +
           " (this library has no CPU path)";
    cudaGetLastError();
    return false;
  }
  int dev = -1;
  for (int d = start_device_id + 1; d < ndev; ++d) {
    if (d < 0) continue;
    if (cudaSetDevice(d) == cudaSuccess && cudaFree(0) == cudaSuccess) {
      dev = d;
      break;
    }
    cudaGetLastError();
  }
  if (dev < 0 && getenv("COS_ALLOW_SHARED_DEVICE") && start_device_id >= 0 && start_device_id < ndev &&
      cudaSetDevice(start_device_id) == cudaSuccess) {
    dev = start_device_id;  // tests on a single-GPU box: several local "devices" share the last GPU
  }
  if (dev < 0) {
    *err = "cannot grab GPU device after id " + std::to_string(start_device_id);
    return false;
  }
  device_ = dev;
  cudaDeviceProp prop;
  COS_RT(cudaGetDeviceProperties(&prop, dev));
  if (prop.major < 10) {
    *err = "device " + std::to_string(dev) + " is sm_" + std::to_string(prop.major * 10 + prop.minor) +
           "; this library is built for sm_100a (B200) only";
    return false;
  }

  // arena = [flags | data_ | diff_ | history | bf16 wire]
  const size_t fbytes = static_cast<size_t>(count_) * sizeof(float);
  size_t off = align_up(kFlagBytes, 4096);
  off_data_ = off;
  off = align_up(off + fbytes, 4096);
  off_diff_ = off;
  off = align_up(off + fbytes, 4096);
  off_hist_ = off;
  off = align_up(off + fbytes, 4096);
  off_wire_ = off;
  if (spec_.grad_dtype == COS_GRAD_BF16) off = align_up(off + static_cast<size_t>(count_) * 2, 4096);
  off_recv_ = off;
  if (world_ > 1) {  // receive slots of the push kernel: one per source rank, ~P/N elements each (<= 4P bytes in all)
    recv_stride_ = push_recv_stride(count_, world_);
    off = align_up(off + static_cast<size_t>(world_) * recv_stride_ * (spec_.grad_dtype == COS_GRAD_BF16 ? 2 : 4), 4096);
  }
  if (world_ >= 2 && world_ <= 8 && fbytes <= kLLRegionMaxBytes) {  // LL kernel slots (small nets)
    ll_slot_words(count_, world_, spec_.grad_dtype == COS_GRAD_BF16, &ll_grad_stride_, &ll_weight_stride_);
    off_llg_ = off;
    off = align_up(off + static_cast<size_t>(world_) * ll_grad_stride_ * 8, 4096);
    off_llw_ = off;
    off = align_up(off + static_cast<size_t>(world_) * ll_weight_stride_ * 8, 4096);
  }
  const char* tr = getenv("COS_PEER_TRANSPORT");
  const bool prefer_vmm = peer_mappable && !(tr && strcmp(tr, "ipc") == 0);
  if (!arena_.create(dev, off, prefer_vmm, err)) return false;
  char* base = static_cast<char*>(arena_.base());
  data_ = reinterpret_cast<float*>(base + off_data_);
  diff_ = reinterpret_cast<float*>(base + off_diff_);
  hist_ = reinterpret_cast<float*>(base + off_hist_);
  wire_ = spec_.grad_dtype == COS_GRAD_BF16 ? reinterpret_cast<uint16_t*>(base + off_wire_) : nullptr;
  peer_data_[rank_] = data_;
  peer_diff_[rank_] = diff_;
  peer_wire_[rank_] = wire_;
  peer_hist_[rank_] = hist_;
  peer_flags_[rank_] = reinterpret_cast<uint32_t*>(base);
  recv_ = recv_stride_ ? static_cast<void*>(base + off_recv_) : nullptr;
  peer_recv_[rank_] = recv_;
  peer_llg_[rank_] = ll_grad_stride_ ? reinterpret_cast<uint64_t*>(base + off_llg_) : nullptr;
  peer_llw_[rank_] = ll_grad_stride_ ? reinterpret_cast<uint64_t*>(base + off_llw_) : nullptr;

  // blob (segment) table: cumulative ends + multipliers
  std::vector<uint64_t> ends;
  std::vector<float> lr, dm;
  uint64_t acc = 0;
  for (size_t k = 0; k < spec_.counts.size(); ++k) {
    if (spec_.counts[k] < 0) {
      *err = "negative blob count";
      return false;
    }
    acc += static_cast<uint64_t>(spec_.counts[k]);
    ends.push_back(acc);
    lr.push_back(k < spec_.lr_mult.size() ? spec_.lr_mult[k] : 1.0f);
    dm.push_back(k < spec_.decay_mult.size() ? spec_.decay_mult[k] : 1.0f);
  }
  if (ends.empty() || acc == 0) {  // net without learnable parameters: size_ == 1
    ends.assign(1, 1);
    lr.assign(1, 1.0f);
    dm.assign(1, 1.0f);
  }
  nseg_ = static_cast<int>(ends.size());
  COS_RT(cudaMalloc(reinterpret_cast<void**>(&seg_end_), nseg_ * sizeof(uint64_t)));
  COS_RT(cudaMalloc(reinterpret_cast<void**>(&seg_lr_), nseg_ * sizeof(float)));
  COS_RT(cudaMalloc(reinterpret_cast<void**>(&seg_dm_), nseg_ * sizeof(float)));
  COS_RT(cudaMemcpy(seg_end_, ends.data(), nseg_ * sizeof(uint64_t), cudaMemcpyHostToDevice));
  COS_RT(cudaMemcpy(seg_lr_, lr.data(), nseg_ * sizeof(float), cudaMemcpyHostToDevice));
  COS_RT(cudaMemcpy(seg_dm_, dm.data(), nseg_ * sizeof(float), cudaMemcpyHostToDevice));

  // host-mapped: [0] device-side error word, [2..11] optional phase timestamps (option "trace")
  COS_RT(cudaHostAlloc(reinterpret_cast<void**>(&status_), 16 * sizeof(unsigned long long), cudaHostAllocMapped));
  memset(status_, 0, 16 * sizeof(unsigned long long));
  COS_RT(cudaMalloc(reinterpret_cast<void**>(&loss_dev_), sizeof(float)));
  COS_RT(cudaMemset(loss_dev_, 0, sizeof(float)));
  COS_RT(cudaHostAlloc(reinterpret_cast<void**>(&loss_host_), 2 * sizeof(float), cudaHostAllocDefault));
  loss_host_[0] = loss_host_[1] = 0.f;
  COS_RT(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
  COS_RT(cudaStreamCreateWithFlags(&copy_stream_, cudaStreamNonBlocking));
  for (InputStage& st : stage_) {
    COS_RT(cudaEventCreateWithFlags(&st.copied, cudaEventDisableTiming));
    COS_RT(cudaEventCreateWithFlags(&st.consumed, cudaEventDisableTiming));
  }
  for (cudaEvent_t& e : loss_ev_) COS_RT(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  COS_RT(cudaEventCreate(&ev_start_));
  COS_RT(cudaEventCreate(&ev_stop_));
  COS_RT(cudaEventCreateWithFlags(&ev_done_, cudaEventDisableTiming));
  return true;
}

int CaffeNet::deviceID(int solver_index) const { return solver_index == 0 ? device_ : -1; }

// CaffeNet.cpp:585-654: per-thread binding to the solver's device.
bool CaffeNet::init(int solver_index, bool enable_nn, std::string* err) {
  (void)enable_nn;
  if (solver_index != 0) {
    *err = "solver_index must be 0";
    return false;
  }
  COS_RT(cudaSetDevice(device_));
  return true;
}

int CaffeNet::resolved_algo() const {
  if (world_ == 1) return kModeLocal;
  if (opt_algo_ == COS_ALGO_TWO_SHOT) return kModeTwoShot;
  if (opt_algo_ == COS_ALGO_ONE_SHOT) return kModeOneShot;
  return static_cast<int64_t>(count_ * sizeof(float)) <= opt_one_shot_max_bytes_ ? kModeOneShot : kModeTwoShot;
}

// Kernel variant (0 LDG/STG pull, 1 TMA bulk-copy pull, 2 push, 3 NVLS).  Depends only on (world, P, wire
// dtype, options, NVLS team) -- all identical on every rank -- so every rank resolves the same variant, which
// the per-CTA barriers require.  AUTO, from the B200 measurements under profiles/:
//   * N >= 6, fp32 wire, multicast team up, 4P >= nvls_min_bytes: NVLS (4P(1+1/N) NVLink bytes per direction
//     instead of 8P(N-1)/N; measured 15-20 % faster than push at N = 8, estimated break-even at N ~ 5);
//   * 4P < ll_max_bytes (N <= 8): LL -- flag-in-data words, no barrier, no fence (latency-bound sizes);
//   * otherwise push (stores only; the bf16 cast costs no extra pass; measured >= the TMA pull pipeline at
//     every size on B200), the TMA pull pipeline above push_max_bytes.
// A forced variant that cannot run the current mode falls back to AUTO's choice.
int CaffeNet::resolved_kernel() const {
  const int algo = resolved_algo();
  const bool fp32 = spec_.grad_dtype == COS_GRAD_FP32;
  const int64_t bytes = static_cast<int64_t>(count_ * sizeof(float));
  const bool nvls_ok = nvls_active_ && fp32 && algo == kModeTwoShot;
  const bool push_ok = world_ > 1 && algo == kModeTwoShot && recv_stride_ > 0;
  const bool ll_ok = world_ > 1 && algo == kModeTwoShot && ll_grad_stride_ > 0;
  if (opt_kernel_ == 0 || opt_kernel_ == 1) return opt_kernel_;
  if (opt_kernel_ == 2 && push_ok) return 2;
  if (opt_kernel_ == 3 && nvls_ok) return 3;
  if (opt_kernel_ == 4 && ll_ok) return 4;
  if (world_ == 1) return 0;
  if (algo != kModeTwoShot) return bytes >= (2 << 20) ? 1 : 0;
  if (nvls_ok && (opt_nvls_ == 1 || (world_ >= kNvlsAutoMinWorld && bytes >= opt_nvls_min_bytes_))) return 3;
  if (ll_ok && bytes < opt_ll_max_bytes_) return 4;
  if (push_ok && (!fp32 || bytes < opt_push_max_bytes_)) return 2;
  return bytes >= (2 << 20) ? 1 : 0;
}

float CaffeNet::current_rate() {
  int step = current_step_;
  float r = 0.f;
  learning_rate(spec_.lr_policy, spec_.base_lr, spec_.gamma, spec_.power, spec_.stepsize,
                spec_.stepvalues.empty() ? nullptr : spec_.stepvalues.data(),
                static_cast<int>(spec_.stepvalues.size()), spec_.max_iter, iter_, &step, &r);
  return r;
}

bool CaffeNet::launch(int mode, cudaStream_t stream, std::string* err) {
  SyncParams p;
  memset(&p, 0, sizeof(p));
  p.world = world_;
  p.rank = rank_;
  p.mode = mode;
  p.grad_bf16 = spec_.grad_dtype == COS_GRAD_BF16;
  p.zero_diff = opt_zero_diff_;
  p.l1 = spec_.regularization_type == "L1" ? 1 : 0;
  p.nseg = nseg_;
  p.count = count_;
  for (int r = 0; r < world_; ++r) {
    p.data[r] = peer_data_[r];
    p.diff[r] = peer_diff_[r];
    p.wire[r] = peer_wire_[r];
    p.flags[r] = peer_flags_[r];
    p.recv[r] = peer_recv_[r];
    p.ll_grad[r] = peer_llg_[r];
    p.ll_weight[r] = peer_llw_[r];
  }
  p.recv_stride = recv_stride_;
  p.ll_grad_stride = ll_grad_stride_;
  p.ll_weight_stride = ll_weight_stride_;
  p.nvls_unroll = opt_nvls_unroll_;
  p.nvls_p2p = opt_nvls_p2p_;
  p.mc_data = nvls_active_ ? reinterpret_cast<float*>(mc_base_ + off_data_) : nullptr;
  p.mc_diff = nvls_active_ ? reinterpret_cast<const float*>(mc_base_ + off_diff_) : nullptr;
  p.hist = hist_;
  p.seg_end = seg_end_;
  p.seg_lr_mult = seg_lr_;
  p.seg_decay_mult = seg_dm_;
  p.momentum = spec_.momentum;
  p.weight_decay = spec_.weight_decay;
  p.inv_scale = static_cast<float>(1.0 / static_cast<double>(world_));  // Dtype(1.0 / solver_count)
  p.timeout_ns = static_cast<unsigned long long>(opt_timeout_ms_) * 1000000ull;
  p.status = status_;
  p.trace = opt_trace_ ? reinterpret_cast<unsigned long long*>(status_) + 2 : nullptr;
  if (mode != kModeAllGather) {
    if (!learning_rate(spec_.lr_policy, spec_.base_lr, spec_.gamma, spec_.power, spec_.stepsize,
                       spec_.stepvalues.empty() ? nullptr : spec_.stepvalues.data(),
                       static_cast<int>(spec_.stepvalues.size()), spec_.max_iter, iter_, &current_step_,
                       &p.rate)) {
      *err = "Unknown learning rate policy: " + spec_.lr_policy;
      return false;
    }
  }
  if (world_ > 1) p.epoch = ++epoch_;
  if (opt_timing_) COS_RT(cudaEventRecord(ev_start_, stream));
  const int grid = opt_grid_;
  const int kern = (mode == kModeAllGather) ? 0 : resolved_kernel();
  cudaError_t e;
  switch (kern) {
    case 1: e = launch_fused_sync_sgd_tma(p, grid, stream); break;
    case 2: e = launch_fused_sync_sgd_push(p, grid, opt_block_, opt_push_vecs_, stream); break;
    case 3: e = launch_fused_sync_sgd_nvls(p, grid, stream); break;
    case 4: e = launch_fused_sync_sgd_ll(p, grid, opt_block_, opt_push_vecs_, stream); break;
    default: e = launch_fused_sync_sgd(p, grid, opt_block_, stream); break;
  }
  if (e != cudaSuccess) {
    *err = rt_err("fused_sync_sgd launch", e);
    return false;
  }
  if (opt_timing_) {
    COS_RT(cudaEventRecord(ev_stop_, stream));
    ev_valid_ = true;
  }
  COS_RT(cudaEventRecord(ev_done_, stream));  // what synchronize() waits on (works for caller-owned streams)
  done_valid_ = true;
  ++launches_;
  return true;
}

bool CaffeNet::sync_step(int solver_index, cudaStream_t stream, bool use_own_stream, std::string* err) {
  if (solver_index != 0) {
    *err = "solver_index must be 0";
    return false;
  }
  if (world_ > 1 && !connected_) {
    *err = "solver was not initialized: connect() has not completed";  // CaffeNet.cpp:720
    return false;
  }
  std::lock_guard<std::mutex> g(mu_);
  COS_RT(cudaSetDevice(device_));
  if (!launch(resolved_algo(), use_own_stream ? stream_ : stream, err)) return false;
  ++iter_;  // solver.cpp:257
  return true;
}

bool CaffeNet::all_gather_weights(cudaStream_t stream, bool use_own_stream, std::string* err) {
  if (world_ == 1) return true;
  if (!connected_) {
    *err = "connect() has not completed";
    return false;
  }
  std::lock_guard<std::mutex> g(mu_);
  COS_RT(cudaSetDevice(device_));
  return launch(kModeAllGather, use_own_stream ? stream_ : stream, err);
}

bool CaffeNet::check_status(std::string* err) {
  int s = *reinterpret_cast<volatile int*>(status_);
  if (s == 0) return true;
  *reinterpret_cast<volatile int*>(status_) = 0;
  std::ostringstream os;
  if (s >= 200 && s < 200 + kMaxRanks) {  // fused_sync_sgd_ll.cu: a peer's flagged words never arrived
    os << "device-side LL exchange timed out after " << opt_timeout_ms_ << " ms waiting for data "
       << (s - 200 == rank_ ? "of a peer" : "of rank " + std::to_string(s - 200)) << " (status " << s << ")";
    *err = os.str();
    return false;
  }
  if (s == 400) {  // fused_sync_sgd_nvls.cu: the zeroing warp never saw an owner finish its reduce phase
    os << "device-side NVLS reduce phase of a peer did not finish within " << opt_timeout_ms_ << " ms (status 400)";
    *err = os.str();
    return false;
  }
  if (s == 300) {  // fused_sync_sgd_tma.cu: an mbarrier never completed (a bulk copy was lost or a peer died mid-tile)
    os << "device-side TMA pipeline timed out after " << opt_timeout_ms_
       << " ms waiting for a bulk copy to complete (status 300)";
    *err = os.str();
    return false;
  }
  int which = (s - 100) / 32, peer = (s - 100) % 32;
  os << "device-side barrier " << (which == 0 ? "A (gradients ready)" : "B (weights landed)") << " timed out after "
     << opt_timeout_ms_ << " ms waiting for rank " << peer << " (status " << s << ")";
  *err = os.str();
  return false;
}

// Waits for the last launch (on whatever stream it went to) and the net's own
// stream.  Deliberately NOT cudaDeviceSynchronize: with several executors in
// one process a device-wide wait from one thread can stall another thread's
// launch while the first one's kernel is spinning on it.
bool CaffeNet::synchronize(std::string* err) {
  COS_RT(cudaSetDevice(device_));
  if (done_valid_) COS_RT(cudaEventSynchronize(ev_done_));
  COS_RT(cudaStreamSynchronize(stream_));
  harvest_losses(true);
  return check_status(err);
}

bool CaffeNet::fill(int which, uint64_t seed, uint64_t stream_id, float amp, std::string* err) {
  float* dst = which == 0 ? data_ : which == 1 ? diff_ : which == 2 ? hist_ : nullptr;
  if (!dst) {
    *err = "fill: which must be 0 (data), 1 (diff) or 2 (history)";
    return false;
  }
  COS_RT(cudaSetDevice(device_));
  COS_RT(launch_fill(dst, count_, seed, stream_id, amp, stream_));
  COS_RT(cudaStreamSynchronize(stream_));
  return true;
}

float CaffeNet::last_kernel_ms() {
  if (!ev_valid_) return -1.f;
  cudaSetDevice(device_);
  if (cudaEventSynchronize(ev_stop_) != cudaSuccess) {
    cudaGetLastError();
    return -1.f;
  }
  float ms = -1.f;
  if (cudaEventElapsedTime(&ms, ev_start_, ev_stop_) != cudaSuccess) {
    cudaGetLastError();
    return -1.f;
  }
  return ms;
}

// CaffeNet.cpp:707-729 train(): feed the batch, Solver::Step(1).
bool CaffeNet::train(int solver_index, const cos_blob* data, int ndata, std::string* err) {
  if (solver_index != 0) {
    *err = "solver_index must be 0";
    return false;
  }
  if (!data) {
    *err = "data is NULL";  // JniCaffeNet.cpp:391-395
    return false;
  }
  if (!fb_fn_) {
    *err = "train: no gradient producer registered (cos_net_set_forward_backward); Net::ForwardBackward is "
           "outside this library";
    return false;
  }
  COS_RT(cudaSetDevice(device_));
  if (!check_status(err)) return false;  // a device-side error of an earlier (pipelined) step surfaces here
  // MemoryInputAdapter::feed (MemoryInputAdapter.cpp:24-32) equivalent: stage the host blobs on the device.
  // Stage k was last read by step t-2: its H2D may only start once that step is done (device-side wait).
  InputStage& st = stage_[stage_idx_];
  if (static_cast<int>(st.dev.size()) < ndata) {
    st.dev.resize(ndata, nullptr);
    st.bytes.resize(ndata, 0);
  }
  if (st.consumed_valid) COS_RT(cudaStreamWaitEvent(copy_stream_, st.consumed, 0));
  std::vector<cos_blob> dev_blobs(ndata);
  for (int i = 0; i < ndata; ++i) {
    if (!data[i].data) {
      *err = "data[" + std::to_string(i) + "] is NULL";
      return false;
    }
    size_t n = static_cast<size_t>(data[i].num) * data[i].channels * data[i].height * data[i].width * sizeof(float);
    if (n > st.bytes[i]) {
      if (st.dev[i]) {
        COS_RT(cudaStreamSynchronize(stream_));  // an earlier step may still read the old buffer
        cudaFree(st.dev[i]);
      }
      st.dev[i] = nullptr;
      COS_RT(cudaMalloc(&st.dev[i], n));
      st.bytes[i] = n;
    }
    COS_RT(cudaMemcpyAsync(st.dev[i], data[i].data, n, cudaMemcpyHostToDevice, copy_stream_));
    dev_blobs[i] = data[i];
    dev_blobs[i].data = static_cast<const float*>(st.dev[i]);
  }
  COS_RT(cudaEventRecord(st.copied, copy_stream_));
  COS_RT(cudaStreamWaitEvent(stream_, st.copied, 0));
  int rc = fb_fn_(fb_user_, solver_index_, dev_blobs.data(), ndata, loss_dev_, stream_);
  if (rc != 0) {
    *err = "gradient producer failed with code " + std::to_string(rc);
    return false;
  }
  if (!sync_step(solver_index, stream_, true, err)) return false;
  COS_RT(cudaEventRecord(st.consumed, stream_));
  st.consumed_valid = true;
  // the step's result (loss): device -> pinned host on the compute stream, harvested when it has arrived
  const int k = loss_idx_;
  if (loss_pending_[k]) COS_RT(cudaEventSynchronize(loss_ev_[k]));
  harvest_losses(false);
  COS_RT(cudaMemcpyAsync(loss_host_ + k, loss_dev_, sizeof(float), cudaMemcpyDeviceToHost, stream_));
  COS_RT(cudaEventRecord(loss_ev_[k], stream_));
  loss_pending_[k] = true;
  loss_idx_ ^= 1;
  stage_idx_ ^= 1;
  if (opt_train_pipeline_) {
    // the caller owns the host blobs again once train() returns: wait for THIS batch's H2D only
    COS_RT(cudaEventSynchronize(st.copied));
    harvest_losses(false);
    return true;
  }
  COS_RT(cudaStreamSynchronize(stream_));
  harvest_losses(true);
  return check_status(err);
}

// Collects the losses whose D2H has completed (oldest first, so last_loss_ ends at the newest one).
void CaffeNet::harvest_losses(bool wait) {
  for (int n = 0; n < 2; ++n) {
    const int k = (loss_idx_ + n) & 1;  // loss_idx_ is the OLDER slot
    if (!loss_pending_[k]) continue;
    cudaError_t e = wait ? cudaEventSynchronize(loss_ev_[k]) : cudaEventQuery(loss_ev_[k]);
    if (e == cudaSuccess) {
      last_loss_ = loss_host_[k];
      loss_pending_[k] = false;
    } else {
      cudaGetLastError();
      if (!wait) break;  // the newer one cannot be done either
    }
  }
}

bool CaffeNet::set_option(const std::string& name, int64_t v, std::string* err) {
  if (name == "algo") {
    if (v < 0 || v > 2) { *err = "algo must be 0..2"; return false; }
    opt_algo_ = static_cast<int>(v);
  } else if (name == "zero_diff") opt_zero_diff_ = v != 0;
  else if (name == "grid") opt_grid_ = static_cast<int>(v);
  else if (name == "block") opt_block_ = static_cast<int>(v);
  else if (name == "kernel") opt_kernel_ = static_cast<int>(v);
  else if (name == "timing") opt_timing_ = v != 0;
  else if (name == "nvls") opt_nvls_ = v < 0 ? -1 : (v != 0);
  else if (name == "nvls_unroll") opt_nvls_unroll_ = static_cast<int>(v);
  else if (name == "nvls_p2p") opt_nvls_p2p_ = static_cast<int>(v);
  else if (name == "push_vecs") opt_push_vecs_ = static_cast<int>(v);
  else if (name == "push_max_bytes") opt_push_max_bytes_ = v;
  else if (name == "ll_max_bytes") opt_ll_max_bytes_ = v;
  else if (name == "nvls_min_bytes") opt_nvls_min_bytes_ = v;
  else if (name == "barrier_timeout_ms") opt_timeout_ms_ = v;
  else if (name == "one_shot_max_bytes") opt_one_shot_max_bytes_ = v;
  else if (name == "iter") { iter_ = static_cast<int>(v); }
  else if (name == "initial_gather") opt_initial_gather_ = v != 0;
  else if (name == "trace") opt_trace_ = v != 0;
  else if (name == "train_pipeline") opt_train_pipeline_ = v != 0;
  else {
    *err = "unknown option '" + name + "'";
    return false;
  }
  return true;
}

int64_t CaffeNet::get_option(const std::string& name) const {
  if (name == "algo") return opt_algo_;
  if (name == "resolved_algo") return resolved_algo();
  if (name == "zero_diff") return opt_zero_diff_;
  if (name == "grid") return opt_grid_;
  if (name == "block") return opt_block_;
  if (name == "kernel") return opt_kernel_;
  if (name == "resolved_kernel") return resolved_kernel();
  if (name == "timing") return opt_timing_;
  if (name == "nvls") return opt_nvls_;
  if (name == "nvls_active") return nvls_active_ ? 1 : 0;
  if (name == "nvls_unroll") return opt_nvls_unroll_;
  if (name == "nvls_p2p") return opt_nvls_p2p_;
  if (name == "push_vecs") return opt_push_vecs_;
  if (name == "push_max_bytes") return opt_push_max_bytes_;
  if (name == "ll_max_bytes") return opt_ll_max_bytes_;
  if (name == "nvls_min_bytes") return opt_nvls_min_bytes_;
  if (name == "barrier_timeout_ms") return opt_timeout_ms_;
  if (name == "one_shot_max_bytes") return opt_one_shot_max_bytes_;
  if (name == "initial_gather") return opt_initial_gather_;
  if (name == "train_pipeline") return opt_train_pipeline_;
  if (name.compare(0, 6, "trace_") == 0 && name.size() >= 7 && name.size() <= 8) {  // trace_0 .. trace_12
    const int k = atoi(name.c_str() + 6);
    if (k >= 0 && k <= 12) return static_cast<int64_t>((reinterpret_cast<volatile unsigned long long*>(status_) + 2)[k]);
  }
  if (name == "transport") return arena_.transport();
  if (name == "default_grid") return default_sync_grid(device_);
  return -1;
}

// ---------------------------------------------------------------- snapshot
// Stock-Caffe binaryproto files (caffe_proto_io.cpp): <prefix>_iter_<n>.caffemodel = NetParameter with one
// LayerParameter per parameterised layer, <prefix>_iter_<n>.solverstate = SolverState {iter, learned_net,
// history[], current_step} -- the names Solver::SnapshotFilename (solver.cpp:446-449) and
// CaffeNet.java:192-207 produce, so FSUtils.GenModelOrState finds them.  Rank 0 is the only caller in the
// reference (CaffeProcessor.scala:454-465); its weights are globally consistent here (the kernel
// all-gathers every step), and the history of the other shards is read straight from the owners' arenas
// over NVLink, which removes the reference's stale-shard quirks (SURVEY App. E-1/E-2).
std::string CaffeNet::snapshot_filename(int iter, bool is_state) const {
  const std::string prefix = spec_.snapshot_prefix.empty() ? std::string("cos_b200") : spec_.snapshot_prefix;
  // CaffeNet.java:203-205 / Solver::SnapshotFilename append ".h5" for snapshot_format: HDF5; those files ARE HDF5
  // (snapshot() below).
  return prefix + "_iter_" + std::to_string(iter) + (is_state ? ".solverstate" : ".caffemodel") +
         (spec_.snapshot_hdf5 ? ".h5" : "");
}

std::vector<BlobView> CaffeNet::blob_views(const float* flat) const {
  std::vector<BlobView> v;
  uint64_t off = 0;
  for (size_t k = 0; k < spec_.counts.size(); ++k) {
    BlobView b;
    b.layer_name = k < spec_.layer_names.size() ? spec_.layer_names[k] : "blob" + std::to_string(k);
    b.layer_type = k < spec_.layer_types.size() ? spec_.layer_types[k] : "Blob";
    if (k < spec_.shapes.size()) b.shape = spec_.shapes[k];
    else b.shape.assign(1, spec_.counts[k]);
    b.count = static_cast<uint64_t>(spec_.counts[k]);
    b.data = flat + off;
    off += b.count;
    v.push_back(std::move(b));
  }
  return v;
}

int CaffeNet::snapshot(std::string* err) {
  std::lock_guard<std::mutex> g(mu_);
  if (cudaSetDevice(device_) != cudaSuccess || (done_valid_ && cudaEventSynchronize(ev_done_) != cudaSuccess) ||
      cudaStreamSynchronize(stream_) != cudaSuccess) {
    *err = rt_err("snapshot: device sync", cudaGetLastError());
    return -1;
  }
  if (!check_status(err)) return -1;
  std::vector<float> w(count_), h(count_);
  cudaError_t e = cudaMemcpy(w.data(), data_, count_ * sizeof(float), cudaMemcpyDeviceToHost);
  const bool sharded_hist = world_ > 1 && resolved_algo() == kModeTwoShot;
  for (int r = 0; r < world_ && e == cudaSuccess; ++r) {
    uint64_t offs = 0, size = count_;
    if (sharded_hist) chunk(count_, world_, r, &offs, &size);
    else if (r != rank_) continue;
    const float* src = (sharded_hist ? peer_hist_[r] : hist_);
    if (!src) {
      *err = "snapshot: history of rank " + std::to_string(r) + " is not mapped (connect() first)";
      return -1;
    }
    if (size) e = cudaMemcpy(h.data() + offs, src + offs, size * sizeof(float), cudaMemcpyDeviceToHost);
  }
  if (e != cudaSuccess) {
    *err = rt_err("snapshot: copy to host", e);
    return -1;
  }
  const std::string model = snapshot_filename(iter_, false), state = snapshot_filename(iter_, true);
  if (spec_.snapshot_hdf5) {  // solver.cpp:417-418 SnapshotToHDF5 + sgd_solver.cpp:251-252 (csrc/hdf5_io.cpp)
    if (!write_caffemodel_h5(model, blob_views(w.data()), err)) return -1;
    if (!write_solverstate_h5(state, iter_, current_step_, model, blob_views(h.data()), err)) return -1;
    return iter_;
  }
  if (!write_caffemodel(model, spec_.net_name, blob_views(w.data()), err)) return -1;
  if (!write_solverstate(state, iter_, current_step_, model, blob_views(h.data()), err)) return -1;
  return iter_;
}

// CaffeNet.cpp:196-205: state + model -> weights from the model file, history / iter / current_step from the
// state (Solver::Restore); model only -> copyLayers (weights by layer NAME, Net::CopyTrainedLayersFrom).
bool CaffeNet::restore(const std::string& model_file, const std::string& state_file, std::string* err) {
  COS_RT(cudaSetDevice(device_));
  std::string model = model_file;
  if (!state_file.empty()) {
    int it = 0, step = 0;
    std::string learned;
    std::vector<ParsedBlob> hist;
    if (!read_solverstate(state_file, &it, &step, &learned, &hist, err)) return false;
    if (hist.size() != spec_.counts.size()) {
      *err = "'" + state_file + "' is not a matching snapshot of this net: " + std::to_string(hist.size()) +
             " history blobs, the net has " + std::to_string(spec_.counts.size()) + " learnable blobs";
      return false;
    }
    std::vector<float> flat(count_, 0.f);
    uint64_t off = 0;
    for (size_t k = 0; k < hist.size(); ++k) {
      if (hist[k].data.size() != static_cast<size_t>(spec_.counts[k])) {
        *err = "'" + state_file + "' is not a matching snapshot of this net: history blob " + std::to_string(k) +
               " has " + std::to_string(hist[k].data.size()) + " elements, expected " +
               std::to_string(spec_.counts[k]);
        return false;
      }
      memcpy(flat.data() + off, hist[k].data.data(), hist[k].data.size() * sizeof(float));
      off += hist[k].data.size();
    }
    COS_RT(cudaMemcpy(hist_, flat.data(), count_ * sizeof(float), cudaMemcpyHostToDevice));
    iter_ = it;
    current_step_ = step;
    spec_.init_iter = it;
    if (model.empty()) model = learned;  // Solver::Restore follows state.learned_net()
  }
  if (!model.empty()) {
    std::vector<ParsedLayer> layers;
    std::string name;
    if (!read_caffemodel(model, &name, &layers, err)) return false;
    std::vector<float> flat(count_);
    COS_RT(cudaMemcpy(flat.data(), data_, count_ * sizeof(float), cudaMemcpyDeviceToHost));
    uint64_t off = 0;
    int matched = 0;
    for (size_t k = 0; k < spec_.counts.size(); ++k) {
      const std::string& lname = k < spec_.layer_names.size() ? spec_.layer_names[k] : std::string();
      size_t j = 0;  // index of blob k inside its layer
      for (size_t q = k; q > 0 && q - 1 < spec_.layer_names.size() && spec_.layer_names[q - 1] == lname; --q) ++j;
      for (const ParsedLayer& L : layers) {
        if (L.name != lname) continue;
        if (j >= L.blobs.size() || L.blobs[j].data.size() != static_cast<size_t>(spec_.counts[k])) {
          *err = "'" + model + "' is not a matching snapshot of this net: layer '" + lname + "' blob " +
                 std::to_string(j) + " does not have " + std::to_string(spec_.counts[k]) + " elements";
          return false;  // CopyTrainedLayersFrom CHECKs the shapes (net.cpp)
        }
        memcpy(flat.data() + off, L.blobs[j].data.data(), L.blobs[j].data.size() * sizeof(float));
        ++matched;
        break;
      }
      off += static_cast<uint64_t>(spec_.counts[k]);
    }
    if (matched == 0 && !spec_.counts.empty()) {
      *err = "'" + model + "' is not a matching snapshot of this net: no layer name matches";
      return false;
    }
    COS_RT(cudaMemcpy(data_, flat.data(), count_ * sizeof(float), cudaMemcpyHostToDevice));
  }
  return true;
}

// ----------------------------------------------------------- NvlinkCaffeNet

NvlinkCaffeNet::NvlinkCaffeNet(const SolverSpec& spec, int cluster_size, int node_rank, bool is_training)
    : CaffeNet(spec, cluster_size, node_rank, is_training) {}

NvlinkCaffeNet::~NvlinkCaffeNet() {
  if (device_ >= 0) {
    cudaSetDevice(device_);
    if (stream_) cudaStreamSynchronize(stream_);
    cudaDeviceSynchronize();
    cudaGetLastError();
  }
  // Peers may still be inside a kernel that touches this arena: give them a
  // short rendezvous.  (The physical allocation is reference-counted by the
  // importers, so a peer that is late still never faults.)
  if (connected_ && adapter_) {
    std::string ignore;
    adapter_->barrier(2000, &ignore);
  }
  mcast_.close();
  mappings_.clear();
  adapter_.reset();
}

void NvlinkCaffeNet::setup_nvls(int timeout_ms) {
  nvls_active_ = false;
  std::string e;
  bool ok = arena_.transport() == kTransportVmmFd && MulticastMapping::supported(device_);
  if (!ok) e = "multicast unsupported or arena not VMM-backed";
  if (rank_ == 0) {
    int fd = -1;
    if (ok) ok = mcast_.create(device_, arena_.bytes(), world_, &fd, &e);
    adapter_->offer("mcast", ok ? fd : -1, ok ? "1" : "0");
    if (fd >= 0) close(fd);
  } else {
    int fd = -1;
    std::string meta, fe;
    bool got = adapter_->fetch(0, "mcast", &fd, &meta, timeout_ms, &fe);
    if (!got || meta != "1" || fd < 0) {
      if (fd >= 0) close(fd);
      if (ok) e = got ? "rank 0 could not create the multicast object" : fe;
      ok = false;
    } else if (ok) {
      ok = mcast_.import(device_, arena_.bytes(), fd, &e);
    } else {
      close(fd);
    }
  }
  if (ok) ok = mcast_.add_device(&e);
  // cuMulticastBindMem blocks until every device of the team was added: agree first
  auto agree = [&](const char* key, bool mine) {
    adapter_->offer(key, -1, mine ? "1" : "0");
    bool all = mine;
    for (int p = 0; p < world_; ++p) {
      if (p == rank_) continue;
      std::string meta, fe;
      if (!adapter_->fetch(p, key, nullptr, &meta, timeout_ms, &fe) || meta != "1") all = false;
    }
    return all;
  };
  bool all = agree("mc_added", ok);
  if (all) ok = mcast_.bind_and_map(arena_, &e);
  all = agree("mc_mapped", all && ok);
  if (all) {
    nvls_active_ = true;
    mc_base_ = static_cast<char*>(mcast_.base());
    nvls_note_ = "nvls active";
  } else {
    mcast_.close();
    nvls_note_ = "nvls off: " + (e.empty() ? std::string("a peer could not join the multicast team") : e);
  }
  if (getenv("COS_VERBOSE")) fprintf(stderr, "[caffedistri_b200] rank %d: %s\n", rank_, nvls_note_.c_str());
}

bool NvlinkCaffeNet::setup(int start_device_id, std::string* err) {
  if (!allocate_device(start_device_id, true, err)) return false;
  // CaffeNet.cpp:253-272: adapter (listener) first, then one channel per peer
  adapter_.reset(new PeerAdapter(world_, rank_));
  if (!adapter_->ok()) {
    *err = "peer adapter: " + adapter_->init_error();
    return false;
  }
  ArenaMeta m = arena_.meta();
  adapter_->offer("arena", arena_.fd(), std::string(reinterpret_cast<const char*>(&m), sizeof(m)));
  mappings_.resize(world_);
  return true;
}

void NvlinkCaffeNet::localAddresses(std::vector<std::string>* vec) {
  vec->assign(world_, std::string());
  for (int i = 0; i < world_; ++i)
    if (i != rank_) (*vec)[i] = adapter_->address();  // "" at the own rank (CaffeNet.cpp:398-401)
}

bool NvlinkCaffeNet::connect(const std::vector<std::string>& addresses, std::string* err) {
  if (connected_) return true;
  if (static_cast<int>(addresses.size()) < world_) {
    *err = "connect: need " + std::to_string(world_) + " addresses, got " + std::to_string(addresses.size());
    return false;
  }
  COS_RT(cudaSetDevice(device_));
  if (!adapter_->connect(addresses, err)) return false;
  const int timeout = static_cast<int>(opt_timeout_ms_);
  for (int n = 1; n < world_; ++n) {
    const int peer = (rank_ + n) % world_;
    int fd = -1;
    std::string meta;
    if (!adapter_->fetch(peer, "arena", &fd, &meta, timeout, err)) return false;
    if (meta.size() != sizeof(ArenaMeta)) {
      if (fd >= 0) close(fd);
      *err = "connect: bad arena metadata from rank " + std::to_string(peer);
      return false;
    }
    ArenaMeta m;
    memcpy(&m, meta.data(), sizeof(m));
    if (m.bytes != arena_.bytes()) {
      if (fd >= 0) close(fd);
      *err = "connect: rank " + std::to_string(peer) + " has a different parameter layout (arena " +
             std::to_string(m.bytes) + " vs " + std::to_string(arena_.bytes()) + " bytes)";
      return false;
    }
    mappings_[peer].reset(new PeerMapping());
    if (!mappings_[peer]->open(m, fd, device_, err)) {
      *err = "connect: mapping rank " + std::to_string(peer) + "'s arena: " + *err;
      return false;
    }
    char* base = static_cast<char*>(mappings_[peer]->base());
    peer_flags_[peer] = reinterpret_cast<uint32_t*>(base);
    peer_data_[peer] = reinterpret_cast<float*>(base + off_data_);
    peer_diff_[peer] = reinterpret_cast<const float*>(base + off_diff_);
    peer_hist_[peer] = reinterpret_cast<const float*>(base + off_hist_);
    peer_wire_[peer] = wire_ ? reinterpret_cast<uint16_t*>(base + off_wire_) : nullptr;
    peer_recv_[peer] = recv_stride_ ? static_cast<void*>(base + off_recv_) : nullptr;
    peer_llg_[peer] = ll_grad_stride_ ? reinterpret_cast<uint64_t*>(base + off_llg_) : nullptr;
    peer_llw_[peer] = ll_grad_stride_ ? reinterpret_cast<uint64_t*>(base + off_llw_) : nullptr;
  }
  connected_ = true;
  // NVLS multicast team: on request, or by default where it pays (N >= 6, message >= nvls_min_bytes, fp32 wire).
  // The decision uses only values that are identical on every rank.
  const bool want_nvls = opt_nvls_ == 1 || (opt_nvls_ < 0 && world_ >= kNvlsAutoMinWorld && spec_.grad_dtype == COS_GRAD_FP32 &&
                                            static_cast<int64_t>(count_ * sizeof(float)) >= opt_nvls_min_bytes_);
  if (want_nvls) setup_nvls(timeout);
  // everyone has mapped everyone; then the first on_start(): all-gather of the
  // owners' weight shards (socket_sync_cpu.cpp:102-105), so that all ranks
  // start from the same weights even if they were initialised differently.
  if (!adapter_->barrier(timeout, err)) return false;
  if (opt_initial_gather_) {
    if (!all_gather_weights(nullptr, true, err)) return false;
    // every rank has LAUNCHED before any rank blocks on the device (matters when several executors
    // live in one process: a thread waiting on the GPU must not be able to delay a peer's launch)
    if (!adapter_->barrier(timeout, err)) return false;
    if (!synchronize(err)) return false;
    if (!adapter_->barrier(timeout, err)) return false;
  }
  return true;
}

bool NvlinkCaffeNet::sync(std::string* err) {
  if (world_ > 1) return adapter_->barrier(static_cast<int>(opt_timeout_ms_), err);
  return true;
}

}  // namespace cosb

// ------------------------------------------------------ MultiDeviceCaffeNet
namespace cosb {

MultiDeviceCaffeNet::MultiDeviceCaffeNet(const SolverSpec& spec, int num_local_devices, int cluster_size,
                                         int node_rank, bool is_training)
    : CaffeNet(spec, cluster_size * num_local_devices, node_rank * num_local_devices, is_training),
      executors_(cluster_size),
      node_rank_(node_rank) {
  for (int i = 0; i < num_local_devices; ++i) {
    ranks_.emplace_back(new NvlinkCaffeNet(spec, cluster_size * num_local_devices, node_rank * num_local_devices + i,
                                           is_training));
    ranks_.back()->set_solver_index(i);
  }
}

MultiDeviceCaffeNet::~MultiDeviceCaffeNet() {
  // the ranks rendezvous with their peers while shutting down: tear them down concurrently
  std::vector<std::thread> th;
  for (auto& r : ranks_) th.emplace_back([&r] { r.reset(); });
  for (auto& t : th) t.join();
}

bool MultiDeviceCaffeNet::setup(int start_device_id, std::string* err) {
  int d = start_device_id;  // CaffeNet.cpp:130-142: d = FindDevice(d + 1) for each local device in turn
  for (auto& r : ranks_) {
    if (!r->setup(d, err)) return false;
    d = r->device();
  }
  return true;
}

void MultiDeviceCaffeNet::localAddresses(std::vector<std::string>* vec) {
  std::string mine;
  for (size_t i = 0; i < ranks_.size(); ++i) {
    std::vector<std::string> a;
    ranks_[i]->localAddresses(&a);
    // every entry of a rank's list except its own is the same endpoint
    const std::string& ep = a[(ranks_[i]->rank() + 1) % a.size()];
    mine += (i ? ";" : "") + ep;
  }
  vec->assign(executors_, std::string());
  for (int e = 0; e < executors_; ++e)
    if (e != node_rank_) (*vec)[e] = mine;  // "" at the own rank (CaffeNet.cpp:398-401)
}

bool MultiDeviceCaffeNet::connect(const std::vector<std::string>& addresses, std::string* err) {
  const int k = static_cast<int>(ranks_.size());
  if (executors_ > 1 && static_cast<int>(addresses.size()) < executors_) {
    *err = "connect: need " + std::to_string(executors_) + " addresses, got " + std::to_string(addresses.size());
    return false;
  }
  std::vector<std::string> table(static_cast<size_t>(executors_) * k);
  for (int e = 0; e < executors_; ++e) {
    if (e == node_rank_) {
      for (int i = 0; i < k; ++i) {
        std::vector<std::string> a;
        ranks_[i]->localAddresses(&a);
        table[static_cast<size_t>(e) * k + i] = a[(ranks_[i]->rank() + 1) % a.size()];
      }
      continue;
    }
    std::string rest = addresses[e];
    for (int i = 0; i < k; ++i) {
      size_t semi = rest.find(';');
      if ((i < k - 1) == (semi == std::string::npos) || rest.empty()) {
        *err = "connect: executor " + std::to_string(e) + " did not publish " + std::to_string(k) +
               " device endpoints: '" + addresses[e] + "'";
        return false;
      }
      table[static_cast<size_t>(e) * k + i] = rest.substr(0, semi);
      rest = semi == std::string::npos ? "" : rest.substr(semi + 1);
    }
  }
  // every rank's connect() rendezvouses with all the others, local ones included: run them concurrently
  std::vector<std::string> errs(k);
  std::vector<char> ok(k, 0);
  std::vector<std::thread> th;
  for (int i = 0; i < k; ++i) th.emplace_back([&, i] { ok[i] = ranks_[i]->connect(table, &errs[i]) ? 1 : 0; });
  for (auto& t : th) t.join();
  for (int i = 0; i < k; ++i) {
    if (!ok[i]) {
      *err = "local device " + std::to_string(i) + ": " + errs[i];
      return false;
    }
  }
  connected_ = true;
  return true;
}

bool MultiDeviceCaffeNet::sync(std::string* err) {
  const int k = static_cast<int>(ranks_.size());
  std::vector<std::string> errs(k);
  std::vector<char> ok(k, 0);
  std::vector<std::thread> th;
  for (int i = 0; i < k; ++i) th.emplace_back([&, i] { ok[i] = ranks_[i]->sync(&errs[i]) ? 1 : 0; });
  for (auto& t : th) t.join();
  for (int i = 0; i < k; ++i) {
    if (!ok[i]) {
      *err = errs[i];
      return false;
    }
  }
  return true;
}

bool MultiDeviceCaffeNet::synchronize(std::string* err) {
  for (auto& r : ranks_)
    if (!r->synchronize(err)) return false;
  return true;
}

void MultiDeviceCaffeNet::set_forward_backward(cos_forward_backward_fn fn, void* user) {
  for (auto& r : ranks_) r->set_forward_backward(fn, user);
}

int64_t MultiDeviceCaffeNet::launch_count() const {
  int64_t n = 0;
  for (auto& r : ranks_) n += r->launch_count();
  return n;
}

bool MultiDeviceCaffeNet::set_option(const std::string& name, int64_t v, std::string* err) {
  for (auto& r : ranks_)
    if (!r->set_option(name, v, err)) return false;
  return true;
}

}  // namespace cosb
