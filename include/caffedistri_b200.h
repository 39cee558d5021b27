/*
 * caffedistri_b200.h -- C ABI of libcaffedistri_b200.so
 *
 * B200-native replacement for the inter-executor gradient-sync hot path of
 * yahoo/CaffeOnSpark's libcaffedistri.so (CaffeNet<float> behind the
 * com.yahoo.ml.jcaffe.CaffeNet JNI class).  Plain pointers and sizes only; no
 * C++/torch types.  Every entry point names the reference interface it
 * replaces (paths relative to the reference repo root):
 *   J  = caffe-distri/src/main/java/com/yahoo/ml/jcaffe/CaffeNet.java
 *   JN = caffe-distri/src/main/cpp/jni/JniCaffeNet.cpp
 *   CN = caffe-distri/src/main/cpp/CaffeNet.cpp
 *   CH = caffe-distri/include/CaffeNet.hpp
 *
 * Conventions (mirroring JN): functions that return `int` status return 1 for
 * true/success and 0 for false/failure unless stated otherwise; integer
 * getters return -1 on failure (JN:235-249,479-580); the message behind a
 * failure is available from cos_last_error() (thread-local), which is what the
 * JNI shim turns into a java.lang.Exception (src/main/cpp/common.cpp:111-116).
 * The handle is the value the reference stores in BaseObject.address (a long).
 *
 * There is NO CPU fallback: every compute entry point fails (0 / -1 with an
 * error string) when no CUDA device is usable.
 */
#ifndef CAFFEDISTRI_B200_H_
#define CAFFEDISTRI_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define COS_API __attribute__((visibility("default")))

/* J:21-23 connection types.  RDMA and SOCKET both select the NVLink peer-memory
 * transport here (there is no socket or verbs data path in this library). */
#define COS_CONNECTION_NONE 0
#define COS_CONNECTION_RDMA 1
#define COS_CONNECTION_SOCKET 2

/* gradient wire precision of the reduce-scatter (weights/history stay fp32) */
#define COS_GRAD_FP32 0
#define COS_GRAD_BF16 1

/* all-reduce algorithm selection (cos_net_set_option "algo") */
#define COS_ALGO_AUTO 0
#define COS_ALGO_TWO_SHOT 1 /* reduce-scatter -> fused SGD -> weight push (sharded PS, reference structure) */
#define COS_ALGO_ONE_SHOT 2 /* every rank reduces + updates everything, no weight push (small P) */

typedef struct cos_net cos_net; /* opaque; == CaffeNet<float>* of the reference (JN:96-99) */

/* One input blob of train()/predict(): what a com.yahoo.ml.jcaffe.FloatBlob
 * hands over (JN:383-413, common.cpp GetFloatBlobVector): host fp32 data in
 * NCHW order owned by the caller for the duration of the call. */
typedef struct cos_blob {
  const float* data;
  int num, channels, height, width;
} cos_blob;

/* Solver + learnable-parameter layout, the information the reference reads
 * from the solver/net prototxt (caffe.proto SolverParameter :102-, ParamSpec
 * :283-304) and from Net::learnable_params() (parallel.cpp:27-57). */
typedef struct cos_solver_desc {
  int nblobs;               /* learnable blobs, learnable_params() order */
  const int64_t* counts;    /* elements per blob */
  const float* lr_mult;     /* ParamSpec.lr_mult   (NULL = all 1.0) */
  const float* decay_mult;  /* ParamSpec.decay_mult (NULL = all 1.0) */
  const char* lr_policy;    /* fixed|step|exp|inv|multistep|poly|sigmoid */
  float base_lr, gamma, power;
  int stepsize;
  const int* stepvalues;
  int nstepvalues;
  int max_iter;
  float momentum, weight_decay;
  int test_iter, test_interval;
  const char* snapshot_prefix; /* may be NULL */
  int grad_dtype;              /* COS_GRAD_FP32 | COS_GRAD_BF16 */
  int init_iter;               /* iteration to resume from (0) */
  int regularization_l1;       /* SolverParameter.regularization_type: 0 = "L2" (default), 1 = "L1" */
  /* SolverParameter.type: "SGD", "Nesterov", "AdaGrad", "RMSProp" or "AdaDelta"; NULL = "SGD".  Other types
   * (Adam among them) fail at allocation, as do momentum != 0 with AdaGrad / RMSProp and rms_decay outside [0, 1)
   * with RMSProp (the checks of the reference's solver constructors, sgd_solvers.hpp:70-100). */
  const char* type;
  float delta;                 /* SolverParameter.delta (AdaGrad, RMSProp, AdaDelta); Caffe's default is 1e-8 */
  float rms_decay;             /* SolverParameter.rms_decay (RMSProp); Caffe's default is 0 */
} cos_solver_desc;

/* Gradient producer = Net::ForwardBackward of the reference (solver.cpp:221-223),
 * out of scope for this library and supplied by the embedding runtime.  Called
 * from cos_net_train on the calling thread after the input blobs were staged
 * to the device: `inputs[i]` are DEVICE pointers (same shapes as the host
 * blobs), it must enqueue on `cuda_stream` work that ACCUMULATES the local
 * gradient into cos_net_diff() using the weights in cos_net_data(), and write
 * the scalar loss to the DEVICE float `loss_dev`.  Return 0 on success. */
typedef int (*cos_forward_backward_fn)(void* user, int solver_index, const cos_blob* inputs, int ninputs,
                                       float* loss_dev, void* cuda_stream);

/* ---------------------------------------------------------------- errors */
COS_API const char* cos_last_error(void);
COS_API const char* cos_version(void);

/* ------------------------------------------ the 18 JNI natives (J:60-230) */

/* J:60-69 allocate / JN:14-89.  cluster_size==1 -> local net (CH LocalCaffeNet),
 * else connection_type RDMA|SOCKET -> NVLink peer net (CH Socket/RDMACaffeNet),
 * anything else fails like the reference's missing switch case (JN:41-64).
 * Parses the solver prototxt and the net it names to derive the layout. */
COS_API int cos_net_allocate(const char* solver_conf_file, const char* model_file, const char* state_file,
                             int num_local_devices, int cluster_size, int node_rank, int is_training,
                             int connection_type, int start_device_id, int validation_net_id, cos_net** out);

/* Same, with the layout given directly instead of parsed from prototxt. */
COS_API int cos_net_allocate_desc(const cos_solver_desc* desc, int num_local_devices, int cluster_size,
                                  int node_rank, int is_training, int connection_type, int start_device_id,
                                  cos_net** out);

/* J:72 deallocate / JN:96-99 */
COS_API void cos_net_deallocate(cos_net* net);

/* J:125 localAddresses / JN:106-159, CN:394-404.  Returns the number of
 * addresses (0 for a local net, cluster_size otherwise; "" at the own rank)
 * or -1.  *addresses points to an array owned by the net, valid until the
 * next call or deallocate. */
COS_API int cos_net_local_addresses(cos_net* net, const char* const** addresses);

/* J:80 connect / JN:184-228, CN:456-480.  `addresses` is indexed by rank; NULL
 * array or NULL entries are allowed (common.cpp:57-77).  A malformed or
 * unreachable address returns 0 (CaffeNetTest.connectbogus). */
COS_API int cos_net_connect(cos_net* net, const char* const* addresses, int naddresses);

/* J:86 sync / JN:166-177, CN:497-504: zero-payload control barrier over all
 * executors (no-op returning 1 on a local net, CH:91). */
COS_API int cos_net_sync(cos_net* net);

/* J:99 init / JN:256-270, CN:585-654: bind the calling thread to the solver's
 * device; solver_index < 0 -> 0. */
COS_API int cos_net_init(cos_net* net, int solver_index, int enable_nn);

/* J:120 train / JN:383-413, CN:707-729: ONE Solver::Step (solver.cpp:194-273):
 * stage the input blobs host->device, run the gradient producer, then the
 * fused scale + reduce-scatter + solver update (SGD, Nesterov, AdaGrad,
 * RMSProp or AdaDelta) + weight all-gather kernel, ++iter.  data==NULL -> 0 with error "data is NULL" (JN:391-395). */
COS_API int cos_net_train(cos_net* net, int solver_index, const cos_blob* data, int ndata);

/* J:110 predict / JN:277-376: forward-only; not on the sync path -> always
 * fails with "predict: not supported" (returns -1).  Kept for symbol parity. */
COS_API int cos_net_predict(cos_net* net, int solver_index, const cos_blob* data, int ndata,
                            const char* const* output_blob_names, int nnames, cos_blob* outputs);

/* J:220,227 validation / aggregateValidationOutputs (JN:420-470): not on the
 * sync path; return 0 with an error string. */
COS_API int cos_net_validation(cos_net* net, const cos_blob* data, int ndata);
COS_API int cos_net_aggregate_validation_outputs(cos_net* net);

/* J:133-165 integer getters / JN:235-249,479-580; -1 on invalid index. */
COS_API int cos_net_device_id(cos_net* net, int solver_index);
COS_API int cos_net_get_init_iter(cos_net* net, int solver_index);
COS_API int cos_net_get_max_iter(cos_net* net, int solver_index);
COS_API int cos_net_get_test_iter(cos_net* net, int solver_index);
COS_API int cos_net_get_test_interval(cos_net* net);

/* J:171 snapshot / JN:537-548, CN:735-738 -> Solver::Snapshot (solver.cpp:400-425):
 * writes stock-Caffe binaryproto files <prefix>_iter_<n>.caffemodel (NetParameter)
 * and .solverstate (SolverState) and returns the iteration, -1 on failure.  With
 * snapshot_format: HDF5 (sgd_solver.cpp:279-323, net.cpp:867-917) the files are
 * <prefix>_iter_<n>.caffemodel.h5 / .solverstate.h5 in HDF5's original file layout,
 * written without libhdf5 (csrc/hdf5_io.cpp): /data/<layer>/<j>, /iter, /learned_net,
 * /current_step, /history/<i>.  Called on rank 0 only, like
 * the reference (CaffeProcessor.scala:454-465); NOT collective: the history
 * shards of the other ranks are read through their mapped arenas. */
COS_API int cos_net_snapshot(cos_net* net);
/* The path snapshot() writes for `iter` (== CaffeNet.java:192-207 snapshotFilename). 1/0. */
COS_API int cos_net_snapshot_filename(cos_net* net, int iter, int is_state, char* buf, int cap);

/* J:177,185 getValidationOutputBlobNames / getValidationOutputBlobs
 * (JN:587-673): no validation net here; return -1 with an error string. */
COS_API int cos_net_get_validation_output_blob_names(cos_net* net, const char* const** names);
COS_API int cos_net_get_validation_output_blobs(cos_net* net, int length, cos_blob* outputs);

/* ------------------- hot-path surface for a native gradient producer ------ */

/* Register Net::ForwardBackward (see cos_forward_backward_fn). */
COS_API int cos_net_set_forward_backward(cos_net* net, cos_forward_backward_fn fn, void* user);

/* Flat device buffers of Params<Dtype> (parallel.hpp:22-45): data_, diff_ and
 * the SGD history, each cos_net_param_count() fp32 elements, blobs laid out
 * back to back in learnable_params() order. */
COS_API float* cos_net_data(cos_net* net, int solver_index);
COS_API float* cos_net_diff(cos_net* net, int solver_index);
COS_API float* cos_net_history(cos_net* net, int solver_index);
/* AdaDelta's second history buffer (the history of updates, history_[n + i] of the reference), laid out like
 * cos_net_history(); NULL for every other solver, which has no second buffer. */
COS_API float* cos_net_update_history(cos_net* net, int solver_index);
COS_API int64_t cos_net_param_count(cos_net* net);

/* SocketSync::chunk (socket_sync_cpu.cpp:46-54): shard of `rank`. 1/0. */
COS_API int cos_net_shard(cos_net* net, int rank, uint64_t* offs, uint64_t* size);

/* Current iteration (Solver::iter()) and the rate GetLearningRate()
 * (sgd_solver.cpp:27-63) yields for it. */
COS_API int cos_net_iter(cos_net* net);
COS_API float cos_net_learning_rate(cos_net* net);
COS_API float cos_net_last_loss(cos_net* net);

/* THE HOT PATH.  Everything of Solver::Step after ForwardBackward plus the
 * next step's on_start, as one kernel launch on `cuda_stream` (NULL = the
 * net's own stream): diff *= 1/N, reduce-scatter over NVLink peer memory in
 * the reference's summation order, L2 / L1 decay, the solver's update (SGD with
 * momentum, Nesterov, AdaGrad, RMSProp or AdaDelta, in the operation order of
 * the reference's CPU branch), w -= update, push of the new weights to every peer, optional diff := 0 (ClearParamDiffs of the next
 * Step), ++iter.  Asynchronous: returns after the launch.  Collective: every
 * rank must call it once per iteration. */
COS_API int cos_net_sync_step(cos_net* net, int solver_index, void* cuda_stream);

/* on_start() alone (socket_sync_cpu.cpp:102-105): all-gather of the owned
 * weight shards.  connect() runs it once; exposed for tests. Collective. */
COS_API int cos_net_all_gather_weights(cos_net* net, int solver_index, void* cuda_stream);

/* Wait for the net's outstanding device work and surface device-side errors
 * (barrier time-outs).  1 = ok. */
COS_API int cos_net_synchronize(cos_net* net);

/* Options: "algo" (COS_ALGO_*), "zero_diff" (0/1, default 1),
 * "grid" (CTAs, 0 = auto), "block" (threads, 0 = auto), "kernel" (-1 = auto,
 * 0 = LDG/STG pull kernel, 1 = TMA bulk-copy pull pipeline, 2 = push kernel
 * (stores only, bf16 cast in registers), 3 = NVLS multimem kernel, 4 = LL kernel
 * (flag-in-data words, no barrier / fence; small nets, cluster_size <= 8); kernels 1 and 3 run SGD only:
 * with another solver a forced 1 runs kernel 0 and a forced 3 AUTO's choice),
 * "barrier_timeout_ms", "one_shot_max_bytes", "ll_max_bytes" / "push_max_bytes" /
 * "nvls_min_bytes" (AUTO thresholds on the message size 4P), "push_vecs" (push / LL
 * kernel grid sizing),
 * "timing" (CUDA events around each launch, default 0), "initial_gather" (0 =
 * connect() skips the first on_start(); the caller then runs
 * cos_net_all_gather_weights itself), "nvls" (-1 = auto: join an NVSwitch
 * multicast team at connect() when cluster_size >= 6, the wire is fp32 and
 * 4P >= nvls_min_bytes (32 MiB); 0 = never; 1 = always try.  The in-switch sum matches the
 * reference to 1e-5, not bitwise: set 0 for bit-exact runs), "nvls_unroll",
 * "nvls_p2p" (share of plain-P2P vectors in the NVLS kernel), "train_pipeline"
 * (1 = cos_net_train returns once its batch has left host memory; 0 = after the
 * whole step), "trace" (record %globaltimer at the kernel's phase boundaries and inside
 * the two barriers).
 * Read-only via get_option: "resolved_algo", "resolved_kernel", "nvls_active",
 * "transport", "default_grid", "trace_0".."trace_12".  1/0. */
COS_API int cos_net_set_option(cos_net* net, const char* name, int64_t value);
COS_API int64_t cos_net_get_option(cos_net* net, const char* name);

/* Device time in ms of the last completed cos_net_sync_step / all_gather
 * launch (CUDA events on the launching stream), -1 if none. */
COS_API float cos_net_last_kernel_ms(cos_net* net);
/* Kernels launched by this net so far (bench.py gpu_launches). */
COS_API int64_t cos_net_launch_count(cos_net* net);
/* Seeded synthetic fill of one flat buffer ON THE DEVICE (which: 0 = data_, 1 = diff_,
 * 2 = history): out[i] = amp * u_i, u_i uniform in [-1, 1) from a counter-based
 * generator keyed by (seed, stream) -- the generator the oracle's driver uses
 * (oracle/ref_driver.cpp), so benchmarks and parity runs need no host copy of the
 * 4P-byte tensors.  Asynchronous on the net's stream; 1/0. */
COS_API int cos_net_fill(cos_net* net, int solver_index, int which, uint64_t seed, uint64_t stream, float amp);

/* --------------------- transport object (reference: util/socket.hpp) ------ */
/* PeerAdapter = SocketAdapter + SocketChannel of the reference
 * (socket.hpp:22-89): a listener thread on a per-process endpoint whose
 * address string travels through Spark; channels carry only control messages
 * and memory handles (file descriptors), never tensor payload. */
typedef struct cos_adapter cos_adapter;
COS_API cos_adapter* cos_adapter_create(int cluster_size, int rank);
COS_API void cos_adapter_destroy(cos_adapter* a);
COS_API const char* cos_adapter_address(cos_adapter* a);
COS_API int cos_adapter_connect(cos_adapter* a, const char* const* addresses, int naddresses);
/* CTRL barrier (socket_sync_cpu.cpp:135-163 with data=false). 1/0. */
COS_API int cos_adapter_barrier(cos_adapter* a, int timeout_ms);
/* Offer a file descriptor under `key` / fetch the one `peer` offered. */
COS_API int cos_adapter_offer_fd(cos_adapter* a, const char* key, int fd, const void* meta, int meta_len);
COS_API int cos_adapter_fetch_fd(cos_adapter* a, int peer, const char* key, void* meta, int meta_cap,
                                 int timeout_ms);

/* ---------------- snapshot file utilities (host only, Caffe binaryproto) ------ */
/* Write / read the subset of caffe.proto the snapshots use (NetParameter.layer[].blobs[],
 * SolverState) without libprotobuf.  Blob k has shape_ndims[k] dims taken in order from
 * dims_flat; consecutive blobs with the same layer name form one layer.  Readers return
 * the element count of the requested blob (copied into `out` when cap allows) or -1. */
COS_API int cos_caffemodel_write(const char* path, const char* net_name, int nblobs, const char* const* layer_names,
                                 const char* const* layer_types, const int* shape_ndims, const int64_t* dims_flat,
                                 const float* const* data);
COS_API int64_t cos_caffemodel_read(const char* path, const char* layer_name, int blob_index, float* out,
                                    int64_t cap);
COS_API int cos_solverstate_write(const char* path, int iter, int current_step, const char* learned_net, int nblobs,
                                  const int* shape_ndims, const int64_t* dims_flat, const float* const* data);
/* blob_index < 0: returns the number of history blobs. */
COS_API int64_t cos_solverstate_read(const char* path, int* iter, int* current_step, char* learned_net,
                                     int learned_cap, int blob_index, float* out, int64_t cap);

/* -------------------------- host helpers (pure functions, no device) ------ */
/* HDF5 twins of the two writers above (snapshot_format: HDF5).  cos_caffemodel_read / cos_solverstate_read
 * recognise HDF5 files by their signature, so they read either format. */
COS_API int cos_caffemodel_write_h5(const char* path, int nblobs, const char* const* layer_names, const int* shape_ndims,
                                    const int64_t* dims_flat, const float* const* data);
COS_API int cos_solverstate_write_h5(const char* path, int iter, int current_step, const char* learned_net, int nblobs,
                                     const int* shape_ndims, const int64_t* dims_flat, const float* const* data);
/* One dataset of ANY old-style HDF5 file by absolute path ("/data", "/history/3"): returns the element count
 * (float32 copied, int32 converted to float), fills up to max_dims dims and *ndims; -1 on failure.  Used to pin the
 * reader on libhdf5-written files. */
COS_API int64_t cos_hdf5_read_dataset(const char* path, const char* dataset, int64_t* dims, int max_dims, int* ndims,
                                      float* out, int64_t cap);

COS_API void cos_chunk(uint64_t param_count, int cluster_size, int peer, uint64_t* offs, uint64_t* size);
COS_API float cos_learning_rate(const char* lr_policy, float base_lr, float gamma, float power, int stepsize,
                                const int* stepvalues, int nstepvalues, int max_iter, int iter,
                                int* current_step);
/* Parse solver prototxt (+ the net prototxt it names) into a layout; arrays
 * are written up to `cap` blobs.  Returns nblobs or -1. */
COS_API int cos_parse_solver(const char* solver_conf_file, cos_solver_desc* desc, int64_t* counts,
                             float* lr_mult, float* decay_mult, int cap, char* lr_policy_buf,
                             char* snapshot_prefix_buf, int strcap, int* stepvalues, int stepcap,
                             int* batch_size);

#ifdef __cplusplus
}
#endif
#endif /* CAFFEDISTRI_B200_H_ */
