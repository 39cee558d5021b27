// solver_spec.hpp -- what the hot path needs to know about the solver and the
// learnable-parameter layout.
//
// The reference obtains this from protobuf (SolverParameter, caffe.proto:102-;
// ParamSpec lr_mult/decay_mult :283-304) and from Net::learnable_params()
// after Caffe has built the net (parallel.cpp:27-57).  Here a small
// text-format reader plus shape inference over the layer types of the
// BASELINE configs recovers the same flat layout, so that
// CaffeNet.allocate(solver.prototxt, ...) keeps working unchanged.
#ifndef COS_SOLVER_SPEC_HPP_
#define COS_SOLVER_SPEC_HPP_

#include <cstdint>
#include <string>
#include <vector>

namespace cosb {

struct SolverSpec {
  // learnable blobs in learnable_params() order
  std::vector<int64_t> counts;
  std::vector<float> lr_mult, decay_mult;
  std::vector<std::string> blob_names;  // "<layer>.<index>" (diagnostics)
  // what Net::ToProto needs to write a stock-Caffe .caffemodel (solver.cpp:452-459)
  std::string net_name;
  std::vector<std::string> layer_names, layer_types;  // per learnable blob: owning layer
  std::vector<std::vector<int64_t>> shapes;            // per learnable blob: Blob shape
  bool snapshot_hdf5 = false;                          // SolverParameter.snapshot_format (caffe.proto:194-198)
  // SolverParameter
  std::string lr_policy = "fixed";
  float base_lr = 0.01f, gamma = 0.1f, power = 0.75f;
  int stepsize = 1;
  std::vector<int> stepvalues;
  int max_iter = 0;
  float momentum = 0.f, weight_decay = 0.f;
  int test_iter = 0, test_interval = 0;
  std::string snapshot_prefix;
  std::string regularization_type = "L2";
  std::string type = "SGD";       // SGD | Nesterov | AdaGrad | RMSProp | AdaDelta (canonical spelling)
  float delta = 1e-8f;             // SolverParameter.delta (caffe.proto: default 1e-8)
  float rms_decay = 0.f;           // SolverParameter.rms_decay (no default: 0)
  int iter_size = 1;
  float clip_gradients = -1.f;
  bool solver_mode_gpu = true;
  // training input layer
  int batch_size = 0;
  std::vector<int> input_shape;  // N,C,H,W of the first top of the data layer
  // this library's extensions
  int grad_dtype = 0;  // COS_GRAD_FP32 / COS_GRAD_BF16
  int init_iter = 0;

  uint64_t param_count() const;  // max(1, sum counts): parallel.cpp:60-68
};

// SocketSync::chunk (socket_sync_cpu.cpp:46-54).
void chunk(uint64_t param_count, int cluster_size, int peer, uint64_t* offs, uint64_t* size);

// SGDSolver::GetLearningRate (sgd_solver.cpp:27-63), Dtype = float.
// Returns false for an unknown policy.
bool learning_rate(const std::string& policy, float base_lr, float gamma, float power, int stepsize,
                   const int* stepvalues, int nstepvalues, int max_iter, int iter, int* current_step,
                   float* rate);

// SolverType (fused_sync_sgd.hpp) of a canonical type name, -1 for any other name.
int solver_type_id(const std::string& type);
// The canonical name of SolverType `id` (static storage), nullptr for any other value.
const char* solver_type_name(int id);
// Checks type, momentum and rms_decay as the reference's solver constructors do (sgd_solvers.hpp:70-100).  Shared
// by the prototxt parser (which maps the deprecated solver_type enum to the type name first) and
// cos_net_allocate_desc.
bool validate_solver(const SolverSpec& spec, std::string* err);

// Parses a solver prototxt and the net it references (net:, train_net: or
// inline net_param/train_net_param) and fills `spec`.
bool parse_solver_prototxt(const std::string& solver_path, SolverSpec* spec, std::string* err);
// Parses only a net prototxt text (TRAIN phase) into the layout part of spec.
bool parse_net_prototxt_text(const std::string& text, SolverSpec* spec, std::string* err);

}  // namespace cosb
#endif
