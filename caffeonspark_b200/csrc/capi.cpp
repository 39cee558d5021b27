// capi.cpp -- the C ABI of include/caffedistri_b200.h over cosb::CaffeNet.
//
// One function per JNI native of com.yahoo.ml.jcaffe.CaffeNet
// (caffe-distri/src/main/cpp/jni/JniCaffeNet.cpp); argument checks and return
// conventions follow that file (solver_index < 0 -> false / -1, null data ->
// "data is NULL", C++ exceptions -> error string instead of a Java exception).
#include <string.h>

#include <exception>
#include <string>
#include <vector>

#include "../../include/caffedistri_b200.h"
#include "caffe_net.hpp"
#include "caffe_proto_io.hpp"
#include "hdf5_io.hpp"
#include "peer_adapter.hpp"
#include "solver_spec.hpp"

using cosb::CaffeNet;
using cosb::SolverSpec;

namespace {
thread_local std::string g_error;

int fail(const std::string& msg, int rc = 0) {
  g_error = msg;
  return rc;
}

CaffeNet* N(cos_net* n) { return reinterpret_cast<CaffeNet*>(n); }
// the object serving local solver `i` (one per local device); nullptr for an invalid index
CaffeNet* R(cos_net* n, int i) { return (n && i >= 0) ? reinterpret_cast<CaffeNet*>(n)->rank_net(i) : nullptr; }

// common.cpp:111-116 ThrowJavaException analogue: never let a C++ exception
// cross the C boundary.
#define COS_GUARD(rc_on_throw, ...)                   \
  try {                                               \
    __VA_ARGS__                                       \
  } catch (const std::exception& ex) {                \
    g_error = std::string("exception: ") + ex.what(); \
    return rc_on_throw;                               \
  } catch (...) {                                     \
    g_error = "unknown exception";                    \
    return rc_on_throw;                               \
  }

bool spec_from_desc(const cos_solver_desc* d, SolverSpec* s, std::string* err) {
  if (!d) {
    *err = "solver description is NULL";
    return false;
  }
  if (d->nblobs < 0 || (d->nblobs > 0 && !d->counts)) {
    *err = "bad blob table";
    return false;
  }
  for (int k = 0; k < d->nblobs; ++k) {
    s->counts.push_back(d->counts[k]);
    s->lr_mult.push_back(d->lr_mult ? d->lr_mult[k] : 1.0f);
    s->decay_mult.push_back(d->decay_mult ? d->decay_mult[k] : 1.0f);
    s->blob_names.push_back("blob." + std::to_string(k));
    s->layer_names.push_back("blob" + std::to_string(k));  // no net definition: one pseudo layer per blob
    s->layer_types.push_back("Blob");
    s->shapes.push_back({d->counts[k]});
  }
  s->net_name = "cos_net";
  s->lr_policy = d->lr_policy ? d->lr_policy : "fixed";
  s->base_lr = d->base_lr;
  s->gamma = d->gamma;
  s->power = d->power;
  s->stepsize = d->stepsize;
  for (int i = 0; i < d->nstepvalues; ++i) s->stepvalues.push_back(d->stepvalues[i]);
  s->max_iter = d->max_iter;
  s->momentum = d->momentum;
  s->weight_decay = d->weight_decay;
  s->test_iter = d->test_iter;
  s->test_interval = d->test_interval;
  s->snapshot_prefix = d->snapshot_prefix ? d->snapshot_prefix : "";
  s->grad_dtype = d->grad_dtype;
  s->init_iter = d->init_iter;
  s->regularization_type = d->regularization_l1 ? "L1" : "L2";
  s->type = d->type ? d->type : "SGD";
  s->delta = d->delta;
  s->rms_decay = d->rms_decay;
  if (!cosb::validate_solver(*s, err)) return false;
  float r;
  int step = 0;
  if (!cosb::learning_rate(s->lr_policy, s->base_lr, s->gamma, s->power, s->stepsize,
                           s->stepvalues.empty() ? nullptr : s->stepvalues.data(),
                           static_cast<int>(s->stepvalues.size()), s->max_iter, 0, &step, &r)) {
    *err = "Unknown learning rate policy: " + s->lr_policy;
    return false;
  }
  return true;
}
}  // namespace

extern "C" {

const char* cos_last_error(void) { return g_error.c_str(); }
const char* cos_version(void) { return "caffedistri_b200 0.1 (sm_100a)"; }

int cos_net_allocate(const char* solver_conf_file, const char* model_file, const char* state_file,
                     int num_local_devices, int cluster_size, int node_rank, int is_training,
                     int connection_type, int start_device_id, int validation_net_id, cos_net** out) {
  (void)validation_net_id;
  COS_GUARD(0, {
    if (!out) return fail("out is NULL");
    *out = nullptr;
    if (!solver_conf_file) return fail("solver_conf_file_chars == NULL");  // JniCaffeNet.cpp:23-26
    SolverSpec spec;
    std::string err;
    if (!cosb::parse_solver_prototxt(solver_conf_file, &spec, &err)) return fail(err);
    if (const char* g = getenv("COS_GRAD_DTYPE")) spec.grad_dtype = strcmp(g, "bf16") == 0 ? COS_GRAD_BF16 : COS_GRAD_FP32;
    CaffeNet* n = CaffeNet::create(spec, num_local_devices, cluster_size, node_rank, is_training != 0,
                                   connection_type, start_device_id, &err);
    if (!n) return fail(err);
    // CaffeNet.cpp:196-205: restore a previous run when files are given
    const std::string model = model_file ? model_file : "", state = state_file ? state_file : "";
    if (!model.empty() || !state.empty()) {
      if (!n->restore(model, state, &err)) {
        delete n;
        return fail(err);
      }
    }
    *out = reinterpret_cast<cos_net*>(n);
    return 1;
  })
}

int cos_net_allocate_desc(const cos_solver_desc* desc, int num_local_devices, int cluster_size, int node_rank,
                          int is_training, int connection_type, int start_device_id, cos_net** out) {
  COS_GUARD(0, {
    if (!out) return fail("out is NULL");
    *out = nullptr;
    SolverSpec spec;
    std::string err;
    if (!spec_from_desc(desc, &spec, &err)) return fail(err);
    CaffeNet* n = CaffeNet::create(spec, num_local_devices, cluster_size, node_rank, is_training != 0,
                                   connection_type, start_device_id, &err);
    if (!n) return fail(err);
    *out = reinterpret_cast<cos_net*>(n);
    return 1;
  })
}

void cos_net_deallocate(cos_net* net) {
  try {
    delete N(net);
  } catch (...) {
  }
}

int cos_net_local_addresses(cos_net* net, const char* const** addresses) {
  COS_GUARD(-1, {
    if (!net) return fail("net is NULL", -1);
    CaffeNet* n = N(net);
    std::vector<std::string>& store = n->address_store();
    n->localAddresses(&store);
    std::vector<const char*>& ptrs = const_cast<std::vector<const char*>&>(n->address_cstrs());
    ptrs.clear();
    for (const std::string& s : store) ptrs.push_back(s.c_str());
    if (addresses) *addresses = ptrs.empty() ? nullptr : ptrs.data();
    return static_cast<int>(store.size());
  })
}

int cos_net_connect(cos_net* net, const char* const* addresses, int naddresses) {
  COS_GUARD(0, {
    if (!net) return fail("net is NULL");
    std::vector<std::string> addrs;
    // common.cpp:57-77 GetStringVector: a null array / null entries are allowed
    for (int i = 0; addresses && i < naddresses; ++i) addrs.push_back(addresses[i] ? addresses[i] : "");
    std::string err;
    if (!N(net)->connect(addrs, &err)) return fail(err);
    return 1;
  })
}

int cos_net_sync(cos_net* net) {
  COS_GUARD(0, {
    if (!net) return fail("net is NULL");
    std::string err;
    if (!N(net)->sync(&err)) return fail(err);
    return 1;
  })
}

int cos_net_init(cos_net* net, int solver_index, int enable_nn) {
  COS_GUARD(0, {
    if (!net) return fail("net is NULL");
    if (solver_index < 0) return fail("invalid solver_index");  // JniCaffeNet.cpp:259-262
    std::string err;
    CaffeNet* r = R(net, solver_index);
    if (!r) return fail("invalid solver_index");
    if (!r->init(0, enable_nn != 0, &err)) return fail(err);
    return 1;
  })
}

int cos_net_train(cos_net* net, int solver_index, const cos_blob* data, int ndata) {
  COS_GUARD(0, {
    if (!net) return fail("net is NULL");
    if (solver_index < 0) return fail("invalid solver_index");
    if (!data) return fail("data is NULL");  // JniCaffeNet.cpp:391-395
    std::string err;
    CaffeNet* r = R(net, solver_index);
    if (!r) return fail("invalid solver_index");
    if (!r->train(0, data, ndata, &err)) return fail(err);
    return 1;
  })
}

int cos_net_predict(cos_net*, int, const cos_blob*, int, const char* const*, int, cos_blob*) {
  return fail("predict: forward-only inference is not part of the gradient-sync library", -1);
}
int cos_net_validation(cos_net*, const cos_blob*, int) {
  return fail("validation: interleaved validation is not part of the gradient-sync library");
}
int cos_net_aggregate_validation_outputs(cos_net*) {
  return fail("aggregateValidationOutputs: not part of the gradient-sync library");
}
int cos_net_get_validation_output_blob_names(cos_net*, const char* const**) {
  return fail("getValidationOutputBlobNames: no validation net in the gradient-sync library", -1);
}
int cos_net_get_validation_output_blobs(cos_net*, int, cos_blob*) {
  return fail("getValidationOutputBlobs: no validation net in the gradient-sync library", -1);
}

int cos_net_device_id(cos_net* net, int solver_index) {
  if (!net || solver_index < 0) return fail("invalid solver_index", -1);  // JniCaffeNet.cpp:238-241
  CaffeNet* r = R(net, solver_index);
  return r ? r->deviceID(0) : fail("invalid solver_index", -1);
}
int cos_net_get_init_iter(cos_net* net, int solver_index) {
  if (!net || solver_index < 0) return fail("invalid solver_index", -1);
  CaffeNet* r = R(net, solver_index);
  return r ? r->getInitIter(0) : fail("invalid solver_index", -1);
}
int cos_net_get_max_iter(cos_net* net, int solver_index) {
  if (!net || solver_index < 0) return fail("invalid solver_index", -1);
  CaffeNet* r = R(net, solver_index);
  return r ? r->getMaxIter(0) : fail("invalid solver_index", -1);
}
int cos_net_get_test_iter(cos_net* net, int solver_index) {
  if (!net || solver_index < 0) return fail("invalid solver_index", -1);
  CaffeNet* r = R(net, solver_index);
  return r ? r->getTestIter(0) : fail("invalid solver_index", -1);
}
int cos_net_get_test_interval(cos_net* net) {
  if (!net) return fail("net is NULL", -1);
  return N(net)->getTestInterval();
}

int cos_net_snapshot(cos_net* net) {
  COS_GUARD(-1, {
    if (!net) return fail("net is NULL", -1);
    std::string err;
    int it = N(net)->snapshot(&err);
    if (it < 0) return fail(err, -1);
    return it;
  })
}

int cos_net_snapshot_filename(cos_net* net, int iter, int is_state, char* buf, int cap) {
  if (!net || !buf || cap <= 0 || iter < 0) return fail("bad argument");
  const std::string s = R(net, 0)->snapshot_filename(iter, is_state != 0);
  if (static_cast<int>(s.size()) >= cap) return fail("buffer too small");
  memcpy(buf, s.c_str(), s.size() + 1);
  return 1;
}

int cos_net_set_forward_backward(cos_net* net, cos_forward_backward_fn fn, void* user) {
  if (!net) return fail("net is NULL");
  N(net)->set_forward_backward(fn, user);
  return 1;
}

float* cos_net_data(cos_net* net, int solver_index) {
  CaffeNet* r = R(net, solver_index);
  return r ? r->data() : nullptr;
}
float* cos_net_diff(cos_net* net, int solver_index) {
  CaffeNet* r = R(net, solver_index);
  return r ? r->diff() : nullptr;
}
float* cos_net_history(cos_net* net, int solver_index) {
  CaffeNet* r = R(net, solver_index);
  return r ? r->history() : nullptr;
}
float* cos_net_update_history(cos_net* net, int solver_index) {
  CaffeNet* r = R(net, solver_index);
  return r ? r->update_history() : nullptr;
}
int64_t cos_net_param_count(cos_net* net) { return net ? static_cast<int64_t>(R(net, 0)->param_count()) : -1; }

int cos_net_shard(cos_net* net, int rank, uint64_t* offs, uint64_t* size) {
  if (!net || !offs || !size) return fail("bad argument");
  CaffeNet* n = N(net);
  if (rank < 0 || rank >= n->cluster_size()) return fail("rank out of range");
  cosb::chunk(n->param_count(), n->cluster_size(), rank, offs, size);
  return 1;
}

int cos_net_iter(cos_net* net) { return net ? R(net, 0)->iter() : -1; }
float cos_net_learning_rate(cos_net* net) { return net ? R(net, 0)->current_rate() : 0.f; }
float cos_net_last_loss(cos_net* net) { return net ? R(net, 0)->last_loss() : 0.f; }

int cos_net_sync_step(cos_net* net, int solver_index, void* cuda_stream) {
  COS_GUARD(0, {
    if (!net) return fail("net is NULL");
    if (solver_index < 0) return fail("invalid solver_index");
    std::string err;
    CaffeNet* r = R(net, solver_index);
    if (!r) return fail("invalid solver_index");
    if (!r->sync_step(0, static_cast<cudaStream_t>(cuda_stream), cuda_stream == nullptr, &err))
      return fail(err);
    return 1;
  })
}

int cos_net_all_gather_weights(cos_net* net, int solver_index, void* cuda_stream) {
  COS_GUARD(0, {
    if (!net) return fail("net is NULL");
    if (solver_index < 0) return fail("invalid solver_index");
    std::string err;
    CaffeNet* r = R(net, solver_index);
    if (!r) return fail("invalid solver_index");
    if (!r->all_gather_weights(static_cast<cudaStream_t>(cuda_stream), cuda_stream == nullptr, &err))
      return fail(err);
    return 1;
  })
}

int cos_net_synchronize(cos_net* net) {
  COS_GUARD(0, {
    if (!net) return fail("net is NULL");
    std::string err;
    if (!N(net)->synchronize(&err)) return fail(err);
    return 1;
  })
}

int cos_net_set_option(cos_net* net, const char* name, int64_t value) {
  if (!net || !name) return fail("bad argument");
  std::string err;
  if (!N(net)->set_option(name, value, &err)) return fail(err);
  return 1;
}
int64_t cos_net_get_option(cos_net* net, const char* name) {
  if (!net || !name) return -1;
  return N(net)->get_option(name);
}
float cos_net_last_kernel_ms(cos_net* net) { return net ? R(net, 0)->last_kernel_ms() : -1.f; }
int64_t cos_net_launch_count(cos_net* net) { return net ? N(net)->launch_count() : 0; }

int cos_net_fill(cos_net* net, int solver_index, int which, uint64_t seed, uint64_t stream, float amp) {
  COS_GUARD(0, {
    if (!net) return fail("net is NULL");
    CaffeNet* r = solver_index < 0 ? nullptr : R(net, solver_index);
    if (!r) return fail("invalid solver_index");
    std::string err;
    if (!r->fill(which, seed, stream, amp, &err)) return fail(err);
    return 1;
  })
}

// ------------------------------------------------------------- adapter API

cos_adapter* cos_adapter_create(int cluster_size, int rank) {
  if (cluster_size < 1 || rank < 0 || rank >= cluster_size) {
    fail("bad cluster_size / rank");
    return nullptr;
  }
  try {
    cosb::PeerAdapter* a = new cosb::PeerAdapter(cluster_size, rank);
    if (!a->ok()) {
      fail(a->init_error());
      delete a;
      return nullptr;
    }
    return reinterpret_cast<cos_adapter*>(a);
  } catch (...) {
    fail("adapter creation failed");
    return nullptr;
  }
}
void cos_adapter_destroy(cos_adapter* a) { delete reinterpret_cast<cosb::PeerAdapter*>(a); }
const char* cos_adapter_address(cos_adapter* a) {
  return a ? reinterpret_cast<cosb::PeerAdapter*>(a)->address().c_str() : "";
}
int cos_adapter_connect(cos_adapter* a, const char* const* addresses, int naddresses) {
  if (!a) return fail("adapter is NULL");
  std::vector<std::string> addrs;
  for (int i = 0; addresses && i < naddresses; ++i) addrs.push_back(addresses[i] ? addresses[i] : "");
  std::string err;
  if (!reinterpret_cast<cosb::PeerAdapter*>(a)->connect(addrs, &err)) return fail(err);
  return 1;
}
int cos_adapter_barrier(cos_adapter* a, int timeout_ms) {
  if (!a) return fail("adapter is NULL");
  std::string err;
  if (!reinterpret_cast<cosb::PeerAdapter*>(a)->barrier(timeout_ms, &err)) return fail(err);
  return 1;
}
int cos_adapter_offer_fd(cos_adapter* a, const char* key, int fd, const void* meta, int meta_len) {
  if (!a || !key) return fail("bad argument");
  reinterpret_cast<cosb::PeerAdapter*>(a)->offer(
      key, fd, meta && meta_len > 0 ? std::string(static_cast<const char*>(meta), meta_len) : std::string());
  return 1;
}
int cos_adapter_fetch_fd(cos_adapter* a, int peer, const char* key, void* meta, int meta_cap, int timeout_ms) {
  if (!a || !key) return fail("bad argument", -2);
  int fd = -1;
  std::string m, err;
  if (!reinterpret_cast<cosb::PeerAdapter*>(a)->fetch(peer, key, &fd, &m, timeout_ms, &err)) return fail(err, -2);
  if (meta && meta_cap > 0) {
    memset(meta, 0, meta_cap);
    memcpy(meta, m.data(), m.size() < static_cast<size_t>(meta_cap) ? m.size() : meta_cap);
  }
  return fd;  // -1: metadata only
}

// ------------------------------------------------- snapshot file utilities
namespace {
std::vector<cosb::BlobView> views_from_c(int nblobs, const char* const* layer_names, const char* const* layer_types,
                                         const int* shape_ndims, const int64_t* dims_flat,
                                         const float* const* data) {
  std::vector<cosb::BlobView> v(nblobs);
  size_t d = 0;
  for (int k = 0; k < nblobs; ++k) {
    v[k].layer_name = layer_names ? layer_names[k] : "";
    v[k].layer_type = layer_types ? layer_types[k] : "";
    v[k].count = 1;
    for (int i = 0; i < shape_ndims[k]; ++i) {
      v[k].shape.push_back(dims_flat[d + i]);
      v[k].count *= static_cast<uint64_t>(dims_flat[d + i]);
    }
    d += shape_ndims[k];
    v[k].data = data[k];
  }
  return v;
}
}  // namespace

int cos_caffemodel_write(const char* path, const char* net_name, int nblobs, const char* const* layer_names,
                         const char* const* layer_types, const int* shape_ndims, const int64_t* dims_flat,
                         const float* const* data) {
  COS_GUARD(0, {
    if (!path || nblobs < 0 || (nblobs && (!layer_names || !shape_ndims || !dims_flat || !data)))
      return fail("bad argument");
    std::string err;
    if (!cosb::write_caffemodel(path, net_name ? net_name : "",
                                views_from_c(nblobs, layer_names, layer_types, shape_ndims, dims_flat, data), &err))
      return fail(err);
    return 1;
  })
}

int64_t cos_caffemodel_read(const char* path, const char* layer_name, int blob_index, float* out, int64_t cap) {
  COS_GUARD(-1, {
    if (!path || !layer_name || blob_index < 0) return fail("bad argument", -1);
    std::vector<cosb::ParsedLayer> layers;
    std::string name, err;
    if (!cosb::read_caffemodel(path, &name, &layers, &err)) return fail(err, -1);
    for (const auto& L : layers) {
      if (L.name != layer_name) continue;
      if (blob_index >= static_cast<int>(L.blobs.size())) return fail("layer has fewer blobs", -1);
      const auto& b = L.blobs[blob_index];
      const int64_t n = static_cast<int64_t>(b.data.size());
      if (out && cap >= n) memcpy(out, b.data.data(), n * sizeof(float));
      return n;
    }
    return fail(std::string("no layer named '") + layer_name + "'", -1);
  })
}

int cos_solverstate_write(const char* path, int iter, int current_step, const char* learned_net, int nblobs,
                          const int* shape_ndims, const int64_t* dims_flat, const float* const* data) {
  COS_GUARD(0, {
    if (!path || nblobs < 0 || (nblobs && (!shape_ndims || !dims_flat || !data))) return fail("bad argument");
    std::string err;
    if (!cosb::write_solverstate(path, iter, current_step, learned_net ? learned_net : "",
                                 views_from_c(nblobs, nullptr, nullptr, shape_ndims, dims_flat, data), &err))
      return fail(err);
    return 1;
  })
}

int cos_caffemodel_write_h5(const char* path, int nblobs, const char* const* layer_names, const int* shape_ndims,
                            const int64_t* dims_flat, const float* const* data) {
  COS_GUARD(0, {
    if (!path || nblobs < 0 || (nblobs && (!layer_names || !shape_ndims || !dims_flat || !data)))
      return fail("bad argument");
    std::string err;
    if (!cosb::write_caffemodel_h5(path, views_from_c(nblobs, layer_names, nullptr, shape_ndims, dims_flat, data), &err))
      return fail(err);
    return 1;
  })
}

int cos_solverstate_write_h5(const char* path, int iter, int current_step, const char* learned_net, int nblobs,
                             const int* shape_ndims, const int64_t* dims_flat, const float* const* data) {
  COS_GUARD(0, {
    if (!path || nblobs < 0 || (nblobs && (!shape_ndims || !dims_flat || !data))) return fail("bad argument");
    std::string err;
    if (!cosb::write_solverstate_h5(path, iter, current_step, learned_net ? learned_net : "",
                                    views_from_c(nblobs, nullptr, nullptr, shape_ndims, dims_flat, data), &err))
      return fail(err);
    return 1;
  })
}

int64_t cos_hdf5_read_dataset(const char* path, const char* dataset, int64_t* dims, int max_dims, int* ndims, float* out,
                              int64_t cap) {
  COS_GUARD(-1, {
    if (!path || !dataset) return fail("bad argument", -1);
    cosb::H5Node root;
    std::string err;
    if (!cosb::h5_read(path, &root, &err)) return fail(err, -1);
    const cosb::H5Node* n = &root;
    std::string rest = dataset;
    while (!rest.empty()) {
      if (rest[0] == '/') {
        rest.erase(0, 1);
        continue;
      }
      const size_t slash = rest.find('/');
      const std::string part = rest.substr(0, slash);
      n = n->find(part);
      if (!n) return fail(std::string("no object '") + dataset + "' in '" + path + "'", -1);
      rest = slash == std::string::npos ? "" : rest.substr(slash + 1);
    }
    if (n->kind != cosb::H5Node::kFloat32 && n->kind != cosb::H5Node::kInt32)
      return fail(std::string("'") + dataset + "' is not a numeric dataset", -1);
    if (ndims) *ndims = static_cast<int>(n->shape.size());
    for (int i = 0; dims && i < max_dims && i < static_cast<int>(n->shape.size()); ++i) dims[i] = n->shape[i];
    const int64_t cnt = static_cast<int64_t>(n->count);
    if (out && cap >= cnt) {
      if (n->kind == cosb::H5Node::kFloat32) memcpy(out, n->f32.data(), cnt * sizeof(float));
      else
        for (int64_t i = 0; i < cnt; ++i) out[i] = static_cast<float>(n->i32[i]);
    }
    return cnt;
  })
}

int64_t cos_solverstate_read(const char* path, int* iter, int* current_step, char* learned_net, int learned_cap,
                             int blob_index, float* out, int64_t cap) {
  COS_GUARD(-1, {
    if (!path) return fail("bad argument", -1);
    int it = 0, st = 0;
    std::string learned, err;
    std::vector<cosb::ParsedBlob> hist;
    if (!cosb::read_solverstate(path, &it, &st, &learned, &hist, &err)) return fail(err, -1);
    if (iter) *iter = it;
    if (current_step) *current_step = st;
    if (learned_net && learned_cap > 0) {
      strncpy(learned_net, learned.c_str(), learned_cap - 1);
      learned_net[learned_cap - 1] = 0;
    }
    if (blob_index < 0) return static_cast<int64_t>(hist.size());  // number of history blobs
    if (blob_index >= static_cast<int>(hist.size())) return fail("no such history blob", -1);
    const int64_t n = static_cast<int64_t>(hist[blob_index].data.size());
    if (out && cap >= n) memcpy(out, hist[blob_index].data.data(), n * sizeof(float));
    return n;
  })
}

// ------------------------------------------------------------ host helpers

void cos_chunk(uint64_t param_count, int cluster_size, int peer, uint64_t* offs, uint64_t* size) {
  cosb::chunk(param_count, cluster_size, peer, offs, size);
}

float cos_learning_rate(const char* lr_policy, float base_lr, float gamma, float power, int stepsize,
                        const int* stepvalues, int nstepvalues, int max_iter, int iter, int* current_step) {
  float r = 0.f;
  int local = 0;
  if (!cosb::learning_rate(lr_policy ? lr_policy : "", base_lr, gamma, power, stepsize, stepvalues, nstepvalues,
                           max_iter, iter, current_step ? current_step : &local, &r)) {
    fail(std::string("Unknown learning rate policy: ") + (lr_policy ? lr_policy : "(null)"));
    return -1.f;
  }
  return r;
}

int cos_parse_solver(const char* solver_conf_file, cos_solver_desc* desc, int64_t* counts, float* lr_mult,
                     float* decay_mult, int cap, char* lr_policy_buf, char* snapshot_prefix_buf, int strcap,
                     int* stepvalues, int stepcap, int* batch_size) {
  COS_GUARD(-1, {
    if (!solver_conf_file || !desc) return fail("bad argument", -1);
    SolverSpec s;
    std::string err;
    if (!cosb::parse_solver_prototxt(solver_conf_file, &s, &err)) return fail(err, -1);
    const int n = static_cast<int>(s.counts.size());
    if (n > cap) return fail("blob table larger than the provided capacity", -1);
    for (int k = 0; k < n; ++k) {
      if (counts) counts[k] = s.counts[k];
      if (lr_mult) lr_mult[k] = s.lr_mult[k];
      if (decay_mult) decay_mult[k] = s.decay_mult[k];
    }
    memset(desc, 0, sizeof(*desc));
    desc->nblobs = n;
    desc->counts = counts;
    desc->lr_mult = lr_mult;
    desc->decay_mult = decay_mult;
    if (lr_policy_buf && strcap > 0) {
      strncpy(lr_policy_buf, s.lr_policy.c_str(), strcap - 1);
      lr_policy_buf[strcap - 1] = 0;
      desc->lr_policy = lr_policy_buf;
    }
    if (snapshot_prefix_buf && strcap > 0) {
      strncpy(snapshot_prefix_buf, s.snapshot_prefix.c_str(), strcap - 1);
      snapshot_prefix_buf[strcap - 1] = 0;
      desc->snapshot_prefix = snapshot_prefix_buf;
    }
    desc->base_lr = s.base_lr;
    desc->gamma = s.gamma;
    desc->power = s.power;
    desc->stepsize = s.stepsize;
    int nsv = static_cast<int>(s.stepvalues.size());
    if (nsv > stepcap) nsv = stepcap;
    for (int i = 0; i < nsv && stepvalues; ++i) stepvalues[i] = s.stepvalues[i];
    desc->stepvalues = stepvalues;
    desc->nstepvalues = stepvalues ? nsv : 0;
    desc->max_iter = s.max_iter;
    desc->momentum = s.momentum;
    desc->weight_decay = s.weight_decay;
    desc->regularization_l1 = s.regularization_type == "L1" ? 1 : 0;
    desc->type = cosb::solver_type_name(cosb::solver_type_id(s.type));
    desc->delta = s.delta;
    desc->rms_decay = s.rms_decay;
    desc->test_iter = s.test_iter;
    desc->test_interval = s.test_interval;
    if (batch_size) *batch_size = s.batch_size;
    return n;
  })
}

}  // extern "C"
