// solver_spec.cpp -- see solver_spec.hpp.
#include "solver_spec.hpp"

#include "fused_sync_sgd.hpp"

#include <math.h>
#include <stdlib.h>

#include <fstream>
#include <map>
#include <memory>
#include <sstream>

namespace cosb {

uint64_t SolverSpec::param_count() const {
  uint64_t n = 0;
  for (int64_t c : counts) n += static_cast<uint64_t>(c);
  return n > 0 ? n : 1;  // "Size have at least one byte" (parallel.cpp:66-67)
}

// socket_sync_cpu.cpp:46-54: size_t arithmetic, multiply before divide.
void chunk(uint64_t param_count, int cluster_size, int peer, uint64_t* offs, uint64_t* size) {
  const uint64_t n = static_cast<uint64_t>(cluster_size);
  const uint64_t start = (static_cast<uint64_t>(peer) + 0) * param_count / n;
  const uint64_t until = (static_cast<uint64_t>(peer) + 1) * param_count / n;
  *offs = start;
  *size = until - start;
}

// sgd_solver.cpp:27-63 with Dtype = float.  The reference's unqualified
// pow()/exp() take float sub-expressions, evaluate in double and the product
// with base_lr is rounded to float when assigned to `Dtype rate`.
bool learning_rate(const std::string& policy, float base_lr, float gamma, float power, int stepsize,
                   const int* stepvalues, int nstepvalues, int max_iter, int iter, int* current_step,
                   float* rate) {
  if (policy == "fixed") {
    *rate = base_lr;
  } else if (policy == "step") {
    if (stepsize <= 0) return false;
    *current_step = iter / stepsize;
    *rate = static_cast<float>(static_cast<double>(base_lr) *
                               pow(static_cast<double>(gamma), static_cast<double>(*current_step)));
  } else if (policy == "exp") {
    *rate = static_cast<float>(static_cast<double>(base_lr) *
                               pow(static_cast<double>(gamma), static_cast<double>(iter)));
  } else if (policy == "inv") {
    const float base = 1.0f + gamma * static_cast<float>(iter);
    const float e = -power;
    *rate = static_cast<float>(static_cast<double>(base_lr) * pow(static_cast<double>(base), static_cast<double>(e)));
  } else if (policy == "multistep") {
    if (*current_step < nstepvalues && iter >= stepvalues[*current_step]) (*current_step)++;
    *rate = static_cast<float>(static_cast<double>(base_lr) *
                               pow(static_cast<double>(gamma), static_cast<double>(*current_step)));
  } else if (policy == "poly") {
    const float base = 1.0f - (static_cast<float>(iter) / static_cast<float>(max_iter));
    *rate = static_cast<float>(static_cast<double>(base_lr) *
                               pow(static_cast<double>(base), static_cast<double>(power)));
  } else if (policy == "sigmoid") {
    const float x = -gamma * (static_cast<float>(iter) - static_cast<float>(stepsize));
    const double d = 1.0 / (1.0 + exp(static_cast<double>(x)));
    *rate = static_cast<float>(static_cast<double>(base_lr) * d);
  } else {
    return false;  // LOG(FATAL) << "Unknown learning rate policy" (:60)
  }
  return true;
}

namespace {
const char* const kSolverNames[] = {"SGD", "Nesterov", "AdaGrad", "RMSProp", "AdaDelta"};
const char* const kSolverEnums[] = {"SGD", "NESTEROV", "ADAGRAD", "RMSPROP", "ADADELTA"};  // caffe.proto SolverType
}  // namespace

const char* solver_type_name(int id) { return id >= 0 && id < 5 ? kSolverNames[id] : nullptr; }

int solver_type_id(const std::string& type) {
  for (int k = 0; k < 5; ++k)
    if (type == kSolverNames[k]) return k;
  return -1;
}

bool validate_solver(const SolverSpec& spec, std::string* err) {
  const int id = solver_type_id(spec.type);
  if (id < 0) {
    *err = "solver type '" + spec.type +
           "' is not on the accelerated path (only SGD, Nesterov, AdaGrad, RMSProp and AdaDelta are)";
    return false;
  }
  if ((id == kSolverAdaGrad || id == kSolverRMSProp) && spec.momentum != 0.f) {
    *err = std::string("Momentum cannot be used with ") + kSolverNames[id] + ".";
    return false;
  }
  if (id == kSolverRMSProp && !(spec.rms_decay >= 0.f && spec.rms_decay < 1.f)) {
    *err = "rms_decay should lie between 0 and 1.";
    return false;
  }
  return true;
}

// ------------------------------------------------- protobuf text-format reader
namespace {

struct Node {
  bool is_msg = false;
  std::string value;                                             // scalar
  std::vector<std::pair<std::string, std::shared_ptr<Node>>> kids;  // message fields, in order

  std::vector<const Node*> all(const std::string& key) const {
    std::vector<const Node*> out;
    for (const auto& kv : kids)
      if (kv.first == key) out.push_back(kv.second.get());
    return out;
  }
  const Node* first(const std::string& key) const {
    for (const auto& kv : kids)
      if (kv.first == key) return kv.second.get();
    return nullptr;
  }
  std::string str(const std::string& key, const std::string& dflt = "") const {
    const Node* n = first(key);
    return (n && !n->is_msg) ? n->value : dflt;
  }
  double num(const std::string& key, double dflt) const {
    const Node* n = first(key);
    return (n && !n->is_msg) ? atof(n->value.c_str()) : dflt;
  }
  long integer(const std::string& key, long dflt) const {
    const Node* n = first(key);
    return (n && !n->is_msg) ? atol(n->value.c_str()) : dflt;
  }
  bool boolean(const std::string& key, bool dflt) const {
    const Node* n = first(key);
    if (!n || n->is_msg) return dflt;
    return n->value == "true" || n->value == "1" || n->value == "True";
  }
};

class TextParser {
 public:
  explicit TextParser(const std::string& s) : s_(s) {}
  bool parse(Node* root, std::string* err) {
    root->is_msg = true;
    if (!message(root, /*top=*/true)) {
      std::ostringstream os;
      os << "prototxt parse error near offset " << pos_ << ": " << err_;
      *err = os.str();
      return false;
    }
    return true;
  }

 private:
  void skip() {
    for (;;) {
      while (pos_ < s_.size() && (isspace(static_cast<unsigned char>(s_[pos_])) || s_[pos_] == ',' || s_[pos_] == ';'))
        ++pos_;
      if (pos_ < s_.size() && s_[pos_] == '#') {
        while (pos_ < s_.size() && s_[pos_] != '\n') ++pos_;
        continue;
      }
      break;
    }
  }
  bool word(std::string* out) {
    skip();
    size_t b = pos_;
    while (pos_ < s_.size()) {
      char c = s_[pos_];
      if (isalnum(static_cast<unsigned char>(c)) || c == '_' || c == '.' || c == '+' || c == '-') ++pos_;
      else break;
    }
    if (pos_ == b) return false;
    *out = s_.substr(b, pos_ - b);
    return true;
  }
  bool quoted(std::string* out) {
    skip();
    if (pos_ >= s_.size() || (s_[pos_] != '"' && s_[pos_] != '\'')) return false;
    out->clear();
    while (pos_ < s_.size() && (s_[pos_] == '"' || s_[pos_] == '\'')) {  // adjacent strings concatenate
      char q = s_[pos_++];
      while (pos_ < s_.size() && s_[pos_] != q) {
        if (s_[pos_] == '\\' && pos_ + 1 < s_.size()) {
          char e = s_[pos_ + 1];
          out->push_back(e == 'n' ? '\n' : e == 't' ? '\t' : e);
          pos_ += 2;
        } else {
          out->push_back(s_[pos_++]);
        }
      }
      if (pos_ >= s_.size()) { err_ = "unterminated string"; return false; }
      ++pos_;
      skip();
    }
    return true;
  }
  bool message(Node* m, bool top) {
    for (;;) {
      skip();
      if (pos_ >= s_.size()) {
        if (top) return true;
        err_ = "missing '}'";
        return false;
      }
      if (s_[pos_] == '}' || s_[pos_] == '>') {
        if (top) { err_ = "unexpected '}'"; return false; }
        ++pos_;
        return true;
      }
      std::string key;
      if (!word(&key)) { err_ = "expected field name"; return false; }
      skip();
      bool colon = false;
      if (pos_ < s_.size() && s_[pos_] == ':') { colon = true; ++pos_; skip(); }
      auto child = std::make_shared<Node>();
      if (pos_ < s_.size() && (s_[pos_] == '{' || s_[pos_] == '<')) {
        ++pos_;
        child->is_msg = true;
        if (!message(child.get(), false)) return false;
      } else if (colon) {
        if (pos_ < s_.size() && s_[pos_] == '[') {  // short repeated form: [a, b]
          ++pos_;
          for (;;) {
            skip();
            if (pos_ < s_.size() && s_[pos_] == ']') { ++pos_; break; }
            auto item = std::make_shared<Node>();
            if (!quoted(&item->value) && !word(&item->value)) { err_ = "bad list item"; return false; }
            m->kids.emplace_back(key, item);
          }
          continue;
        }
        if (!quoted(&child->value) && !word(&child->value)) { err_ = "expected value for '" + key + "'"; return false; }
      } else {
        err_ = "expected ':' or '{' after '" + key + "'";
        return false;
      }
      m->kids.emplace_back(key, child);
    }
  }
  const std::string& s_;
  size_t pos_ = 0;
  std::string err_;
};

bool read_file(const std::string& path, std::string* out) {
  std::ifstream f(path.c_str(), std::ios::in | std::ios::binary);
  if (!f) return false;
  std::ostringstream ss;
  ss << f.rdbuf();
  *out = ss.str();
  return true;
}

// NetStateRule filtering for phase TRAIN (net.cpp FilterNet/StateMeetsRule;
// only the phase criterion is modelled).
bool in_train_phase(const Node& layer) {
  auto includes = layer.all("include");
  auto excludes = layer.all("exclude");
  if (!includes.empty()) {
    for (const Node* r : includes) {
      std::string ph = r->str("phase");
      if (ph.empty() || ph == "TRAIN") return true;
    }
    return false;
  }
  for (const Node* r : excludes) {
    std::string ph = r->str("phase");
    if (ph.empty() || ph == "TRAIN") return false;
  }
  std::string own = layer.str("phase");  // rarely used layer-level phase
  return own.empty() || own == "TRAIN";
}

typedef std::vector<long> Shape;

long prod(const Shape& s, size_t from = 0) {
  long p = 1;
  for (size_t i = from; i < s.size(); ++i) p *= s[i];
  return p;
}

struct HW { long h, w; };

// kernel_size / kernel_h,kernel_w style repeated-or-pair fields
HW pair_field(const Node& p, const std::string& rep, const std::string& h, const std::string& w, long dflt) {
  HW r{dflt, dflt};
  auto reps = p.all(rep);
  if (reps.size() == 1) r.h = r.w = atol(reps[0]->value.c_str());
  else if (reps.size() >= 2) { r.h = atol(reps[0]->value.c_str()); r.w = atol(reps[1]->value.c_str()); }
  if (p.first(h)) r.h = p.integer(h, dflt);
  if (p.first(w)) r.w = p.integer(w, dflt);
  return r;
}

bool net_layout(const Node& net, SolverSpec* spec, std::string* err) {
  std::map<std::string, Shape> blobs;
  spec->counts.clear();
  spec->lr_mult.clear();
  spec->decay_mult.clear();
  spec->blob_names.clear();
  spec->layer_names.clear();
  spec->layer_types.clear();
  spec->shapes.clear();
  spec->net_name = net.str("name");
  // legacy "input:" / "input_shape" / "input_dim" net-level inputs
  {
    auto inputs = net.all("input");
    auto shapes = net.all("input_shape");
    auto dims = net.all("input_dim");
    for (size_t i = 0; i < inputs.size(); ++i) {
      Shape s;
      if (i < shapes.size()) for (const Node* d : shapes[i]->all("dim")) s.push_back(atol(d->value.c_str()));
      else for (size_t k = 4 * i; k < 4 * i + 4 && k < dims.size(); ++k) s.push_back(atol(dims[k]->value.c_str()));
      blobs[inputs[i]->value] = s;
    }
  }
  auto layers = net.all("layer");
  if (layers.empty() && !net.all("layers").empty()) {
    *err = "V1 'layers' net definitions are not supported";
    return false;
  }
  bool first_data = true;
  for (const Node* L : layers) {
    if (!in_train_phase(*L)) continue;
    const std::string type = L->str("type");
    const std::string name = L->str("name");
    std::vector<std::string> bottoms, tops;
    for (const Node* b : L->all("bottom")) bottoms.push_back(b->value);
    for (const Node* t : L->all("top")) tops.push_back(t->value);
    auto bottom_shape = [&](size_t i, Shape* s) -> bool {
      if (i >= bottoms.size() || !blobs.count(bottoms[i])) {
        *err = "layer '" + name + "' (" + type + "): unknown bottom blob";
        return false;
      }
      *s = blobs[bottoms[i]];
      return true;
    };
    std::vector<long> param_counts;  // learnable blobs this layer owns, in order
    std::vector<std::vector<int64_t>> param_shapes;
    if (type == "MemoryData") {
      const Node* p = L->first("memory_data_param");
      if (!p) { *err = "MemoryData layer without memory_data_param"; return false; }
      Shape s{p->integer("batch_size", 0), p->integer("channels", 0), p->integer("height", 0), p->integer("width", 0)};
      if (!tops.empty()) blobs[tops[0]] = s;
      if (tops.size() > 1) blobs[tops[1]] = Shape{s[0]};
      if (first_data) { spec->batch_size = static_cast<int>(s[0]); spec->input_shape.assign(s.begin(), s.end()); first_data = false; }
    } else if (type == "CoSData") {
      const Node* p = L->first("cos_data_param");
      if (!p) { *err = "CoSData layer without cos_data_param"; return false; }
      long batch = p->integer("batch_size", 0);
      auto tb = p->all("top");
      for (size_t i = 0; i < tops.size(); ++i) {
        Shape s{batch};
        if (i < tb.size()) {
          long c = tb[i]->integer("out_channels", 0), h = tb[i]->integer("out_height", 0), w = tb[i]->integer("out_width", 0);
          if (!c) c = tb[i]->integer("channels", 0);
          if (!h) h = tb[i]->integer("height", 0);
          if (!w) w = tb[i]->integer("width", 0);
          long axes = tb[i]->integer("sample_num_axes", 3);
          Shape full{c, h, w};
          for (long a = 0; a < axes && a < 3; ++a) s.push_back(full[a] ? full[a] : 1);
        }
        blobs[tops[i]] = s;
        if (first_data && i == 0) { spec->batch_size = static_cast<int>(batch); spec->input_shape.assign(s.begin(), s.end()); first_data = false; }
      }
    } else if (type == "Input") {
      const Node* p = L->first("input_param");
      auto shapes = p ? p->all("shape") : std::vector<const Node*>();
      for (size_t i = 0; i < tops.size(); ++i) {
        Shape s;
        const Node* sh = shapes.empty() ? nullptr : shapes[std::min(i, shapes.size() - 1)];
        if (sh) for (const Node* d : sh->all("dim")) s.push_back(atol(d->value.c_str()));
        blobs[tops[i]] = s;
        if (first_data && i == 0 && !s.empty()) { spec->batch_size = static_cast<int>(s[0]); spec->input_shape.assign(s.begin(), s.end()); first_data = false; }
      }
    } else if (type == "Convolution" || type == "Deconvolution") {
      const Node* p = L->first("convolution_param");
      Shape in;
      if (!p || !bottom_shape(0, &in) || in.size() != 4) { if (err->empty()) *err = "layer '" + name + "': bad Convolution"; return false; }
      long nout = p->integer("num_output", 0), group = p->integer("group", 1);
      HW k = pair_field(*p, "kernel_size", "kernel_h", "kernel_w", 0);
      HW st = pair_field(*p, "stride", "stride_h", "stride_w", 1);
      HW pad = pair_field(*p, "pad", "pad_h", "pad_w", 0);
      HW dil = pair_field(*p, "dilation", "dilation_h", "dilation_w", 1);
      bool bias = p->boolean("bias_term", true);
      if (nout <= 0 || k.h <= 0 || k.w <= 0 || group <= 0 || in[1] % group || nout % group || st.h <= 0 || st.w <= 0 ||
          dil.h <= 0 || dil.w <= 0 || pad.h < 0 || pad.w < 0) {
        *err = "layer '" + name + "': bad convolution_param";
        return false;
      }
      Shape out(4);
      out[0] = in[0];
      if (type == "Convolution") {
        param_counts.push_back(nout * (in[1] / group) * k.h * k.w);  // conv_layer / base_conv_layer.cpp weight shape
        param_shapes.push_back({nout, in[1] / group, k.h, k.w});
        out[1] = nout;
        out[2] = (in[2] + 2 * pad.h - (dil.h * (k.h - 1) + 1)) / st.h + 1;
        out[3] = (in[3] + 2 * pad.w - (dil.w * (k.w - 1) + 1)) / st.w + 1;
      } else {
        param_counts.push_back(in[1] * (nout / group) * k.h * k.w);
        param_shapes.push_back({in[1], nout / group, k.h, k.w});
        out[1] = nout;
        out[2] = st.h * (in[2] - 1) + (dil.h * (k.h - 1) + 1) - 2 * pad.h;
        out[3] = st.w * (in[3] - 1) + (dil.w * (k.w - 1) + 1) - 2 * pad.w;
      }
      if (bias) {
        param_counts.push_back(nout);
        param_shapes.push_back({nout});
      }
      if (!tops.empty()) blobs[tops[0]] = out;
    } else if (type == "Pooling") {
      const Node* p = L->first("pooling_param");
      Shape in;
      if (!p || !bottom_shape(0, &in) || in.size() != 4) { if (err->empty()) *err = "layer '" + name + "': bad Pooling"; return false; }
      HW k = pair_field(*p, "kernel_size", "kernel_h", "kernel_w", 0);
      HW st = pair_field(*p, "stride", "stride_h", "stride_w", 1);
      HW pad = pair_field(*p, "pad", "pad_h", "pad_w", 0);
      if (p->boolean("global_pooling", false)) { k.h = in[2]; k.w = in[3]; }
      if (k.h <= 0 || k.w <= 0 || st.h <= 0 || st.w <= 0 || pad.h < 0 || pad.w < 0) {
        *err = "layer '" + name + "': bad pooling_param";
        return false;
      }
      // pooling_layer.cpp: ceil((H + 2p - k) / s) + 1, clipped so the last window starts inside
      long oh = static_cast<long>(ceil(static_cast<float>(in[2] + 2 * pad.h - k.h) / st.h)) + 1;
      long ow = static_cast<long>(ceil(static_cast<float>(in[3] + 2 * pad.w - k.w) / st.w)) + 1;
      if (pad.h || pad.w) {
        if ((oh - 1) * st.h >= in[2] + pad.h) --oh;
        if ((ow - 1) * st.w >= in[3] + pad.w) --ow;
      }
      for (const std::string& t : tops) blobs[t] = Shape{in[0], in[1], oh, ow};
    } else if (type == "InnerProduct") {
      const Node* p = L->first("inner_product_param");
      Shape in;
      if (!p || !bottom_shape(0, &in)) { if (err->empty()) *err = "layer '" + name + "': bad InnerProduct"; return false; }
      long nout = p->integer("num_output", 0);
      long axis = p->integer("axis", 1);
      if (axis < 0) axis += static_cast<long>(in.size());
      if (nout <= 0 || axis < 0 || axis > static_cast<long>(in.size())) { *err = "layer '" + name + "': bad inner_product_param"; return false; }
      param_counts.push_back(nout * prod(in, static_cast<size_t>(axis)));
      param_shapes.push_back({nout, prod(in, static_cast<size_t>(axis))});  // inner_product_layer.cpp: N x K
      if (p->boolean("bias_term", true)) {
        param_counts.push_back(nout);
        param_shapes.push_back({nout});
      }
      Shape out(in.begin(), in.begin() + axis);
      out.push_back(nout);
      if (!tops.empty()) blobs[tops[0]] = out;
    } else if (type == "ReLU" || type == "LRN" || type == "Dropout" || type == "Sigmoid" || type == "TanH" ||
               type == "Softmax" || type == "Power" || type == "AbsVal" || type == "BNLL" || type == "ELU" ||
               type == "Exp" || type == "Log" || type == "Threshold" || type == "Split" || type == "Eltwise") {
      Shape in;
      if (!bottom_shape(0, &in)) return false;
      for (const std::string& t : tops) blobs[t] = in;
    } else if (type == "Flatten") {
      Shape in;
      if (!bottom_shape(0, &in) || in.empty()) return false;
      if (!tops.empty()) blobs[tops[0]] = Shape{in[0], prod(in, 1)};
    } else if (type == "Concat") {
      Shape out;
      if (!bottom_shape(0, &out)) return false;
      const Node* p = L->first("concat_param");
      long axis = p ? p->integer("axis", 1) : 1;
      if (axis < 0) axis += static_cast<long>(out.size());
      for (size_t i = 1; i < bottoms.size(); ++i) {
        Shape s;
        if (!bottom_shape(i, &s) || s.size() != out.size()) return false;
        out[axis] += s[axis];
      }
      if (!tops.empty()) blobs[tops[0]] = out;
    } else if (type == "SoftmaxWithLoss" || type == "Accuracy" || type == "EuclideanLoss" ||
               type == "SigmoidCrossEntropyLoss" || type == "HingeLoss" || type == "MultinomialLogisticLoss") {
      for (const std::string& t : tops) blobs[t] = Shape{};
    } else if (type == "Silence") {
    } else {
      *err = "layer '" + name + "' of type '" + type +
             "' is not understood by the layout parser; pass the layout with cos_net_allocate_desc";
      return false;
    }
    auto pspecs = L->all("param");
    for (size_t i = 0; i < param_counts.size(); ++i) {
      spec->counts.push_back(param_counts[i]);
      // ParamSpec defaults lr_mult = 1, decay_mult = 1 (caffe.proto:297-304)
      spec->lr_mult.push_back(i < pspecs.size() ? static_cast<float>(pspecs[i]->num("lr_mult", 1.0)) : 1.0f);
      spec->decay_mult.push_back(i < pspecs.size() ? static_cast<float>(pspecs[i]->num("decay_mult", 1.0)) : 1.0f);
      spec->blob_names.push_back(name + "." + std::to_string(i));
      spec->layer_names.push_back(name);
      spec->layer_types.push_back(type);
      spec->shapes.push_back(param_shapes[i]);
    }
  }
  return true;
}

}  // namespace

bool parse_net_prototxt_text(const std::string& text, SolverSpec* spec, std::string* err) {
  Node net;
  TextParser tp(text);
  if (!tp.parse(&net, err)) return false;
  return net_layout(net, spec, err);
}

bool parse_solver_prototxt(const std::string& solver_path, SolverSpec* spec, std::string* err) {
  std::string text;
  if (!read_file(solver_path, &text)) {
    *err = "cannot read solver file '" + solver_path + "'";
    return false;
  }
  Node s;
  TextParser tp(text);
  if (!tp.parse(&s, err)) return false;
  spec->lr_policy = s.str("lr_policy", "fixed");
  spec->base_lr = static_cast<float>(s.num("base_lr", 0.0));
  spec->gamma = static_cast<float>(s.num("gamma", 0.0));
  spec->power = static_cast<float>(s.num("power", 0.0));
  spec->stepsize = static_cast<int>(s.integer("stepsize", 0));
  spec->stepvalues.clear();
  for (const Node* v : s.all("stepvalue")) spec->stepvalues.push_back(atoi(v->value.c_str()));
  spec->max_iter = static_cast<int>(s.integer("max_iter", 0));
  spec->momentum = static_cast<float>(s.num("momentum", 0.0));
  spec->weight_decay = static_cast<float>(s.num("weight_decay", 0.0));
  // repeated test_iter: the reference reads test_iter(0) (CaffeNet.cpp getTestIter)
  spec->test_iter = static_cast<int>(s.integer("test_iter", 0));
  spec->test_interval = static_cast<int>(s.integer("test_interval", 0));
  spec->snapshot_prefix = s.str("snapshot_prefix", "");
  spec->regularization_type = s.str("regularization_type", "L2");
  spec->iter_size = static_cast<int>(s.integer("iter_size", 1));
  spec->clip_gradients = static_cast<float>(s.num("clip_gradients", -1.0));
  spec->solver_mode_gpu = s.str("solver_mode", "GPU") != "CPU";
  spec->snapshot_hdf5 = s.str("snapshot_format", "BINARYPROTO") == "HDF5";
  std::string type = s.str("type", "");
  if (type.empty()) {  // deprecated enum field solver_type (caffe.proto SolverType), upgraded to the type name
    type = s.str("solver_type", "SGD");
    for (int k = 0; k < 5; ++k)
      if (type == kSolverEnums[k]) type = kSolverNames[k];
  }
  spec->type = type;
  spec->delta = static_cast<float>(s.num("delta", 1e-8));
  spec->rms_decay = static_cast<float>(s.num("rms_decay", 0.0));
  if (!validate_solver(*spec, err)) return false;
  if (spec->regularization_type != "L2" && spec->regularization_type != "L1") {
    *err = "Unknown regularization type: " + spec->regularization_type;  // sgd_solver.cpp:169-171
    return false;
  }
  if (spec->iter_size != 1) {
    *err = "iter_size != 1 is not supported";
    return false;
  }
  if (spec->clip_gradients >= 0.f) {
    *err = "clip_gradients is not supported";
    return false;
  }
  // locate the net definition
  if (const Node* inl = s.first("net_param") ? s.first("net_param") : s.first("train_net_param")) {
    return net_layout(*inl, spec, err);
  }
  std::string net_path = s.str("net", "");
  if (net_path.empty()) net_path = s.str("train_net", "");
  if (net_path.empty()) {
    *err = "solver file names no net (net / train_net / net_param)";
    return false;
  }
  std::string net_text;
  bool ok = read_file(net_path, &net_text);
  if (!ok) {  // relative to the solver file's directory, then by basename there
    size_t slash = solver_path.find_last_of('/');
    std::string dir = slash == std::string::npos ? "." : solver_path.substr(0, slash);
    ok = read_file(dir + "/" + net_path, &net_text);
    if (!ok) {
      size_t s2 = net_path.find_last_of('/');
      if (s2 != std::string::npos) ok = read_file(dir + "/" + net_path.substr(s2 + 1), &net_text);
    }
  }
  if (!ok) {
    *err = "cannot read net file '" + net_path + "' named by '" + solver_path + "'";
    return false;
  }
  return parse_net_prototxt_text(net_text, spec, err);
}

}  // namespace cosb
