// ONNX graph loader for the CLAP audio encoder: protobuf wire-format reader + graph-driven lowering.
//
// The reference creates an onnxruntime session straight from CLAP_AUDIO_MODEL_PATH
// (tasks/clap_analyzer.py:109-116, external-data fallback :132-147) and feeds it
// {'mel_spectrogram': f32[1,1,n_mels,T]} (:534).  The file comes out of
// torch.onnx.export(opset 17, do_constant_folding=True) (student_clap/models/student_onnx_model.py:611-626).
// am_clap_load() accepts that file directly: this translation unit reads the ModelProto by hand (there is no
// protobuf / onnx dependency in the image) and lowers the node list to the engine's layer program
// (model_spec.cuh).  Nothing about the architecture is assumed: the walk follows the graph's data flow and maps
//
//   Squeeze / Unsqueeze / Transpose / BatchNormalization / Pad on the input      -> an input VIEW (axis order + per-mel affine)
//   Conv on the view (Cin = 1)                                                   -> kConvFirst (kStem when it is the
//                                                                                    rank-1 3x3 stride-2 separable stem)
//   Conv 1x1 / depthwise KxK / BatchNormalization / Clip / Relu / HardSwish / Add -> kPointwise / kDepthwise with the
//                                                                                    activation and the residual fused
//   GlobalAveragePool|ReduceMean -> Conv -> Relu -> Conv -> HardSigmoid|Sigmoid -> Mul   -> kSqueezeExcite
//   [Conv 1x1 stride s ->] ReduceMean|GlobalAveragePool (+ Flatten / Squeeze / Reshape)  -> kVecPool (+ kVecLinear)
//   MatMul / Gemm / Add / Mul / Erf-GELU / LayerNorm (op or decomposed) / ReduceL2-normalise / unary ops -> head program
//
// and rejects everything else with the node's name and operator in am_last_error().
#include "common.cuh"
#include "model_spec.cuh"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <map>
#include <memory>
#include <set>

#include "onnx_proto.cuh"

namespace am {
namespace {

// ------------------------------------------------------------------------------------------- lowering
enum ValKind { kView, kAct, kStridedPw, kVec, kShape };

struct Val {
  int kind = kAct;
  // kView: logical axis -> axis of the graph input [B, 1, n_mels, T] (or -1 for an inserted unit axis)
  std::vector<int> perm;
  std::vector<float> sc, sh;                  // per-mel affine applied so far (empty: identity)
  int pad_t = 0, pad_b = 0, pad_l = 0, pad_r = 0;  // explicit Pad waiting for its convolution
  // kAct: a trunk activation.  layer = index of the layer that wrote it (-1: none yet)
  int layer = -1, channels = 0;
  // kStridedPw: 1x1 convolution with stride > 1 over an activation, waiting for the spatial mean
  std::vector<float> w, bias;
  int stride = 1, cout = 0;
  // kVec
  int reg = -1, dim = 0;
};

#define LOWER_FAIL(node, ...)                                                                     \
  do {                                                                                            \
    char _b[512];                                                                                 \
    std::snprintf(_b, sizeof _b, __VA_ARGS__);                                                    \
    set_error("onnx: cannot lower node '%s' (%s): %s", (node).name.empty() ? (node).out[0].c_str() : (node).name.c_str(), \
              (node).op.c_str(), _b);                                                             \
    return AM_ERR_INVALID;                                                                        \
  } while (0)

struct Lowerer {
  OGraph& g;
  ModelSpec& spec;
  std::map<std::string, Val> vals;
  std::map<std::string, std::vector<int>> consumers;
  std::map<std::string, const OTensor*> consts;
  std::vector<std::unique_ptr<OTensor>> owned;
  std::vector<std::string> layer_input;  // value name each emitted layer reads
  std::string cur;                        // value name of the trunk's latest activation
  std::set<std::string> graph_outputs;

  Lowerer(OGraph& g_, ModelSpec& s_) : g(g_), spec(s_) {}

  const OTensor* cst(const std::string& name) const {
    auto it = consts.find(name);
    return it == consts.end() ? nullptr : it->second;
  }
  const OTensor* cin(const ONode& n, size_t idx) const { return idx < n.in.size() && !n.in[idx].empty() ? cst(n.in[idx]) : nullptr; }
  // the single consumer of a value (or -1 when it has several / is a graph output)
  int sole_consumer(const std::string& name) const {
    auto it = consumers.find(name);
    if (it == consumers.end() || it->second.size() != 1 || graph_outputs.count(name)) return -1;
    return it->second[0];
  }
  static int64_t attr_i(const ONode& n, const char* k, int64_t dflt) {
    auto it = n.attrs.find(k);
    return it != n.attrs.end() && it->second.has_i ? it->second.i : dflt;
  }
  static float attr_f(const ONode& n, const char* k, float dflt) {
    auto it = n.attrs.find(k);
    return it != n.attrs.end() && it->second.has_f ? it->second.f : dflt;
  }
  static std::vector<int64_t> attr_ints(const ONode& n, const char* k) {
    auto it = n.attrs.find(k);
    return it != n.attrs.end() ? it->second.ints : std::vector<int64_t>();
  }
  // integer list given as attribute `k` (older opsets / torch's serializer) or as constant input `idx`
  bool ints_of(const ONode& n, const char* k, size_t idx, std::vector<int64_t>* out) const {
    if (const OTensor* t = cin(n, idx)) {
      out->clear();
      for (size_t q = 0; q < t->count(); ++q) out->push_back((int64_t)t->at(q));
      return true;
    }
    auto it = n.attrs.find(k);
    if (it == n.attrs.end()) return false;
    *out = it->second.ints;
    return true;
  }
  bool scalar_of(const ONode& n, const char* k, size_t idx, float* out) const {
    if (const OTensor* t = cin(n, idx)) {
      if (t->count() != 1) return false;
      *out = (float)t->at(0);
      return true;
    }
    auto it = n.attrs.find(k);
    if (it == n.attrs.end() || !it->second.has_f) return false;
    *out = it->second.f;
    return true;
  }
  int new_reg(int dim) {
    spec.reg_dim.push_back(dim);
    return spec.n_regs++;
  }
  // a block starts at the first layer and after every linear 1x1 projection
  bool rule_block_start(size_t i) const {
    if (i == 0 || i >= spec.layers.size()) return false;
    if (i == 1) return true;
    const LayerSpec& p = spec.layers[i - 1];
    return p.type == kPointwise && p.act == kActNone;
  }
  void alias(const ONode& n, const std::string& src) { vals[n.out[0]] = vals[src]; if (cur == src) cur = n.out[0]; }

  // activation kind of a node applied elementwise, or -1
  int act_of(const ONode& n) const {
    if (n.op == "Relu") return kActRelu;
    if (n.op == "HardSwish") return kActHardSwish;
    if (n.op == "Sigmoid") return kActSigmoid;
    if (n.op == "Tanh") return kActTanh;
    if (n.op == "HardSigmoid") {
      const float a = attr_f(n, "alpha", 0.2f), b = attr_f(n, "beta", 0.5f);
      return (std::fabs(a - 1.0f / 6.0f) < 1e-6f && std::fabs(b - 0.5f) < 1e-6f) ? kActHardSigmoid : -1;
    }
    if (n.op == "Clip") {
      float lo = -INFINITY, hi = INFINITY;
      const bool has_lo = scalar_of(n, "min", 1, &lo), has_hi = scalar_of(n, "max", 2, &hi);
      if (has_lo && lo == 0.f && has_hi && hi == 6.f) return kActRelu6;
      if (has_lo && lo == 0.f && (!has_hi || std::isinf(hi))) return kActRelu;
      return -1;
    }
    return -1;
  }

  int run();
  int lower_view_op(ONode& n, const Val& v);
  int lower_conv(ONode& n);
  int lower_trunk_pool(ONode& n, int ni);
  int lower_vec(ONode& n, int ni);
  int finish();
};

static bool is_spatial_axes(const std::vector<int64_t>& axes) {
  if (axes.size() != 2) return false;
  const int64_t a = axes[0] < 0 ? axes[0] + 4 : axes[0], b = axes[1] < 0 ? axes[1] + 4 : axes[1];
  return (a == 2 && b == 3) || (a == 3 && b == 2);
}

int Lowerer::lower_view_op(ONode& n, const Val& v) {
  Val o = v;
  if (n.op == "Squeeze") {
    std::vector<int64_t> axes;
    if (!ints_of(n, "axes", 1, &axes)) LOWER_FAIL(n, "Squeeze without constant axes");
    std::vector<int> keep;
    const int r = (int)v.perm.size();
    std::set<int> drop;
    for (int64_t a : axes) drop.insert((int)(a < 0 ? a + r : a));
    for (int q = 0; q < r; ++q) {
      if (!drop.count(q)) keep.push_back(v.perm[q]);
      else if (v.perm[q] != 1 && v.perm[q] != -1) LOWER_FAIL(n, "squeezes axis %d of the input, which is not a unit axis", v.perm[q]);
    }
    o.perm = keep;
  } else if (n.op == "Unsqueeze") {
    std::vector<int64_t> axes;
    if (!ints_of(n, "axes", 1, &axes)) LOWER_FAIL(n, "Unsqueeze without constant axes");
    const int r = (int)v.perm.size() + (int)axes.size();
    std::set<int> ins;
    for (int64_t a : axes) ins.insert((int)(a < 0 ? a + r : a));
    std::vector<int> p;
    size_t src = 0;
    for (int q = 0; q < r; ++q) p.push_back(ins.count(q) ? -1 : v.perm[src++]);
    o.perm = p;
  } else if (n.op == "Transpose") {
    const std::vector<int64_t> perm = attr_ints(n, "perm");
    if (perm.size() != v.perm.size()) LOWER_FAIL(n, "perm of rank %zu on a rank-%zu view", perm.size(), v.perm.size());
    for (size_t q = 0; q < perm.size(); ++q) o.perm[q] = v.perm[(size_t)perm[q]];
  } else if (n.op == "BatchNormalization") {
    if (v.perm.size() < 2) LOWER_FAIL(n, "rank-%zu input", v.perm.size());
    const OTensor *ga = cin(n, 1), *be = cin(n, 2), *mu = cin(n, 3), *var = cin(n, 4);
    if (!ga || !be || !mu || !var) LOWER_FAIL(n, "non-constant statistics");
    const float eps = attr_f(n, "epsilon", 1e-5f);
    const int ax = v.perm[1];
    const size_t c = ga->count();
    if (v.pad_t || v.pad_b || v.pad_l || v.pad_r) LOWER_FAIL(n, "normalisation after an explicit Pad");
    if (ax == 2) {  // per-mel statistics (PhiNet bn0, student_onnx_model.py:49-51)
      if ((int)c != spec.n_mels && spec.n_mels) LOWER_FAIL(n, "%zu channels on a %d-bin mel axis", c, spec.n_mels);
      spec.n_mels = (int)c;
      std::vector<float> sc(c), sh(c);
      for (size_t q = 0; q < c; ++q) {
        const double s = (double)ga->f[q] / std::sqrt((double)var->f[q] + eps);
        sc[q] = (float)s;
        sh[q] = (float)((double)be->f[q] - (double)mu->f[q] * s);
      }
      if (o.sc.empty()) {
        o.sc = sc;
        o.sh = sh;
      } else {
        for (size_t q = 0; q < c; ++q) {
          o.sh[q] = o.sh[q] * sc[q] + sh[q];
          o.sc[q] = o.sc[q] * sc[q];
        }
      }
    } else if ((ax == 1 || ax == -1) && c == 1) {  // scalar affine over the single input channel
      const double s = (double)ga->f[0] / std::sqrt((double)var->f[0] + eps);
      const double t = (double)be->f[0] - (double)mu->f[0] * s;
      if (o.sc.empty()) {
        if (!spec.n_mels) LOWER_FAIL(n, "mel width still unknown");
        o.sc.assign((size_t)spec.n_mels, 1.f);
        o.sh.assign((size_t)spec.n_mels, 0.f);
      }
      for (size_t q = 0; q < o.sc.size(); ++q) {
        o.sh[q] = (float)(o.sh[q] * s + t);
        o.sc[q] = (float)(o.sc[q] * s);
      }
    } else {
      LOWER_FAIL(n, "normalises input axis %d (only the mel axis or the unit channel are supported)", ax);
    }
  } else if (n.op == "Pad") {
    std::vector<int64_t> pads;
    if (!ints_of(n, "pads", 1, &pads) || pads.size() != 8) LOWER_FAIL(n, "needs 8 constant pads on a rank-4 view");
    float val = 0.f;
    scalar_of(n, "value", 2, &val);
    auto it = n.attrs.find("mode");
    if ((it != n.attrs.end() && it->second.s != "constant") || val != 0.f) LOWER_FAIL(n, "only constant zero padding");
    if (pads[0] || pads[1] || pads[4] || pads[5]) LOWER_FAIL(n, "pads batch / channel axes");
    o.pad_t += (int)pads[2];
    o.pad_l += (int)pads[3];
    o.pad_b += (int)pads[6];
    o.pad_r += (int)pads[7];
  } else {
    LOWER_FAIL(n, "operator not supported on the input view");
  }
  vals[n.out[0]] = o;
  return AM_OK;
}

int Lowerer::lower_conv(ONode& n) {
  const Val& v = vals[n.in[0]];
  const OTensor* w = cin(n, 1);
  const OTensor* b = cin(n, 2);
  if (!w || w->dims.size() != 4) LOWER_FAIL(n, "weights must be a constant rank-4 tensor");
  const int cout = (int)w->dims[0], cin_g = (int)w->dims[1], kh = (int)w->dims[2], kw = (int)w->dims[3];
  const int group = (int)attr_i(n, "group", 1);
  std::vector<int64_t> strides = attr_ints(n, "strides"), pads = attr_ints(n, "pads"), dil = attr_ints(n, "dilations");
  if (strides.empty()) strides = {1, 1};
  if (pads.empty()) pads = {0, 0, 0, 0};
  for (int64_t d : dil)
    if (d != 1) LOWER_FAIL(n, "dilated convolution");
  auto ap = n.attrs.find("auto_pad");
  if (ap != n.attrs.end() && !ap->second.s.empty() && ap->second.s != "NOTSET") LOWER_FAIL(n, "auto_pad %s", ap->second.s.c_str());
  if (strides[0] != strides[1]) LOWER_FAIL(n, "anisotropic stride %lld x %lld", (long long)strides[0], (long long)strides[1]);
  std::vector<float> bias((size_t)cout, 0.f);
  if (b) {
    if ((int)b->count() != cout) LOWER_FAIL(n, "bias of %zu for %d channels", b->count(), cout);
    bias = b->f;
  }
  if (v.kind == kView) {
    if (v.perm.size() != 4 || v.perm[0] != 0 || (v.perm[1] != 1 && v.perm[1] != -1) || cin_g != 1 || group != 1)
      LOWER_FAIL(n, "first convolution needs a [B, 1, H, W] view of the input (got rank %zu, Cin %d)", v.perm.size(), cin_g);
    const bool h_time = v.perm[2] == 3 && v.perm[3] == 2, h_mel = v.perm[2] == 2 && v.perm[3] == 3;
    if (!h_time && !h_mel) LOWER_FAIL(n, "spatial axes of the view are not the (mel, time) axes of the input");
    if (kh > 7 || kw > 7) LOWER_FAIL(n, "%d x %d kernel", kh, kw);
    LayerSpec L;
    L.type = kConvFirst;
    L.cin = 1;
    L.cout = cout;
    L.kh = kh;
    L.kw = kw;
    L.stride = (int)strides[0];
    L.pad_t = v.pad_t + (int)pads[0];
    L.pad_l = v.pad_l + (int)pads[1];
    L.pad_b = v.pad_b + (int)pads[2];
    L.pad_r = v.pad_r + (int)pads[3];
    L.h_is_time = h_time ? 1 : 0;
    L.aux0 = v.sc;
    L.aux1 = v.sh;
    L.w = w->f;
    L.bias = bias;
    spec.layers.push_back(std::move(L));
    layer_input.push_back(n.in[0]);
  } else if (v.kind == kAct) {
    if (n.in[0] != cur) LOWER_FAIL(n, "reads '%s', which is not the trunk's latest activation ('%s')", n.in[0].c_str(), cur.c_str());
    const int C = v.channels;
    if (group == 1 && kh == 1 && kw == 1) {
      if (cin_g != C) LOWER_FAIL(n, "expects %d input channels, the trunk carries %d", cin_g, C);
      for (int64_t p : pads)
        if (p) LOWER_FAIL(n, "padded 1x1 convolution");
      // the separable stem: Conv(1 -> 1, KxK) immediately followed by Conv(1 -> C, 1x1): one rank-1 first convolution
      if (!spec.layers.empty() && spec.layers.back().type == kConvFirst && spec.layers.size() == 1 &&
          spec.layers.back().cout == 1 && spec.layers.back().act == kActNone && strides[0] == 1 && C == 1) {
        LayerSpec& F = spec.layers.back();
        const std::vector<float> k0 = F.w;
        const float b0 = F.bias[0];
        const int taps = F.kh * F.kw;
        F.aux2.assign(w->f.begin(), w->f.end());  // rank-1 factor (kept for the kStem fast path)
        F.aux2.insert(F.aux2.end(), k0.begin(), k0.end());
        F.w.assign((size_t)cout * taps, 0.f);
        F.bias.assign((size_t)cout, 0.f);
        for (int c = 0; c < cout; ++c) {
          for (int t = 0; t < taps; ++t) F.w[(size_t)c * taps + t] = w->f[c] * k0[t];
          F.bias[c] = w->f[c] * b0 + bias[c];
        }
        F.cout = cout;
        vals[n.out[0]].kind = kAct;
        vals[n.out[0]].layer = 0;
        vals[n.out[0]].channels = cout;
        cur = n.out[0];
        return AM_OK;
      }
      if (strides[0] != 1) {  // only as "1x1 stride-s conv -> spatial mean" (the mean commutes with the conv)
        Val o;
        o.kind = kStridedPw;
        o.w = w->f;
        o.bias = bias;
        o.stride = (int)strides[0];
        o.cout = cout;
        o.channels = C;
        vals[n.out[0]] = o;
        return AM_OK;
      }
      LayerSpec L;
      L.type = kPointwise;
      L.cin = C;
      L.cout = cout;
      L.w = w->f;
      L.bias = bias;
      spec.layers.push_back(std::move(L));
      layer_input.push_back(n.in[0]);
    } else if (group == C && cin_g == 1 && cout == C) {
      if (kh != kw || kh > 7 || !(kh & 1)) LOWER_FAIL(n, "%d x %d depthwise kernel", kh, kw);
      if (strides[0] != 1 && strides[0] != 2) LOWER_FAIL(n, "depthwise stride %lld", (long long)strides[0]);
      LayerSpec L;
      L.type = kDepthwise;
      L.cin = L.cout = C;
      L.kh = kh;
      L.kw = kw;
      L.stride = (int)strides[0];
      L.pad_t = v.pad_t + (int)pads[0];
      L.pad_l = v.pad_l + (int)pads[1];
      L.pad_b = v.pad_b + (int)pads[2];
      L.pad_r = v.pad_r + (int)pads[3];
      L.w = w->f;
      L.bias = bias;
      spec.layers.push_back(std::move(L));
      layer_input.push_back(n.in[0]);
    } else {
      LOWER_FAIL(n, "convolution with group %d, %d -> %d channels, %d x %d kernel is neither 1x1 nor depthwise", group,
                 cin_g * group, cout, kh, kw);
    }
  } else {
    LOWER_FAIL(n, "input is not an activation");
  }
  Val o;
  o.kind = kAct;
  o.layer = (int)spec.layers.size() - 1;
  o.channels = cout;
  vals[n.out[0]] = o;
  cur = n.out[0];
  return AM_OK;
}

// GlobalAveragePool / ReduceMean over (H, W): squeeze-excite gate or the head's pooling
int Lowerer::lower_trunk_pool(ONode& n, int ni) {
  const Val v = vals[n.in[0]];
  bool keep = true;
  if (n.op != "GlobalAveragePool") {
    std::vector<int64_t> axes;
    if (!ints_of(n, "axes", 1, &axes) || !is_spatial_axes(axes)) LOWER_FAIL(n, "reduction is not over the two spatial axes");
    keep = attr_i(n, "keepdims", 1) != 0;
  }
  // ---- squeeze-excite: pool -> Conv -> act -> Conv -> gate -> Mul(x, gate)
  if (v.kind == kAct && keep && n.in[0] == cur) {
    do {
      const int c1 = sole_consumer(n.out[0]);
      if (c1 < 0 || g.nodes[c1].op != "Conv") break;
      ONode& f1 = g.nodes[c1];
      const int a1 = sole_consumer(f1.out[0]);
      if (a1 < 0) break;
      const int inner = act_of(g.nodes[a1]);
      if (inner != kActRelu && inner != kActHardSwish && inner != kActRelu6) break;
      const int c2 = sole_consumer(g.nodes[a1].out[0]);
      if (c2 < 0 || g.nodes[c2].op != "Conv") break;
      ONode& f2 = g.nodes[c2];
      const int a2 = sole_consumer(f2.out[0]);
      if (a2 < 0) break;
      const int gate = act_of(g.nodes[a2]);
      if (gate != kActHardSigmoid && gate != kActSigmoid) break;
      const int mu = sole_consumer(g.nodes[a2].out[0]);
      if (mu < 0 || g.nodes[mu].op != "Mul") break;
      ONode& mul = g.nodes[mu];
      const std::string& other = mul.in[0] == g.nodes[a2].out[0] ? mul.in[1] : mul.in[0];
      if (other != n.in[0]) break;
      const OTensor *w1 = cin(f1, 1), *b1 = cin(f1, 2), *w2 = cin(f2, 1), *b2 = cin(f2, 2);
      const int C = v.channels;
      if (!w1 || !w2 || w1->dims.size() != 4 || w2->dims.size() != 4 || w1->dims[2] != 1 || w1->dims[3] != 1 ||
          w2->dims[2] != 1 || w2->dims[3] != 1 || (int)w1->dims[1] != C || (int)w2->dims[0] != C || w1->dims[0] != w2->dims[1])
        LOWER_FAIL(n, "squeeze-excite gate with unexpected weight shapes");
      LayerSpec L;
      L.type = kSqueezeExcite;
      L.cin = L.cout = C;
      L.cmid = (int)w1->dims[0];
      L.act = inner;
      L.gate_act = gate;
      L.w = w1->f;
      L.bias = b1 ? b1->f : std::vector<float>((size_t)L.cmid, 0.f);
      L.aux0 = w2->f;
      L.aux1 = b2 ? b2->f : std::vector<float>((size_t)C, 0.f);
      spec.layers.push_back(std::move(L));
      layer_input.push_back(n.in[0]);
      for (int q : {ni, c1, a1, c2, a2, mu}) g.nodes[q].done = true;
      Val o;
      o.kind = kAct;
      o.layer = (int)spec.layers.size() - 1;
      o.channels = C;
      vals[mul.out[0]] = o;
      cur = mul.out[0];
      return AM_OK;
    } while (false);
  }
  // ---- head pooling
  VecOp p;
  p.kind = kVecPool;
  p.stride = v.kind == kStridedPw ? v.stride : 1;
  p.N = v.channels;
  p.dst = new_reg(v.channels);
  if (v.kind == kAct && n.in[0] != cur) LOWER_FAIL(n, "pools '%s', which is not the trunk's latest activation", n.in[0].c_str());
  if (!spec.head.empty()) LOWER_FAIL(n, "second spatial pooling");
  spec.head.push_back(p);
  int reg = p.dst, dim = v.channels;
  if (v.kind == kStridedPw) {
    VecOp l;
    l.kind = kVecLinear;
    l.a = reg;
    l.K = v.channels;
    l.N = v.cout;
    l.w = v.w;
    l.bias = v.bias;
    l.dst = new_reg(v.cout);
    spec.head.push_back(l);
    reg = l.dst;
    dim = v.cout;
  }
  Val o;
  o.kind = kVec;
  o.reg = reg;
  o.dim = dim;
  vals[n.out[0]] = o;
  cur.clear();
  return AM_OK;
}

static bool close_to(double a, double b, double tol = 1e-5) { return std::fabs(a - b) <= tol * std::max(1.0, std::fabs(b)); }

int Lowerer::lower_vec(ONode& n, int ni) {
  auto vec_in = [&](size_t idx) -> const Val* {
    if (idx >= n.in.size()) return nullptr;
    auto it = vals.find(n.in[idx]);
    return it != vals.end() && it->second.kind == kVec ? &it->second : nullptr;
  };
  auto emit = [&](VecOp op, int dim) {
    op.dst = new_reg(dim);
    if (!op.N) op.N = dim;
    spec.head.push_back(op);
    Val o;
    o.kind = kVec;
    o.reg = op.dst;
    o.dim = dim;
    return o;
  };
  const Val* x0 = vec_in(0);
  const Val* x1 = vec_in(1);
  const std::string& op = n.op;
  if (op == "Flatten" || op == "Reshape" || op == "Squeeze" || op == "Unsqueeze" || op == "Identity" || op == "Dropout") {
    if (!x0) LOWER_FAIL(n, "input is not a pooled feature row");
    vals[n.out[0]] = *x0;  // [B, C, 1, 1] <-> [B, C]: same register
    return AM_OK;
  }
  if (op == "MatMul" || op == "Gemm") {
    const OTensor* w = cin(n, 1);
    if (!x0 || !w || w->dims.size() != 2) LOWER_FAIL(n, "needs (feature rows) x (constant matrix)");
    const bool tb = op == "Gemm" && attr_i(n, "transB", 0) != 0;
    if (op == "Gemm" && (attr_i(n, "transA", 0) != 0 || attr_f(n, "alpha", 1.f) != 1.f || attr_f(n, "beta", 1.f) != 1.f))
      LOWER_FAIL(n, "Gemm with transA / alpha / beta");
    const int K = (int)(tb ? w->dims[1] : w->dims[0]), N = (int)(tb ? w->dims[0] : w->dims[1]);
    if (K != x0->dim) LOWER_FAIL(n, "matrix expects %d inputs, the row has %d", K, x0->dim);
    VecOp l;
    l.kind = kVecLinear;
    l.a = x0->reg;
    l.K = K;
    l.N = N;
    l.w.resize((size_t)N * K);
    for (int o = 0; o < N; ++o)
      for (int k = 0; k < K; ++k) l.w[(size_t)o * K + k] = tb ? w->f[(size_t)o * K + k] : w->f[(size_t)k * N + o];
    if (op == "Gemm") {
      if (const OTensor* b = cin(n, 2)) {
        if ((int)b->count() != N) LOWER_FAIL(n, "bias of %zu for %d outputs", b->count(), N);
        l.bias = b->f;
      }
    }
    vals[n.out[0]] = emit(l, N);
    return AM_OK;
  }
  if (op == "LayerNormalization") {
    const OTensor *ga = cin(n, 1), *be = cin(n, 2);
    if (!x0 || !ga || (int)ga->count() != x0->dim) LOWER_FAIL(n, "needs a feature row and a constant scale of its width");
    VecOp l;
    l.kind = kVecLayerNorm;
    l.a = x0->reg;
    l.eps = attr_f(n, "epsilon", 1e-5f);
    l.w = ga->f;
    l.bias = be ? be->f : std::vector<float>((size_t)x0->dim, 0.f);
    vals[n.out[0]] = emit(l, x0->dim);
    return AM_OK;
  }
  int act = act_of(n);
  if (act >= 0 && x0) {
    std::string act_out = n.out[0];
    if (act == kActHardSigmoid) {  // x * HardSigmoid(x) == HardSwish(x)
      const int mu = sole_consumer(n.out[0]);
      if (mu >= 0 && g.nodes[mu].op == "Mul" && (g.nodes[mu].in[0] == n.in[0] || g.nodes[mu].in[1] == n.in[0])) {
        act = kActHardSwish;
        act_out = g.nodes[mu].out[0];
        g.nodes[mu].done = true;
      }
    }
    VecOp u;
    u.kind = kVecUnary;
    u.a = x0->reg;
    u.act = act;
    vals[act_out] = emit(u, x0->dim);
    return AM_OK;
  }
  // ---- GELU, exact form: x * 0.5 * (1 + erf(x / sqrt(2)))  exported as Div, Erf, Add, Mul, Mul
  if (op == "Div" && x0 && cin(n, 1) && cin(n, 1)->count() == 1 && close_to(cin(n, 1)->at(0), std::sqrt(2.0), 1e-4)) {
    do {
      int er = -1;
      for (int c : consumers[n.out[0]])
        if (g.nodes[c].op == "Erf") er = c;
      if (er < 0 || consumers[n.out[0]].size() != 1) break;
      const int ad = sole_consumer(g.nodes[er].out[0]);
      if (ad < 0 || g.nodes[ad].op != "Add") break;
      const OTensor* one = cin(g.nodes[ad], 1) ? cin(g.nodes[ad], 1) : cin(g.nodes[ad], 0);
      if (!one || one->count() != 1 || !close_to(one->at(0), 1.0)) break;
      const int m1 = sole_consumer(g.nodes[ad].out[0]);
      if (m1 < 0 || g.nodes[m1].op != "Mul") break;
      const std::string& xin = g.nodes[m1].in[0] == g.nodes[ad].out[0] ? g.nodes[m1].in[1] : g.nodes[m1].in[0];
      if (xin != n.in[0]) break;
      const int m2 = sole_consumer(g.nodes[m1].out[0]);
      if (m2 < 0 || g.nodes[m2].op != "Mul") break;
      const OTensor* half = cin(g.nodes[m2], 1) ? cin(g.nodes[m2], 1) : cin(g.nodes[m2], 0);
      if (!half || half->count() != 1 || !close_to(half->at(0), 0.5)) break;
      VecOp u;
      u.kind = kVecUnary;
      u.a = x0->reg;
      u.act = kActGelu;
      vals[g.nodes[m2].out[0]] = emit(u, x0->dim);
      for (int q : {ni, er, ad, m1, m2}) g.nodes[q].done = true;
      return AM_OK;
    } while (false);
    LOWER_FAIL(n, "division by sqrt(2) that is not part of an exact-GELU pattern");
  }
  // ---- LayerNorm, decomposed: ReduceMean, Sub, Pow 2, ReduceMean, Add eps, Sqrt, Div, Mul g, Add b
  if (op == "ReduceMean" && x0) {
    do {
      std::vector<int64_t> axes;
      if (!ints_of(n, "axes", 1, &axes) || axes.size() != 1 || (axes[0] != -1 && axes[0] != 1)) break;
      int sb = -1;
      for (int c : consumers[n.out[0]])
        if (g.nodes[c].op == "Sub" && g.nodes[c].in[0] == n.in[0]) sb = c;
      if (sb < 0 || consumers[n.out[0]].size() != 1) break;
      const std::string& cen = g.nodes[sb].out[0];
      int pw = -1, dv = -1;
      for (int c : consumers[cen]) {
        if (g.nodes[c].op == "Pow") pw = c;
        if (g.nodes[c].op == "Div" && g.nodes[c].in[0] == cen) dv = c;
      }
      if (pw < 0 || dv < 0 || consumers[cen].size() != 2) break;
      const OTensor* two = cin(g.nodes[pw], 1);
      if (!two || two->count() != 1 || !close_to(two->at(0), 2.0)) break;
      const int rm = sole_consumer(g.nodes[pw].out[0]);
      if (rm < 0 || g.nodes[rm].op != "ReduceMean") break;
      const int ae = sole_consumer(g.nodes[rm].out[0]);
      if (ae < 0 || g.nodes[ae].op != "Add") break;
      const OTensor* eps = cin(g.nodes[ae], 1) ? cin(g.nodes[ae], 1) : cin(g.nodes[ae], 0);
      if (!eps || eps->count() != 1) break;
      const int sq = sole_consumer(g.nodes[ae].out[0]);
      if (sq < 0 || g.nodes[sq].op != "Sqrt") break;
      if (sole_consumer(g.nodes[sq].out[0]) != dv) break;
      VecOp l;
      l.kind = kVecLayerNorm;
      l.a = x0->reg;
      l.eps = (float)eps->at(0);
      l.w.assign((size_t)x0->dim, 1.f);
      l.bias.assign((size_t)x0->dim, 0.f);
      std::vector<int> used = {ni, sb, pw, rm, ae, sq, dv};
      std::string out = g.nodes[dv].out[0];
      const int mg = sole_consumer(out);
      if (mg >= 0 && g.nodes[mg].op == "Mul") {
        const OTensor* ga = cin(g.nodes[mg], 1) ? cin(g.nodes[mg], 1) : cin(g.nodes[mg], 0);
        if (ga && (int)ga->count() == x0->dim) {
          l.w = ga->f;
          used.push_back(mg);
          out = g.nodes[mg].out[0];
          const int ab = sole_consumer(out);
          if (ab >= 0 && g.nodes[ab].op == "Add") {
            const OTensor* be = cin(g.nodes[ab], 1) ? cin(g.nodes[ab], 1) : cin(g.nodes[ab], 0);
            if (be && (int)be->count() == x0->dim) {
              l.bias = be->f;
              used.push_back(ab);
              out = g.nodes[ab].out[0];
            }
          }
        }
      }
      vals[out] = emit(l, x0->dim);
      for (int q : used) g.nodes[q].done = true;
      return AM_OK;
    } while (false);
    LOWER_FAIL(n, "row mean that is not part of a LayerNorm pattern");
  }
  // ---- F.normalize: ReduceL2(keepdims) -> Clip(min eps) -> [Expand(., Shape(x))] -> Div(x, .)
  if (op == "ReduceL2" && x0) {
    do {
      std::vector<int64_t> axes;
      if (!ints_of(n, "axes", 1, &axes) || axes.size() != 1 || (axes[0] != -1 && axes[0] != 1)) break;
      int at = sole_consumer(n.out[0]);
      float eps = 0.f;
      std::vector<int> used = {ni};
      if (at >= 0 && g.nodes[at].op == "Clip") {
        if (!scalar_of(g.nodes[at], "min", 1, &eps)) break;
        used.push_back(at);
        at = sole_consumer(g.nodes[at].out[0]);
      }
      if (at >= 0 && g.nodes[at].op == "Expand") {
        used.push_back(at);
        at = sole_consumer(g.nodes[at].out[0]);
      }
      if (at < 0 || g.nodes[at].op != "Div" || g.nodes[at].in[0] != n.in[0]) break;
      used.push_back(at);
      VecOp l;
      l.kind = kVecL2Norm;
      l.a = x0->reg;
      l.eps2 = eps;
      vals[g.nodes[at].out[0]] = emit(l, x0->dim);
      for (int q : used) g.nodes[q].done = true;
      return AM_OK;
    } while (false);
    LOWER_FAIL(n, "row norm that is not part of an L2-normalise pattern");
  }
  if (op == "Add" && x0 && x1) {
    if (x0->dim != x1->dim) LOWER_FAIL(n, "adds rows of %d and %d", x0->dim, x1->dim);
    VecOp a;
    a.kind = kVecAdd;
    a.a = x0->reg;
    a.b = x1->reg;
    vals[n.out[0]] = emit(a, x0->dim);
    return AM_OK;
  }
  if ((op == "Add" || op == "Mul" || op == "Sub" || op == "Div") && (x0 || x1)) {
    const Val* x = x0 ? x0 : x1;
    const OTensor* c = cin(n, x0 ? 1 : 0);
    if (!c || (c->count() != 1 && (int)c->count() != x->dim)) LOWER_FAIL(n, "second operand is neither a feature row nor a constant of its width");
    if (!x0 && (op == "Sub" || op == "Div")) LOWER_FAIL(n, "constant %s row", op == "Sub" ? "minus" : "over");
    VecOp a;
    a.kind = kVecAffine;
    a.a = x->reg;
    std::vector<float> cv((size_t)x->dim);
    for (int q = 0; q < x->dim; ++q) cv[q] = (float)c->at(c->count() == 1 ? 0 : q);
    if (op == "Add") a.bias = cv;
    else if (op == "Sub") {
      for (float& f : cv) f = -f;
      a.bias = cv;
    } else if (op == "Mul") a.w = cv;
    else {
      for (float& f : cv) f = 1.0f / f;
      a.w = cv;
    }
    vals[n.out[0]] = emit(a, x->dim);
    return AM_OK;
  }
  if (op == "Shape") {
    Val o;
    o.kind = kShape;
    vals[n.out[0]] = o;
    return AM_OK;
  }
  LOWER_FAIL(n, "operator is not supported in the head (inputs are%s feature rows)", x0 ? "" : " not");
}

int Lowerer::run() {
  if (g.inputs.size() != 1) {
    set_error("onnx: the encoder graph must have exactly one input (found %zu)", g.inputs.size());
    return AM_ERR_INVALID;
  }
  if (g.outputs.empty()) {
    set_error("onnx: the graph has no output");
    return AM_ERR_INVALID;
  }
  for (const auto& o : g.outputs) graph_outputs.insert(o);
  for (auto& kv : g.init) consts[kv.first] = &kv.second;
  for (size_t i = 0; i < g.nodes.size(); ++i)
    for (const auto& in : g.nodes[i].in)
      if (!in.empty()) consumers[in].push_back((int)i);
  {
    Val in;
    in.kind = kView;
    in.perm = {0, 1, 2, 3};
    vals[g.inputs[0]] = in;
  }
  // constants first: the pattern matchers look ahead of the node being lowered
  for (ONode& n : g.nodes) {
    if (n.op != "Constant" || n.out.empty()) continue;
    auto it = n.attrs.find("value");
    if (it != n.attrs.end() && it->second.has_t) {
      consts[n.out[0]] = &it->second.t;
      continue;
    }
    auto fi = n.attrs.find("value_float");
    auto ii = n.attrs.find("value_int");
    auto t = std::make_unique<OTensor>();
    if (fi != n.attrs.end() && fi->second.has_f) t->f.push_back(fi->second.f);
    else if (ii != n.attrs.end() && ii->second.has_i) {
      t->is_int = true;
      t->i.push_back(ii->second.i);
    } else LOWER_FAIL(n, "Constant without a tensor value");
    consts[n.out[0]] = t.get();
    owned.push_back(std::move(t));
  }
  for (size_t ni = 0; ni < g.nodes.size(); ++ni) {
    ONode& n = g.nodes[ni];
    if (n.done) continue;
    if (n.out.empty()) continue;
    if (n.op == "Constant") continue;  // registered by the pre-pass above
    if (n.in.empty() || n.in[0].empty()) LOWER_FAIL(n, "node without a data input");
    // which kind of value does it read?
    auto it0 = vals.find(n.in[0]);
    auto it1 = n.in.size() > 1 ? vals.find(n.in[1]) : vals.end();
    const bool in0 = it0 != vals.end(), in1 = it1 != vals.end();
    if (!in0 && !in1) LOWER_FAIL(n, "reads '%s', which no supported node produced", n.in[0].c_str());
    const Val& v = (in1 && !cur.empty() && n.in[1] == cur) ? it1->second : (in0 ? it0->second : it1->second);
    if (v.kind == kShape) {
      if (n.op == "Expand") continue;  // consumed by the L2-normalise pattern
      LOWER_FAIL(n, "shape arithmetic is only supported inside F.normalize");
    }
    if (v.kind == kVec || (in1 && it1->second.kind == kVec)) {
      AM_TRY(lower_vec(n, (int)ni));
      continue;
    }
    if (n.op == "Conv") {
      AM_TRY(lower_conv(n));
      continue;
    }
    if (v.kind == kView) {
      AM_TRY(lower_view_op(n, v));
      continue;
    }
    if (n.op == "GlobalAveragePool" || n.op == "ReduceMean") {
      AM_TRY(lower_trunk_pool(n, (int)ni));
      continue;
    }
    if (v.kind == kStridedPw) LOWER_FAIL(n, "a strided 1x1 convolution is only supported directly before the spatial mean");
    // ---- trunk activation ops
    if (n.op == "Identity" || n.op == "Dropout") {
      alias(n, n.in[0]);
      continue;
    }
    if (n.op == "Pad") {  // explicit padding before a depthwise convolution
      std::vector<int64_t> pads;
      if (!ints_of(n, "pads", 1, &pads) || pads.size() != 8 || pads[0] || pads[1] || pads[4] || pads[5])
        LOWER_FAIL(n, "needs 8 constant pads on the spatial axes");
      float val = 0.f;
      scalar_of(n, "value", 2, &val);
      if (val != 0.f) LOWER_FAIL(n, "non-zero pad value");
      Val o = v;
      o.pad_t += (int)pads[2];
      o.pad_l += (int)pads[3];
      o.pad_b += (int)pads[6];
      o.pad_r += (int)pads[7];
      vals[n.out[0]] = o;
      if (cur == n.in[0]) cur = n.out[0];
      continue;
    }
    if (n.in[0] != cur && !(n.in.size() > 1 && n.in[1] == cur))
      LOWER_FAIL(n, "reads '%s' while the trunk's latest activation is '%s' (only chain-structured trunks are supported)",
                 n.in[0].c_str(), cur.c_str());
    if (v.layer < 0 || v.layer != (int)spec.layers.size() - 1) LOWER_FAIL(n, "activation has no producing layer");
    LayerSpec& L = spec.layers[(size_t)v.layer];
    int act = act_of(n);
    std::string act_out = n.out[0];
    if (act == kActHardSigmoid) {  // HardSwish as exported by older symbolic functions: x * HardSigmoid(x)
      const int mu = sole_consumer(n.out[0]);
      if (mu >= 0 && g.nodes[mu].op == "Mul" && (g.nodes[mu].in[0] == n.in[0] || g.nodes[mu].in[1] == n.in[0])) {
        act = kActHardSwish;
        act_out = g.nodes[mu].out[0];
        g.nodes[mu].done = true;
      }
    }
    if (act >= 0) {
      if (act != kActRelu6 && act != kActRelu && act != kActHardSwish) LOWER_FAIL(n, "activation is not supported in the trunk");
      if (L.act != kActNone || L.residual || L.type == kSqueezeExcite) LOWER_FAIL(n, "second activation / activation after a residual add");
      L.act = act;
      vals[act_out] = vals[n.in[0]];
      if (cur == n.in[0]) cur = act_out;
      continue;
    }
    if (n.op == "BatchNormalization") {  // not folded by the exporter: fold it into the producing convolution
      const OTensor *ga = cin(n, 1), *be = cin(n, 2), *mu = cin(n, 3), *var = cin(n, 4);
      if (!ga || !be || !mu || !var || (int)ga->count() != L.cout) LOWER_FAIL(n, "statistics do not match %d channels", L.cout);
      if (L.act != kActNone || L.residual || L.type == kSqueezeExcite || L.type == kStem) LOWER_FAIL(n, "normalisation after an activation");
      const float eps = attr_f(n, "epsilon", 1e-5f);
      const size_t per = L.w.size() / (size_t)L.cout;
      for (int c = 0; c < L.cout; ++c) {
        const double s = (double)ga->f[c] / std::sqrt((double)var->f[c] + eps);
        for (size_t q = 0; q < per; ++q) L.w[(size_t)c * per + q] = (float)(L.w[(size_t)c * per + q] * s);
        L.bias[c] = (float)(L.bias[c] * s + ((double)be->f[c] - (double)mu->f[c] * s));
      }
      alias(n, n.in[0]);
      continue;
    }
    if (n.op == "Add" && in0 && in1 && it0->second.kind == kAct && it1->second.kind == kAct) {
      const std::string& other = n.in[0] == cur ? n.in[1] : n.in[0];
      if (L.type != kPointwise || L.act != kActNone || L.residual) LOWER_FAIL(n, "residual add must follow a linear 1x1 projection");
      // the residual source must be the input of the block this projection closes
      int bs = -1;
      for (int q = (int)spec.layers.size() - 1; q >= 1; --q)
        if (layer_input[(size_t)q] == other) {
          bs = q;
          break;
        }
      if (bs < 0) LOWER_FAIL(n, "residual source '%s' is not the input of an earlier layer", other.c_str());
      // the executor keeps ONE residual source: the input of the latest block-start layer (see finish())
      if (!rule_block_start((size_t)bs)) LOWER_FAIL(n, "residual source '%s' is not the input of a block", other.c_str());
      for (int q = bs + 1; q < (int)spec.layers.size(); ++q)
        if (rule_block_start((size_t)q)) LOWER_FAIL(n, "overlapping residual connections");
      if (vals[other].channels != L.cout) LOWER_FAIL(n, "residual of %d channels onto %d", vals[other].channels, L.cout);
      L.residual = 1;
      alias(n, cur);
      continue;
    }
    LOWER_FAIL(n, "operator is not supported on a trunk activation");
  }
  return finish();
}

int Lowerer::finish() {
  auto ito = vals.find(g.outputs[0]);
  if (ito == vals.end() || ito->second.kind != kVec) {
    set_error("onnx: graph output '%s' is not produced by the head program", g.outputs[0].c_str());
    return AM_ERR_INVALID;
  }
  if (spec.layers.empty() || spec.layers[0].type != kConvFirst) {
    set_error("onnx: the graph does not start with a convolution on the mel spectrogram");
    return AM_ERR_INVALID;
  }
  if (!spec.n_mels) spec.n_mels = 128;  // no per-mel statistics in the graph: the reference's fixed width (config.py:386)
  spec.emb = ito->second.dim;
  // block starts: first layer, and every layer that follows a linear projection (the fused-block matcher and the
  // executor's residual bookkeeping key on them)
  for (size_t i = 1; i < spec.layers.size(); ++i) spec.layers[i].block_start = rule_block_start(i) ? 1 : 0;
  // the separable PhiNet stem (bn0 + pad + 3x3 s2 + 1x1 + ReLU6) has a dedicated kernel
  {
    LayerSpec& F = spec.layers[0];
    if (F.kh == 3 && F.kw == 3 && F.stride == 2 && F.h_is_time && F.act == kActRelu6 && F.aux2.size() == (size_t)F.cout + 9) {
      LayerSpec S = F;
      S.type = kStem;
      S.w.assign(F.aux2.begin() + F.cout, F.aux2.end());  // dw[9]
      S.aux2.assign(F.aux2.begin(), F.aux2.begin() + F.cout);  // pw scale
      if (S.aux0.empty()) {
        S.aux0.assign((size_t)spec.n_mels, 1.f);
        S.aux1.assign((size_t)spec.n_mels, 0.f);
      }
      F = S;
    } else {
      F.aux2.clear();
    }
  }
  // ---- head peepholes
  std::vector<int> uses((size_t)spec.n_regs, 0);
  for (const VecOp& o : spec.head) {
    if (o.a >= 0) ++uses[(size_t)o.a];
    if (o.b >= 0) ++uses[(size_t)o.b];
  }
  const int out_reg = ito->second.reg;
  ++uses[(size_t)out_reg];
  auto producer = [&](int reg) -> int {
    for (size_t q = 0; q < spec.head.size(); ++q)
      if (spec.head[q].dst == reg) return (int)q;
    return -1;
  };
  // bias add after a bias-free linear
  for (size_t q = 0; q < spec.head.size(); ++q) {
    VecOp& o = spec.head[q];
    if (o.kind != kVecAffine || !o.w.empty() || o.bias.empty() || uses[(size_t)o.a] != 1) continue;
    const int p = producer(o.a);
    if (p < 0 || spec.head[(size_t)p].kind != kVecLinear || !spec.head[(size_t)p].bias.empty()) continue;
    spec.head[(size_t)p].bias = o.bias;
    spec.head[(size_t)p].dst = o.dst;
    spec.head.erase(spec.head.begin() + (long)q);
    --q;
  }
  // activation feeding only a linear: applied while the linear stages its input
  for (size_t q = 0; q < spec.head.size(); ++q) {
    VecOp& o = spec.head[q];
    if (o.kind != kVecLinear || o.act != kActNone || uses[(size_t)o.a] != 1) continue;
    const int p = producer(o.a);
    if (p < 0 || spec.head[(size_t)p].kind != kVecUnary) continue;
    o.act = spec.head[(size_t)p].act;
    o.a = spec.head[(size_t)p].a;
    spec.head.erase(spec.head.begin() + p);
    --q;
  }
  // Add -> LayerNorm -> L2 at the very end: one kernel
  if (spec.head.size() >= 3) {
    const size_t z = spec.head.size();
    VecOp &a = spec.head[z - 3], &l = spec.head[z - 2], &n2 = spec.head[z - 1];
    if (a.kind == kVecAdd && l.kind == kVecLayerNorm && n2.kind == kVecL2Norm && l.a == a.dst && n2.a == l.dst &&
        uses[(size_t)a.dst] == 1 && uses[(size_t)l.dst] == 1 && n2.dst == out_reg) {
      VecOp f;
      f.kind = kVecAddLnL2;
      f.a = a.a;
      f.b = a.b;
      f.dst = n2.dst;
      f.N = l.N;
      f.eps = l.eps;
      f.eps2 = n2.eps2;
      f.w = l.w;
      f.bias = l.bias;
      spec.head.resize(z - 3);
      spec.head.push_back(f);
    }
  }
  if (spec.head.empty() || spec.head.back().dst != out_reg) {
    set_error("onnx: the graph output is not the last value the head computes");
    return AM_ERR_INVALID;
  }
  return AM_OK;
}

}  // namespace

bool looks_like_onnx(const void* data, size_t nbytes) {
  if (!data || nbytes < 8 || std::memcmp(data, "AMW1", 4) == 0) return false;
  // a ModelProto starts with field 1 (ir_version, varint): key byte 0x08
  return ((const uint8_t*)data)[0] == 0x08;
}

int load_onnx_spec(const void* data, size_t nbytes, const char* path, ModelSpec* out) {
  OGraph g;
  AM_TRY(parse_model(data, nbytes, dir_of(path), &g));
  *out = ModelSpec{};
  Lowerer lw(g, *out);
  AM_TRY(lw.run());
  char src[128];
  std::snprintf(src, sizeof src, "ONNX (ir %lld, opset %lld, %zu nodes)", (long long)g.ir_version, (long long)g.opset, g.nodes.size());
  out->source = src;
  return AM_OK;
}

}  // namespace am
