// MusiCNN tower (tasks/analysis.py:324-573): ONNX lowering + sm_100a kernels.
//
// The reference runs two onnxruntime sessions per track: musicnn_embedding.onnx ([n, 187, 96] log-mel patches ->
// [n, 200] `model/dense/BiasAdd:0`) and musicnn_prediction.onnx ([n, 200] -> [n, 50] logits).  am_musicnn_load reads
// either file (onnx_proto.cuh) and lowers it to one of two programs:
//
//   embedding:  input scalar affine (BatchNorm on the single channel, applied where the patch is staged, i.e. before
//               the zero padding) -> front-end branches (Conv k_h x k_w on the input, ReLU, BatchNorm, max over
//               frequency; one tcgen05 implicit GEMM launch per branch, the frequency max in the epilogue, the
//               pre-pool tensor never leaves the SM) -> mid-end (7-tap convolutions over time: im2col + the tcgen05
//               GEMM with bias + ReLU, then BatchNorm + residual in a row pass) -> time max + mean pooling -> head row
//               program (BatchNorm affine, dense);
//   prediction: head row program only (ReLU, BatchNorm affine, dense).
//
// Two spellings of each graph are accepted: torch's exporter (Unsqueeze(1), BatchNormalization, Conv with pads or
// auto_pad SAME_*, ReduceMax over frequency, Conv1d mid-end, Gemm) and tf2onnx's (Unsqueeze(3) + Transpose NHWC ->
// NCHW, BatchNorm as constant Mul [+ Add], explicit Pad, MaxPool [1, W] + Squeeze over frequency, the mid-end as a
// Conv [cout, 1, k, C] over the Transpose + Unsqueeze + Pad image of the series, MatMul + Add).
//
// Every width comes from the graph (branch count, kernel sizes, filters, mid-end depth, dense widths).  BatchNorm
// after a ReLU is NOT folded into the convolution: a negative scale turns the max into a min, so it is applied per
// filter before the frequency max.
#include "common.cuh"
#include "gemm_tcgen05.cuh"
#include "model_spec.cuh"
#include "ptx_sm100.cuh"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <map>
#include <memory>
#include <set>

#include "onnx_proto.cuh"

namespace am {

// ------------------------------------------------------------------------------------------- program
struct MxBranch {
  int kh = 0, kw = 0, cout = 0, pad_top = 0, ch_off = 0;
  int pool_w = 0;                  // MaxPool [1, W] window (0: ReduceMax); must cover the whole frequency axis
  float in_s = 1.f, in_h = 0.f;    // input affine on the path into this branch
  std::vector<float> w;            // [cout, kh, kw]
  std::vector<float> bias, s, h;   // conv bias, BatchNorm scale / shift after the ReLU
};
struct MxMid {
  int cin = 0, cout = 0, k = 0, residual = 0;
  std::vector<float> w;            // [cout, cin, k]
  std::vector<float> bias, s, h;
};
struct MusicnnSpec {
  int is_embedding = 0;
  float in_s = 1.f, in_h = 0.f;
  std::vector<MxBranch> br;
  int c_front = 0;
  std::vector<MxMid> mid;
  std::vector<int> pool_segs;  // concat order of the pooled series: -1 = front-end output, j >= 0 = mid-end layer j
  int pool_max_first = 1;
  int in_dim = 0, out_dim = 0;  // prediction: row widths; embedding: out_dim = dense width
  std::vector<VecOp> head;      // row program on f32 [n, dim]; registers: 0 = program input
  std::vector<int> reg_dim;
  std::string source;
  std::string in_name, out_name;  // the graph's input / output tensor names
};

namespace {

#define MX_FAIL(node, ...)                                                                                         \
  do {                                                                                                             \
    char _b[512];                                                                                                  \
    std::snprintf(_b, sizeof _b, __VA_ARGS__);                                                                     \
    set_error("musicnn onnx: cannot lower node '%s' (%s): %s", (node).name.empty() ? (node).out[0].c_str()        \
                                                                                    : (node).name.c_str(),        \
              (node).op.c_str(), _b);                                                                              \
    return AM_ERR_INVALID;                                                                                         \
  } while (0)

enum MxKind { kMxIn, kMxBranch, kMxSeries, kMxMid, kMxPoolMax, kMxPoolMean, kMxVec };

// Series segment codes: -1 - b = front-end branch b; j = mid-end layer j after its residual add;
// kRaw + j = mid-end layer j's BatchNorm output (the same tensor as j when the layer has no residual)
constexpr int kRaw = 1000;

struct MxVal {
  int kind = kMxIn;
  // kMxIn: layout 0 = [n, T, F], 1 = [n, 1, T, F], 3 = [n, T, F, 1]; scalar affine applied so far; time padding
  int layout = 0, pad_t = 0, pad_b = 0;
  float s = 1.f, h = 0.f;
  // kMxBranch / kMxMid: index + stage (0 conv, 1 relu, 2 normalised); mul_open: normalised by a Mul whose shift
  // Add may follow
  int idx = -1, stage = 0;
  bool mul_open = false;
  // kMxBranch / kMxMid / kMxSeries: a trailing unit axis waiting for its Squeeze
  int r4 = 0;
  // kMxSeries / pools: segments; tmaj: [n, T, C]; img: [n, 1, T, C] (+ time padding in pad_t / pad_b)
  std::vector<int> segs;
  int tmaj = 0, img = 0;
  // kMxVec
  int reg = -1, dim = 0;
};

struct MxLowerer {
  OGraph& g;
  MusicnnSpec& spec;
  std::map<std::string, MxVal> vals;
  std::map<std::string, const OTensor*> consts;
  std::set<int> raw_used;  // mid-end layers whose pre-residual output is read
  MxLowerer(OGraph& g_, MusicnnSpec& s_) : g(g_), spec(s_) {}

  const OTensor* cst(const ONode& n, size_t i) const {
    if (i >= n.in.size() || n.in[i].empty()) return nullptr;
    auto it = consts.find(n.in[i]);
    return it == consts.end() ? nullptr : it->second;
  }
  static int64_t attr_i(const ONode& n, const char* k, int64_t d) {
    auto it = n.attrs.find(k);
    return it != n.attrs.end() && it->second.has_i ? it->second.i : d;
  }
  static float attr_f(const ONode& n, const char* k, float d) {
    auto it = n.attrs.find(k);
    return it != n.attrs.end() && it->second.has_f ? it->second.f : d;
  }
  static std::vector<int64_t> attr_ints(const ONode& n, const char* k) {
    auto it = n.attrs.find(k);
    return it != n.attrs.end() ? it->second.ints : std::vector<int64_t>();
  }
  bool ints_of(const ONode& n, const char* k, size_t idx, std::vector<int64_t>* out) const {
    if (const OTensor* t = cst(n, idx)) {
      out->clear();
      for (size_t q = 0; q < t->count(); ++q) out->push_back((int64_t)t->at(q));
      return true;
    }
    auto it = n.attrs.find(k);
    if (it == n.attrs.end()) return false;
    *out = it->second.ints;
    return true;
  }
  bool one_axis(const ONode& n, int want, int rank) const {
    std::vector<int64_t> axes;
    if (!ints_of(n, "axes", 1, &axes) || axes.size() != 1) return false;
    return (axes[0] < 0 ? axes[0] + rank : axes[0]) == want;
  }
  int new_reg(int dim) {
    spec.reg_dim.push_back(dim);
    return (int)spec.reg_dim.size() - 1;
  }
  // BatchNormalization statistics -> per-channel scale / shift
  int bn_affine(const ONode& n, std::vector<float>* s, std::vector<float>* h) const {
    const OTensor *ga = cst(n, 1), *be = cst(n, 2), *mu = cst(n, 3), *var = cst(n, 4);
    if (!ga || !be || !mu || !var) MX_FAIL(n, "non-constant statistics");
    const double eps = attr_f(n, "epsilon", 1e-5f);
    const size_t c = ga->count();
    s->resize(c);
    h->resize(c);
    for (size_t q = 0; q < c; ++q) {
      const double sc = ga->at(q) / std::sqrt(var->at(q) + eps);
      (*s)[q] = (float)sc;
      (*h)[q] = (float)(be->at(q) - mu->at(q) * sc);
    }
    return AM_OK;
  }
  // a constant operand of Mul / Add that broadcasts per channel over axis 1 of a value with `c` channels
  const OTensor* per_channel(const ONode& n, int c) const {
    const OTensor* t = cst(n, 1);
    if (!t || (int)t->count() != c || t->is_int) return nullptr;
    for (size_t d = 0; d < t->dims.size(); ++d)
      if (t->dims[d] != 1 && !(t->dims[d] == c && (d == 1 || t->dims.size() == 1))) return nullptr;
    return t;
  }
  int seg_of(int code) {
    if (code >= kRaw) {
      raw_used.insert(code - kRaw);
      return code - kRaw;
    }
    return code;
  }
  int series_channels(const std::vector<int>& segs) const {
    int c = 0;
    for (int sg : segs) c += sg < 0 ? spec.br[(size_t)(-1 - sg)].cout : spec.mid[(size_t)(sg % kRaw)].cout;
    return c;
  }
  int emit_vec(const ONode& n, VecOp op, int dim) {
    op.dst = new_reg(dim);
    spec.head.push_back(std::move(op));
    MxVal v;
    v.kind = kMxVec;
    v.reg = spec.head.back().dst;
    v.dim = dim;
    vals[n.out[0]] = v;
    return AM_OK;
  }
  int conv_front(ONode& n, const MxVal& v);
  int conv_mid(ONode& n, const MxVal& v);
  int stage_op(ONode& n, const MxVal& v);
  int series_op(ONode& n, MxVal v);
  int node(ONode& n);
  int run();
};

int MxLowerer::conv_front(ONode& n, const MxVal& v) {
  const OTensor* w = cst(n, 1);
  const OTensor* b = cst(n, 2);
  if (v.layout != 1 || !w || w->dims.size() != 4 || w->dims[1] != 1)
    MX_FAIL(n, "front-end convolution must take the single-channel [n, 1, time, mel] input with constant rank-4 weights");
  if (attr_i(n, "group", 1) != 1) MX_FAIL(n, "grouped convolution");
  for (int64_t s : attr_ints(n, "strides"))
    if (s != 1) MX_FAIL(n, "strided convolution");
  for (int64_t d : attr_ints(n, "dilations"))
    if (d != 1) MX_FAIL(n, "dilated convolution");
  MxBranch br;
  br.cout = (int)w->dims[0];
  br.kh = (int)w->dims[2];
  br.kw = (int)w->dims[3];
  int pt = v.pad_t, pb = v.pad_b;
  auto ap = n.attrs.find("auto_pad");
  const std::string aps = ap != n.attrs.end() ? ap->second.s : std::string();
  if (aps == "SAME_UPPER" || aps == "SAME_LOWER") {
    const int tot = br.kh - 1;
    if (br.kw != 1) MX_FAIL(n, "same padding along frequency");
    pt += aps == "SAME_UPPER" ? tot / 2 : tot - tot / 2;
    pb += aps == "SAME_UPPER" ? tot - tot / 2 : tot / 2;
  } else if (!aps.empty() && aps != "NOTSET" && aps != "VALID") {
    MX_FAIL(n, "auto_pad %s", aps.c_str());
  } else {
    const std::vector<int64_t> p = attr_ints(n, "pads");
    if (!p.empty()) {
      if (p.size() != 4 || p[1] || p[3]) MX_FAIL(n, "pads along frequency");
      pt += (int)p[0];
      pb += (int)p[2];
    }
  }
  if (pt + pb != br.kh - 1) MX_FAIL(n, "time padding %d + %d does not keep the %d-tap output as long as the input", pt, pb, br.kh);
  if (br.kh > 256 || br.kw > 384) MX_FAIL(n, "kernel %dx%d too large", br.kh, br.kw);
  br.pad_top = pt;
  br.in_s = v.s;
  br.in_h = v.h;
  br.w = w->f;
  br.bias.assign((size_t)br.cout, 0.f);
  if (b) br.bias = b->f;
  spec.br.push_back(std::move(br));
  MxVal o;
  o.kind = kMxBranch;
  o.idx = (int)spec.br.size() - 1;
  vals[n.out[0]] = o;
  return AM_OK;
}

// mid-end convolution over time: Conv1d [cout, cin, k] on a [n, C, T] series, or Conv2d [cout, 1, k, C] on the padded
// [n, 1, T, C] image of one
int MxLowerer::conv_mid(ONode& n, const MxVal& v) {
  const OTensor* w = cst(n, 1);
  const OTensor* b = cst(n, 2);
  if (attr_i(n, "group", 1) != 1) MX_FAIL(n, "grouped convolution");
  for (int64_t s : attr_ints(n, "strides"))
    if (s != 1) MX_FAIL(n, "strided convolution");
  for (int64_t d : attr_ints(n, "dilations"))
    if (d != 1) MX_FAIL(n, "dilated convolution");
  auto ap = n.attrs.find("auto_pad");
  if (ap != n.attrs.end() && !ap->second.s.empty() && ap->second.s != "NOTSET" && ap->second.s != "VALID")
    MX_FAIL(n, "auto_pad %s on a mid-end convolution", ap->second.s.c_str());
  const int C = series_channels(v.segs);
  MxMid m;
  int pt = 0, pb = 0;
  const std::vector<int64_t> p = attr_ints(n, "pads");
  if (!v.img) {
    if (v.tmaj || v.r4 || !w || w->dims.size() != 3) MX_FAIL(n, "mid-end convolution needs a [n, C, T] series and constant [cout, cin, k] weights");
    m.cout = (int)w->dims[0];
    m.cin = (int)w->dims[1];
    m.k = (int)w->dims[2];
    if (!p.empty() && p.size() != 2) MX_FAIL(n, "pads of rank %zu", p.size());
    pt = p.empty() ? 0 : (int)p[0];
    pb = p.empty() ? 0 : (int)p[1];
    m.w = w->f;
  } else {
    if (!w || w->dims.size() != 4 || w->dims[1] != 1) MX_FAIL(n, "mid-end convolution over the (time, channel) image needs constant [cout, 1, k, C] weights");
    m.cout = (int)w->dims[0];
    m.k = (int)w->dims[2];
    m.cin = (int)w->dims[3];
    if (!p.empty() && (p.size() != 4 || p[1] || p[3])) MX_FAIL(n, "pads along channels");
    pt = v.pad_t + (p.empty() ? 0 : (int)p[0]);
    pb = v.pad_b + (p.empty() ? 0 : (int)p[2]);
    m.w.assign((size_t)m.cout * m.cin * m.k, 0.f);
    for (int o = 0; o < m.cout; ++o)
      for (int t = 0; t < m.k; ++t)
        for (int c = 0; c < m.cin; ++c)
          m.w[((size_t)o * m.cin + c) * m.k + t] = w->f[((size_t)o * m.k + t) * m.cin + c];
  }
  if (m.k % 2 == 0 || pt != (m.k - 1) / 2 || pb != (m.k - 1) / 2)
    MX_FAIL(n, "mid-end convolution must be odd-sized with symmetric zero padding that keeps its length (k=%d, pads %d/%d)", m.k, pt, pb);
  if (m.cin != C) MX_FAIL(n, "%d input channels on a %d-channel series", m.cin, C);
  const size_t j = spec.mid.size();
  bool ok = true;
  if (j == 0) {
    ok = v.segs.size() == spec.br.size();
    for (size_t q = 0; ok && q < v.segs.size(); ++q) ok = v.segs[q] == -1 - (int)q;
  } else {
    ok = v.segs.size() == 1 && v.segs[0] % kRaw == (int)j - 1 && v.segs[0] >= 0;
    if (ok) seg_of(v.segs[0]);
  }
  if (!ok) MX_FAIL(n, "mid-end layer %zu must read %s", j, j == 0 ? "the concatenated front-end branches" : "the previous mid-end output");
  m.bias.assign((size_t)m.cout, 0.f);
  if (b) m.bias = b->f;
  spec.mid.push_back(std::move(m));
  MxVal o;
  o.kind = kMxMid;
  o.idx = (int)j;
  o.r4 = v.img;
  vals[n.out[0]] = o;
  return AM_OK;
}

// Relu -> BatchNormalization | Mul [-> Add] after a front-end or mid-end convolution, and the front-end frequency max
int MxLowerer::stage_op(ONode& n, const MxVal& v) {
  MxVal o = v;
  const bool is_mid = v.kind == kMxMid;
  const int c = is_mid ? spec.mid[(size_t)v.idx].cout : spec.br[(size_t)v.idx].cout;
  std::vector<float>& S = is_mid ? spec.mid[(size_t)v.idx].s : spec.br[(size_t)v.idx].s;
  std::vector<float>& H = is_mid ? spec.mid[(size_t)v.idx].h : spec.br[(size_t)v.idx].h;
  const std::string& op = n.op;
  o.mul_open = false;
  if (op == "Relu" && v.stage == 0) {
    o.stage = 1;
  } else if (op == "BatchNormalization" && v.stage == 1) {
    std::vector<float> s, h;
    AM_TRY(bn_affine(n, &s, &h));
    if ((int)s.size() != c) MX_FAIL(n, "%zu statistics for %d filters", s.size(), c);
    S = s;
    H = h;
    o.stage = 2;
  } else if (op == "Mul" && v.stage == 1) {
    const OTensor* t = per_channel(n, c);
    if (!t) MX_FAIL(n, "a normalisation Mul needs a constant per-filter scale of %d", c);
    S = t->f;
    H.assign((size_t)c, 0.f);
    o.stage = 2;
    o.mul_open = true;
  } else if (op == "Add" && v.stage == 2 && v.mul_open && per_channel(n, c)) {
    const OTensor* t = per_channel(n, c);
    for (int q = 0; q < c; ++q) H[(size_t)q] += t->f[(size_t)q];
  } else if (!is_mid && v.stage == 2 && (op == "ReduceMax" || op == "MaxPool")) {
    if (op == "ReduceMax") {
      if (!one_axis(n, 3, 4)) MX_FAIL(n, "the front-end pool must reduce the frequency axis 3");
      o.r4 = (int)attr_i(n, "keepdims", 1);
    } else {
      const std::vector<int64_t> k = attr_ints(n, "kernel_shape"), pads = attr_ints(n, "pads");
      if (k.size() != 2 || k[0] != 1) MX_FAIL(n, "the front-end pool must be a [1, W] window over frequency");
      for (int64_t q : pads)
        if (q) MX_FAIL(n, "padded max pool");
      if (attr_i(n, "ceil_mode", 0)) MX_FAIL(n, "ceil_mode");
      spec.br[(size_t)v.idx].pool_w = (int)k[1];
      o.r4 = 1;
    }
    o.kind = kMxSeries;
    o.segs = {-1 - v.idx};
  } else if (is_mid && v.stage == 2) {
    // the normalised mid-end output is a series from here on
    o.kind = kMxSeries;
    o.segs = {kRaw + v.idx};
    return series_op(n, o);
  } else {
    MX_FAIL(n, "unexpected after the %s convolution (expected Relu -> BatchNormalization or Mul [-> Add]%s)",
            is_mid ? "mid-end" : "front-end", is_mid ? "" : " -> ReduceMax / MaxPool over frequency");
  }
  vals[n.out[0]] = o;
  return AM_OK;
}

int MxLowerer::series_op(ONode& n, MxVal v) {
  const std::string& op = n.op;
  MxVal o = v;
  if (op == "Squeeze") {
    if (!v.r4 || !one_axis(n, 3, 4)) MX_FAIL(n, "only the trailing unit axis 3 may be squeezed from a series");
    o.r4 = 0;
    vals[n.out[0]] = o;
    return AM_OK;
  }
  if (op == "Conv") return conv_mid(n, v);
  if (v.r4) MX_FAIL(n, "a series with a trailing unit axis (squeeze it first)");
  if (op == "Transpose") {
    const std::vector<int64_t> perm = attr_ints(n, "perm");
    if (v.tmaj || v.img || perm != std::vector<int64_t>{0, 2, 1}) MX_FAIL(n, "only [n, C, T] -> [n, T, C] is supported on a series");
    o.tmaj = 1;
  } else if (op == "Unsqueeze") {
    if (!v.tmaj || v.img || !one_axis(n, 1, 4)) MX_FAIL(n, "only a [n, T, C] series may gain the unit axis 1");
    o.img = 1;
  } else if (op == "Pad") {
    std::vector<int64_t> pads;
    if (!v.img || !ints_of(n, "pads", 1, &pads) || pads.size() != 8) MX_FAIL(n, "needs 8 constant pads on a [n, 1, T, C] image");
    auto it = n.attrs.find("mode");
    if (it != n.attrs.end() && it->second.s != "constant") MX_FAIL(n, "only constant zero padding");
    if (const OTensor* c = cst(n, 2))
      if (c->count() && c->at(0) != 0.0) MX_FAIL(n, "only zero padding");
    if (pads[0] || pads[1] || pads[3] || pads[4] || pads[5] || pads[7]) MX_FAIL(n, "pads an axis other than time");
    o.pad_t += (int)pads[2];
    o.pad_b += (int)pads[6];
  } else if (v.tmaj || v.img) {
    MX_FAIL(n, "operator not supported on a time-major series");
  } else if (op == "Concat") {
    if (attr_i(n, "axis", 0) != 1) MX_FAIL(n, "concatenates axis %lld, not channels", (long long)attr_i(n, "axis", 0));
    o.segs.clear();
    for (const auto& in : n.in) {
      auto it = vals.find(in);
      MxVal u = it == vals.end() ? MxVal() : it->second;
      if (u.kind == kMxMid && u.stage == 2) {
        u.kind = kMxSeries;
        u.segs = {kRaw + u.idx};
      }
      if (it == vals.end() || u.kind != kMxSeries || u.r4 || u.tmaj || u.img)
        MX_FAIL(n, "input '%s' is not a [n, C, T] channel series", in.c_str());
      o.segs.insert(o.segs.end(), u.segs.begin(), u.segs.end());
    }
  } else if (op == "Add") {
    // BatchNorm(ReLU(conv(x))) + x: the residual of a mid-end layer
    auto it = n.in.size() == 2 ? vals.find(n.in[1]) : vals.end();
    if (it == vals.end()) MX_FAIL(n, "residual operand missing");
    MxVal u = it->second;
    if (u.kind == kMxMid && u.stage == 2) {
      u.kind = kMxSeries;
      u.segs = {kRaw + u.idx};
    }
    const int j = (int)spec.mid.size() - 1;
    const MxVal *a = &v, *r = &u;
    if (!(a->segs.size() == 1 && a->segs[0] == kRaw + j)) std::swap(a, r);
    if (j < 1 || a->kind != kMxSeries || a->segs.size() != 1 || a->segs[0] != kRaw + j || r->kind != kMxSeries ||
        r->r4 || r->tmaj || r->img || r->segs.size() != 1 || r->segs[0] < 0 || r->segs[0] % kRaw != j - 1)
      MX_FAIL(n, "only the residual add of the latest mid-end layer and its own input is supported");
    MxMid& m = spec.mid.back();
    if (m.residual || m.cin != m.cout) MX_FAIL(n, "residual over %d -> %d channels", m.cin, m.cout);
    seg_of(r->segs[0]);
    m.residual = 1;
    o.segs = {j};
  } else if (op == "ReduceMax" || op == "ReduceMean") {
    if (!one_axis(n, 2, 3) || attr_i(n, "keepdims", 1) != 0) MX_FAIL(n, "the back-end pool must reduce the time axis 2 without keepdims");
    o.kind = op == "ReduceMax" ? kMxPoolMax : kMxPoolMean;
  } else {
    MX_FAIL(n, "operator not supported on a channel series");
  }
  vals[n.out[0]] = o;
  return AM_OK;
}

int MxLowerer::node(ONode& n) {
  if (n.op == "Constant") {
    auto it = n.attrs.find("value");
    if (it == n.attrs.end() || !it->second.has_t) MX_FAIL(n, "Constant without a tensor value");
    consts[n.out[0]] = &it->second.t;
    return AM_OK;
  }
  if (n.in.empty() || !vals.count(n.in[0])) {
    // a binary op with the constant first
    if ((n.op == "Mul" || n.op == "Add") && n.in.size() == 2 && consts.count(n.in[0]) && vals.count(n.in[1])) {
      std::swap(n.in[0], n.in[1]);
    } else {
      MX_FAIL(n, "input '%s' is not produced by a supported node", n.in.empty() ? "" : n.in[0].c_str());
    }
  }
  const MxVal v = vals[n.in[0]];
  const std::string& op = n.op;

  if (v.kind == kMxIn) {
    MxVal o = v;
    if (op == "Unsqueeze") {
      if (v.layout != 0) MX_FAIL(n, "input already has a unit axis");
      if (one_axis(n, 1, 4)) o.layout = 1;
      else if (one_axis(n, 3, 4)) o.layout = 3;
      else MX_FAIL(n, "only the channel axis (1, or 3 for NHWC) may be inserted into the [n, time, mel] input");
    } else if (op == "Transpose") {
      if (v.layout != 3 || attr_ints(n, "perm") != std::vector<int64_t>{0, 3, 1, 2}) MX_FAIL(n, "only NHWC -> NCHW of the input");
      o.layout = 1;
    } else if (op == "BatchNormalization" || op == "Mul" || op == "Add") {
      if (v.layout != 1 || v.pad_t || v.pad_b) MX_FAIL(n, "input normalisation must act on the [n, 1, time, mel] input before any padding");
      if (op == "BatchNormalization") {
        std::vector<float> s, h;
        AM_TRY(bn_affine(n, &s, &h));
        if (s.size() != 1) MX_FAIL(n, "%zu channels on the single-channel input", s.size());
        o.s = v.s * s[0];
        o.h = v.h * s[0] + h[0];
      } else {
        const OTensor* t = cst(n, 1);
        if (!t || t->count() != 1) MX_FAIL(n, "only a constant scalar on the input");
        const float c = (float)t->at(0);
        if (op == "Mul") {
          o.s = v.s * c;
          o.h = v.h * c;
        } else {
          o.h = v.h + c;
        }
      }
    } else if (op == "Pad") {
      std::vector<int64_t> pads;
      if (v.layout != 1 || !ints_of(n, "pads", 1, &pads) || pads.size() != 8) MX_FAIL(n, "needs 8 constant pads on the [n, 1, time, mel] input");
      auto it = n.attrs.find("mode");
      if (it != n.attrs.end() && it->second.s != "constant") MX_FAIL(n, "only constant zero padding");
      if (const OTensor* c = cst(n, 2))
        if (c->count() && c->at(0) != 0.0) MX_FAIL(n, "only zero padding");
      if (pads[0] || pads[1] || pads[3] || pads[4] || pads[5] || pads[7]) MX_FAIL(n, "pads an axis other than time");
      o.pad_t += (int)pads[2];
      o.pad_b += (int)pads[6];
    } else if (op == "Conv") {
      return conv_front(n, v);
    } else {
      MX_FAIL(n, "operator not supported on the patch input");
    }
    vals[n.out[0]] = o;
    return AM_OK;
  }
  if (v.kind == kMxBranch || v.kind == kMxMid) return stage_op(n, v);
  if (v.kind == kMxSeries) return series_op(n, v);

  if (v.kind == kMxPoolMax || v.kind == kMxPoolMean) {
    if (op != "Concat" || attr_i(n, "axis", 0) != 1 || n.in.size() != 2 || !vals.count(n.in[1]))
      MX_FAIL(n, "the time max and mean must be concatenated along channels");
    const MxVal& u = vals[n.in[1]];
    if (u.kind == v.kind || (u.kind != kMxPoolMax && u.kind != kMxPoolMean) || u.segs != v.segs)
      MX_FAIL(n, "needs the max and the mean of the same series");
    if (!spec.pool_segs.empty()) MX_FAIL(n, "a second back-end pool");
    // front-end branches are one buffer: they must appear together and in order
    std::vector<int> segs;
    for (size_t q = 0; q < v.segs.size();) {
      if (v.segs[q] < 0) {
        for (size_t b = 0; b < spec.br.size(); ++b, ++q)
          if (q >= v.segs.size() || v.segs[q] != -1 - (int)b) MX_FAIL(n, "the pooled series splits the front-end branches");
        segs.push_back(-1);
      } else {
        segs.push_back(seg_of(v.segs[q++]));
      }
    }
    spec.pool_segs = segs;
    spec.pool_max_first = v.kind == kMxPoolMax ? 1 : 0;
    const int c = series_channels(v.segs);
    MxVal o;
    o.kind = kMxVec;
    o.reg = 0;
    o.dim = 2 * c;
    spec.reg_dim = {2 * c};
    vals[n.out[0]] = o;
    return AM_OK;
  }

  if (v.kind == kMxVec) {
    VecOp vo;
    vo.a = v.reg;
    vo.N = v.dim;
    if (op == "Relu") {
      vo.kind = kVecUnary;
      vo.act = kActRelu;
      return emit_vec(n, vo, v.dim);
    }
    if (op == "BatchNormalization") {
      AM_TRY(bn_affine(n, &vo.w, &vo.bias));
      if ((int)vo.w.size() != v.dim) MX_FAIL(n, "%zu statistics on a %d-wide row", vo.w.size(), v.dim);
      vo.kind = kVecAffine;
      return emit_vec(n, vo, v.dim);
    }
    if (op == "Mul") {
      const OTensor* t = per_channel(n, v.dim);
      if (!t) MX_FAIL(n, "only a constant per-column scale of %d on a row", v.dim);
      vo.kind = kVecAffine;
      vo.w = t->f;
      return emit_vec(n, vo, v.dim);
    }
    if (op == "Add") {
      const OTensor* t = per_channel(n, v.dim);
      if (!t) MX_FAIL(n, "only a constant per-column shift of %d on a row", v.dim);
      VecOp* last = spec.head.empty() ? nullptr : &spec.head.back();
      if (last && last->dst == v.reg && (last->kind == kVecLinear || last->kind == kVecAffine) && last->bias.empty()) {
        last->bias = t->f;  // bias of a MatMul, shift of a Mul
        vals[n.out[0]] = v;
        return AM_OK;
      }
      vo.kind = kVecAffine;
      vo.bias = t->f;
      return emit_vec(n, vo, v.dim);
    }
    if (op == "Gemm" || op == "MatMul") {
      const OTensor* w = cst(n, 1);
      if (!w || w->dims.size() != 2) MX_FAIL(n, "needs constant 2-D weights");
      const bool tb = op == "Gemm" && attr_i(n, "transB", 0);
      if (op == "Gemm" && (attr_i(n, "transA", 0) || attr_f(n, "alpha", 1.f) != 1.f || attr_f(n, "beta", 1.f) != 1.f))
        MX_FAIL(n, "transA / alpha / beta");
      const int K = (int)(tb ? w->dims[1] : w->dims[0]), N = (int)(tb ? w->dims[0] : w->dims[1]);
      if (K != v.dim) MX_FAIL(n, "%d inputs on a %d-wide row", K, v.dim);
      vo.kind = kVecLinear;
      vo.K = K;
      vo.N = N;
      vo.w.assign((size_t)N * K, 0.f);
      for (int r = 0; r < N; ++r)
        for (int k = 0; k < K; ++k) vo.w[(size_t)r * K + k] = tb ? w->f[(size_t)r * K + k] : w->f[(size_t)k * N + r];
      if (const OTensor* b = cst(n, 2)) {
        if ((int)b->count() != N) MX_FAIL(n, "bias of %zu for %d outputs", b->count(), N);
        vo.bias = b->f;
      }
      return emit_vec(n, vo, N);
    }
    MX_FAIL(n, "operator not supported on a row vector");
  }
  MX_FAIL(n, "unsupported data flow");
}

int MxLowerer::run() {
  if (g.inputs.size() != 1 || g.outputs.size() != 1) {
    set_error("musicnn onnx: expected one graph input and one output (%zu / %zu)", g.inputs.size(), g.outputs.size());
    return AM_ERR_INVALID;
  }
  for (auto& kv : g.init) consts[kv.first] = &kv.second;
  // the input is a patch tensor [n, time, mel] unless the first consumer treats it as a row
  bool row_input = false;
  for (const ONode& n : g.nodes)
    if (std::find(n.in.begin(), n.in.end(), g.inputs[0]) != n.in.end()) {
      row_input = n.op == "Relu" || n.op == "Gemm" || n.op == "MatMul" || n.op == "BatchNormalization";
      break;
    }
  MxVal in;
  if (row_input) {
    in.kind = kMxVec;
    in.reg = 0;
    in.dim = 0;
    // width from the first weight that reads it
    for (const ONode& n : g.nodes) {
      const OTensor* t = nullptr;
      if (n.op == "BatchNormalization") t = cst(n, 1);
      if ((n.op == "Gemm" || n.op == "MatMul") && cst(n, 1)) {
        const OTensor* w = cst(n, 1);
        in.dim = (int)((n.op == "Gemm" && attr_i(n, "transB", 0)) ? w->dims[1] : w->dims[0]);
        break;
      }
      if (t) {
        in.dim = (int)t->count();
        break;
      }
    }
    if (in.dim <= 0) {
      set_error("musicnn onnx: cannot infer the row width of input '%s'", g.inputs[0].c_str());
      return AM_ERR_INVALID;
    }
    spec.reg_dim = {in.dim};
    spec.in_dim = in.dim;
  }
  vals[g.inputs[0]] = in;
  for (ONode& n : g.nodes) AM_TRY(node(n));
  auto it = vals.find(g.outputs[0]);
  if (it == vals.end() || it->second.kind != kMxVec || spec.head.empty() || spec.head.back().dst != it->second.reg) {
    set_error("musicnn onnx: graph output '%s' is not the end of a row program", g.outputs[0].c_str());
    return AM_ERR_INVALID;
  }
  spec.is_embedding = row_input ? 0 : 1;
  for (int j : raw_used)
    if (spec.mid[(size_t)j].residual) {
      set_error("musicnn onnx: mid-end layer %d's output is read before its residual add as well as after it", j);
      return AM_ERR_INVALID;
    }
  if (spec.is_embedding) {
    for (const auto& b : spec.br)
      if (b.in_s != spec.br[0].in_s || b.in_h != spec.br[0].in_h) {
        set_error("musicnn onnx: the front-end branches read the input under different normalisations");
        return AM_ERR_INVALID;
      }
    spec.in_s = spec.br.empty() ? 1.f : spec.br[0].in_s;
    spec.in_h = spec.br.empty() ? 0.f : spec.br[0].in_h;
    if (spec.br.empty() || spec.pool_segs.empty()) {
      set_error("musicnn onnx: no front-end branches or no back-end pool");
      return AM_ERR_INVALID;
    }
    for (const auto& b : spec.br)
      if (b.s.empty()) {
        set_error("musicnn onnx: a front-end branch has no BatchNormalization");
        return AM_ERR_INVALID;
      }
    for (const auto& m : spec.mid)
      if (m.s.empty()) {
        set_error("musicnn onnx: a mid-end layer has no BatchNormalization");
        return AM_ERR_INVALID;
      }
    int off = 0;
    for (auto& b : spec.br) {
      b.ch_off = off;
      off += b.cout;
    }
    spec.c_front = off;
  }
  spec.out_dim = it->second.dim;
  char src[128];
  std::snprintf(src, sizeof src, "ONNX (ir %lld, opset %lld, %zu nodes)", (long long)g.ir_version, (long long)g.opset, g.nodes.size());
  spec.source = src;
  spec.in_name = g.inputs[0];
  spec.out_name = g.outputs[0];
  return AM_OK;
}

}  // namespace

int load_musicnn_spec(const void* data, size_t nbytes, const char* path, MusicnnSpec* out) {
  OGraph g;
  AM_TRY(parse_model(data, nbytes, dir_of(path), &g));
  MxLowerer L(g, *out);
  return L.run();
}

static std::string describe_spec(const MusicnnSpec& s) {
  std::string r;
  char b[512];
  std::snprintf(b, sizeof b, "musicnn %s: %s\n", s.is_embedding ? "embedding" : "prediction", s.source.c_str());
  r += b;
  if (s.is_embedding) {
    std::snprintf(b, sizeof b, "input affine scale=%.6g shift=%.6g (applied before zero padding)\n", s.in_s, s.in_h);
    r += b;
    for (size_t i = 0; i < s.br.size(); ++i) {
      const auto& x = s.br[i];
      std::snprintf(b, sizeof b, "front %zu: conv %dx%d cout=%d pad_time=%d/%d relu bn max_freq -> channels [%d, %d)%s\n", i,
                    x.kh, x.kw, x.cout, x.pad_top, x.kh - 1 - x.pad_top, x.ch_off, x.ch_off + x.cout,
                    x.pool_w ? (" (window " + std::to_string(x.pool_w) + ")").c_str() : "");
      r += b;
    }
    for (size_t j = 0; j < s.mid.size(); ++j) {
      const auto& m = s.mid[j];
      std::snprintf(b, sizeof b, "mid %zu: conv1d k=%d %d->%d relu bn%s\n", j, m.k, m.cin, m.cout, m.residual ? " +residual" : "");
      r += b;
    }
    std::string segs;
    for (int sg : s.pool_segs) segs += sg < 0 ? std::string(" front") : " mid" + std::to_string(sg);
    std::snprintf(b, sizeof b, "pool time %s over [%s ] -> %d\n", s.pool_max_first ? "max|mean" : "mean|max", segs.c_str(), s.reg_dim[0]);
    r += b;
  } else {
    std::snprintf(b, sizeof b, "input rows %d\n", s.in_dim);
    r += b;
  }
  for (const auto& h : s.head) {
    if (h.kind == kVecUnary) std::snprintf(b, sizeof b, "head unary act=%d width=%d\n", h.act, h.N);
    else if (h.kind == kVecAffine) std::snprintf(b, sizeof b, "head affine width=%d\n", h.N);
    else std::snprintf(b, sizeof b, "head linear %d->%d%s\n", h.K, h.N, h.bias.empty() ? "" : " +bias");
    r += b;
  }
  return r;
}

// ------------------------------------------------------------------------------------------- front-end kernel
// One branch = one implicit GEMM on the tensor cores, transposed so that a TMEM lane is a FILTER and the columns are
// output pixels:  D[filter, (tt, f)] = sum_{df, dt} W[filter, dt, df] * x[t0 + tt + dt - pad, f + df].
// K is ordered (df, dt) with dt padded to kh8 = round_up(kh, 8): for a fixed df, eight consecutive taps are eight
// consecutive TIME samples of one mel bin, so a 16-byte K chunk of the im2col row is a (shifted) 16-byte run of the
// staged, time-contiguous window xwin[mel][time].  A = weights (pre-swizzled K-major SW128 image, one bulk copy per
// k-block), B = the im2col tile built in shared memory by the producer warps.  Epilogue: each thread owns one filter
// and its columns: ReLU(acc + bias), BatchNorm (may be negative), max over the F_out columns of each time step, one
// bf16 store per (time step, filter).  The [filter, pixel] tile never leaves TMEM.
namespace mxk {
constexpr int kEpiWarps = 4, kMmaWarp = 4, kProdWarp0 = 5, kProdWarps = 8;
constexpr int kThreads = (kProdWarp0 + kProdWarps) * 32;
constexpr int kStages = 3;
constexpr int kProdThreads = kProdWarps * 32;

struct FrontArgs {
  const float* x;  // [P, T, F] patches
  int P, T, F;
  float in_s, in_h;
  int kh8, pad_top, F_out, TT, N, mtiles, nkb, nk16, kw;
  int items_per_patch;
  int64_t n_items;
  const uint8_t* wimg;  // [nkb][mtiles][16 KB]
  const float *bias, *bs, *bh;  // [mtiles * 128]
  int cout, ch_off;
  __nv_bfloat16* out;  // [P, out_rows, out_ld]
  int out_ld, out_rows, out_row0;
  int xw_pitch;  // elements per mel row of the window (multiple of 8)
  int xw_len;    // time samples staged per item (multiple of 8)
  uint32_t stage_bytes, a_bytes;
};

__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   ptx::smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(ptx::smem_u32(bar))
               : "memory");
}

__global__ void __launch_bounds__(kThreads, 1) musicnn_front_kernel(const FrontArgs a) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t* stages = smem;
  __nv_bfloat16* xwin = (__nv_bfloat16*)(smem + (size_t)kStages * a.stage_bytes);
  uint64_t* bars = (uint64_t*)((uint8_t*)xwin + (size_t)a.F * a.xw_pitch * 2 + 64);
  uint64_t *full = bars, *empty = bars + kStages, *tfull = bars + 2 * kStages, *tempty = bars + 2 * kStages + 2;
  uint32_t* tmem_slot = (uint32_t*)(bars + 2 * kStages + 4);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      ptx::mbar_init(&full[s], kProdWarps + 1);
      ptx::mbar_init(&empty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      ptx::mbar_init(&tfull[b], 1);
      ptx::mbar_init(&tempty[b], kEpiWarps);
    }
    ptx::fence_barrier_init();
  }
  if (warp == kMmaWarp) ptx::tmem_alloc(tmem_slot, 512);
  ptx::tcgen05_fence_before();
  __syncthreads();
  ptx::tcgen05_fence_after();
  const uint32_t tmem = *tmem_slot;
  const int ncols = a.mtiles * a.N;  // TMEM columns of one accumulator set

  if (warp >= kProdWarp0) {
    // ---------------------------------------------------------------- producers
    const int pt = threadIdx.x - kProdWarp0 * 32;
    int s = 0;
    uint32_t ph = 0;
    const int xw_chunks = a.xw_len >> 3;
    const int kc_per_df = a.kh8 >> 3;
    const int nvalid_rows = a.TT * a.F_out;
    for (int64_t item = blockIdx.x; item < a.n_items; item += gridDim.x) {
      const int p = (int)(item / a.items_per_patch);
      const int t0 = (int)(item % a.items_per_patch) * a.TT;
      ptx::named_bar_sync_1<kProdThreads>();  // every builder is done with the previous window
      // stage the window: xwin[f][j] = in_s * x[p, t0 - pad + j, f] + in_h (zero outside the patch)
      const float* xp = a.x + (int64_t)p * a.T * a.F;
      for (int task = pt; task < a.F * xw_chunks; task += kProdThreads) {
        const int f = task % a.F, jc = task / a.F;
        float v[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int t = t0 - a.pad_top + jc * 8 + e;
          v[e] = (t >= 0 && t < a.T) ? fmaf(__ldg(xp + (int64_t)t * a.F + f), a.in_s, a.in_h) : 0.f;
        }
        uint4 pk;
        __nv_bfloat162 q;
        q = __floats2bfloat162_rn(v[0], v[1]); pk.x = *reinterpret_cast<uint32_t*>(&q);
        q = __floats2bfloat162_rn(v[2], v[3]); pk.y = *reinterpret_cast<uint32_t*>(&q);
        q = __floats2bfloat162_rn(v[4], v[5]); pk.z = *reinterpret_cast<uint32_t*>(&q);
        q = __floats2bfloat162_rn(v[6], v[7]); pk.w = *reinterpret_cast<uint32_t*>(&q);
        *reinterpret_cast<uint4*>(xwin + (size_t)f * a.xw_pitch + jc * 8) = pk;
      }
      ptx::named_bar_sync_1<kProdThreads>();
      for (int kb = 0; kb < a.nkb; ++kb) {
        ptx::mbar_wait(&empty[s], ph ^ 1);
        uint8_t* st = stages + (size_t)s * a.stage_bytes;
        if (pt == 0) {
          ptx::mbar_expect_tx(&full[s], a.a_bytes);
          bulk_g2s(st, a.wimg + (size_t)kb * a.a_bytes, a.a_bytes, &full[s]);
        }
        uint8_t* bt = st + a.a_bytes;
        // B tile: N rows x 8 chunks of 8 K-values; lanes walk rows (consecutive mel bins)
        for (int task = pt; task < a.N * 8; task += kProdThreads) {
          const int n = task % a.N, c = task / a.N;
          const int kc = kb * 8 + c;  // global chunk index
          const int df = kc / kc_per_df, dt0 = (kc - df * kc_per_df) * 8;
          uint4 o = make_uint4(0, 0, 0, 0);
          if (n < nvalid_rows && df < a.kw) {
            const int tt = n / a.F_out, f = n - tt * a.F_out;
            const int e = tt + dt0;
            const uint4* row = reinterpret_cast<const uint4*>(xwin + (size_t)(f + df) * a.xw_pitch);
            const uint4 q0 = row[e >> 3];
            const int r = e & 7;
            if (r == 0) {
              o = q0;
            } else {
              const uint4 q1 = row[(e >> 3) + 1];
              const uint64_t E0 = ((uint64_t)q0.y << 32) | q0.x, E1 = ((uint64_t)q0.w << 32) | q0.z;
              const uint64_t E2 = ((uint64_t)q1.y << 32) | q1.x, E3 = ((uint64_t)q1.w << 32) | q1.z;
              const bool hi = r >= 4;
              const int sh = 16 * (r & 3);
              const uint64_t a0 = hi ? E1 : E0, a1 = hi ? E2 : E1, a2 = hi ? E3 : E2;
              uint64_t o0, o1;
              if (sh == 0) {
                o0 = a0;
                o1 = a1;
              } else {
                o0 = (a0 >> sh) | (a1 << (64 - sh));
                o1 = (a1 >> sh) | (a2 << (64 - sh));
              }
              o = make_uint4((uint32_t)o0, (uint32_t)(o0 >> 32), (uint32_t)o1, (uint32_t)(o1 >> 32));
            }
          }
          *reinterpret_cast<uint4*>(bt + ptx::sw128_offset((uint32_t)n, (uint32_t)c)) = o;
        }
        ptx::fence_proxy_async();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&full[s]);
        if (++s == kStages) {
          s = 0;
          ph ^= 1;
        }
      }
    }
  } else if (warp == kMmaWarp) {
    // ---------------------------------------------------------------- MMA issuer
    const uint32_t idesc = ptx::make_idesc(128, a.N);
    int s = 0;
    uint32_t ph = 0;
    int it = 0;
    for (int64_t item = blockIdx.x; item < a.n_items; item += gridDim.x, ++it) {
      const int buf = it & 1;
      const uint32_t tph = (uint32_t)(it >> 1) & 1u;
      ptx::mbar_wait(&tempty[buf], tph ^ 1);
      ptx::tcgen05_fence_after();
      const uint32_t d0 = tmem + (uint32_t)(buf * ncols);
      for (int kb = 0; kb < a.nkb; ++kb) {
        ptx::mbar_wait(&full[s], ph);
        ptx::tcgen05_fence_after();
        const uint32_t st = ptx::smem_u32(stages + (size_t)s * a.stage_bytes);
        const int ksteps = min(4, a.nk16 - kb * 4);
        if (ptx::elect_one_sync()) {
          for (int mt = 0; mt < a.mtiles; ++mt) {
            for (int ks = 0; ks < ksteps; ++ks) {
              const uint64_t da = ptx::make_smem_desc(st + (uint32_t)mt * 16384u + (uint32_t)ks * 32u);
              const uint64_t db = ptx::make_smem_desc(st + a.a_bytes + (uint32_t)ks * 32u);
              ptx::umma_f16(d0 + (uint32_t)(mt * a.N), da, db, idesc, (kb | ks) ? 1u : 0u);
            }
          }
          ptx::umma_commit(&empty[s]);
          if (kb == a.nkb - 1) ptx::umma_commit(&tfull[buf]);
        }
        __syncwarp();
        if (++s == kStages) {
          s = 0;
          ph ^= 1;
        }
      }
    }
  } else {
    // ---------------------------------------------------------------- epilogue (warp w reads TMEM lanes 32w..32w+31)
    int it = 0;
    for (int64_t item = blockIdx.x; item < a.n_items; item += gridDim.x, ++it) {
      const int p = (int)(item / a.items_per_patch);
      const int t0 = (int)(item % a.items_per_patch) * a.TT;
      const int tv = min(a.TT, a.T - t0);
      const int buf = it & 1;
      ptx::mbar_wait(&tfull[buf], (uint32_t)(it >> 1) & 1u);
      ptx::tcgen05_fence_after();
      for (int mt = 0; mt < a.mtiles; ++mt) {
        const int filt = mt * 128 + warp * 32 + lane;
        const float bias = a.bias[filt], bs = a.bs[filt], bh = a.bh[filt];
        const uint32_t taddr = tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)(buf * ncols + mt * a.N);
        __nv_bfloat16* o = a.out + ((int64_t)p * a.out_rows + a.out_row0 + t0) * a.out_ld + a.ch_off + filt;
        const bool store = filt < a.cout;
        float m = -INFINITY;
        int tt = 0, next = a.F_out;
        const int ncol = tv * a.F_out;
        for (int c0 = 0; c0 < ncol; c0 += 16) {
          uint32_t v[16];
          ptx::tmem_ld_x16(taddr + (uint32_t)c0, v);
          ptx::tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int col = c0 + j;
            if (col < ncol) {
              const float y = fmaf(fmaxf(__uint_as_float(v[j]) + bias, 0.f), bs, bh);
              m = fmaxf(m, y);
              if (col + 1 == next) {
                if (store) o[(int64_t)tt * a.out_ld] = __float2bfloat16_rn(m);
                m = -INFINITY;
                ++tt;
                next += a.F_out;
              }
            }
          }
        }
      }
      ptx::tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&tempty[buf]);
    }
  }
  ptx::tcgen05_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    ptx::tcgen05_fence_after();
    ptx::tmem_dealloc(tmem, 512);
  }
}
}  // namespace mxk

// ------------------------------------------------------------------------------------------- small kernels
// A[(p*T + t), dt*cin_p + c] = in[p, row0 - pad + t + dt, c]   (16-byte vectors; in has zero pad rows)
__global__ void __launch_bounds__(256) mx_im2col_kernel(const __nv_bfloat16* __restrict__ in, int P, int T, int rows,
                                                        int row0, int cin_p, int k, __nv_bfloat16* __restrict__ A) {
  const int vec = cin_p >> 3, pad = (k - 1) / 2;
  const int64_t n = (int64_t)P * T * k * vec;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int cv = (int)(i % vec);
    int64_t r = i / vec;
    const int dt = (int)(r % k);
    r /= k;
    const int t = (int)(r % T);
    const int p = (int)(r / T);
    const uint4 q = *reinterpret_cast<const uint4*>(in + ((int64_t)p * rows + row0 - pad + t + dt) * cin_p + cv * 8);
    *reinterpret_cast<uint4*>(A + i * 8) = q;
  }
}

// out[p, row0 + t, c] = bf16(D[p*T + t, c] * s[c] + h[c] (+ res[p, row0 + t, c]))   (D already holds relu(conv + bias))
__global__ void __launch_bounds__(256) mx_mid_post_kernel(const float* __restrict__ D, int P, int T, int C,
                                                          const float* __restrict__ s, const float* __restrict__ h,
                                                          const __nv_bfloat16* __restrict__ res, int res_ld,
                                                          __nv_bfloat16* __restrict__ out, int rows, int row0) {
  const int64_t n = (int64_t)P * T * C;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    const int64_t pt = i / C;
    const int t = (int)(pt % T), p = (int)(pt / T);
    const int64_t orow = (int64_t)p * rows + row0 + t;
    float v = fmaf(D[i], s[c], h[c]);
    if (res) v += __bfloat162float(res[orow * res_ld + c]);
    out[orow * C + c] = __float2bfloat16_rn(v);
  }
}

struct PoolSeg {
  const __nv_bfloat16* buf;
  int ld, ch;
};
struct PoolArgs {
  PoolSeg seg[8];
  int n_seg;
  int C;  // total pooled channels
  int rows, row0, T, max_first;
};
// one CTA per patch: vec[p, c] = max_t, vec[p, C + c] = mean_t (or the other way round)
__global__ void __launch_bounds__(256) mx_pool_kernel(const PoolArgs a, float* __restrict__ vec) {
  const int p = blockIdx.x;
  for (int c = threadIdx.x; c < a.C; c += blockDim.x) {
    int cc = c, q = 0;
    while (q < a.n_seg - 1 && cc >= a.seg[q].ch) cc -= a.seg[q++].ch;
    const __nv_bfloat16* b = a.seg[q].buf + ((int64_t)p * a.rows + a.row0) * a.seg[q].ld + cc;
    float mx = -INFINITY, sm = 0.f;
    for (int t = 0; t < a.T; ++t) {
      const float v = __bfloat162float(b[(int64_t)t * a.seg[q].ld]);
      mx = fmaxf(mx, v);
      sm += v;
    }
    float* o = vec + (int64_t)p * 2 * a.C;
    o[a.max_first ? c : a.C + c] = mx;
    o[a.max_first ? a.C + c : c] = sm / (float)a.T;
  }
}

__global__ void mx_affine_kernel(const float* __restrict__ x, int64_t n, int dim, const float* __restrict__ s,
                                 const float* __restrict__ h, int relu, float* __restrict__ y) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float v = x[i];
    if (relu) v = fmaxf(v, 0.f);
    if (s) v *= s[i % dim];
    if (h) v += h[i % dim];
    y[i] = v;
  }
}

// y[r, n] = sum_k x[r, k] W[n, k] + b[n]   (fp32, 32 x 32 tiles)
__global__ void __launch_bounds__(256) mx_linear_kernel(const float* __restrict__ x, int R, int K, const float* __restrict__ W,
                                                        const float* __restrict__ b, int N, float* __restrict__ y) {
  __shared__ float xs[32][33], ws[32][33];
  const int r0 = blockIdx.y * 32, n0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 8 rows of threads, 4 outputs each
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  for (int k0 = 0; k0 < K; k0 += 32) {
    for (int q = ty; q < 32; q += 8) {
      const int r = r0 + q, n = n0 + q, k = k0 + tx;
      xs[q][tx] = (r < R && k < K) ? x[(int64_t)r * K + k] : 0.f;
      ws[q][tx] = (n < N && k < K) ? W[(int64_t)n * K + k] : 0.f;
    }
    __syncthreads();
#pragma unroll 8
    for (int k = 0; k < 32; ++k) {
      const float w = ws[tx][k];
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[j] = fmaf(xs[ty + 8 * j][k], w, acc[j]);
    }
    __syncthreads();
  }
  const int n = n0 + tx;
  if (n < N)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = r0 + ty + 8 * j;
      if (r < R) y[(int64_t)r * N + n] = acc[j] + (b ? b[n] : 0.f);
    }
}

// per track: emb = mean of its patch embeddings, moods = sigmoid(mean(sigmoid(logits)))
__global__ void mx_track_kernel(const float* __restrict__ E, int de, const float* __restrict__ L, int dl,
                                const int* __restrict__ off, float* __restrict__ emb, float* __restrict__ moods) {
  const int tr = blockIdx.x;
  const int a = off[tr], b = off[tr + 1], n = b - a;
  for (int c = threadIdx.x; c < de; c += blockDim.x) {
    float s = 0.f;
    for (int q = a; q < b; ++q) s += E[(int64_t)q * de + c];
    emb[(int64_t)tr * de + c] = n ? s / (float)n : 0.f;
  }
  if (moods)
    for (int c = threadIdx.x; c < dl; c += blockDim.x) {
      float s = 0.f;
      for (int q = a; q < b; ++q) s += 1.f / (1.f + expf(-L[(int64_t)q * dl + c]));
      moods[(int64_t)tr * dl + c] = n ? 1.f / (1.f + expf(-s / (float)n)) : 0.f;
    }
}

}  // namespace am

// ------------------------------------------------------------------------------------------- model object
using namespace am;

struct DevHeadOp {
  int kind = 0, K = 0, N = 0, act = 0;
  DevBuf<float> w, bias;
};
struct DevBranch {
  mxk::FrontArgs args{};
  int pool_w = 0;
  DevBuf<uint8_t> wimg;
  DevBuf<float> bias, bs, bh;
};
struct DevMid {
  int cin = 0, cin_p = 0, cout = 0, k = 0, residual = 0;
  DevBuf<__nv_bfloat16> w;  // [cout, k * cin_p]
  DevBuf<float> bias, s, h;
};

struct am_musicnn {
  MusicnnSpec spec;
  int cf_p = 0, pad_rows = 0;
  std::vector<std::unique_ptr<DevBranch>> br;
  std::vector<std::unique_ptr<DevMid>> mid;
  std::vector<std::unique_ptr<DevHeadOp>> head;
  Stream stream;
  // workspace (per sub-batch of patches)
  int ws_T = 0, ws_P = 0;
  DevBuf<__nv_bfloat16> fbuf, a_col;
  std::vector<std::unique_ptr<DevBuf<__nv_bfloat16>>> mbuf;
  DevBuf<float> d_mid, vec0, vec1, vec2;
  DevBuf<float> io_in, io_out;
  // track path
  DevBuf<float> t_pcm, t_mel, t_emb, t_logit, t_out_e, t_out_m;
  DevBuf<int> t_off;
};

namespace {
constexpr int kSubBatch = 512;

int upload_f(DevBuf<float>& d, const std::vector<float>& h, size_t n = 0) {
  std::vector<float> v(h);
  if (n > v.size()) v.resize(n, 0.f);
  AM_TRY(d.alloc(std::max<size_t>(v.size(), 1)));
  if (!v.empty()) AM_CUDA(cudaMemcpy(d.p, v.data(), v.size() * 4, cudaMemcpyHostToDevice));
  return AM_OK;
}

int build_branch(const MxBranch& b, DevBranch* d) {
  mxk::FrontArgs& a = d->args;
  a.kh8 = (int)round_up((size_t)b.kh, 8);
  a.kw = b.kw;
  a.pad_top = b.pad_top;
  a.mtiles = (b.cout + 127) / 128;
  AM_CHECK(a.mtiles <= 2, "musicnn: %d filters in one branch (at most 256)", b.cout);
  const int K = b.kw * a.kh8;
  a.nk16 = (K + 15) / 16;
  a.nkb = (a.nk16 + 3) / 4;
  a.a_bytes = (uint32_t)a.mtiles * 16384u;
  a.cout = b.cout;
  a.ch_off = b.ch_off;
  d->pool_w = b.pool_w;
  // pre-swizzled K-major SW128 image: block (kb, mt) = 128 rows x 128 B
  std::vector<__nv_bfloat16> img((size_t)a.nkb * a.mtiles * 8192, __float2bfloat16_rn(0.f));
  for (int kb = 0; kb < a.nkb; ++kb)
    for (int mt = 0; mt < a.mtiles; ++mt)
      for (int r = 0; r < 128; ++r) {
        const int filt = mt * 128 + r;
        if (filt >= b.cout) continue;
        for (int k = 0; k < 64; ++k) {
          const int kg = kb * 64 + k, df = kg / a.kh8, dt = kg % a.kh8;
          if (df >= b.kw || dt >= b.kh) continue;
          const float w = b.w[((size_t)filt * b.kh + dt) * b.kw + df];
          const uint32_t off = (uint32_t)((r >> 3) * 1024 + (r & 7) * 128 + ((((uint32_t)k >> 3) ^ (uint32_t)(r & 7)) << 4) + (k & 7) * 2);
          img[((size_t)kb * a.mtiles + mt) * 8192 + off / 2] = __float2bfloat16_rn(w);
        }
      }
  AM_TRY(d->wimg.alloc(img.size() * 2));
  AM_CUDA(cudaMemcpy(d->wimg.p, img.data(), img.size() * 2, cudaMemcpyHostToDevice));
  AM_TRY(upload_f(d->bias, b.bias, (size_t)a.mtiles * 128));
  AM_TRY(upload_f(d->bs, b.s, (size_t)a.mtiles * 128));
  AM_TRY(upload_f(d->bh, b.h, (size_t)a.mtiles * 128));
  a.wimg = d->wimg.p;
  a.bias = d->bias.p;
  a.bs = d->bs.p;
  a.bh = d->bh.p;
  return AM_OK;
}

int build(am_musicnn* m) {
  const MusicnnSpec& s = m->spec;
  for (const auto& b : s.br) {
    m->br.emplace_back(new DevBranch());
    AM_TRY(build_branch(b, m->br.back().get()));
  }
  m->cf_p = (int)round_up((size_t)std::max(s.c_front, 1), 16);
  m->pad_rows = 0;
  for (const auto& x : s.mid) m->pad_rows = std::max(m->pad_rows, (x.k - 1) / 2);
  for (size_t j = 0; j < s.mid.size(); ++j) {
    const MxMid& x = s.mid[j];
    std::unique_ptr<DevMid> d(new DevMid());
    d->cin = x.cin;
    d->cin_p = j == 0 ? m->cf_p : (int)round_up((size_t)x.cin, 16);
    d->cout = x.cout;
    d->k = x.k;
    d->residual = x.residual;
    std::vector<__nv_bfloat16> w((size_t)x.cout * x.k * d->cin_p, __float2bfloat16_rn(0.f));
    for (int o = 0; o < x.cout; ++o)
      for (int c = 0; c < x.cin; ++c)
        for (int t = 0; t < x.k; ++t)
          w[(size_t)o * x.k * d->cin_p + (size_t)t * d->cin_p + c] = __float2bfloat16_rn(x.w[((size_t)o * x.cin + c) * x.k + t]);
    AM_TRY(d->w.alloc(w.size()));
    AM_CUDA(cudaMemcpy(d->w.p, w.data(), w.size() * 2, cudaMemcpyHostToDevice));
    AM_TRY(upload_f(d->bias, x.bias));
    AM_TRY(upload_f(d->s, x.s));
    AM_TRY(upload_f(d->h, x.h));
    m->mid.push_back(std::move(d));
  }
  for (const auto& x : s.mid) AM_CHECK(x.cout % 16 == 0, "musicnn: mid-end width %d is not a multiple of 16", x.cout);
  for (const auto& h : s.head) {
    std::unique_ptr<DevHeadOp> d(new DevHeadOp());
    d->kind = h.kind;
    d->K = h.K;
    d->N = h.N;
    d->act = h.act;
    if (!h.w.empty()) AM_TRY(upload_f(d->w, h.w));
    if (!h.bias.empty()) AM_TRY(upload_f(d->bias, h.bias));
    m->head.push_back(std::move(d));
  }
  return m->stream.create();
}

int max_dim(const am_musicnn* m) {
  int d = 1;
  for (int x : m->spec.reg_dim) d = std::max(d, x);
  return d;
}

// head row program: rows f32 [n, reg_dim[0]] in `in` -> out f32 [n, out_dim]
int run_head(am_musicnn* m, const float* in, int n, float* out, cudaStream_t st) {
  const float* cur = in;
  const size_t nh = m->head.size();
  for (size_t q = 0; q < nh; ++q) {
    const DevHeadOp& h = *m->head[q];
    float* dst = q + 1 == nh ? out : ((cur == m->vec1.p) ? m->vec2.p : m->vec1.p);
    const int dim = m->spec.head[q].N;
    const int64_t tot = (int64_t)n * dim;
    const int grid = (int)std::min<int64_t>((tot + 255) / 256, (int64_t)sm_count() * 8);
    if (h.kind == kVecLinear) {
      AM_LAUNCH(mx_linear_kernel, dim3((unsigned)ceil_div(h.N, 32), (unsigned)ceil_div(n, 32)), 256, 0, st, cur, n, h.K,
                h.w.p, h.bias.p, h.N, dst);
    } else if (h.kind == kVecAffine) {
      AM_LAUNCH(mx_affine_kernel, std::max(grid, 1), 256, 0, st, cur, tot, dim, h.w.p, h.bias.p, 0, dst);
    } else {
      AM_LAUNCH(mx_affine_kernel, std::max(grid, 1), 256, 0, st, cur, tot, dim, nullptr, nullptr, 1, dst);
    }
    cur = dst;
  }
  return AM_OK;
}

int ensure_ws(am_musicnn* m, int T, int n, cudaStream_t st) {
  const int P = std::min(n, kSubBatch);
  if (m->ws_T == T && m->ws_P >= P) return AM_OK;
  const MusicnnSpec& s = m->spec;
  const int rows = T + 2 * m->pad_rows;
  m->ws_T = 0;
  AM_TRY(m->fbuf.alloc((size_t)P * rows * m->cf_p));
  AM_CUDA(cudaMemsetAsync(m->fbuf.p, 0, (size_t)P * rows * m->cf_p * 2, st));
  m->mbuf.clear();
  size_t acol = 8, dmid = 8;
  for (size_t j = 0; j < s.mid.size(); ++j) {
    m->mbuf.emplace_back(new DevBuf<__nv_bfloat16>());
    AM_TRY(m->mbuf.back()->alloc((size_t)P * rows * s.mid[j].cout));
    AM_CUDA(cudaMemsetAsync(m->mbuf.back()->p, 0, (size_t)P * rows * s.mid[j].cout * 2, st));
    acol = std::max(acol, (size_t)P * T * m->mid[j]->k * m->mid[j]->cin_p);
    dmid = std::max(dmid, (size_t)P * T * s.mid[j].cout);
  }
  AM_TRY(m->a_col.alloc(acol));
  AM_TRY(m->d_mid.alloc(dmid));
  const size_t vd = (size_t)P * max_dim(m);
  AM_TRY(m->vec0.alloc(vd));
  AM_TRY(m->vec1.alloc(vd));
  AM_TRY(m->vec2.alloc(vd));
  m->ws_T = T;
  m->ws_P = P;
  return AM_OK;
}

int front_smem(const mxk::FrontArgs& a) {
  return mxk::kStages * (int)a.stage_bytes + a.F * a.xw_pitch * 2 + 64 + 128 + 1024;
}

// embedding trunk for P <= kSubBatch patches x f32 [P, T, F] -> rows f32 [P, emb]
int embed_sub(am_musicnn* m, const float* x, int P, int T, int F, float* out, cudaStream_t st) {
  const MusicnnSpec& s = m->spec;
  const int rows = T + 2 * m->pad_rows;
  for (auto& bp : m->br) {
    mxk::FrontArgs a = bp->args;
    a.x = x;
    a.P = P;
    a.T = T;
    a.F = F;
    a.in_s = s.in_s;
    a.in_h = s.in_h;
    a.F_out = F - a.kw + 1;
    AM_CHECK(a.F_out >= 1, "musicnn: %d mel bins under a %d-wide kernel", F, a.kw);
    AM_CHECK(bp->pool_w == 0 || bp->pool_w == a.F_out,
             "musicnn: the graph pools %d of the %d frequency outputs; only a max over the whole axis is supported",
             bp->pool_w, a.F_out);
    a.TT = 1;
    while (a.TT < 8 && (int)round_up((size_t)(a.TT + 1) * a.F_out, 16) * a.mtiles <= 256) ++a.TT;
    a.N = (int)round_up((size_t)a.TT * a.F_out, 16);
    AM_CHECK(a.N * a.mtiles <= 256, "musicnn: %d output bins do not fit one tile", a.F_out);
    a.items_per_patch = ceil_div(T, a.TT);
    a.n_items = (int64_t)P * a.items_per_patch;
    a.out = m->fbuf.p;
    a.out_ld = m->cf_p;
    a.out_rows = rows;
    a.out_row0 = m->pad_rows;
    a.xw_len = (int)round_up((size_t)(a.TT - 1 + a.kh8), 8) + 8;
    a.xw_pitch = ((a.xw_len / 8) | 1) * 8;
    a.stage_bytes = a.a_bytes + (uint32_t)a.N * 128u;
    const int smem = front_smem(a);
    AM_CHECK(smem <= 232448, "musicnn: front-end branch needs %d bytes of shared memory", smem);
    AM_CUDA(cudaFuncSetAttribute(mxk::musicnn_front_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    const int grid = (int)std::min<int64_t>(a.n_items, sm_count());
    AM_LAUNCH(mxk::musicnn_front_kernel, grid, mxk::kThreads, smem, st, a);
  }
  const __nv_bfloat16* cur = m->fbuf.p;
  int cur_c = m->cf_p;
  for (size_t j = 0; j < m->mid.size(); ++j) {
    const DevMid& d = *m->mid[j];
    const int64_t vecs = (int64_t)P * T * d.k * (d.cin_p / 8);
    AM_LAUNCH(mx_im2col_kernel, (int)std::min<int64_t>((vecs + 255) / 256, (int64_t)sm_count() * 16), 256, 0, st, cur, P,
              T, rows, m->pad_rows, d.cin_p, d.k, m->a_col.p);
    gemm::Epilogue ep;
    ep.bias = d.bias.p;
    ep.act = kActRelu;
    const int K = d.k * d.cin_p;
    AM_TRY(gemm::gemm_bf16(m->a_col.p, (int64_t)P * T, K, d.w.p, d.cout, K, K, m->d_mid.p, d.cout, true, ep, false, st));
    const int64_t tot = (int64_t)P * T * d.cout;
    AM_LAUNCH(mx_mid_post_kernel, (int)std::min<int64_t>((tot + 255) / 256, (int64_t)sm_count() * 16), 256, 0, st,
              m->d_mid.p, P, T, d.cout, d.s.p, d.h.p, d.residual ? cur : nullptr, cur_c, m->mbuf[j]->p, rows, m->pad_rows);
    cur = m->mbuf[j]->p;
    cur_c = d.cout;
  }
  PoolArgs pa{};
  AM_CHECK(s.pool_segs.size() <= 8, "musicnn: more than 8 pooled series");
  pa.n_seg = (int)s.pool_segs.size();
  pa.C = 0;
  for (int q = 0; q < pa.n_seg; ++q) {
    const int sg = s.pool_segs[(size_t)q];
    if (sg < 0) pa.seg[q] = {m->fbuf.p, m->cf_p, s.c_front};
    else pa.seg[q] = {m->mbuf[(size_t)sg]->p, s.mid[(size_t)sg].cout, s.mid[(size_t)sg].cout};
    pa.C += pa.seg[q].ch;
  }
  pa.rows = rows;
  pa.row0 = m->pad_rows;
  pa.T = T;
  pa.max_first = s.pool_max_first;
  AM_LAUNCH(mx_pool_kernel, P, 256, 0, st, pa, m->vec0.p);
  return run_head(m, m->vec0.p, P, out, st);
}

int run_dev(am_musicnn* m, const float* in, int n, int T, int F, float* out, cudaStream_t st) {
  const MusicnnSpec& s = m->spec;
  if (n <= 0) return AM_OK;
  if (!s.is_embedding) {
    AM_CHECK(T == s.in_dim && F == 1, "musicnn prediction: rows of %d expected, got [%d, %d]", s.in_dim, T, F);
    AM_TRY(ensure_ws(m, 1, kSubBatch, st));
    for (int b0 = 0; b0 < n; b0 += kSubBatch) {
      const int nb = std::min(kSubBatch, n - b0);
      AM_TRY(run_head(m, in + (int64_t)b0 * s.in_dim, nb, out + (int64_t)b0 * s.out_dim, st));
    }
    return AM_OK;
  }
  AM_CHECK(T >= 1 && F >= 1, "musicnn embedding: bad patch shape [%d, %d]", T, F);
  AM_TRY(ensure_ws(m, T, n, st));
  for (int b0 = 0; b0 < n; b0 += kSubBatch) {
    const int nb = std::min(kSubBatch, n - b0);
    AM_TRY(embed_sub(m, in + (int64_t)b0 * T * F, nb, T, F, out + (int64_t)b0 * s.out_dim, st));
  }
  return AM_OK;
}

int read_file(const char* path, std::vector<uint8_t>* buf) {
  FILE* f = std::fopen(path, "rb");
  if (!f) {
    set_error("musicnn: cannot open %s", path);
    return AM_ERR_IO;
  }
  std::fseek(f, 0, SEEK_END);
  const long n = std::ftell(f);
  std::fseek(f, 0, SEEK_SET);
  buf->resize(n > 0 ? (size_t)n : 0);
  const size_t got = buf->empty() ? 0 : std::fread(buf->data(), 1, buf->size(), f);
  std::fclose(f);
  if (got != buf->size()) {
    set_error("musicnn: short read of %s", path);
    return AM_ERR_IO;
  }
  return AM_OK;
}

int load_common(const void* blob, size_t nbytes, const char* path, am_musicnn** out) {
  AM_CHECK(out != nullptr, "am_musicnn_load: out is NULL");
  *out = nullptr;
  std::unique_ptr<am_musicnn> m(new am_musicnn());
  AM_TRY(load_musicnn_spec(blob, nbytes, path, &m->spec));
  AM_TRY(ensure_init());
  AM_CHECK(gemm::available(), "am_musicnn_load: the tcgen05 path is unavailable on this device; no fallback is shipped");
  AM_TRY(build(m.get()));
  *out = m.release();
  return AM_OK;
}
}  // namespace

extern "C" int am_musicnn_load(const char* path, am_musicnn** out) {
  AM_CHECK(path != nullptr, "am_musicnn_load: path is NULL");
  std::vector<uint8_t> buf;
  AM_TRY(read_file(path, &buf));
  return load_common(buf.data(), buf.size(), path, out);
}

extern "C" int am_musicnn_load_mem(const void* blob, size_t nbytes, am_musicnn** out) {
  AM_CHECK(blob != nullptr && nbytes > 0, "am_musicnn_load_mem: empty blob");
  return load_common(blob, nbytes, nullptr, out);
}

extern "C" int am_musicnn_describe_file(const char* path, char* buf, int cap) {
  AM_CHECK(path != nullptr, "am_musicnn_describe_file: path is NULL");
  std::vector<uint8_t> data;
  AM_TRY(read_file(path, &data));
  MusicnnSpec s;
  AM_TRY(load_musicnn_spec(data.data(), data.size(), path, &s));
  const std::string d = describe_spec(s);
  if (buf && cap > 0) {
    const size_t k = std::min(d.size(), (size_t)cap - 1);
    std::memcpy(buf, d.data(), k);
    buf[k] = 0;
  }
  return (int)d.size() + 1;
}

extern "C" void am_musicnn_free(am_musicnn* m) {
  if (m) {
    cudaDeviceSynchronize();
    delete m;
  }
}

extern "C" int am_musicnn_release_workspace(am_musicnn* m) {
  AM_CHECK(m != nullptr, "am_musicnn_release_workspace: NULL model");
  // am_musicnn_run_dev may have queued work on a caller's stream: wait for the whole device
  AM_CUDA(cudaDeviceSynchronize());
  m->fbuf.release();
  m->a_col.release();
  m->mbuf.clear();
  m->d_mid.release();
  m->vec0.release();
  m->vec1.release();
  m->vec2.release();
  m->io_in.release();
  m->io_out.release();
  m->t_pcm.release();
  m->t_mel.release();
  m->t_emb.release();
  m->t_logit.release();
  m->t_out_e.release();
  m->t_out_m.release();
  m->t_off.release();
  m->ws_T = m->ws_P = 0;
  return AM_OK;
}

extern "C" int am_musicnn_dims(const am_musicnn* m, int* is_embedding, int* in_dim, int* out_dim) {
  AM_CHECK(m != nullptr, "am_musicnn_dims: NULL model");
  if (is_embedding) *is_embedding = m->spec.is_embedding;
  if (in_dim) *in_dim = m->spec.is_embedding ? 0 : m->spec.in_dim;
  if (out_dim) *out_dim = m->spec.out_dim;
  return AM_OK;
}

extern "C" int am_musicnn_io_names(const am_musicnn* m, char* in_name, char* out_name, int cap) {
  AM_CHECK(m != nullptr, "am_musicnn_io_names: NULL model");
  const int need = (int)std::max(m->spec.in_name.size(), m->spec.out_name.size()) + 1;
  if (cap >= need && in_name && out_name) {
    std::memcpy(in_name, m->spec.in_name.c_str(), m->spec.in_name.size() + 1);
    std::memcpy(out_name, m->spec.out_name.c_str(), m->spec.out_name.size() + 1);
  }
  return need;
}

extern "C" double am_musicnn_flops_per_patch(const am_musicnn* m, int T, int F, double* front_flops) {
  if (!m) return -1.0;
  const MusicnnSpec& s = m->spec;
  double fr = 0.0, tot = 0.0;
  if (s.is_embedding) {
    for (const auto& b : s.br) fr += 2.0 * T * (double)(F - b.kw + 1) * b.cout * b.kh * b.kw;
    tot = fr;
    for (const auto& x : s.mid) tot += 2.0 * T * (double)x.cout * x.cin * x.k;
  }
  for (const auto& h : s.head)
    if (h.kind == kVecLinear) tot += 2.0 * h.K * h.N;
  if (front_flops) *front_flops = fr;
  return tot;
}

extern "C" int am_musicnn_run_dev(am_musicnn* m, const float* in_dev, int n, int T, int F, float* out_dev, void* stream) {
  AM_CHECK(m && in_dev && out_dev, "am_musicnn_run_dev: NULL argument");
  return run_dev(m, in_dev, n, T, F, out_dev, (cudaStream_t)stream);
}

extern "C" int am_musicnn_run(am_musicnn* m, const float* in, int n, int T, int F, float* out) {
  AM_CHECK(m && in && out, "am_musicnn_run: NULL argument");
  AM_CHECK(n >= 0, "am_musicnn_run: n < 0");
  if (n == 0) return AM_OK;
  const size_t nin = (size_t)n * T * F, nout = (size_t)n * m->spec.out_dim;
  AM_TRY(m->io_in.ensure(nin));
  AM_TRY(m->io_out.ensure(nout));
  cudaStream_t st = m->stream.s;
  AM_CUDA(cudaMemcpyAsync(m->io_in.p, in, nin * 4, cudaMemcpyHostToDevice, st));
  AM_TRY(run_dev(m, m->io_in.p, n, T, F, m->io_out.p, st));
  AM_CUDA(cudaMemcpyAsync(out, m->io_out.p, nout * 4, cudaMemcpyDeviceToHost, st));
  AM_CUDA(cudaStreamSynchronize(st));
  return AM_OK;
}

extern "C" int am_musicnn_analyze_tracks(am_musicnn* emb, am_musicnn* pred, const float* pcm, const int64_t* offsets,
                                         int n_tracks, float* emb_out, float* moods_out, int* n_patches) {
  AM_CHECK(emb && emb->spec.is_embedding, "am_musicnn_analyze_tracks: first model must be the embedding graph");
  AM_CHECK(!pred || (!pred->spec.is_embedding && pred->spec.in_dim == emb->spec.out_dim),
           "am_musicnn_analyze_tracks: prediction model must take the %d-wide embedding", emb->spec.out_dim);
  AM_CHECK(pcm && offsets && emb_out && n_patches && n_tracks >= 0, "am_musicnn_analyze_tracks: NULL argument");
  AM_CHECK(!moods_out || pred, "am_musicnn_analyze_tracks: moods need the prediction model");
  if (n_tracks == 0) return AM_OK;
  // tasks/analysis.py:371-381: 16 kHz, n_fft 512, hop 256, 96 mels, center=False, log10(1 + 10000 x), 187-frame patches
  const int kFrames = 187, kMels = 96;
  am_mel_cfg cfg{16000, 512, 256, kMels, 0.f, 8000.f, 1};
  std::vector<int> poff((size_t)n_tracks + 1, 0);
  std::vector<int> frames((size_t)n_tracks, 0);
  for (int t = 0; t < n_tracks; ++t) {
    const int64_t L = offsets[t + 1] - offsets[t];
    AM_CHECK(L >= 0 && L < ((int64_t)1 << 31), "am_musicnn_analyze_tracks: track %d has %lld samples", t, (long long)L);
    const int T = L >= 512 ? am_mel_num_frames_ex(&cfg, 0, (int)L) : 0;
    frames[(size_t)t] = T;
    n_patches[t] = T / kFrames;
    poff[(size_t)t + 1] = poff[(size_t)t] + n_patches[t];
  }
  const int NP = poff[(size_t)n_tracks];
  const int de = emb->spec.out_dim, dl = pred ? pred->spec.out_dim : 0;
  cudaStream_t st = emb->stream.s;
  const int64_t total = offsets[n_tracks] - offsets[0];
  AM_TRY(emb->t_pcm.ensure((size_t)std::max<int64_t>(total, 1)));
  AM_CUDA(cudaMemcpyAsync(emb->t_pcm.p, pcm + offsets[0], (size_t)total * 4, cudaMemcpyHostToDevice, st));
  AM_TRY(emb->t_mel.ensure((size_t)std::max(NP, 1) * kFrames * kMels + (size_t)kFrames * kMels));
  AM_TRY(emb->t_emb.ensure((size_t)std::max(NP, 1) * de));
  if (pred) AM_TRY(emb->t_logit.ensure((size_t)std::max(NP, 1) * dl));
  AM_TRY(emb->t_out_e.ensure((size_t)n_tracks * de));
  AM_TRY(emb->t_out_m.ensure((size_t)n_tracks * std::max(dl, 1)));
  AM_TRY(emb->t_off.ensure((size_t)n_tracks + 1));
  am_mel_plan* plan = nullptr;
  AM_TRY(am_mel_plan_create_ex(&cfg, 0, 1, &plan));
  std::unique_ptr<am_mel_plan, void (*)(am_mel_plan*)> guard(plan, am_mel_plan_free);
  // mel in [T, 96] layout: the first n * 187 frames of a track ARE its n patches
  for (int t = 0; t < n_tracks; ++t) {
    if (n_patches[t] == 0) continue;
    const int64_t L = offsets[t + 1] - offsets[t];
    // only the samples of whole patches: frames [0, n*187) need (n*187 - 1) * 256 + 512 samples
    const int64_t need = (int64_t)(n_patches[t] * kFrames - 1) * 256 + 512;
    AM_TRY(am_mel_batch_dev(plan, emb->t_pcm.p + (offsets[t] - offsets[0]), 0, 1, (int)std::min(L, need),
                            emb->t_mel.p + (size_t)poff[(size_t)t] * kFrames * kMels, st));
  }
  if (NP > 0) {
    AM_TRY(run_dev(emb, emb->t_mel.p, NP, kFrames, kMels, emb->t_emb.p, st));
    if (pred) AM_TRY(run_dev(pred, emb->t_emb.p, NP, de, 1, emb->t_logit.p, st));
  }
  AM_CUDA(cudaMemcpyAsync(emb->t_off.p, poff.data(), poff.size() * 4, cudaMemcpyHostToDevice, st));
  AM_LAUNCH(mx_track_kernel, n_tracks, 256, 0, st, emb->t_emb.p, de, pred ? emb->t_logit.p : nullptr, dl, emb->t_off.p,
            emb->t_out_e.p, pred ? emb->t_out_m.p : nullptr);
  AM_CUDA(cudaMemcpyAsync(emb_out, emb->t_out_e.p, (size_t)n_tracks * de * 4, cudaMemcpyDeviceToHost, st));
  if (moods_out) AM_CUDA(cudaMemcpyAsync(moods_out, emb->t_out_m.p, (size_t)n_tracks * dl * 4, cudaMemcpyDeviceToHost, st));
  AM_CUDA(cudaStreamSynchronize(st));
  return AM_OK;
}
