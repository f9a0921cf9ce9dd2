// ONNX ModelProto reader shared by the graph loaders (onnx_model.cu: CLAP encoder, musicnn.cu: MusiCNN tower):
// a hand-rolled protobuf wire-format walk into OGraph (nodes, initialisers incl. external data, graph inputs /
// outputs).  There is no protobuf / onnx dependency in the image.
#pragma once

#include "common.cuh"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <map>
#include <string>
#include <vector>

namespace am {
namespace {

// ------------------------------------------------------------------------------------------- protobuf
struct Pb {
  const uint8_t* p;
  const uint8_t* end;
  bool ok = true;
  Pb(const void* d, size_t n) : p((const uint8_t*)d), end((const uint8_t*)d + n) {}
  bool more() const { return ok && p < end; }
  uint64_t varint() {
    uint64_t r = 0;
    for (int s = 0; s < 64; s += 7) {
      if (p >= end) {
        ok = false;
        return 0;
      }
      const uint8_t c = *p++;
      r |= (uint64_t)(c & 0x7f) << s;
      if (!(c & 0x80)) return r;
    }
    ok = false;
    return 0;
  }
  // one field: number, wire type; value in `v` (varint / fixed) or [sub, sub + len)
  bool field(uint32_t* fn, uint32_t* wt, uint64_t* v, const uint8_t** sub, size_t* len) {
    const uint64_t key = varint();
    if (!ok) return false;
    *fn = (uint32_t)(key >> 3);
    *wt = (uint32_t)(key & 7);
    *v = 0;
    *sub = nullptr;
    *len = 0;
    switch (*wt) {
      case 0:
        *v = varint();
        return ok;
      case 1:
        if (end - p < 8) return ok = false;
        std::memcpy(v, p, 8);
        p += 8;
        return true;
      case 5:
        if (end - p < 4) return ok = false;
        std::memcpy(v, p, 4);
        p += 4;
        return true;
      case 2: {
        const uint64_t n = varint();
        if (!ok || n > (uint64_t)(end - p)) return ok = false;
        *sub = p;
        *len = (size_t)n;
        p += n;
        return true;
      }
      default:
        return ok = false;
    }
  }
};

static void packed_ints(uint32_t wt, uint64_t v, const uint8_t* sub, size_t len, std::vector<int64_t>* out) {
  if (wt == 0) {
    out->push_back((int64_t)v);
    return;
  }
  Pb q(sub, len);
  while (q.more()) {
    const uint64_t x = q.varint();
    if (q.ok) out->push_back((int64_t)x);
  }
}
static void packed_floats(uint32_t wt, uint64_t v, const uint8_t* sub, size_t len, std::vector<float>* out) {
  if (wt == 5) {
    float f;
    const uint32_t u = (uint32_t)v;
    std::memcpy(&f, &u, 4);
    out->push_back(f);
    return;
  }
  for (size_t i = 0; i + 4 <= len; i += 4) {
    float f;
    std::memcpy(&f, sub + i, 4);
    out->push_back(f);
  }
}

static float half_to_float(uint16_t h) {
  const uint32_t s = (h >> 15) & 1u, e = (h >> 10) & 31u, m = h & 1023u;
  float v;
  if (e == 0) v = std::ldexp((float)m, -24);
  else if (e == 31) v = m ? NAN : INFINITY;
  else v = std::ldexp((float)(m | 1024u), (int)e - 25);
  return s ? -v : v;
}

struct OTensor {
  std::vector<int64_t> dims;
  int dtype = 1;
  bool is_int = false;
  std::vector<float> f;    // float-typed payloads, converted to fp32
  std::vector<int64_t> i;  // integer-typed payloads
  size_t count() const { return is_int ? i.size() : f.size(); }
  double at(size_t k) const { return is_int ? (double)i[k] : (double)f[k]; }
};

struct OAttr {
  bool has_f = false, has_i = false, has_t = false;
  float f = 0.f;
  int64_t i = 0;
  std::string s;
  OTensor t;
  std::vector<float> floats;
  std::vector<int64_t> ints;
};

struct ONode {
  std::string op, name;
  std::vector<std::string> in, out;
  std::map<std::string, OAttr> attrs;
  bool done = false;
};

struct OGraph {
  std::vector<ONode> nodes;
  std::map<std::string, OTensor> init;
  std::vector<std::string> inputs, outputs;
  int64_t ir_version = 0, opset = 0;
};

static std::string dir_of(const char* path) {
  if (!path) return std::string();
  std::string s(path);
  const size_t k = s.find_last_of('/');
  return k == std::string::npos ? std::string(".") : s.substr(0, k);
}

static int parse_tensor(const uint8_t* d, size_t n, const std::string& base_dir, std::string* name, OTensor* t) {
  Pb pb(d, n);
  uint32_t fn, wt;
  uint64_t v;
  const uint8_t* sub;
  size_t len;
  const uint8_t* raw = nullptr;
  size_t raw_len = 0;
  std::vector<float> f32;
  std::vector<int64_t> i32, i64;
  std::vector<double> f64;
  std::map<std::string, std::string> ext;
  int64_t location = 0;
  while (pb.more() && pb.field(&fn, &wt, &v, &sub, &len)) {
    switch (fn) {
      case 1: packed_ints(wt, v, sub, len, &t->dims); break;
      case 2: t->dtype = (int)v; break;
      case 4: packed_floats(wt, v, sub, len, &f32); break;
      case 5: packed_ints(wt, v, sub, len, &i32); break;
      case 7: packed_ints(wt, v, sub, len, &i64); break;
      case 8: name->assign((const char*)sub, len); break;
      case 9: raw = sub; raw_len = len; break;
      case 10:
        if (wt == 1) {
          double x;
          std::memcpy(&x, &v, 8);
          f64.push_back(x);
        } else {
          for (size_t k = 0; k + 8 <= len; k += 8) {
            double x;
            std::memcpy(&x, sub + k, 8);
            f64.push_back(x);
          }
        }
        break;
      case 13: {
        Pb kv(sub, len);
        std::string key, val;
        uint32_t f2, w2;
        uint64_t v2;
        const uint8_t* s2;
        size_t l2;
        while (kv.more() && kv.field(&f2, &w2, &v2, &s2, &l2)) {
          if (f2 == 1) key.assign((const char*)s2, l2);
          if (f2 == 2) val.assign((const char*)s2, l2);
        }
        ext[key] = val;
        break;
      }
      case 14: location = (int64_t)v; break;
      default: break;
    }
  }
  if (!pb.ok) {
    set_error("onnx: malformed TensorProto");
    return AM_ERR_IO;
  }
  std::vector<uint8_t> ext_buf;
  if (location == 1 || !ext.empty()) {  // external data (model.onnx.data next to the model, clap_analyzer.py:132-147)
    if (base_dir.empty() || !ext.count("location")) {
      set_error("onnx: tensor %s uses external data but the model was given without a path", name->c_str());
      return AM_ERR_IO;
    }
    const std::string fp = base_dir + "/" + ext["location"];
    FILE* f = std::fopen(fp.c_str(), "rb");
    if (!f) {
      set_error("onnx: cannot open external data file %s (tensor %s)", fp.c_str(), name->c_str());
      return AM_ERR_IO;
    }
    const long long off = ext.count("offset") ? std::atoll(ext["offset"].c_str()) : 0;
    long long length = ext.count("length") ? std::atoll(ext["length"].c_str()) : -1;
    if (length < 0) {
      std::fseek(f, 0, SEEK_END);
      length = std::ftell(f) - off;
    }
    ext_buf.resize((size_t)std::max<long long>(length, 0));
    std::fseek(f, (long)off, SEEK_SET);
    const size_t got = ext_buf.empty() ? 0 : std::fread(ext_buf.data(), 1, ext_buf.size(), f);
    std::fclose(f);
    if (got != ext_buf.size()) {
      set_error("onnx: short read of external data for tensor %s", name->c_str());
      return AM_ERR_IO;
    }
    raw = ext_buf.data();
    raw_len = ext_buf.size();
  }
  size_t count = 1;
  for (int64_t x : t->dims) count *= (size_t)std::max<int64_t>(x, 0);
  switch (t->dtype) {
    case 1:  // float
      if (raw) {
        t->f.resize(raw_len / 4);
        std::memcpy(t->f.data(), raw, t->f.size() * 4);
      } else {
        t->f = f32;
      }
      break;
    case 10:  // float16 (raw, or int32_data holding the bit patterns)
      if (raw) {
        t->f.resize(raw_len / 2);
        for (size_t k = 0; k < t->f.size(); ++k) {
          uint16_t h;
          std::memcpy(&h, raw + 2 * k, 2);
          t->f[k] = half_to_float(h);
        }
      } else {
        for (int64_t h : i32) t->f.push_back(half_to_float((uint16_t)h));
      }
      break;
    case 11:  // double
      if (raw) {
        t->f.resize(raw_len / 8);
        for (size_t k = 0; k < t->f.size(); ++k) {
          double x;
          std::memcpy(&x, raw + 8 * k, 8);
          t->f[k] = (float)x;
        }
      } else {
        for (double x : f64) t->f.push_back((float)x);
      }
      break;
    case 7:  // int64
      t->is_int = true;
      if (raw) {
        t->i.resize(raw_len / 8);
        std::memcpy(t->i.data(), raw, t->i.size() * 8);
      } else {
        t->i = i64;
      }
      break;
    case 6:  // int32
      t->is_int = true;
      if (raw) {
        t->i.resize(raw_len / 4);
        for (size_t k = 0; k < t->i.size(); ++k) {
          int32_t x;
          std::memcpy(&x, raw + 4 * k, 4);
          t->i[k] = x;
        }
      } else {
        t->i = i32;
      }
      break;
    case 9:  // bool
      t->is_int = true;
      if (raw) for (size_t k = 0; k < raw_len; ++k) t->i.push_back(raw[k]);
      else t->i = i32;
      break;
    default:
      set_error("onnx: tensor %s has unsupported data_type %d", name->c_str(), t->dtype);
      return AM_ERR_INVALID;
  }
  if (t->count() != count) {
    set_error("onnx: tensor %s holds %zu elements, its dims say %zu", name->c_str(), t->count(), count);
    return AM_ERR_IO;
  }
  return AM_OK;
}

static int parse_attr(const uint8_t* d, size_t n, const std::string& base_dir, std::string* name, OAttr* a) {
  Pb pb(d, n);
  uint32_t fn, wt;
  uint64_t v;
  const uint8_t* sub;
  size_t len;
  while (pb.more() && pb.field(&fn, &wt, &v, &sub, &len)) {
    switch (fn) {
      case 1: name->assign((const char*)sub, len); break;
      case 2: {
        const uint32_t u = (uint32_t)v;
        std::memcpy(&a->f, &u, 4);
        a->has_f = true;
        break;
      }
      case 3: a->i = (int64_t)v; a->has_i = true; break;
      case 4: a->s.assign((const char*)sub, len); break;
      case 5: {
        std::string tn;
        AM_TRY(parse_tensor(sub, len, base_dir, &tn, &a->t));
        a->has_t = true;
        break;
      }
      case 7: packed_floats(wt, v, sub, len, &a->floats); break;
      case 8: packed_ints(wt, v, sub, len, &a->ints); break;
      default: break;
    }
  }
  if (!pb.ok) {
    set_error("onnx: malformed AttributeProto");
    return AM_ERR_IO;
  }
  return AM_OK;
}

static int parse_node(const uint8_t* d, size_t n, const std::string& base_dir, ONode* node) {
  Pb pb(d, n);
  uint32_t fn, wt;
  uint64_t v;
  const uint8_t* sub;
  size_t len;
  while (pb.more() && pb.field(&fn, &wt, &v, &sub, &len)) {
    switch (fn) {
      case 1: node->in.emplace_back((const char*)sub, len); break;
      case 2: node->out.emplace_back((const char*)sub, len); break;
      case 3: node->name.assign((const char*)sub, len); break;
      case 4: node->op.assign((const char*)sub, len); break;
      case 5: {
        std::string an;
        OAttr a;
        AM_TRY(parse_attr(sub, len, base_dir, &an, &a));
        node->attrs[an] = std::move(a);
        break;
      }
      default: break;
    }
  }
  if (!pb.ok) {
    set_error("onnx: malformed NodeProto");
    return AM_ERR_IO;
  }
  return AM_OK;
}

static std::string value_info_name(const uint8_t* d, size_t n) {
  Pb pb(d, n);
  uint32_t fn, wt;
  uint64_t v;
  const uint8_t* sub;
  size_t len;
  while (pb.more() && pb.field(&fn, &wt, &v, &sub, &len))
    if (fn == 1) return std::string((const char*)sub, len);
  return std::string();
}

static int parse_model(const void* data, size_t nbytes, const std::string& base_dir, OGraph* g) {
  Pb pb(data, nbytes);
  uint32_t fn, wt;
  uint64_t v;
  const uint8_t* sub;
  size_t len;
  bool saw_graph = false;
  while (pb.more() && pb.field(&fn, &wt, &v, &sub, &len)) {
    if (fn == 1 && wt == 0) g->ir_version = (int64_t)v;
    if (fn == 8 && wt == 2) {  // opset_import
      Pb q(sub, len);
      uint32_t f2, w2;
      uint64_t v2;
      const uint8_t* s2;
      size_t l2;
      std::string domain;
      int64_t ver = 0;
      while (q.more() && q.field(&f2, &w2, &v2, &s2, &l2)) {
        if (f2 == 1) domain.assign((const char*)s2, l2);
        if (f2 == 2) ver = (int64_t)v2;
      }
      if (domain.empty() || domain == "ai.onnx") g->opset = std::max(g->opset, ver);
    }
    if (fn == 7 && wt == 2) {  // graph
      saw_graph = true;
      Pb q(sub, len);
      uint32_t f2, w2;
      uint64_t v2;
      const uint8_t* s2;
      size_t l2;
      while (q.more() && q.field(&f2, &w2, &v2, &s2, &l2)) {
        if (f2 == 1) {
          ONode node;
          AM_TRY(parse_node(s2, l2, base_dir, &node));
          g->nodes.push_back(std::move(node));
        } else if (f2 == 5) {
          std::string tn;
          OTensor t;
          AM_TRY(parse_tensor(s2, l2, base_dir, &tn, &t));
          g->init[tn] = std::move(t);
        } else if (f2 == 11) {
          g->inputs.push_back(value_info_name(s2, l2));
        } else if (f2 == 12) {
          g->outputs.push_back(value_info_name(s2, l2));
        }
      }
      if (!q.ok) {
        set_error("onnx: malformed GraphProto");
        return AM_ERR_IO;
      }
    }
  }
  if (!pb.ok || !saw_graph || g->nodes.empty()) {
    set_error("onnx: not a ModelProto with a graph (parse %s, %zu nodes)", pb.ok ? "ok" : "failed", g->nodes.size());
    return AM_ERR_IO;
  }
  std::vector<std::string> real_inputs;
  for (const auto& s : g->inputs)
    if (!g->init.count(s)) real_inputs.push_back(s);
  g->inputs = real_inputs;
  return AM_OK;
}

}  // namespace
}  // namespace am
