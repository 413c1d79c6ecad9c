// weights.cc — safetensors reader + BatchNorm folding for the policy/value net.
//
// Replaces the weight hand-off of the reference: VarStore::save (ref: src/learner.rs:192,
// src/learner_concurrent.rs:155-156) -> VarStore::load (ref: src/main.rs:61).  The network
// architecture is model/mod.rs:152-184 + model/connect_four.rs:50-73 (tictactoe.rs:50-73).
//
// Two naming schemes are accepted:
//  (1) explicit: conv{i}.{weight,bias}, bn{i}.{weight,bias,running_mean,running_var} for
//      i = 0 (stem), 1..8 (residual convs), 9 (policy conv), 10 (value conv);
//      policy_fc.{weight,bias}, value_fc.{weight,bias}.
//  (2) tch VarStore root-path names: every layer is created on the SAME nn::Path (model/mod.rs:155-159,
//      connect_four.rs:55-71), so tch de-duplicates names by appending "__{n}" where n is the number
//      of variables created so far.  Tensors are therefore matched by CREATION ORDER (the numeric
//      suffix) within each (name, rank) class.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <functional>
#include <map>
#include <string>
#include <vector>

#include "chess_net.cuh"
#include "evaluator.cuh"
#include "weights.cuh"

namespace spb {
namespace {

// Minimal JSON reader for the safetensors header: {"name": {"dtype": "..", "shape": [..], "data_offsets": [b, e]}, ...}
struct JsonCursor {
  const char* p;
  const char* e;
  bool fail = false;
  void ws() { while (p < e && (*p == ' ' || *p == '\n' || *p == '\t' || *p == '\r')) ++p; }
  bool eat(char c) { ws(); if (p < e && *p == c) { ++p; return true; } return false; }
  std::string str() {
    ws();
    std::string s;
    if (p >= e || *p != '"') { fail = true; return s; }
    ++p;
    while (p < e && *p != '"') {
      if (*p == '\\' && p + 1 < e) { ++p; }
      s.push_back(*p++);
    }
    if (p >= e) { fail = true; return s; }
    ++p;
    return s;
  }
  int64_t num() {
    ws();
    int64_t v = 0;
    bool any = false, neg = false;
    if (p < e && *p == '-') { neg = true; ++p; }
    while (p < e && *p >= '0' && *p <= '9') { v = v * 10 + (*p - '0'); ++p; any = true; }
    if (!any) fail = true;
    return neg ? -v : v;
  }
  void skip_value() {   // skips any JSON value (used for __metadata__)
    ws();
    if (p >= e) { fail = true; return; }
    if (*p == '"') { str(); return; }
    if (*p == '{' || *p == '[') {
      char open = *p, close = (open == '{') ? '}' : ']';
      int depth = 0;
      while (p < e) {
        if (*p == '"') { str(); continue; }
        if (*p == open) ++depth;
        else if (*p == close) { --depth; if (depth == 0) { ++p; return; } }
        ++p;
      }
      fail = true;
      return;
    }
    while (p < e && *p != ',' && *p != '}' && *p != ']') ++p;
  }
};

bool parse_header(const uint8_t* blob, size_t n, std::vector<WeightEntry>* out, size_t* data_off, std::string* err) {
  if (n < 8) { *err = "blob shorter than the 8-byte header length"; return false; }
  uint64_t hlen = 0;
  std::memcpy(&hlen, blob, 8);
  if (hlen > n - 8 || hlen > (1ull << 26)) { *err = "header length out of range"; return false; }
  JsonCursor c{reinterpret_cast<const char*>(blob + 8), reinterpret_cast<const char*>(blob + 8 + hlen)};
  *data_off = 8 + (size_t)hlen;
  if (!c.eat('{')) { *err = "header is not a JSON object"; return false; }
  if (c.eat('}')) return true;
  do {
    std::string name = c.str();
    if (c.fail || !c.eat(':')) { *err = "malformed header near key"; return false; }
    if (name == "__metadata__") { c.skip_value(); if (c.fail) { *err = "malformed __metadata__"; return false; } continue; }
    WeightEntry t;
    t.name = name;
    if (!c.eat('{')) { *err = "tensor entry is not an object: " + name; return false; }
    do {
      std::string k = c.str();
      if (c.fail || !c.eat(':')) { *err = "malformed tensor entry: " + name; return false; }
      if (k == "dtype") t.dtype = c.str();
      else if (k == "shape") {
        if (!c.eat('[')) { *err = "shape is not an array: " + name; return false; }
        if (!c.eat(']')) { do { t.shape.push_back(c.num()); } while (c.eat(',')); if (!c.eat(']')) { *err = "malformed shape: " + name; return false; } }
      } else if (k == "data_offsets") {
        if (!c.eat('[')) { *err = "data_offsets is not an array: " + name; return false; }
        t.begin = (size_t)c.num();
        if (!c.eat(',')) { *err = "malformed data_offsets: " + name; return false; }
        t.end = (size_t)c.num();
        if (!c.eat(']')) { *err = "malformed data_offsets: " + name; return false; }
      } else c.skip_value();
      if (c.fail) { *err = "malformed tensor entry: " + name; return false; }
    } while (c.eat(','));
    if (!c.eat('}')) { *err = "unterminated tensor entry: " + name; return false; }
    out->push_back(t);
  } while (c.eat(','));
  if (!c.eat('}')) { *err = "unterminated header"; return false; }
  return true;
}

bool load_f32(const uint8_t* blob, size_t n, size_t data_off, const WeightEntry& t, std::vector<float>* out, std::string* err) {
  size_t count = 0;
  const size_t esz = element_size(t, &count, err);
  if (esz == 0) return false;
  if (t.end < t.begin || t.end - t.begin != count * esz || data_off + t.end > n) { *err = "data_offsets do not match shape: " + t.name; return false; }
  const uint8_t* src = blob + data_off + t.begin;
  out->resize(count);
  if (t.dtype == "F32") std::memcpy(out->data(), src, count * 4);
  else if (t.dtype == "F64") { for (size_t i = 0; i < count; ++i) { double d; std::memcpy(&d, src + i * 8, 8); (*out)[i] = (float)d; } }
  else { for (size_t i = 0; i < count; ++i) { uint16_t h; std::memcpy(&h, src + i * 2, 2); uint32_t u = (uint32_t)h << 16; std::memcpy(&(*out)[i], &u, 4); } }
  return true;
}

bool shape_is(const WeightEntry& t, std::initializer_list<int64_t> s) { return t.shape == std::vector<int64_t>(s); }

// splits "weight__12" into ("weight", 12); no suffix -> index -1 (the first variable of that name).
void split_suffix(const std::string& name, std::string* base, long* idx) {
  size_t pos = name.rfind("__");
  *base = name;
  *idx = -1;
  if (pos != std::string::npos && pos + 2 < name.size()) {
    bool digits = true;
    for (size_t i = pos + 2; i < name.size(); ++i) digits &= (name[i] >= '0' && name[i] <= '9');
    if (digits) { *base = name.substr(0, pos); *idx = std::stol(name.substr(pos + 2)); }
  }
  // tolerate a leading path component ("net.weight__3")
  size_t dot = base->rfind('.');
  if (dot != std::string::npos) *base = base->substr(dot + 1);
}

// The tch creation-order classes: weights by rank (4: conv, 1: BatchNorm, 2: Linear), biases, running statistics, each
// sorted by the numeric suffix.
struct Census {
  std::vector<size_t> w4, w1, w2, bias, rmean, rvar;
  explicit Census(const std::vector<WeightEntry>& entries) {
    struct Item { long idx; size_t e; };
    std::vector<Item> c[6];
    for (size_t e = 0; e < entries.size(); ++e) {
      const WeightEntry& t = entries[e];
      std::string base; long idx;
      split_suffix(t.name, &base, &idx);
      if (base == "weight") {
        if (t.shape.size() == 4) c[0].push_back({idx, e});
        else if (t.shape.size() == 1) c[1].push_back({idx, e});
        else if (t.shape.size() == 2) c[2].push_back({idx, e});
      } else if (base == "bias") c[3].push_back({idx, e});
      else if (base == "running_mean") c[4].push_back({idx, e});
      else if (base == "running_var") c[5].push_back({idx, e});
    }
    std::vector<size_t>* out[6] = {&w4, &w1, &w2, &bias, &rmean, &rvar};
    for (int k = 0; k < 6; ++k) {
      std::stable_sort(c[k].begin(), c[k].end(), [](const Item& a, const Item& b) { return a.idx < b.idx; });
      for (const Item& it : c[k]) out[k]->push_back(it.e);
    }
  }
};

// Assigns roles and calls take in order; `set(role, entry)` records and takes one role.
struct Assign {
  size_t* role_entry;
  const TakeRole& take;
  std::string* err;
  bool operator()(int role, size_t e) const { role_entry[role] = e; return take(role, e, err); }
};

// The explicit names of conv i: conv{i}.{weight,bias}, bn{i}.{weight,bias,running_mean,running_var}, taken in that order.
bool take_explicit_conv(const std::map<std::string, size_t>& by_name, int i, const Assign& set, std::string* err) {
  const std::string c = "conv" + std::to_string(i), b = "bn" + std::to_string(i);
  const std::string names[6] = {c + ".weight", c + ".bias", b + ".weight", b + ".bias", b + ".running_mean", b + ".running_var"};
  for (int k = 0; k < 6; ++k) {
    auto it = by_name.find(names[k]);
    if (it == by_name.end()) { *err = "missing tensor " + names[k]; return false; }
    if (!set(6 * i + k, it->second)) return false;
  }
  return true;
}

bool take_named(const std::map<std::string, size_t>& by_name, const char* name, int role, const Assign& set, std::string* err) {
  auto it = by_name.find(name);
  if (it == by_name.end()) { *err = std::string("missing tensor ") + name; return false; }
  return set(role, it->second);
}

// The shapes of conv i's six roles: weight [oc][ic][3][3], the rest [oc].
bool conv_shapes_are(const std::vector<WeightEntry>& t, const size_t* re, int i, int oc, int ic) {
  if (!shape_is(t[re[6 * i + ROLE_W]], {oc, ic, 3, 3})) return false;
  for (int k = ROLE_B; k <= ROLE_VAR; ++k)
    if (!shape_is(t[re[6 * i + k]], {oc})) return false;
  return true;
}

// BatchNorm (eval mode) folded into conv i: y = (conv(x)+b - mean) * g / sqrt(var + eps) + beta
template <class Conv>
void fold_conv(const std::vector<float>* raw, int i, int oc, int ic, float eps, Conv* h) {
  const std::vector<float> &w = raw[6 * i + ROLE_W], &b = raw[6 * i + ROLE_B], &g = raw[6 * i + ROLE_G], &beta = raw[6 * i + ROLE_BETA],
                           &mean = raw[6 * i + ROLE_MEAN], &var = raw[6 * i + ROLE_VAR];
  h->oc = oc; h->ic = ic;
  h->w.resize((size_t)oc * ic * 9);
  h->b.resize(oc);
  for (int o = 0; o < oc; ++o) {
    const double s = (double)g[o] / std::sqrt((double)var[o] + (double)eps);
    for (int k = 0; k < ic * 9; ++k) h->w[(size_t)o * ic * 9 + k] = (float)((double)w[(size_t)o * ic * 9 + k] * s);
    h->b[o] = (float)(((double)b[o] - (double)mean[o]) * s + (double)beta[o]);
  }
}

}  // namespace

size_t element_size(const WeightEntry& t, size_t* count, std::string* err) {
  *count = 1;
  for (int64_t d : t.shape) { if (d < 0) { *err = "negative dim: " + t.name; return 0; } *count *= (size_t)d; }
  size_t esz = t.dtype == "F32" ? 4 : (t.dtype == "F64" ? 8 : (t.dtype == "BF16" || t.dtype == "F16" ? 2 : 0));
  if (esz == 0 || t.dtype == "F16") { *err = "unsupported dtype " + t.dtype + " for " + t.name + " (expected F32)"; return 0; }
  return esz;
}

bool resolve_net(const std::vector<WeightEntry>& entries, int game, size_t* re, const TakeRole& take, std::string* err) {
  const int P = game == SPB_GAME_CONNECT4 ? 42 : 9, A = game == SPB_GAME_CONNECT4 ? 7 : 9;
  std::map<std::string, size_t> by_name;
  for (size_t e = 0; e < entries.size(); ++e) by_name[entries[e].name] = e;
  const Assign set{re, take, err};
  if (by_name.count("conv0.weight")) {
    for (int i = 0; i < NET_CONVS; ++i)
      if (!take_explicit_conv(by_name, i, set, err)) return false;
    if (!take_named(by_name, "policy_fc.weight", NET_ROLE_PFC_W, set, err) || !take_named(by_name, "policy_fc.bias", NET_ROLE_PFC_B, set, err) ||
        !take_named(by_name, "value_fc.weight", NET_ROLE_VFC_W, set, err) || !take_named(by_name, "value_fc.bias", NET_ROLE_VFC_B, set, err))
      return false;
  } else {
    // tch creation-order scheme
    const Census c(entries);
    if (c.w4.size() != NET_CONVS || c.w1.size() != NET_CONVS || c.rmean.size() != NET_CONVS || c.rvar.size() != NET_CONVS ||
        c.w2.size() != 2 || c.bias.size() != 2 * NET_CONVS + 2) {
      *err = "unexpected tensor census for the 4x64 ResNet: conv weights " + std::to_string(c.w4.size()) + ", bn weights " +
             std::to_string(c.w1.size()) + ", linear weights " + std::to_string(c.w2.size()) + ", biases " + std::to_string(c.bias.size()) +
             ", running_mean " + std::to_string(c.rmean.size()) + ", running_var " + std::to_string(c.rvar.size());
      return false;
    }
    // bias order: conv0, bn0, ..., conv8, bn8, conv9, bn9, policy_fc, conv10, bn10, value_fc
    int bi = 0;
    for (int i = 0; i < NET_CONVS; ++i) {
      if (!set(6 * i + ROLE_W, c.w4[i]) || !set(6 * i + ROLE_G, c.w1[i]) || !set(6 * i + ROLE_MEAN, c.rmean[i]) || !set(6 * i + ROLE_VAR, c.rvar[i]))
        return false;
      if (!set(6 * i + ROLE_B, c.bias[bi++]) || !set(6 * i + ROLE_BETA, c.bias[bi++])) return false;
      if (i == 9 && !set(NET_ROLE_PFC_B, c.bias[bi++])) return false;
      if (i == 10 && !set(NET_ROLE_VFC_B, c.bias[bi++])) return false;
    }
    if (!set(NET_ROLE_PFC_W, c.w2[0]) || !set(NET_ROLE_VFC_W, c.w2[1])) return false;
  }
  for (int i = 0; i < NET_CONVS; ++i) {
    const int ic = i == 0 ? 3 : NET_HIDDEN;
    const int oc = i <= 8 ? NET_HIDDEN : (i == 9 ? NET_POLICY_CH : NET_VALUE_CH);
    if (!conv_shapes_are(entries, re, i, oc, ic)) { *err = "shape mismatch in conv/bn layer " + std::to_string(i); return false; }
  }
  if (!shape_is(entries[re[NET_ROLE_PFC_W]], {A, NET_POLICY_CH * P}) || !shape_is(entries[re[NET_ROLE_PFC_B]], {A}) ||
      !shape_is(entries[re[NET_ROLE_VFC_W]], {1, NET_VALUE_CH * P}) || !shape_is(entries[re[NET_ROLE_VFC_B]], {1})) {
    *err = "shape mismatch in the policy/value linear layers";
    return false;
  }
  return true;
}

bool parse_safetensors_net(const void* blob_v, size_t n, int game, HostNet* out, std::string* err) {
  const uint8_t* blob = static_cast<const uint8_t*>(blob_v);
  std::vector<WeightEntry> infos;
  size_t data_off = 0;
  if (!parse_header(blob, n, &infos, &data_off, err)) return false;
  out->game = game; out->rows = game == SPB_GAME_CONNECT4 ? 6 : 3; out->cols = game == SPB_GAME_CONNECT4 ? 7 : 3;
  out->actions = game == SPB_GAME_CONNECT4 ? 7 : 9;
  std::vector<float> raw[NET_ROLES];
  size_t re[NET_ROLES];
  const TakeRole load = [&](int role, size_t e, std::string* er) { return load_f32(blob, n, data_off, infos[e], &raw[role], er); };
  if (!resolve_net(infos, game, re, load, err)) return false;
  for (int i = 0; i < NET_CONVS; ++i)
    fold_conv(raw, i, i <= 8 ? NET_HIDDEN : (i == 9 ? NET_POLICY_CH : NET_VALUE_CH), i == 0 ? 3 : NET_HIDDEN, BN_EPS, &out->conv[i]);
  out->pfc_w = raw[NET_ROLE_PFC_W]; out->pfc_b = raw[NET_ROLE_PFC_B]; out->vfc_w = raw[NET_ROLE_VFC_W]; out->vfc_b = raw[NET_ROLE_VFC_B];
  return true;
}


// ---- chess network (ref: src/model/chess.rs:50-73) -------------------------------------------------------------------
// Explicit names: conv{i}.{weight,bias} + bn{i}.{weight,bias,running_mean,running_var} for i = 0 (stem), 1..20 (residual
// convs); policy_conv1 / policy_conv2 / value_conv / value_fc1 / value_fc2 .{weight,bias}.  tch VarStore names: creation
// order as for the small nets — torso (conv, bn) x 21, policy convs, value conv, the two Linear layers.
bool resolve_chess(const std::vector<WeightEntry>& entries, size_t* re, const TakeRole& take, std::string* err) {
  using chess::NET_CONV3; using chess::NET_IN; using chess::NET_MOVE_PLANES;
  constexpr int NET_HIDDEN = chess::NET_HIDDEN;
  std::map<std::string, size_t> by_name;
  for (size_t e = 0; e < entries.size(); ++e) by_name[entries[e].name] = e;
  const Assign set{re, take, err};
  if (by_name.count("conv0.weight")) {
    for (int i = 0; i < NET_CONV3; ++i)
      if (!take_explicit_conv(by_name, i, set, err)) return false;
    static const char* const heads[10] = {"policy_conv1.weight", "policy_conv1.bias", "policy_conv2.weight", "policy_conv2.bias", "value_conv.weight",
                                          "value_conv.bias",     "value_fc1.weight",  "value_fc1.bias",      "value_fc2.weight",  "value_fc2.bias"};
    for (int k = 0; k < 10; ++k)
      if (!take_named(by_name, heads[k], CH_ROLE_P1_W + k, set, err)) return false;
  } else {
    const Census c(entries);
    if (c.w4.size() != NET_CONV3 + 3 || c.w1.size() != NET_CONV3 || c.rmean.size() != NET_CONV3 || c.rvar.size() != NET_CONV3 || c.w2.size() != 2 ||
        c.bias.size() != 2 * NET_CONV3 + 5) {
      *err = "unexpected tensor census for the chess 10x256 ResNet: conv weights " + std::to_string(c.w4.size()) + ", bn weights " +
             std::to_string(c.w1.size()) + ", linear weights " + std::to_string(c.w2.size()) + ", biases " + std::to_string(c.bias.size());
      return false;
    }
    int bi = 0;
    for (int i = 0; i < NET_CONV3; ++i)
      if (!set(6 * i + ROLE_W, c.w4[i]) || !set(6 * i + ROLE_G, c.w1[i]) || !set(6 * i + ROLE_MEAN, c.rmean[i]) || !set(6 * i + ROLE_VAR, c.rvar[i]) ||
          !set(6 * i + ROLE_B, c.bias[bi++]) || !set(6 * i + ROLE_BETA, c.bias[bi++]))
        return false;
    if (!set(CH_ROLE_P1_W, c.w4[NET_CONV3]) || !set(CH_ROLE_P1_B, c.bias[bi++]) || !set(CH_ROLE_P2_W, c.w4[NET_CONV3 + 1]) ||
        !set(CH_ROLE_P2_B, c.bias[bi++]) || !set(CH_ROLE_V_W, c.w4[NET_CONV3 + 2]) || !set(CH_ROLE_V_B, c.bias[bi++]) ||
        !set(CH_ROLE_F1_W, c.w2[0]) || !set(CH_ROLE_F1_B, c.bias[bi++]) || !set(CH_ROLE_F2_W, c.w2[1]) || !set(CH_ROLE_F2_B, c.bias[bi++]))
      return false;
  }
  for (int i = 0; i < NET_CONV3; ++i)
    if (!conv_shapes_are(entries, re, i, NET_HIDDEN, i == 0 ? NET_IN : NET_HIDDEN)) {
      *err = "shape mismatch in conv/bn layer " + std::to_string(i) + " of the chess net";
      return false;
    }
  auto is = [&](int role, std::initializer_list<int64_t> s) { return shape_is(entries[re[role]], s); };
  if (!is(CH_ROLE_P1_W, {NET_HIDDEN, NET_HIDDEN, 1, 1}) || !is(CH_ROLE_P1_B, {NET_HIDDEN}) || !is(CH_ROLE_P2_W, {NET_MOVE_PLANES, NET_HIDDEN, 1, 1}) ||
      !is(CH_ROLE_P2_B, {NET_MOVE_PLANES}) || !is(CH_ROLE_V_W, {1, NET_HIDDEN, 1, 1}) || !is(CH_ROLE_V_B, {1}) || !is(CH_ROLE_F1_W, {256, 64}) ||
      !is(CH_ROLE_F1_B, {256}) || !is(CH_ROLE_F2_W, {1, 256}) || !is(CH_ROLE_F2_B, {1})) {
    *err = "shape mismatch in the heads of the chess net";
    return false;
  }
  return true;
}

namespace chess {

bool parse_safetensors_chess(const void* blob_v, size_t n, HostNet* out, std::string* err) {
  const uint8_t* blob = static_cast<const uint8_t*>(blob_v);
  std::vector<WeightEntry> infos;
  size_t data_off = 0;
  if (!parse_header(blob, n, &infos, &data_off, err)) return false;
  std::vector<float> raw[CH_ROLES];
  size_t re[CH_ROLES];
  const TakeRole load = [&](int role, size_t e, std::string* er) { return load_f32(blob, n, data_off, infos[e], &raw[role], er); };
  if (!resolve_chess(infos, re, load, err)) return false;
  for (int i = 0; i < NET_CONV3; ++i) {
    fold_conv(raw, i, NET_HIDDEN, i == 0 ? NET_IN : NET_HIDDEN, NET_BN_EPS, &out->conv3[i]);
    out->conv3[i].k = 3;
  }
  auto set1x1 = [&](HostNet::Conv& h, int role_w, int oc) { h.oc = oc; h.ic = NET_HIDDEN; h.k = 1; h.w = raw[role_w]; h.b = raw[role_w + 1]; };
  set1x1(out->p1, CH_ROLE_P1_W, NET_HIDDEN);
  set1x1(out->p2, CH_ROLE_P2_W, NET_MOVE_PLANES);
  set1x1(out->vconv, CH_ROLE_V_W, 1);
  out->fc1_w = raw[CH_ROLE_F1_W]; out->fc1_b = raw[CH_ROLE_F1_B]; out->fc2_w = raw[CH_ROLE_F2_W]; out->fc2_b = raw[CH_ROLE_F2_B];
  return true;
}

}  // namespace chess
}  // namespace spb
