// forest.cpp — model-file readers/writers and the depth-ordered flattening.  See forest.hpp.
//
// File formats follow XGBoost 1.6.0 (the version the reference pins,
// /root/reference/Shared/CMakeLists.txt:8) as published:
//   legacy binary: LearnerIO::LoadModel (src/learner.cc), GBTreeModel::Load
//                  (src/gbm/gbtree_model.cc), RegTree::Load (src/tree/tree_model.cc);
//                  strings / vectors are dmlc-serializer uint64-length-prefixed
//   JSON / UBJSON: doc/model.schema; UBJSON is draft-12, big-endian, typed arrays
#include "forest.hpp"
#include "kernels.hpp"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <map>
#include <memory>
#include <stdexcept>

namespace qcoh {
namespace {

[[noreturn]] void fail(const std::string &m) { throw std::runtime_error(m); }

// ------------------------------------------------------------------------------------
// tiny DOM shared by the JSON and UBJSON readers
// ------------------------------------------------------------------------------------
struct JV {
  enum Kind { Null, Bool, Num, Str, Arr, Obj, F32A, I64A } kind = Null;
  bool b = false;
  double num = 0;
  float f32 = 0;  // the same token parsed straight to float (strtof), no double rounding
  bool is_int = false;
  int64_t i64 = 0;
  std::string str;
  std::vector<JV> arr;
  std::vector<std::pair<std::string, JV>> obj;
  std::vector<float> f32a;    // UBJSON typed arrays
  std::vector<int64_t> i64a;

  const JV &at(const char *key) const {
    if (kind != Obj) fail(std::string("model: expected an object around key '") + key + "'");
    for (auto &kv : obj)
      if (kv.first == key) return kv.second;
    fail(std::string("model: missing key '") + key + "'");
  }
  const JV *find(const char *key) const {
    if (kind != Obj) return nullptr;
    for (auto &kv : obj)
      if (kv.first == key) return &kv.second;
    return nullptr;
  }
  size_t size() const {
    switch (kind) {
      case Arr: return arr.size();
      case F32A: return f32a.size();
      case I64A: return i64a.size();
      default: fail("model: expected an array");
    }
  }
  int64_t as_int() const {
    if (kind == Num) return is_int ? i64 : (int64_t)num;
    if (kind == Bool) return b;
    if (kind == Str) return strtoll(str.c_str(), nullptr, 10);
    fail("model: expected an integer");
  }
  float as_float() const {
    if (kind == Num) return f32;
    if (kind == Str) return strtof(str.c_str(), nullptr);
    fail("model: expected a number");
  }
  int64_t int_at(size_t i) const {
    if (kind == I64A) return i64a[i];
    if (kind == F32A) return (int64_t)f32a[i];
    return arr[i].as_int();
  }
  float float_at(size_t i) const {
    if (kind == F32A) return f32a[i];
    if (kind == I64A) return (float)i64a[i];
    return arr[i].as_float();
  }
};

struct JsonReader {
  const char *p, *end;
  void ws() {
    while (p < end && (*p == ' ' || *p == '\n' || *p == '\t' || *p == '\r')) ++p;
  }
  [[noreturn]] void err(const char *what) {
    fail(std::string("JSON model: ") + what + " at byte " + std::to_string((long)(p - (end - (end - p)))));
  }
  std::string string() {
    if (*p != '"') fail("JSON model: expected string");
    ++p;
    std::string s;
    while (p < end && *p != '"') {
      if (*p == '\\' && p + 1 < end) {
        ++p;
        switch (*p) {
          case 'n': s += '\n'; break;
          case 't': s += '\t'; break;
          case 'r': s += '\r'; break;
          case 'b': s += '\b'; break;
          case 'f': s += '\f'; break;
          case 'u': {
            if (p + 4 >= end) fail("JSON model: bad \\u escape");
            unsigned cp = (unsigned)strtoul(std::string(p + 1, p + 5).c_str(), nullptr, 16);
            if (cp < 0x80) s += (char)cp;
            else if (cp < 0x800) { s += (char)(0xC0 | (cp >> 6)); s += (char)(0x80 | (cp & 0x3F)); }
            else { s += (char)(0xE0 | (cp >> 12)); s += (char)(0x80 | ((cp >> 6) & 0x3F)); s += (char)(0x80 | (cp & 0x3F)); }
            p += 4;
            break;
          }
          default: s += *p;
        }
        ++p;
      } else {
        s += *p++;
      }
    }
    if (p >= end) fail("JSON model: unterminated string");
    ++p;
    return s;
  }
  JV value(int depth = 0) {
    if (depth > 64) fail("JSON model: nesting too deep");
    ws();
    if (p >= end) fail("JSON model: unexpected end of file");
    JV v;
    char c = *p;
    if (c == '{') {
      v.kind = JV::Obj;
      ++p;
      ws();
      if (p < end && *p == '}') { ++p; return v; }
      while (true) {
        ws();
        std::string k = string();
        ws();
        if (p >= end || *p != ':') fail("JSON model: expected ':'");
        ++p;
        v.obj.emplace_back(std::move(k), value(depth + 1));
        ws();
        if (p < end && *p == ',') { ++p; continue; }
        if (p < end && *p == '}') { ++p; break; }
        fail("JSON model: expected ',' or '}'");
      }
    } else if (c == '[') {
      v.kind = JV::Arr;
      ++p;
      ws();
      if (p < end && *p == ']') { ++p; return v; }
      while (true) {
        v.arr.push_back(value(depth + 1));
        ws();
        if (p < end && *p == ',') { ++p; continue; }
        if (p < end && *p == ']') { ++p; break; }
        fail("JSON model: expected ',' or ']'");
      }
    } else if (c == '"') {
      v.kind = JV::Str;
      v.str = string();
    } else if (c == 't' && end - p >= 4 && !memcmp(p, "true", 4)) {
      v.kind = JV::Bool, v.b = true, p += 4;
    } else if (c == 'f' && end - p >= 5 && !memcmp(p, "false", 5)) {
      v.kind = JV::Bool, v.b = false, p += 5;
    } else if (c == 'n' && end - p >= 4 && !memcmp(p, "null", 4)) {
      p += 4;
    } else {
      // number (XGBoost also writes NaN / Infinity / -Infinity tokens)
      char tok[64];
      size_t n = 0;
      while (p < end && n < sizeof tok - 1 &&
             (strchr("+-.eE", *p) || (*p >= '0' && *p <= '9') || (*p >= 'A' && *p <= 'Z') || (*p >= 'a' && *p <= 'z')))
        tok[n++] = *p++;
      tok[n] = 0;
      if (!n) fail("JSON model: unexpected character");
      char *e1 = nullptr;
      v.kind = JV::Num;
      v.num = strtod(tok, &e1);
      if (e1 == tok) fail(std::string("JSON model: bad number '") + tok + "'");
      v.f32 = strtof(tok, nullptr);
      v.is_int = !strpbrk(tok, ".eEnN");
      if (v.is_int) v.i64 = strtoll(tok, nullptr, 10);
    }
    return v;
  }
};

struct UbjReader {
  const unsigned char *p, *end;
  void need(size_t n) {
    if ((size_t)(end - p) < n) fail("UBJSON model: truncated");
  }
  template <class T>
  T be() {
    need(sizeof(T));
    unsigned char t[sizeof(T)];
    for (size_t i = 0; i < sizeof(T); ++i) t[i] = p[sizeof(T) - 1 - i];
    p += sizeof(T);
    T v;
    memcpy(&v, t, sizeof(T));
    return v;
  }
  int64_t integer(char m) {
    switch (m) {
      case 'i': return be<int8_t>();
      case 'U': return be<uint8_t>();
      case 'I': return be<int16_t>();
      case 'l': return be<int32_t>();
      case 'L': return be<int64_t>();
      default: fail("UBJSON model: expected an integer marker");
    }
  }
  char marker() {
    need(1);
    return (char)*p++;
  }
  std::string string() {
    int64_t n = integer(marker());
    if (n < 0) fail("UBJSON model: negative string length");
    need((size_t)n);
    std::string s((const char *)p, (size_t)n);
    p += n;
    return s;
  }
  JV value(char m = 0, int depth = 0) {
    if (depth > 64) fail("UBJSON model: nesting too deep");
    if (!m) m = marker();
    JV v;
    switch (m) {
      case '{': {
        v.kind = JV::Obj;
        while (true) {
          need(1);
          if (*p == '}') { ++p; break; }
          std::string k = string();
          v.obj.emplace_back(std::move(k), value(0, depth + 1));
        }
        break;
      }
      case '[': {
        need(1);
        if (*p == '$') {
          ++p;
          char ty = marker();
          if (marker() != '#') fail("UBJSON model: typed array without count");
          int64_t n = integer(marker());
          if (n < 0) fail("UBJSON model: negative array length");
          const size_t elem = ty == 'D' || ty == 'L' ? 8 : ty == 'd' || ty == 'l' ? 4 : ty == 'I' ? 2 : 1;
          if ((uint64_t)n > (uint64_t)(end - p) / elem) fail("UBJSON model: typed array longer than the file");
          if (ty == 'd' || ty == 'D') {
            v.kind = JV::F32A;
            v.f32a.resize((size_t)n);
            for (int64_t i = 0; i < n; ++i) v.f32a[i] = ty == 'd' ? be<float>() : (float)be<double>();
          } else {
            v.kind = JV::I64A;
            v.i64a.resize((size_t)n);
            for (int64_t i = 0; i < n; ++i) v.i64a[i] = integer(ty);
          }
        } else if (*p == '#') {
          ++p;
          int64_t n = integer(marker());
          v.kind = JV::Arr;
          for (int64_t i = 0; i < n; ++i) v.arr.push_back(value(0, depth + 1));
        } else {
          v.kind = JV::Arr;
          while (true) {
            need(1);
            if (*p == ']') { ++p; break; }
            v.arr.push_back(value(0, depth + 1));
          }
        }
        break;
      }
      case 'S': v.kind = JV::Str, v.str = string(); break;
      case 'C': v.kind = JV::Str, v.str = std::string(1, marker()); break;
      case 'T': v.kind = JV::Bool, v.b = true; break;
      case 'F': v.kind = JV::Bool, v.b = false; break;
      case 'Z': case 'N': break;
      case 'd': v.kind = JV::Num, v.f32 = be<float>(), v.num = v.f32; break;
      case 'D': v.kind = JV::Num, v.num = be<double>(), v.f32 = (float)v.num; break;
      case 'i': case 'U': case 'I': case 'l': case 'L':
        v.kind = JV::Num, v.is_int = true, v.i64 = integer(m), v.num = (double)v.i64, v.f32 = (float)v.i64;
        break;
      default: fail(std::string("UBJSON model: unknown marker '") + m + "'");
    }
    return v;
  }
};

void check_objective(const std::string &name) {
  // Only identity PredTransform objectives (src/objective/regression_obj.cu); reg:linear is the
  // pre-1.0 alias found in 0.81-era files (OH_instance_OH.rc:18).
  if (name != "reg:squarederror" && name != "reg:linear")
    fail("Unsupported objective '" + name + "': libqcoh implements reg:squarederror (identity transform) only");
}

void validate_tree(const HostTree &t, uint32_t num_feature, size_t ti) {
  const int32_t n = t.num_nodes();
  if (n <= 0) fail("tree " + std::to_string(ti) + ": no nodes");
  for (int32_t i = 0; i < n; ++i) {
    if (t.cleft[i] == -1) continue;
    if (t.cleft[i] < 0 || t.cleft[i] >= n || t.cright[i] < 0 || t.cright[i] >= n)
      fail("tree " + std::to_string(ti) + " node " + std::to_string(i) + ": child index out of range");
    if ((t.sindex[i] & 0x7FFFFFFFu) >= num_feature)
      fail("tree " + std::to_string(ti) + " node " + std::to_string(i) + ": split feature out of range");
  }
}

HostForest from_dom(const JV &root, ModelFormat fmt) {
  HostForest f;
  f.format = fmt;
  if (const JV *ver = root.find("version"))
    for (size_t i = 0; i < 3 && i < ver->size(); ++i) f.version[i] = (uint32_t)ver->int_at(i);
  const JV &lr = root.at("learner");
  const JV &lmp = lr.at("learner_model_param");
  f.base_score = lmp.at("base_score").as_float();
  f.num_feature = (uint32_t)lmp.at("num_feature").as_int();
  if (const JV *nc = lmp.find("num_class"))
    if (nc->as_int() > 1) fail("multi-class boosters are not supported");
  f.objective = lr.at("objective").at("name").str;
  check_objective(f.objective);
  if (const JV *at = lr.find("attributes"))
    if (at->kind == JV::Obj)
      for (auto &kv : at->obj) f.attributes.emplace_back(kv.first, kv.second.str);
  const JV &gb = lr.at("gradient_booster");
  if (gb.at("name").str != "gbtree") fail("Unsupported booster '" + gb.at("name").str + "' (gbtree only)");
  const JV &model = gb.at("model");
  const int64_t ntree = model.at("gbtree_model_param").at("num_trees").as_int();
  const JV &trees = model.at("trees");
  if ((int64_t)trees.size() != ntree) fail("JSON model: num_trees does not match the trees array");
  const JV &ti = model.at("tree_info");
  for (size_t i = 0; i < ti.size(); ++i) f.tree_info.push_back((int32_t)ti.int_at(i));
  f.trees.resize((size_t)ntree);
  for (int64_t t = 0; t < ntree; ++t) {
    const JV &jt = trees.arr[(size_t)t];
    const JV &L = jt.at("left_children"), &R = jt.at("right_children"), &P = jt.at("parents");
    const JV &SI = jt.at("split_indices"), &SC = jt.at("split_conditions"), &DL = jt.at("default_left");
    const size_t n = L.size();
    if ((int64_t)n != jt.at("tree_param").at("num_nodes").as_int() || R.size() != n || SI.size() != n ||
        SC.size() != n || DL.size() != n)
      fail("JSON model: tree " + std::to_string(t) + " array lengths disagree with num_nodes");
    if (const JV *st = jt.find("split_type"))
      for (size_t i = 0; i < st->size(); ++i)
        if (st->int_at(i) != 0) fail("categorical splits are not supported");
    HostTree &ht = f.trees[(size_t)t];
    ht.cleft.resize(n), ht.cright.resize(n), ht.parent.resize(n), ht.sindex.resize(n), ht.info.resize(n);
    ht.loss_chg.assign(n, 0.f), ht.sum_hess.assign(n, 0.f), ht.base_weight.assign(n, 0.f), ht.leaf_child_cnt.assign(n, 0);
    const JV *LC = jt.find("loss_changes"), *SH = jt.find("sum_hessian"), *BW = jt.find("base_weights");
    for (size_t i = 0; i < n; ++i) {
      ht.cleft[i] = (int32_t)L.int_at(i);
      ht.cright[i] = (int32_t)R.int_at(i);
      ht.info[i] = SC.float_at(i);
      ht.sindex[i] = (uint32_t)SI.int_at(i) | (DL.int_at(i) ? 0x80000000u : 0u);
      if (LC && LC->size() == n) ht.loss_chg[i] = LC->float_at(i);
      if (SH && SH->size() == n) ht.sum_hess[i] = SH->float_at(i);
      if (BW && BW->size() == n) ht.base_weight[i] = BW->float_at(i);
    }
    // legacy parent encoding: bit31 = is-left-child, root = -1
    for (size_t i = 0; i < n; ++i) ht.parent[i] = -1;
    for (size_t i = 0; i < n; ++i) {
      if (ht.cleft[i] == -1) continue;
      if (ht.cleft[i] < 0 || (size_t)ht.cleft[i] >= n || ht.cright[i] < 0 || (size_t)ht.cright[i] >= n)
        fail("tree " + std::to_string(t) + " node " + std::to_string(i) + ": child index out of range");
      ht.parent[(size_t)ht.cleft[i]] = (int32_t)((uint32_t)i | 0x80000000u);
      ht.parent[(size_t)ht.cright[i]] = (int32_t)i;
    }
    (void)P;
    validate_tree(ht, f.num_feature, (size_t)t);
  }
  return f;
}

// ------------------------------------------------------------------------------------
// legacy binary
// ------------------------------------------------------------------------------------
struct Rd {
  const unsigned char *p, *end;
  void bytes(void *dst, size_t n) {
    if ((size_t)(end - p) < n) fail("Truncated legacy binary model file");
    memcpy(dst, p, n);
    p += n;
  }
  std::string str() {
    uint64_t n;
    bytes(&n, 8);
    if ((uint64_t)(end - p) < n) fail("Truncated legacy binary model file");
    std::string s((const char *)p, (size_t)n);
    p += n;
    return s;
  }
};

#pragma pack(push, 1)
struct LearnerModelParamLegacy {  // 136 B
  float base_score;
  uint32_t num_feature;
  int32_t num_class, contain_extra_attrs, contain_eval_metrics;
  uint32_t major_version, minor_version, num_target;
  int32_t reserved[26];
};
struct GBTreeModelParam {  // 160 B
  int32_t num_trees, num_roots, num_feature, pad;
  int64_t num_pbuffer;
  int32_t num_output_group, size_leaf_vector;
  int32_t reserved[32];
};
struct TreeParam {  // 148 B
  int32_t num_roots, num_nodes, num_deleted, max_depth, num_feature, size_leaf_vector;
  int32_t reserved[31];
};
struct DiskNode {  // 20 B
  int32_t parent, cleft, cright;
  uint32_t sindex;
  float info;
};
struct DiskStat {  // 16 B
  float loss_chg, sum_hess, base_weight;
  int32_t leaf_child_cnt;
};
#pragma pack(pop)
static_assert(sizeof(LearnerModelParamLegacy) == 136 && sizeof(GBTreeModelParam) == 160 && sizeof(TreeParam) == 148 &&
                  sizeof(DiskNode) == 20 && sizeof(DiskStat) == 16,
              "legacy layouts");

HostForest load_legacy(const unsigned char *buf, size_t len) {
  Rd r{buf, buf + len};
  if (len >= 4 && !memcmp(buf, "binf", 4)) r.p += 4;
  HostForest f;
  f.format = kLegacyBinary;
  LearnerModelParamLegacy mp;
  r.bytes(&mp, sizeof mp);
  f.base_score = mp.base_score;
  f.num_feature = mp.num_feature;
  f.version[0] = mp.major_version, f.version[1] = mp.minor_version, f.version[2] = 0;
  if (mp.num_class > 1) fail("multi-class boosters are not supported");
  f.objective = r.str();
  std::string booster = r.str();
  if (booster != "gbtree") fail("Unsupported booster '" + booster + "' (gbtree only)");
  check_objective(f.objective);
  GBTreeModelParam gp;
  r.bytes(&gp, sizeof gp);
  if (gp.num_trees < 0) fail("Invalid legacy binary model: negative num_trees");
  if (gp.size_leaf_vector != 0) fail("size_leaf_vector != 0 is not supported");
  f.trees.resize((size_t)gp.num_trees);
  for (int32_t t = 0; t < gp.num_trees; ++t) {
    TreeParam tp;
    r.bytes(&tp, sizeof tp);
    if (tp.num_nodes <= 0) fail("Invalid legacy binary model: tree " + std::to_string(t) + " has no nodes");
    if ((uint64_t)(r.end - r.p) < (uint64_t)tp.num_nodes * 36) fail("Truncated legacy binary model file");
    const size_t n = (size_t)tp.num_nodes;
    HostTree &ht = f.trees[(size_t)t];
    ht.cleft.resize(n), ht.cright.resize(n), ht.parent.resize(n), ht.sindex.resize(n), ht.info.resize(n);
    ht.loss_chg.resize(n), ht.sum_hess.resize(n), ht.base_weight.resize(n), ht.leaf_child_cnt.resize(n);
    for (size_t i = 0; i < n; ++i) {
      DiskNode d;
      r.bytes(&d, sizeof d);
      ht.parent[i] = d.parent, ht.cleft[i] = d.cleft, ht.cright[i] = d.cright, ht.sindex[i] = d.sindex, ht.info[i] = d.info;
    }
    for (size_t i = 0; i < n; ++i) {
      DiskStat s;
      r.bytes(&s, sizeof s);
      ht.loss_chg[i] = s.loss_chg, ht.sum_hess[i] = s.sum_hess, ht.base_weight[i] = s.base_weight;
      ht.leaf_child_cnt[i] = s.leaf_child_cnt;
    }
    validate_tree(ht, f.num_feature, (size_t)t);
  }
  f.tree_info.resize((size_t)gp.num_trees);
  if (gp.num_trees) r.bytes(f.tree_info.data(), sizeof(int32_t) * (size_t)gp.num_trees);
  if (mp.contain_extra_attrs && r.p < r.end) {
    uint64_t na;
    r.bytes(&na, 8);
    for (uint64_t i = 0; i < na; ++i) {
      std::string k = r.str();
      std::string v = r.str();
      f.attributes.emplace_back(k, v);
    }
  }
  // metric names (contain_eval_metrics) do not affect prediction
  return f;
}

void wstr(std::string &o, const std::string &s) {
  uint64_t n = s.size();
  o.append((const char *)&n, 8);
  o += s;
}

std::string legacy_bytes(const HostForest &f) {
  std::string o = "binf";
  LearnerModelParamLegacy mp;
  memset(&mp, 0, sizeof mp);
  mp.base_score = f.base_score, mp.num_feature = f.num_feature;
  mp.contain_extra_attrs = f.attributes.empty() ? 0 : 1;
  mp.major_version = f.version[0], mp.minor_version = f.version[1], mp.num_target = 1;
  o.append((const char *)&mp, sizeof mp);
  wstr(o, f.objective);
  wstr(o, "gbtree");
  GBTreeModelParam gp;
  memset(&gp, 0, sizeof gp);
  gp.num_trees = (int32_t)f.trees.size(), gp.num_roots = 1, gp.num_feature = (int32_t)f.num_feature, gp.num_output_group = 1;
  o.append((const char *)&gp, sizeof gp);
  for (auto &t : f.trees) {
    TreeParam tp;
    memset(&tp, 0, sizeof tp);
    tp.num_roots = 1, tp.num_nodes = t.num_nodes(), tp.num_feature = (int32_t)f.num_feature;
    o.append((const char *)&tp, sizeof tp);
    for (int32_t i = 0; i < t.num_nodes(); ++i) {
      DiskNode d{t.parent[i], t.cleft[i], t.cright[i], t.sindex[i], t.info[i]};
      o.append((const char *)&d, sizeof d);
    }
    for (int32_t i = 0; i < t.num_nodes(); ++i) {
      DiskStat s{t.loss_chg[i], t.sum_hess[i], t.base_weight[i], t.leaf_child_cnt[i]};
      o.append((const char *)&s, sizeof s);
    }
  }
  for (size_t i = 0; i < f.trees.size(); ++i) {
    int32_t g = i < f.tree_info.size() ? f.tree_info[i] : 0;
    o.append((const char *)&g, 4);
  }
  if (!f.attributes.empty()) {
    uint64_t na = f.attributes.size();
    o.append((const char *)&na, 8);
    for (auto &kv : f.attributes) wstr(o, kv.first), wstr(o, kv.second);
  }
  return o;
}

// shortest decimal that round-trips through float32
std::string f32_repr(float v) {
  if (std::isnan(v)) return "NaN";
  if (std::isinf(v)) return v > 0 ? "Infinity" : "-Infinity";
  char b[40];
  for (int prec = 1; prec <= 9; ++prec) {
    snprintf(b, sizeof b, "%.*E", prec - 1, (double)v);
    if (strtof(b, nullptr) == v) break;
  }
  return b;
}

int32_t json_parent(const HostTree &t, int32_t i) {
  return t.parent[i] == -1 ? 2147483647 : (int32_t)((uint32_t)t.parent[i] & 0x7FFFFFFFu);
}

std::string json_text(const HostForest &f) {
  std::string o;
  o.reserve(64 + 200 * (size_t)f.trees.size());
  auto arr = [&](const char *key, size_t n, auto &&item) {
    o += '"', o += key, o += "\":[";
    for (size_t i = 0; i < n; ++i) {
      if (i) o += ',';
      o += item(i);
    }
    o += ']';
  };
  o += "{\"learner\":{\"attributes\":{";
  for (size_t i = 0; i < f.attributes.size(); ++i) {
    if (i) o += ',';
    o += '"' + f.attributes[i].first + "\":\"" + f.attributes[i].second + '"';
  }
  o += "},\"feature_names\":[],\"feature_types\":[],\"gradient_booster\":{\"model\":{\"gbtree_model_param\":{"
       "\"num_parallel_tree\":\"1\",\"num_trees\":\"" + std::to_string(f.trees.size()) + "\",\"size_leaf_vector\":\"0\"},";
  arr("tree_info", f.trees.size(), [&](size_t i) { return std::to_string(i < f.tree_info.size() ? f.tree_info[i] : 0); });
  o += ",\"trees\":[";
  for (size_t ti = 0; ti < f.trees.size(); ++ti) {
    const HostTree &t = f.trees[ti];
    const size_t n = (size_t)t.num_nodes();
    if (ti) o += ',';
    o += '{';
    arr("base_weights", n, [&](size_t i) { return f32_repr(t.base_weight[i]); });
    o += ",\"categories\":[],\"categories_nodes\":[],\"categories_segments\":[],\"categories_sizes\":[],";
    arr("default_left", n, [&](size_t i) { return std::string((t.sindex[i] >> 31) ? "1" : "0"); });
    o += ",\"id\":" + std::to_string(ti) + ",";
    arr("left_children", n, [&](size_t i) { return std::to_string(t.cleft[i]); });
    o += ',';
    arr("loss_changes", n, [&](size_t i) { return f32_repr(t.loss_chg[i]); });
    o += ',';
    arr("parents", n, [&](size_t i) { return std::to_string(json_parent(t, (int32_t)i)); });
    o += ',';
    arr("right_children", n, [&](size_t i) { return std::to_string(t.cright[i]); });
    o += ',';
    arr("split_conditions", n, [&](size_t i) { return f32_repr(t.info[i]); });
    o += ',';
    arr("split_indices", n, [&](size_t i) { return std::to_string(t.sindex[i] & 0x7FFFFFFFu); });
    o += ',';
    arr("split_type", n, [&](size_t) { return std::string("0"); });
    o += ',';
    arr("sum_hessian", n, [&](size_t i) { return f32_repr(t.sum_hess[i]); });
    o += ",\"tree_param\":{\"num_deleted\":\"0\",\"num_feature\":\"" + std::to_string(f.num_feature) +
         "\",\"num_nodes\":\"" + std::to_string(n) + "\",\"size_leaf_vector\":\"0\"}}";
  }
  o += "]},\"name\":\"gbtree\"},\"learner_model_param\":{\"base_score\":\"" + f32_repr(f.base_score) +
       "\",\"num_class\":\"0\",\"num_feature\":\"" + std::to_string(f.num_feature) +
       "\",\"num_target\":\"1\"},\"objective\":{\"name\":\"" + f.objective +
       "\",\"reg_loss_param\":{\"scale_pos_weight\":\"1\"}}},\"version\":[" + std::to_string(f.version[0]) + "," +
       std::to_string(f.version[1]) + "," + std::to_string(f.version[2]) + "]}";
  return o;
}

// UBJSON writer (big-endian, typed arrays for the per-node vectors)
struct UbjW {
  std::string o;
  template <class T>
  void be(T v) {
    unsigned char t[sizeof(T)];
    memcpy(t, &v, sizeof(T));
    for (size_t i = 0; i < sizeof(T); ++i) o += (char)t[sizeof(T) - 1 - i];
  }
  void len(int64_t n) { o += 'L', be<int64_t>(n); }
  void key(const std::string &k) { len((int64_t)k.size()), o += k; }
  void str(const std::string &s) { o += 'S', key(s); }
  void kstr(const std::string &k, const std::string &s) { key(k), str(s); }
  template <class T, class F>
  void typed(const std::string &k, char ty, size_t n, F &&get) {
    key(k), o += "[$", o += ty, o += '#', len((int64_t)n);
    for (size_t i = 0; i < n; ++i) be<T>(get(i));
  }
};

std::string ubj_bytes(const HostForest &f) {
  UbjW w;
  w.o += '{';
  w.key("learner"), w.o += '{';
  w.key("attributes"), w.o += '{';
  for (auto &kv : f.attributes) w.kstr(kv.first, kv.second);
  w.o += '}';
  w.key("feature_names"), w.o += "[]";
  w.key("feature_types"), w.o += "[]";
  w.key("gradient_booster"), w.o += '{';
  w.key("model"), w.o += '{';
  w.key("gbtree_model_param"), w.o += '{';
  w.kstr("num_parallel_tree", "1"), w.kstr("num_trees", std::to_string(f.trees.size())), w.kstr("size_leaf_vector", "0");
  w.o += '}';
  w.typed<int32_t>("tree_info", 'l', f.trees.size(), [&](size_t i) { return i < f.tree_info.size() ? f.tree_info[i] : 0; });
  w.key("trees"), w.o += '[';
  for (size_t ti = 0; ti < f.trees.size(); ++ti) {
    const HostTree &t = f.trees[ti];
    const size_t n = (size_t)t.num_nodes();
    w.o += '{';
    w.typed<float>("base_weights", 'd', n, [&](size_t i) { return t.base_weight[i]; });
    for (const char *k : {"categories", "categories_nodes", "categories_segments", "categories_sizes"})
      w.typed<int32_t>(k, 'l', 0, [&](size_t) { return 0; });
    w.typed<uint8_t>("default_left", 'U', n, [&](size_t i) { return (uint8_t)(t.sindex[i] >> 31); });
    w.key("id"), w.o += 'l', w.be<int32_t>((int32_t)ti);
    w.typed<int32_t>("left_children", 'l', n, [&](size_t i) { return t.cleft[i]; });
    w.typed<float>("loss_changes", 'd', n, [&](size_t i) { return t.loss_chg[i]; });
    w.typed<int32_t>("parents", 'l', n, [&](size_t i) { return json_parent(t, (int32_t)i); });
    w.typed<int32_t>("right_children", 'l', n, [&](size_t i) { return t.cright[i]; });
    w.typed<float>("split_conditions", 'd', n, [&](size_t i) { return t.info[i]; });
    w.typed<int32_t>("split_indices", 'l', n, [&](size_t i) { return (int32_t)(t.sindex[i] & 0x7FFFFFFFu); });
    w.typed<uint8_t>("split_type", 'U', n, [&](size_t) { return (uint8_t)0; });
    w.typed<float>("sum_hessian", 'd', n, [&](size_t i) { return t.sum_hess[i]; });
    w.key("tree_param"), w.o += '{';
    w.kstr("num_deleted", "0"), w.kstr("num_feature", std::to_string(f.num_feature));
    w.kstr("num_nodes", std::to_string(n)), w.kstr("size_leaf_vector", "0");
    w.o += "}}";
  }
  w.o += ']';
  w.o += '}';  // model
  w.kstr("name", "gbtree");
  w.o += '}';  // gradient_booster
  w.key("learner_model_param"), w.o += '{';
  w.kstr("base_score", f32_repr(f.base_score)), w.kstr("num_class", "0");
  w.kstr("num_feature", std::to_string(f.num_feature)), w.kstr("num_target", "1");
  w.o += '}';
  w.key("objective"), w.o += '{';
  w.kstr("name", f.objective);
  w.key("reg_loss_param"), w.o += '{', w.kstr("scale_pos_weight", "1"), w.o += '}';
  w.o += '}';
  w.o += '}';  // learner
  w.key("version"), w.o += '[';
  for (int i = 0; i < 3; ++i) w.o += 'l', w.be<int32_t>((int32_t)f.version[i]);
  w.o += ']';
  w.o += '}';
  return w.o;
}

bool ends_with(const std::string &s, const char *suf) {
  size_t n = strlen(suf);
  return s.size() >= n && !s.compare(s.size() - n, n, suf);
}

}  // namespace

HostForest load_model_buffer(const unsigned char *buf, size_t len) {
  if (len == 0) fail("Empty model file");
  if (len >= 4 && !memcmp(buf, "bs64", 4)) fail("Base64 model format is not supported");
  if (buf[0] == '{') {
    // '{' followed by '"' or whitespace is text JSON; UBJSON objects start "{L", "{U", "{i" ...
    size_t i = 1;
    while (i < len && (buf[i] == ' ' || buf[i] == '\n' || buf[i] == '\t' || buf[i] == '\r')) ++i;
    if (i < len && (buf[i] == '"' || buf[i] == '}')) {
      JsonReader r{(const char *)buf, (const char *)buf + len};
      return from_dom(r.value(), kJson);
    }
    UbjReader u{buf, buf + len};
    return from_dom(u.value(), kUbjson);
  }
  return load_legacy(buf, len);
}

HostForest load_model_file(const std::string &path) {
  FILE *fp = fopen(path.c_str(), "rb");
  if (!fp) fail("Opening " + path + " failed: " + strerror(errno));
  std::vector<unsigned char> buf;
  unsigned char chunk[1 << 16];
  size_t n;
  while ((n = fread(chunk, 1, sizeof chunk, fp)) > 0) buf.insert(buf.end(), chunk, chunk + n);
  fclose(fp);
  return load_model_buffer(buf.data(), buf.size());
}

void save_model_file(const HostForest &f, const std::string &path) {
  std::string bytes = ends_with(path, ".json") ? json_text(f) : ends_with(path, ".ubj") ? ubj_bytes(f) : legacy_bytes(f);
  FILE *fp = fopen(path.c_str(), "wb");
  if (!fp) fail("Opening " + path + " for writing failed: " + strerror(errno));
  size_t w = fwrite(bytes.data(), 1, bytes.size(), fp);
  fclose(fp);
  if (w != bytes.size()) fail("Short write on " + path);
}

FlatForest flatten(const HostForest &f) {
  if (f.num_feature > kMaxFeatures)
    fail("num_feature = " + std::to_string(f.num_feature) + " exceeds the " + std::to_string(kMaxFeatures) +
         " features the sm_100a node layout encodes");
  FlatForest out;
  out.tree_offset.push_back(0);
  for (size_t ti = 0; ti < f.trees.size(); ++ti) {
    const HostTree &t = f.trees[ti];
    const uint32_t base = (uint32_t)out.orig_id.size();
    // breadth-first renumbering; (old id, depth)
    std::vector<int32_t> order;
    std::vector<int32_t> depth;
    std::vector<int32_t> newpos((size_t)t.num_nodes(), -1);
    order.reserve((size_t)t.num_nodes());
    order.push_back(0), depth.push_back(0);
    newpos[0] = 0;
    for (size_t h = 0; h < order.size(); ++h) {
      const int32_t o = order[h];
      if (t.cleft[o] == -1) continue;
      const int32_t l = t.cleft[o], r = t.cright[o];
      // GetNextNode (xgboost src/predictor/predict_fn.h) takes `cleft + !(fvalue < cond)` for
      // present values and DefaultChild() for missing ones; both agree only if cright == cleft+1,
      // which every XGBoost-grown tree satisfies (children are allocated as a pair).
      if (r != l + 1)
        fail("tree " + std::to_string(ti) + " node " + std::to_string(o) + ": cright != cleft + 1 (not an XGBoost-grown tree)");
      if (newpos[(size_t)l] != -1 || newpos[(size_t)r] != -1)
        fail("tree " + std::to_string(ti) + ": node reachable twice (not a tree)");
      newpos[(size_t)l] = (int32_t)order.size();
      order.push_back(l), depth.push_back(depth[h] + 1);
      newpos[(size_t)r] = (int32_t)order.size();
      order.push_back(r), depth.push_back(depth[h] + 1);
    }
    if (order.size() > kMetaRelMask) fail("tree " + std::to_string(ti) + " has too many nodes for the 23-bit child offset");
    int32_t maxd = 0, mind = 1 << 30;
    for (size_t h = 0; h < order.size(); ++h) {
      const int32_t o = order[h];
      uint32_t xbits, meta;
      memcpy(&xbits, &t.info[(size_t)o], 4);
      if (t.cleft[o] == -1) {
        meta = (f.num_feature << kMetaFeatShift) | kMetaDefaultLeftBit;  // rel = 0: self-loop
        if (depth[h] > maxd) maxd = depth[h];
        if (depth[h] < mind) mind = depth[h];
        if (!std::isfinite(t.info[(size_t)o]))
          fail("tree " + std::to_string(ti) + " node " + std::to_string(o) + ": non-finite leaf value");
      } else {
        const uint32_t rel = (uint32_t)(newpos[(size_t)t.cleft[o]] - (int32_t)h);
        meta = ((t.sindex[o] & 0x7FFFFFFFu) << kMetaFeatShift) | ((t.sindex[o] >> 31) ? kMetaDefaultLeftBit : 0u) | rel;
      }
      out.nodes_xy.push_back(xbits);
      out.nodes_xy.push_back(meta);
      out.orig_id.push_back(o);
    }
    (void)base;
    out.tree_depth.push_back(maxd);
    out.tree_min_leaf_depth.push_back(mind);
    if (maxd > out.max_depth) out.max_depth = maxd;
    out.tree_offset.push_back((uint32_t)out.orig_id.size());
  }
  return out;
}

// ---- two-level records --------------------------------------------------------------------------
static bool build_duo_with(const FlatForest &f, uint32_t num_feature, int blk_shift, DuoForest &out) {
  const bool dlbits = blk_shift == 18;
  out.blk_shift = blk_shift, out.has_default_bits = dlbits;
  const size_t ntree = f.tree_depth.size();
  auto X = [&](uint32_t n) { return f.nodes_xy[2 * (size_t)n]; };
  auto REL = [&](uint32_t n) { return f.nodes_xy[2 * (size_t)n + 1] & kMetaRelMask; };
  auto FEAT = [&](uint32_t n) { return f.nodes_xy[2 * (size_t)n + 1] >> kMetaFeatShift; };
  auto DL = [&](uint32_t n) { return REL(n) != 0 && (f.nodes_xy[2 * (size_t)n + 1] & kMetaDefaultLeftBit) != 0; };
  auto thr_word = [&](uint32_t n) -> uint32_t {
    if (REL(n) == 0) return 0u;  // leaf child: compared against key 0 of the sentinel slot, never carries
    float thr;
    const uint32_t b = X(n);
    memcpy(&thr, &b, 4);
    return neg_threshold_key(thr);
  };
  constexpr uint32_t kRow = 1u << kDuoTop;  // heap entries per tree (entry 0 unused), and level-kDuoTop roots
  for (size_t t = 0; t < ntree; ++t) {
    const uint32_t n0 = f.tree_offset[t];
    // complete heap-ordered top: node[i] = the real node at heap position i, or the leaf it pads
    uint32_t node[2 * kRow];
    bool pad[2 * kRow];
    node[1] = n0, pad[1] = false;
    out.top_xy.resize(out.top_xy.size() + 2 * kRow, 0u);
    uint32_t *top = out.top_xy.data() + out.top_xy.size() - 2 * kRow;
    for (uint32_t i = 1; i < kRow; ++i) {
      const uint32_t n = node[i];
      if (!pad[i] && REL(n) != 0) {
        top[2 * i] = thr_word(n), top[2 * i + 1] = (FEAT(n) << kMetaFeatShift) | (DL(n) ? kTopDefaultLeftBit : 0u);
        node[2 * i] = n + REL(n), node[2 * i + 1] = n + REL(n) + 1;
        pad[2 * i] = pad[2 * i + 1] = false;
      } else {  // a leaf above level kDuoTop, or padding below one: never right
        top[2 * i] = 0u, top[2 * i + 1] = num_feature << kMetaFeatShift;
        node[2 * i] = node[2 * i + 1] = n;
        pad[2 * i] = pad[2 * i + 1] = true;
      }
    }
    // tree bases on 128-byte lines
    while ((out.rec.size() / 4) % 8) out.rec.insert(out.rec.end(), 4, 0u);
    const size_t base = out.rec.size() / 4;
    out.tree_slot.push_back((uint32_t)base);
    std::vector<uint32_t> root_of;  // tree-local slot -> root node (global index), ~0u = unused slot
    for (uint32_t i = kRow; i < 2 * kRow; ++i) root_of.push_back(node[i]);  // padded leaves become terminal records
    for (size_t s = 0; s < root_of.size(); ++s) {
      const uint32_t n = root_of[s];
      uint32_t w[4] = {0u, 0u, 0u, 0u};
      if (n != ~0u) {
        if (REL(n) == 0) {
          w[0] = X(n), w[1] = (uint32_t)f.orig_id[n];  // terminal: value bits, XGBoost node id
        } else {
          const uint32_t kids[2] = {n + REL(n), n + REL(n) + 1};
          const size_t blk = root_of.size() / 4;
          if (blk >= (1u << (32 - blk_shift))) {
            out.why = "tree " + std::to_string(t) + " needs more than 2^" + std::to_string(32 - blk_shift) + " record blocks";
            return false;
          }
          for (int c = 0; c < 2; ++c) {
            if (REL(kids[c]) == 0) {
              root_of.push_back(kids[c]), root_of.push_back(~0u);
            } else {
              root_of.push_back(kids[c] + REL(kids[c])), root_of.push_back(kids[c] + REL(kids[c]) + 1);
            }
          }
          w[0] = thr_word(n), w[1] = thr_word(kids[0]), w[2] = thr_word(kids[1]);
          const uint32_t fl = REL(kids[0]) ? FEAT(kids[0]) : num_feature, fr = REL(kids[1]) ? FEAT(kids[1]) : num_feature;
          w[3] = ((uint32_t)blk << blk_shift) | (fl << 10) | (fr << 5) | FEAT(n);
          if (dlbits) w[3] |= (DL(n) ? kDuoDlRoot : 0u) | (DL(kids[0]) ? kDuoDlLeft : 0u) | (DL(kids[1]) ? kDuoDlRight : 0u);
        }
      }
      out.rec.insert(out.rec.end(), w, w + 4);
    }
    if (out.rec.size() / 4 > 0x7FFFFFFFull) {
      out.why = "forest needs more than 2^31 records";
      return false;
    }
  }
  out.ok = true;
  return true;
}

DuoForest build_duo(const FlatForest &f, uint32_t num_feature) {
  // with the three default-direction bits a tree may use 2^14 record blocks (1 MB of records); a bigger tree
  // gets the 17-bit block pointer and no default bits (matrices with missing entries then walk the 8-byte nodes)
  DuoForest out;
  if (build_duo_with(f, num_feature, 18, out)) return out;
  DuoForest wide;
  if (build_duo_with(f, num_feature, 15, wide)) return wide;
  wide.rec.clear(), wide.tree_slot.clear(), wide.top_xy.clear();
  return wide;
}

// ---- contributions: node means and root-to-leaf paths ---------------------------------------------------
namespace {
// libxgboost 1.6.0 FillNodeMeanValue (src/predictor/cpu_predictor.cc), float32 in its order
float fill_mean(const HostTree &t, int32_t n, std::vector<float> &mean) {
  float r;
  if (t.cleft[n] == -1) {
    r = t.info[n];
  } else {
    r = fill_mean(t, t.cleft[n], mean) * t.sum_hess[t.cleft[n]];
    r += fill_mean(t, t.cright[n], mean) * t.sum_hess[t.cright[n]];
    r /= t.sum_hess[n];
  }
  mean[n] = r;
  return r;
}

struct PathElem {
  uint32_t feat, lo, hi, miss;
  double zero;
};

uint32_t threshold_key(float thr) { return 0u - neg_threshold_key(thr); }

// The kernels keep an element's one fraction in the sign of its float32 zero fraction, so every stored zero fraction
// must be a positive, finite float32; covers that are each finite and positive can still multiply past that range.
void collect_paths(size_t ti, const HostTree &t, int32_t n, std::vector<PathElem> &path,
                   std::vector<std::pair<std::vector<PathElem>, float>> &out) {
  if (t.cleft[n] == -1) {
    for (const PathElem &e : path) {
      const float z = (float)e.zero;
      if (!(z > 0.f) || !std::isfinite(z)) {
        char msg[320];
        snprintf(msg, sizeof msg,
                 "contributions need every path's product of cover(child) / cover(parent) over the splits on one "
                 "feature to be a positive, finite float32, but tree %zu leaf %d has %g on feature %u: this booster "
                 "cannot be explained",
                 ti, n, e.zero, e.feat);
        fail(msg);
      }
    }
    out.emplace_back(path, t.info[n]);
    return;
  }
  const uint32_t f = t.sindex[n] & 0x7FFFFFFFu;
  const bool dl = (t.sindex[n] >> 31) != 0;
  const uint32_t k = threshold_key(t.info[n]);
  for (int side = 0; side < 2; ++side) {
    const int32_t c = side ? t.cright[n] : t.cleft[n];
    std::vector<PathElem> p(path);
    size_t i = 0;
    while (i < p.size() && p[i].feat != f) ++i;
    if (i == p.size()) p.push_back({f, 0u, 0xFFFFFFFFu, 1u, 1.0});
    if (side) p[i].lo = std::max(p[i].lo, k);
    else p[i].hi = std::min(p[i].hi, k);
    p[i].miss &= (dl == (side == 0)) ? 1u : 0u;
    p[i].zero *= (double)t.sum_hess[c] / (double)t.sum_hess[n];
    collect_paths(ti, t, c, p, out);
  }
}
}  // namespace

ShapForest build_shap(const HostForest &h, const FlatForest &f) {
  ShapForest s;
  s.mean.assign((size_t)f.num_nodes(), 0.f);
  s.tree_bin.push_back(0);
  for (size_t ti = 0; ti < h.trees.size(); ++ti) {
    const HostTree &t = h.trees[ti];
    for (int32_t n = 0; n < t.num_nodes(); ++n)
      if (!std::isfinite(t.sum_hess[n]) || !(t.sum_hess[n] > 0.f))
        fail("contributions need the node covers (sum_hess), but tree " + std::to_string(ti) + " node " + std::to_string(n) +
             " has cover " + std::to_string(t.sum_hess[n]) +
             ": this booster cannot be explained (a JSON model without sum_hessian, or trees converted without covers)");
    std::vector<float> m((size_t)t.num_nodes());
    fill_mean(t, 0, m);
    const uint32_t n0 = f.tree_offset[ti];
    for (uint32_t i = n0; i < f.tree_offset[ti + 1]; ++i) s.mean[i] = m[(size_t)f.orig_id[i]];
    std::vector<std::pair<std::vector<PathElem>, float>> paths;
    std::vector<PathElem> root;
    collect_paths(ti, t, 0, root, paths);
    // first-fit decreasing into 32-lane bins; lengths include the bias element (<= kMaxFeatures + 1 = 32)
    std::vector<size_t> order(paths.size());
    for (size_t i = 0; i < order.size(); ++i) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return paths[a].first.size() > paths[b].first.size(); });
    std::vector<int> fill;                      // lanes used per bin of this tree
    std::vector<std::vector<size_t>> members;   // paths per bin, in placement order
    std::map<int, std::vector<size_t>> by_free;  // free lanes -> bins with that many free lanes (ascending index)
    for (size_t pi : order) {
      const int len = (int)paths[pi].first.size() + 1;
      size_t bin = fill.size();
      int have = -1;
      for (auto it = by_free.lower_bound(len); it != by_free.end(); ++it)
        if (!it->second.empty() && it->second.front() < bin) bin = it->second.front(), have = it->first;
      if (have < 0) {
        fill.push_back(0), members.emplace_back();
      } else {
        auto &v = by_free[have];
        v.erase(v.begin());
      }
      fill[bin] += len;
      members[bin].push_back(pi);
      auto &v = by_free[32 - fill[bin]];
      v.insert(std::lower_bound(v.begin(), v.end(), bin), bin);
      s.max_path_len = std::max(s.max_path_len, len);
      s.num_paths += 1, s.num_elements += len;
    }
    for (size_t b = 0; b < members.size(); ++b) {
      uint32_t w[32][4];
      for (uint32_t l = 0; l < 32; ++l) w[l][0] = 0u, w[l][1] = 0xFFFFFFFFu, w[l][2] = kShapNoFeature | (l << 16), w[l][3] = 0u;
      uint32_t lane = 0;
      for (size_t pi : members[b]) {
        const auto &p = paths[pi];
        const uint32_t g0 = lane, len = (uint32_t)p.first.size() + 1;
        const uint32_t grp = (g0 << 16) | (len << 24);
        float v = p.second;
        w[lane][2] = kShapNoFeature | (1u << 8) | grp;
        memcpy(&w[lane][3], &v, 4);
        ++lane;
        for (const PathElem &e : p.first) {
          const float z = (float)e.zero;
          w[lane][0] = e.lo, w[lane][1] = e.hi, w[lane][2] = e.feat | (e.miss << 8) | grp;
          memcpy(&w[lane][3], &z, 4);
          ++lane;
        }
      }
      s.bins.insert(s.bins.end(), &w[0][0], &w[0][0] + 128);
    }
    s.tree_bin.push_back(s.num_bins());
  }
  s.ok = true;
  return s;
}

void build_shap_by_feature(ShapForest &s, uint32_t nfeat) {
  std::vector<std::vector<uint32_t>> lists(nfeat);
  const int64_t nb = s.num_bins();
  for (int64_t b = 0; b < nb; ++b) {
    uint32_t seen = 0u;  // features < kMaxFeatures = 31
    for (int l = 0; l < 32; ++l) {
      const uint32_t f = s.bins[(size_t)(b * 32 + l) * 4 + 2] & 0xFFu;
      if (f < nfeat && !((seen >> f) & 1u)) seen |= 1u << f, lists[f].push_back((uint32_t)b);
    }
  }
  s.feat_off.assign(1, 0);
  s.feat_bins.clear();
  for (const auto &v : lists) {
    s.feat_bins.insert(s.feat_bins.end(), v.begin(), v.end());
    s.feat_off.push_back((int64_t)s.feat_bins.size());
  }
}

float shap_bias(const ShapForest &s, const HostForest &h, const FlatForest &f, int ntree) {
  float b = 0.f;
  for (int t = 0; t < ntree; ++t) b += 0.f + s.mean[f.tree_offset[t]];
  return b + h.base_score;
}

namespace {
JV parse_json_object(const char *json, const std::string &what) {
  if (!json) fail(what + " is NULL");
  JV root;
  try {
    JsonReader r{json, json + strlen(json)};
    root = r.value();
  } catch (const std::exception &e) {
    fail(what + " is not valid JSON (" + e.what() + ")");
  }
  if (root.kind != JV::Obj) fail(what + " must be a JSON object");
  return root;
}
JV parse_json_value(const char *json, const std::string &what) {
  if (!json) fail(what + " is NULL");
  try {
    JsonReader r{json, json + strlen(json)};
    return r.value();
  } catch (const std::exception &e) {
    fail(what + " is not valid JSON (" + e.what() + ")");
  }
  return JV();
}

// The fields a 2-D array interface and a 1-D column share, read in the order of their refusals, each message starting
// with `pre`: typestr and mask; then layout(need) reads the shape and strides (need(key) refuses a missing key) and
// returns what a NULL data address is refused for, empty when the array has no elements; then the data and stream.
struct InterfaceFields {
  uint64_t addr = 0;
  bool has_stream = false;
  uint64_t stream = 0;
};
template <class Layout>
InterfaceFields read_interface(const JV &obj, const std::string &pre, Layout &&layout) {
  auto need = [&](const char *key) -> const JV & {
    const JV *v = obj.find(key);
    if (!v) fail(pre + "array interface is missing the key '" + key + "'");
    return *v;
  };
  const JV &ty = need("typestr");
  if (ty.kind != JV::Str || ty.str != "<f4")
    fail(pre + "typestr '" + (ty.kind == JV::Str ? ty.str : std::string("?")) + "': only little-endian float32 ('<f4') is accepted");
  if (obj.find("mask")) fail(pre + "masked arrays are not supported (the array interface has a 'mask' entry)");
  const std::string null_for = layout(need);
  const JV &data = need("data");
  if (data.kind != JV::Arr || data.arr.empty()) fail(pre + "'data' must be [address, readonly]");
  InterfaceFields f;
  f.addr = (uint64_t)data.arr[0].as_int();
  if (f.addr == 0 && !null_for.empty()) fail(pre + "the data address is NULL for " + null_for);
  const JV *s = obj.find("stream");
  if (s && s->kind != JV::Null) {
    f.stream = (uint64_t)s->as_int();
    if (f.stream == 0) fail(pre + "stream 0 is not valid in the CUDA Array Interface (1: legacy default stream, 2: per-thread default stream)");
    f.has_stream = true;
  }
  return f;
}
}  // namespace

PredictConfig parse_predict_config(const char *json, const char *caller, bool inplace) {
  const std::string pre = std::string(caller) + ": ";
  const JV root = parse_json_object(json, pre + "config");
  auto need = [&](const char *key) -> const JV & {
    const JV *v = root.find(key);
    if (!v) fail(pre + "config is missing the key '" + key + "'");
    return *v;
  };
  PredictConfig c;
  c.type = (int)need("type").as_int();
  if (inplace) {
    const JV &m = need("missing");
    if (m.kind != JV::Num) fail(pre + "config: 'missing' must be a number (NaN is written NaN)");
    c.missing = m.f32;
  } else {
    c.training = need("training").as_int() != 0;
  }
  c.iteration_begin = need("iteration_begin").as_int();
  c.iteration_end = need("iteration_end").as_int();
  c.strict_shape = need("strict_shape").as_int() != 0;
  return c;
}

ArrayInterface parse_array_interface(const char *json, const char *caller) {
  const std::string pre = std::string(caller) + ": ";
  const JV root = parse_json_object(json, pre + "array interface");
  ArrayInterface a;
  const InterfaceFields f = read_interface(root, pre, [&](auto &&need) {
    const JV &shape = need("shape");
    if (shape.kind != JV::Arr || shape.arr.size() != 2)
      fail(pre + "the array must be 2-D [nrow, ncol]; its shape has " + std::to_string(shape.kind == JV::Arr ? shape.arr.size() : 0) + " dimensions");
    const int64_t nr = shape.arr[0].as_int(), nc = shape.arr[1].as_int();
    if (nr < 0 || nc < 0) fail(pre + "negative shape [" + std::to_string(nr) + ", " + std::to_string(nc) + "]");
    a.nrow = (uint64_t)nr, a.ncol = (uint64_t)nc;
    a.row_bytes = 4 * nc;
    const JV *st = root.find("strides");
    if (st && st->kind != JV::Null) {
      if (st->kind != JV::Arr || st->arr.size() != 2) fail(pre + "strides must be null or [row_bytes, col_bytes]");
      const int64_t rb = st->arr[0].as_int(), cb = st->arr[1].as_int();
      if (rb < 0 || cb < 0 || rb % 4 || cb % 4)
        fail(pre + "strides [" + std::to_string(rb) + ", " + std::to_string(cb) + "]: they must be non-negative multiples of 4 bytes");
      a.row_bytes = rb, a.col_bytes = cb;
    }
    return a.nrow * a.ncol > 0 ? "a " + std::to_string(nr) + " x " + std::to_string(nc) + " array" : std::string();
  });
  a.addr = f.addr, a.has_stream = f.has_stream, a.stream = f.stream;
  return a;
}

float parse_dmatrix_config(const char *json, const char *caller) {
  const std::string pre = std::string(caller) + ": ";
  const JV root = parse_json_object(json, pre + "config");
  const JV *m = root.find("missing");
  if (!m) fail(pre + "config is missing the key 'missing'");
  if (m->kind != JV::Num) fail(pre + "config: 'missing' must be a number (NaN is written NaN)");
  return m->f32;
}

ColumnarInterface parse_columnar_interface(const char *json, const char *caller) {
  const std::string pre = std::string(caller) + ": ";
  const JV root = parse_json_value(json, pre + "columnar interface");
  if (root.kind != JV::Arr) fail(pre + "the columnar interface must be a JSON list of 1-D array interfaces, one per column");
  if (root.arr.empty()) fail(pre + "the list of columns is empty");
  if (root.arr.size() > kMaxMatrixCols)
    fail(pre + std::to_string(root.arr.size()) + " columns; libqcoh's tile form holds at most " + std::to_string(kMaxMatrixCols));
  ColumnarInterface ci;
  for (size_t c = 0; c < root.arr.size(); ++c) {
    const JV &col = root.arr[c];
    const std::string at = pre + "column " + std::to_string(c) + ": ";
    if (col.kind != JV::Obj) fail(at + "must be an array interface (a JSON object)");
    int64_t sb = 4;
    const InterfaceFields f = read_interface(col, at, [&](auto &&need) {
      const JV &shape = need("shape");
      if (shape.kind != JV::Arr || shape.arr.size() != 1)
        fail(at + "a column must be 1-D [nrow]; its shape has " + std::to_string(shape.kind == JV::Arr ? shape.arr.size() : 0) + " dimensions");
      const int64_t nr = shape.arr[0].as_int();
      if (nr < 0) fail(at + "negative shape [" + std::to_string(nr) + "]");
      if (c == 0) ci.nrow = (uint64_t)nr;
      else if ((uint64_t)nr != ci.nrow)
        fail(at + "the columns differ in length: column " + std::to_string(c) + " has " + std::to_string(nr) + " rows, column 0 has " +
             std::to_string(ci.nrow));
      const JV *st = col.find("strides");
      if (st && st->kind != JV::Null) {
        if (st->kind != JV::Arr || st->arr.size() != 1) fail(at + "strides must be null or [bytes]");
        sb = st->arr[0].as_int();
        if (sb <= 0 || sb % 4) fail(at + "strides [" + std::to_string(sb) + "]: the stride must be a positive multiple of 4 bytes");
      }
      return nr > 0 ? "a column of " + std::to_string(nr) + " rows" : std::string();
    });
    if (f.has_stream && std::find(ci.streams.begin(), ci.streams.end(), f.stream) == ci.streams.end()) ci.streams.push_back(f.stream);
    ci.addr.push_back(f.addr);
    ci.stride_bytes.push_back(sb);
  }
  return ci;
}

}  // namespace qcoh
