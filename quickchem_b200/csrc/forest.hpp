// forest.hpp — host-side booster: XGBoost model files -> in-memory trees -> flattened,
// depth-ordered structure-of-nodes that the sm_100a predict kernel walks.
//
// Replaces what `XGBoosterLoadModel` does inside libxgboost 1.6.0 for the reference
// (/root/reference/OH_GridComp/OH_GridCompMod.F90:261 via Shared/xgb_fortran_api.F90:18-24).
// Pure C++ (no CUDA), so it is testable on a box without a GPU.
#pragma once
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

namespace qcoh {

// One tree as XGBoost stores it (RegTree::Node + RTreeNodeStat), node 0 = root.
struct HostTree {
  std::vector<int32_t> cleft, cright, parent;  // parent: raw legacy encoding (bit31 = is-left-child, -1 root)
  std::vector<uint32_t> sindex;                // bit31 default_left | split feature
  std::vector<float> info;                     // split_cond, or leaf_value at leaves
  std::vector<float> loss_chg, sum_hess, base_weight;
  std::vector<int32_t> leaf_child_cnt;
  int32_t num_nodes() const { return (int32_t)cleft.size(); }
};

enum ModelFormat { kLegacyBinary = 0, kJson = 1, kUbjson = 2 };

struct HostForest {
  float base_score = 0.5f;
  uint32_t num_feature = 0;
  uint32_t version[3] = {1, 6, 0};
  std::string objective = "reg:squarederror";
  std::vector<HostTree> trees;
  std::vector<int32_t> tree_info;
  std::vector<std::pair<std::string, std::string>> attributes;
  ModelFormat format = kLegacyBinary;
};

// Flattened layout (see DESIGN.md "Node layout").  Per tree the nodes are renumbered in
// breadth-first (depth) order, siblings adjacent (right = left + 1).  One node = 8 bytes:
//   x: float bits — split threshold, or the leaf value at a leaf
//   y: meta = feat << 26 | default_left << 23 | rel   (rel = left-child index - own index; the top byte is
//      feat * 4, so one byte-permute turns it into the byte offset feat * 1024 of the kernel's feature tile)
// A leaf has rel = 0 and feat = num_feature: the predict kernel keeps one extra per-row
// slot holding key 0 at that feature index, so the compare never says "right" and the walk
// self-loops without a leaf test.
constexpr uint32_t kMetaFeatShift = 26;
constexpr uint32_t kMetaDefaultLeftBit = 1u << 23;
constexpr uint32_t kMetaRelMask = (1u << 23) - 1;
constexpr uint32_t kMaxFeatures = 31;  // the 5-bit feature fields of the two-level records also hold the leaf slot num_feature

struct FlatForest {
  std::vector<uint32_t> nodes_xy;     // 2 words per node
  std::vector<uint32_t> tree_offset;  // [ntree + 1], in nodes
  std::vector<int32_t> tree_depth;    // [ntree] depth of the deepest leaf (root = 0)
  std::vector<int32_t> tree_min_leaf_depth;  // [ntree] depth of the shallowest leaf
  std::vector<int32_t> orig_id;       // flattened position -> XGBoost node id (pred_leaf output)
  int32_t max_depth = 0;
  int64_t num_nodes() const { return (int64_t)orig_id.size(); }
};

// Device form of a split threshold: -key(thr) mod 2^32, key = order-preserving integer image of the
// float with -0.0 folded into +0.0 (kernels.cu "Order-preserving integer keys").  Never 0.
inline uint32_t neg_threshold_key(float thr) {
  thr += 0.0f;
  uint32_t bits;
  memcpy(&bits, &thr, 4);
  return 0u - (bits ^ ((bits >> 31) ? 0xFFFFFFFFu : 0x80000000u));
}

// Two-level records (DESIGN.md "Two levels per gather").  Levels 0..kDuoTop-1 of every tree are a COMPLETE
// heap-ordered top (entry i = 1..15, children 2i and 2i+1; `top_xy` row of 16 {x, feat << 26 | default_left} pairs
// per tree, entry 0 unused) served from constant memory; a leaf above level kDuoTop is padded downwards with
// never-right dummy nodes (x = 0, feat = num_feature).  Below, one 16-byte record holds a node at even depth
// AND its two children, so one gather decides two levels.  {w0, w1, w2} = -key(threshold) of root / left / right
// (0 where that child is a leaf), w3 = blk << blk_shift | [default-left bits] | feat(left) << 10 | feat(right) << 5 |
// feat(root); the four grandchild records sit contiguously at tree-local slots blk*4 + 2*right1 + right2.  A leaf
// is a terminal record (w3 == 0, w0 = value bits, w1 = XGBoost node id); a leaf CHILD has feature num_feature
// (whose key is 0: never "right") and its terminal record sits at slot blk*4 + 2*side.
//   blk_shift = 18: bits 17 / 16 / 15 of w3 are default_left of root / left / right (the missing-value direction,
//                   xgboost RegTree::Node::DefaultLeft), leaving 14 bits for blk: every tree needs < 2^14 blocks
//   blk_shift = 15: no default bits (a matrix with missing entries then walks the 8-byte nodes), 17-bit blk
constexpr int kDuoTop = 4;
constexpr uint32_t kDuoDlRoot = 1u << 17, kDuoDlLeft = 1u << 16, kDuoDlRight = 1u << 15;
constexpr uint32_t kTopDefaultLeftBit = 1u;  // bit 0 of a top_xy y word
struct DuoForest {
  bool ok = false;                    // false: some tree does not qualify (reason in `why`)
  std::string why;
  int blk_shift = 18;
  bool has_default_bits = true;       // blk_shift == 18
  std::vector<uint32_t> rec;          // 4 words per slot
  std::vector<uint32_t> tree_slot;    // [ntree] global slot of the tree's 16 level-kDuoTop records
  std::vector<uint32_t> top_xy;       // [ntree][16][2] heap-ordered tops for the constant-memory table
  int64_t num_slots() const { return (int64_t)(rec.size() / 4); }
};
DuoForest build_duo(const struct FlatForest &f, uint32_t num_feature);

// Per-feature contributions (DESIGN.md "Contributions"), built at the first contributions call.
//   mean: FillNodeMeanValue of libxgboost 1.6.0 in float32, by flat (depth-ordered) node index
//   bins: every root-to-leaf path of every tree as one lane group of a 32-lane bin, 4 words per lane:
//     {lo_key, hi_key, feat | missing_goes_here << 8 | group_start << 16 | group_len << 24, float bits}
//   Lane group_start is the path's bias element (feat 0xFF; its float is the leaf value); the others hold one
//   feature each — repeated splits on a path merged: key bounds intersected, zero fractions (cover(child) /
//   cover(parent)) multiplied, missing flags ANDed; their float is the zero fraction.  A present value with key k
//   follows the path iff lo_key <= k < hi_key, a missing one iff the flag is set.  Unused lanes: feat 0xFF, len 0.
//   Paths never straddle a bin, and a tree's bins are contiguous: bins [tree_bin[t], tree_bin[t + 1]).
constexpr uint32_t kShapNoFeature = 0xFF;
struct ShapForest {
  bool ok = false;
  std::vector<float> mean;
  std::vector<uint32_t> bins;      // [num_bins][32][4]
  std::vector<int64_t> tree_bin;   // [ntree + 1]
  int32_t max_path_len = 0;        // elements of the longest path, bias included
  int64_t num_paths = 0, num_elements = 0;
  // interactions only (build_shap_by_feature, at the first interactions call): the bins holding a path that contains
  // feature f are feat_bins[feat_off[f] .. feat_off[f + 1]), ascending, so the bins of the first t trees are a prefix
  std::vector<int64_t> feat_off;
  std::vector<uint32_t> feat_bins;
  int64_t num_bins() const { return (int64_t)(bins.size() / 128); }
};
// Throws unless every node of every tree has a finite, positive cover (sum_hess).
ShapForest build_shap(const struct HostForest &h, const struct FlatForest &f);
// Fills s.feat_off / s.feat_bins for features [0, nfeat).
void build_shap_by_feature(ShapForest &s, uint32_t nfeat);
// The bias column of a contributions row: ((0 + mean_0(root)) + mean_1(root) + ...) + base_score in float32.
float shap_bias(const ShapForest &s, const struct HostForest &h, const struct FlatForest &f, int ntree);

// The config of XGBoosterPredictFromDMatrix (libxgboost 1.6.0 keys); throws naming a missing key.  `inplace`: the
// config of the inplace predicts, which require `missing` instead of `training`; messages start with `caller`.
struct PredictConfig {
  int type = 0;
  bool training = false;
  int64_t iteration_begin = 0, iteration_end = 0;
  bool strict_shape = false;
  float missing = 0.f;  // inplace only
};
PredictConfig parse_predict_config(const char *json, const char *caller = "XGBoosterPredictFromDMatrix", bool inplace = false);

// A 2-D float32 array interface (numpy __array_interface__ / CUDA Array Interface v3, as JSON) for the inplace
// predicts: {"data": [address, readonly], "shape": [nrow, ncol], "strides": null | [row_bytes, col_bytes],
// "typestr": "<f4", "version": 3[, "stream": s]}.  Throws, prefixed with `caller`, on any other type, a mask, a shape
// that is not 2-D, negative strides or strides that are not a multiple of 4, a NULL address for a non-empty array, and
// stream 0.
struct ArrayInterface {
  uint64_t addr = 0;
  uint64_t nrow = 0, ncol = 0;
  int64_t row_bytes = 0, col_bytes = 4;  // C-contiguous when "strides" is null
  bool has_stream = false;
  uint64_t stream = 0;                   // CUDA Array Interface: 1 legacy default stream, 2 per-thread default stream
};
ArrayInterface parse_array_interface(const char *json, const char *caller);

// Throws std::runtime_error with libxgboost-style messages on malformed / unsupported input.
HostForest load_model_file(const std::string &path);
HostForest load_model_buffer(const unsigned char *buf, size_t len);
void save_model_file(const HostForest &f, const std::string &path);
FlatForest flatten(const HostForest &f);

}  // namespace qcoh
