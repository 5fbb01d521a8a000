// kernels.hpp — launch interface of the sm_100a kernels (kernels.cu), used by capi_xgb.cpp / capi_oh.cpp.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

namespace qcoh {

// Device copy of a FlatForest (forest.hpp) and of its two-level records, as upload() builds it.
struct DeviceForest {
  const uint2 *nodes = nullptr;          // {value bits, meta}
  const uint32_t *tree_offset = nullptr; // [ntree + 1]
  const int32_t *tree_depth = nullptr;   // [ntree]
  const int32_t *orig_id = nullptr;      // [num_nodes]
  cudaTextureObject_t tex = 0;           // the same nodes as a 1-D linear uint2 texture (TEX pipe)
  const uint4 *recs = nullptr;           // two-level records (forest.hpp DuoForest), or nullptr
  cudaTextureObject_t tex4 = 0;          // the records as a 1-D linear uint4 texture
  int duo_has_dl = 0;                    // the records carry the default-direction bits (DuoForest::has_default_bits)
  uint32_t duo_blk_mul = 0;              // 1 << (32 - DuoForest::blk_shift): blk = mulhi(w3, duo_blk_mul)
  int32_t ntree = 0;
  int32_t nfeat = 0;
  int duo_shallow = 0;                   // records average < kShallowRecBytesPerTree per tree (picks the launch shape)
  float base_score = 0.f;
};

// What the constant-memory tables of tree tops hold: one window of trees [tree0, tree0 + ntree) of one booster, as
// the first levels of its 8-byte nodes or as the heap-ordered tops of its two-level records.  The tables exist once
// per device; capi_xgb.cpp hold() fills them and returns the window, and the launchers take it as an argument.
enum class TopLayout { kNone, kRecordTops, kNodeTops };
struct ConstWindow {
  TopLayout layout = TopLayout::kNone;
  int32_t tree0 = 0, ntree = 0;
  bool holds(TopLayout l, int t0, int t1) const { return layout == l && tree0 <= t0 && t1 <= tree0 + ntree; }
};

// How many trees the constant-memory tables hold at once (4 levels x 16 entries per tree in 61 440 B), and how
// many of them one launch walks.  Measured (profiles/README.md "trees per launch"): warps drift apart through a
// forest, and when a launch walks hundreds of trees their tops and shallow records no longer share the constant
// cache and L1 — 500 trees x depth 10 take 75 ms in one 480-tree launch and 25 ms in launches of 120 (the tile
// stream is re-read per launch: 0.23 ms of the 5 ms a 120-tree range takes at C180).
constexpr int kConstTreesMax = 480;
constexpr int kRangeTrees = 120;
// A forest whose records average less than this per tree (depth <= ~7) is "shallow": 4 trees in flight and 6
// resident CTAs instead of 6 and 5 (100 trees x depth 6: 3.2 ms against 8.0 ms).
constexpr int64_t kShallowRecBytesPerTree = 4096;

// The device form of a DMatrix: order-preserving integer KEYS (kernels.cu) in feature-major tiles of 256 rows,
// Xt[tile][1 + col][256] — what a CTA's transposed shared-memory tile holds, so that a tile arrives with one bulk
// async copy (TMA) and needs no staging arithmetic.  Missing entries (NaN or == missing) are key 0xFFFFFFFF.
// Word-row 0 of a tile is its ROW ORDER: within a tile the rows without a missing entry come first (stable), the
// rows with one last; word p of the order row = original row index in the tile | has_missing << 8.  A predict launch
// on a matrix with missing entries reads it, so that a warp whose 32 rows are all clean walks without the
// default-direction test: what missing entries cost is proportional to the rows that have them.  (A clean matrix has
// the identity order and its launches skip that word-row.)
// Built by seal_tiles from the row-major float matrix, like libxgboost builds its SparsePage in
// XGDMatrixCreateFromMat (OH_GridCompMod.F90:347).
constexpr int kTileRows = 256;
constexpr uint64_t kMaxMatrixCols = 192;  // seal stages a 256 x ncol tile in shared memory; boosters take <= 31 features anyway
inline uint64_t tile_count(uint64_t nrow) { return (nrow + kTileRows - 1) / kTileRows; }
inline size_t tile_words(uint64_t nrow, uint64_t ncol) { return (size_t)tile_count(nrow) * (size_t)(ncol + 1) * kTileRows; }
// words from the start of Xt to the tile that holds row `row0` (a multiple of 256)
inline size_t tile_offset_words(uint64_t row0, uint64_t ncol) { return (size_t)(row0 / kTileRows) * (size_t)(ncol + 1) * kTileRows; }

struct PredictArgs {
  const uint32_t *Xt = nullptr;  // key tiles, device
  uint64_t nrow = 0;
  int32_t ncol = 0;
  int has_missing = 1;       // 0: the sealed matrix holds no NaN / == missing entry
  int pred_leaf = 0;         // option_mask & 2
  int32_t tree_begin = 0;    // this launch walks trees [tree_begin, tree_end) ...
  int32_t tree_end = 0;
  int32_t out_stride = 0;    // pred_leaf: floats per row in `out` (= trees used by the whole call)
  int first = 1;             // sums: 1 = start from base_score, 0 = continue from the partial sum in out[row]
  int last = 1;              // sums: 1 = apply the export transform, 0 = store the partial sum
  int exp10 = 0;             // fused export transform, OH_GridCompMod.F90:369,1569
  float scale = 1.f;
  float *out = nullptr;      // device: [nrow] or [nrow][out_stride]
  int32_t ctree0 = 0;        // first tree of the constant-table window (set by launch_predict)
};

uint64_t launch_count();
// launches per kernel family since load, and the family that served the last predict launch
// ("duo", "duo_missing", "duo_leaf", "duo_missing_leaf", "nodes8", "nodes8_missing", "nodes8_leaf", ...)
uint64_t kernel_launches(const char *family);
const char *last_predict_kernel();

// 8-byte-node layout: levels 0..kDuoTop-1 of every tree into the tree-top table
cudaError_t upload_const_top(const uint32_t *dev_nodes_xy, const uint32_t *tree_offset, int ntree, cudaStream_t s);
// two-level layout: DuoForest::top_xy into the tree-top table and DuoForest::tree_slot into its base table
cudaError_t upload_const_duo(const uint32_t *top_xy, const uint32_t *tree_slot, int ntree, cudaStream_t s);

// Row-major float matrix -> key tiles.  flags[0] |= 1 if any entry is NaN or == missing; flags[0] |= 2 if any
// entry is +-inf (and `missing` is finite) — what XGDMatrixCreateFromMat checks (xgboost src/data/data.cc).
// X and Xt cover `nrow` rows starting at a tile boundary.
cudaError_t launch_seal_tiles(const float *X, uint64_t nrow, int ncol, float missing, uint32_t *Xt, int *flags, cudaStream_t s);

cudaError_t launch_predict(const DeviceForest &f, const ConstWindow &w, const PredictArgs &a, cudaStream_t s);

// Inplace prediction from a dense float array (XGBoosterPredictFromDense / FromCudaArray): row r, column c of the
// array is X[r * row_stride + c * col_stride].  The predict kernel builds its key tiles from it in shared memory
// (value / margin sums only); PredictArgs::Xt and has_missing are not read.
struct DenseArgs {
  const float *X = nullptr;  // device
  int64_t row_stride = 0;    // in floats
  int64_t col_stride = 1;
  float missing = -999.f;    // entries that are NaN or == missing are missing
  int *flags = nullptr;      // |= 2 on +-inf input when `missing` is finite
};
cudaError_t launch_predict_dense(const DeviceForest &f, const ConstWindow &w, const PredictArgs &a, const DenseArgs &d, cudaStream_t s);

// Per-feature contributions (forest.hpp ShapForest).  out: [nrow][nfeat + 1] floats, column nfeat = `bias`.
//   exact (TreeSHAP on the path bins): launch_shap writes float64 partial sums of bin slice s to
//   part[s][nrow][nfeat]; launch_shap_reduce adds the slices in slice order and rounds once.  The slicing depends
//   only on the number of bins, so every row gets the same sums in the same order whatever the launch shape.
//   approximate (Saabas): launch_shap_approx walks the 8-byte nodes with the node means, float32 in libxgboost's order.
constexpr int kShapSlices = 16;             // bin slices of one call (a 4096-row call is 16 tiles x 16 slices = 256 CTAs)
constexpr uint64_t kShapChunkRows = 32768;  // rows per exact launch: part[] holds kShapSlices x 32768 x nfeat doubles
struct ContribArgs {
  const uint32_t *Xt = nullptr;  // key tiles of rows [0, nrow) (nrow <= kShapChunkRows for launch_shap)
  uint64_t nrow = 0;
  int32_t ncol = 0;
  int32_t nfeat = 0;
  float bias = 0.f;
  float *out = nullptr;
};
cudaError_t launch_shap(const uint4 *bins, int64_t nbins, int nslices, const ContribArgs &a, double *part, cudaStream_t s);
cudaError_t launch_shap_reduce(const double *part, int nslices, const ContribArgs &a, cudaStream_t s);
cudaError_t launch_shap_approx(const DeviceForest &f, const float *mean, int ntree, const ContribArgs &a, cudaStream_t s);

// SHAP interaction values (libxgboost 1.6.0 PredictInteractionContributions).  out: [nrow][nfeat + 1][nfeat + 1]
// floats, row i the conditioning feature, index nfeat the bias.
//   exact: launch_shap_inter runs, for every conditioning feature c, the paths of c's bins (ShapForest::feat_bins,
//   the first nbins of the booster only) extended without c's element, and writes float64 partial sums of slice s of
//   c's list to part[c][s][nrow][nfeat]; launch_shap_inter_reduce adds the slices in slice order, halves them for the
//   off-diagonal and takes the diagonal as phi_c (the slices of launch_shap in shap_part) minus the row's
//   off-diagonal sum, rounding each output once.  The slicing of c's list depends only on the list and nbins.
//   approximate: launch_shap_inter_expand puts the Saabas row contribs[nrow][nfeat + 1] of launch_shap_approx on the
//   diagonal (0 + phi) and +0 elsewhere, as libxgboost's loop does when on == off.
constexpr int kInterSlices = 16;
constexpr uint64_t kInterChunkRows = 4096;  // part[] holds nfeat x 16 x 4096 x nfeat doubles: 382 MB at 27 features
cudaError_t launch_shap_inter(const uint4 *bins, const int64_t *feat_off, const uint32_t *feat_bins, int64_t nbins,
                              const ContribArgs &a, double *part, cudaStream_t s);
cudaError_t launch_shap_inter_reduce(const double *part, const double *shap_part, int shap_slices, const ContribArgs &a,
                                     cudaStream_t s);
cudaError_t launch_shap_inter_expand(const float *contribs, const ContribArgs &a, cudaStream_t s);

// Where the 27 Run1 features come from, in feature order (filled by qcoh_oh_run1): feature f of cell e in column c is
// src3[f][e], or src2[f][c] for a 2-D field; feature 1 is PL_BST / 100, computed from ple.  kernels.cu run1_feature
// reads it for both the fused predict and the matrix pack.
struct Run1Features {
  const float *src3[27];     // [km][ncol] source of feature f, or nullptr if it is a 2-D field
  const float *src2[27];     // [ncol] source of a 2-D feature
  const float *ple = nullptr;  // PLE_BST [km+1][ncol]
};

// Fused Run1 predict: the tile of every CTA is assembled straight from the feature sources
struct SoaArgs {
  Run1Features feat;
  int32_t ncol = 0;
  uint64_t e0 = 0;           // cell index of slab row 0: (k1 - 1) * ncol
  uint64_t nrow = 0;         // ncol * ksub
  float missing = -999.f;
  int32_t ntree_used = 0;
  int32_t ctree0 = 0;        // first tree of the constant-table window (set by launch_predict_soa)
  int exp10 = 1;
  float scale = 1.f;
  float *out = nullptr;      // OH_ML slab
  float *pred = nullptr;     // optional raw booster output
  int *flags = nullptr;      // |= 2 on +-inf input
};
cudaError_t launch_predict_soa(const DeviceForest &f, const ConstWindow &w, const SoaArgs &a, cudaStream_t s);
// The same features as the row-major [npred][27] matrix xx_carr: row m is cell e0 + m
cudaError_t launch_oh_pack(const Run1Features &x, uint64_t e0, int32_t ncol, uint64_t npred, float *X, cudaStream_t s);

// ---- fused Run1 pieces (OH_GridCompMod.F90:1232-1599) ---------------------------------
struct Run1Dev {
  int32_t ncol = 0, km = 0;
  float eps = 0, avogad = 0, runiv = 0, r2d = 0;
  float ohscale = 1.f, tropp_min = 4000.f, missing = -999.f;
  int dynamic_k = 0;
  // Inputs the four kernels read (the 27 features reach the predict and the pack through Run1Features).  The order is
  // part of the kernels' code: when a kernel reads both pointers of one 16-byte word of its parameters, the compiler
  // loads them at once, so moving a field changes the SASS of oh_state / oh_sums (tools/compare_sass.py shows it).
  const float *T_MOD, *Q_MOD, *PLE_MOD, *TROPP;
  const float *PLE_BST, *ZLE_BST;
  const float *TAUCLW, *TAUCLI, *CH4;
  const float *SCA[7];
  const float *OH_CLIM;
  const float *GMITO3, *GMITTO3, *LATS;
  // work / outputs (device)
  float *PL_MOD, *NDWET;             // [km][ncol]
  float *sums[6];                    // wdn idn iup wup aup adn, [km][ncol]
  float *lat_deg, *so3;              // [ncol] latarr, stratO3 (written by oh_sums)
  float *aod, *pl_bst;               // [km][ncol] aod (:1451-1466) and PL_BST (:1488), written by oh_sums
  float *OH_ML;                      // persistent [km][ncol]
  float *OH, *OH_boost;              // [km][ncol]
  float *LOSS_CH4, *LOSS_CO;         // optional [km][ncol] 1/s (build-defined, SURVEY.md 8(f)4)
  int *ctl;                          // [0] ksub (atomicMax) [1] tropp<=tropp_min count [2] the slab's missing / inf
                                     // flags (predict_soa or seal_tiles)
  const float *AREA;                 // [ncol] m2, input of the optional diagnostic
  double *diag;                      // [4] its partial sums
};

cudaError_t launch_oh_state(const Run1Dev &r, cudaStream_t s);
cudaError_t launch_oh_sums(const Run1Dev &r, cudaStream_t s);
cudaError_t launch_oh_finalize(const Run1Dev &r, cudaStream_t s);
cudaError_t launch_oh_diag(const Run1Dev &r, cudaStream_t s);
cudaError_t launch_fill(float *p, uint64_t n, float v, cudaStream_t s);

}  // namespace qcoh
