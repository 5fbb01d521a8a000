/* qcoh.h — C ABI of libqcoh.so, the B200 (sm_100a) replacement for the one hot path of
 * GEOS-ESM/QuickChem: per-grid-cell OH prediction (OH_GridComp -> xgb_fortran_api -> libxgboost).
 *
 * Two groups of entry points:
 *
 *  (1) The eleven XGBoost-named symbols that the reference's Fortran interface module binds
 *      (/root/reference/Shared/xgb_fortran_api.F90:18-120).  Same names, argument meaning,
 *      ownership and 0 / -1 return convention as libxgboost 1.6.0, so the reference's
 *      `predict_OH_with_XGB` (OH_GridComp/OH_GridCompMod.F90:123-398) links against libqcoh.so
 *      unchanged.  Everything numerical runs on the GPU; there is no CPU fallback: without a
 *      CUDA device every compute call returns -1 and XGBGetLastError() says why.
 *
 *  (2) qcoh_* — the device-resident, fused extension a patched Run1 calls
 *      (OH_GridCompMod.F90:1232-1599): feature assembly, prediction, export transform and the
 *      build-defined global-mean diagnostic without ever forming the [N x 27] matrix on the host.
 *
 * Plain pointers and sizes only.  Thread model: a host thread is one "rank" bound to one GPU — one process per
 * GPU (as the reference: `SAVE` booster, OH_GridCompMod.F90:182,209), or one process with one host thread per GPU.
 * All library state (device context, handles, buffer pools, model cache, last-error string) is thread-local: a
 * handle belongs to the thread that created it, and a second thread cannot bind to a GPU that already has one.
 */
#ifndef QCOH_H
#define QCOH_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void *DMatrixHandle;
typedef void *BoosterHandle;
typedef uint64_t bst_ulong;

/* =====================================================================================
 * (1) xgb_fortran_api boundary
 * ================================================================================== */

/* replaces libxgboost XGBoosterLoadModel — xgb_fortran_api.F90:18-24 (wrapper :123-131);
 * call site OH_GridCompMod.F90:261.  Reads XGBoost legacy binary ("binf" optional; what
 * `*.model` / `*.bin` of OH_instance_OH.rc:17-20 are), JSON and UBJSON; flattens the trees
 * into the depth-ordered device layout and uploads them once. */
int XGBoosterLoadModel(BoosterHandle handle, const char *fname);

/* xgb_fortran_api.F90:26-32 (wrapper :133-141).  Unused by OH.  Writes legacy binary, or
 * JSON / UBJSON when fname ends in .json / .ubj (libxgboost 1.6.0 rule). */
int XGBoosterSaveModel(BoosterHandle handle, const char *fname);

/* xgb_fortran_api.F90:34-41 (wrapper :143-152).  Unused by OH.  Writes the dense matrix in
 * libqcoh's own container ("QCDM" magic), readable by XGDMatrixCreateFromFile below. */
int XGDMatrixSaveBinary(DMatrixHandle handle, const char *fname, int silent);

/* xgb_fortran_api.F90:44-49 (wrapper :156-161); call sites OH_GridCompMod.F90:264,377. */
int XGDMatrixFree(DMatrixHandle handle);

/* xgb_fortran_api.F90:52-59 (wrapper :165-174).  Unused by OH.  Reads a "QCDM" file, libsvm text, or
 * csv ("<path>?format=csv[&label_column=N]") like libxgboost's URI; XGBoost's binary DMatrix is not read. */
int XGDMatrixCreateFromFile(const char *fname, int silent, DMatrixHandle *out);

/* xgb_fortran_api.F90:61-73; call site OH_GridCompMod.F90:356 (option_mask=0, ntree_limit=0,
 * training=0).  option_mask: 0 value, 1 margin, 2 leaf index per tree ([nrow][ntree] floats).
 * *out_result points at a pinned host buffer owned by the booster, valid until the next
 * predict / free on that booster (libxgboost's thread-local-entry contract). */
int XGBoosterPredict(BoosterHandle handle, DMatrixHandle dmat, int option_mask, unsigned ntree_limit,
                     int training, bst_ulong *out_len, const float **out_result);

/* libxgboost 1.6.0's JSON-configured predict (not bound by xgb_fortran_api; fortran/qcoh_fortran_api.F90 binds
 * it).  config: {"type", "training", "iteration_begin", "iteration_end", "strict_shape"}, all required.  type 0 value,
 * 1 margin, 6 leaf index (the kernels of XGBoosterPredict), 2 exact per-feature contributions (TreeSHAP), 3
 * approximate contributions (Saabas); 4 / 5 (interactions) fail.  iteration_end = 0: all trees; iteration_begin
 * must be 0.  Shapes: value / margin (nrow), leaf (nrow, ntree), contributions (nrow, num_feature + 1) — the last
 * column is the bias; strict_shape: (nrow, 1), (nrow, ntree, 1, 1), (nrow, 1, num_feature + 1).  *out_shape and
 * *out_result are booster-owned (pinned), valid until the next predict / free on that booster.  Contributions
 * need the node covers (sum_hess > 0 everywhere) and fail on a booster without them. */
int XGBoosterPredictFromDMatrix(BoosterHandle handle, DMatrixHandle dmat, const char *config,
                                const bst_ulong **out_shape, bst_ulong *out_dim, const float **out_result);

/* libxgboost 1.6.0's inplace predicts (what xgboost's Python Booster.inplace_predict calls; fortran/qcoh_fortran_api.F90
 * binds them): prediction straight from a dense float32 array, without a DMatrix.  The predict kernel builds its key
 * tiles from the array in shared memory, so nothing but the result is written to HBM — no copy of the matrix, no key
 * tiles.  values: a JSON array interface {"data": [address, readonly], "shape": [nrow, ncol], "strides": null |
 * [row_bytes, col_bytes], "typestr": "<f4", "version": 3}; other types, masks, shapes that are not 2-D, negative strides
 * or strides that are not a multiple of 4, and a NULL address for a non-empty array fail.  ncol <= the booster's
 * num_feature; absent columns are missing.  config: {"type", "missing", "iteration_begin", "iteration_end",
 * "strict_shape"}, all required (other keys are ignored); type 0 value or 1 margin (both the float32 margin, no
 * transform); entries that are NaN or == missing are missing (NaN is written NaN), +-inf with a finite missing fails
 * like XGDMatrixCreateFromMat; iteration_begin must be 0, iteration_end = 0: all trees.  m (the proxy DMatrix) must be
 * NULL.  Shape (nrow), or (nrow, 1) with strict_shape.  Both return when the result is complete; result and shape are
 * booster-owned, valid until the next predict / free on that booster.
 *   FromDense: HOST memory (pinned or pageable), C-contiguous; it is copied to HBM in chunks, each predicted as it lands,
 *   and read completely before the call returns.  A device address (detected) is read like FromCudaArray.  The
 *   result is a pinned host buffer.
 *   FromCudaArray: DEVICE memory, any strides (a feature-major [ncol][nrow] array is [4, 4 * nrow]).  An optional
 *   "stream" entry (CUDA Array Interface v3: 1 legacy default stream, 2 per-thread default stream, else a cudaStream_t;
 *   0 is invalid) is waited for before the array is read.  The result is a DEVICE buffer. */
int XGBoosterPredictFromDense(BoosterHandle handle, const char *values, const char *config, DMatrixHandle m,
                              const bst_ulong **out_shape, bst_ulong *out_dim, const float **out_result);
int XGBoosterPredictFromCudaArray(BoosterHandle handle, const char *values, const char *config, DMatrixHandle m,
                                  const bst_ulong **out_shape, bst_ulong *out_dim, const float **out_result);

/* xgb_fortran_api.F90:75-83; call site OH_GridCompMod.F90:256.  The reference passes a DMatrix
 * handle *by value* as `dmats` with len = 0; dmats is never dereferenced when len == 0. */
int XGBoosterCreate(const DMatrixHandle dmats[], bst_ulong len, BoosterHandle *out);

/* xgb_fortran_api.F90:85-95; call sites OH_GridCompMod.F90:251,347 (missing = -999.0).
 * data is row-major [nrow][ncol] HOST memory (or device memory: detected), borrowed for the
 * call only.  Entries that are NaN or == missing are missing; +-inf with a finite `missing`
 * fails like libxgboost.  The matrix is copied to HBM here. */
int XGDMatrixCreateFromMat(const float *data, bst_ulong nrow, bst_ulong ncol, float missing,
                           DMatrixHandle *out);

/* xgb_fortran_api.F90:97-104 and :106-113.  Unused by OH. */
int XGDMatrixNumRow(DMatrixHandle handle, bst_ulong *out);
int XGDMatrixNumCol(DMatrixHandle handle, bst_ulong *out);

/* xgb_fortran_api.F90:115-120.  Commented out at OH_GridCompMod.F90:389-392. */
int XGBoosterFree(BoosterHandle handle);

/* libxgboost's error channel (not bound by xgb_fortran_api, but part of the same C API). */
const char *XGBGetLastError(void);

/* =====================================================================================
 * (2) qcoh_* extension
 * ================================================================================== */

/* ---- library / device -------------------------------------------------------------- */
const char *qcoh_version(void);
/* Number of visible CUDA devices (0 without a GPU; never fails). */
int qcoh_device_count(void);
/* Bind this process to one GPU (one process per GPU; default = $LOCAL_RANK or 0). */
int qcoh_set_device(int device);
/* Pinned host memory for callers that want full-speed H2D/D2H (cudaHostAlloc / cudaFreeHost). */
int qcoh_host_alloc(size_t bytes, void **out);
int qcoh_host_free(void *p);
/* Raw device memory + copies, so that a Fortran/C host can keep fields resident in HBM. */
int qcoh_device_alloc(size_t bytes, void **out);
int qcoh_device_free(void *p);
int qcoh_memcpy_h2d(void *dst_dev, const void *src_host, size_t bytes);
int qcoh_memcpy_d2h(void *dst_host, const void *src_dev, size_t bytes);
int qcoh_device_synchronize(void);
/* Device-side timing of library work (CUDA events on the library's stream). */
int qcoh_timer_start(void);
int qcoh_timer_stop(float *elapsed_ms);
/* Overwrite a > L2-sized scratch buffer (cache flush between timed iterations). */
int qcoh_flush_l2(void);

/* ---- booster introspection (host side only; works without a GPU) -------------------- */
typedef struct {
  int32_t num_trees;
  int32_t num_feature;
  int32_t max_depth;       /* deepest leaf over all trees */
  int64_t num_nodes;       /* total nodes */
  float base_score;
  int32_t format;          /* 0 legacy binary, 1 JSON, 2 UBJSON */
  uint32_t version[3];
} qcoh_booster_info;
/* Parse a model file into a booster WITHOUT touching the GPU (upload happens lazily at the
 * first predict).  XGBoosterLoadModel == this + upload. */
int qcoh_booster_parse(BoosterHandle handle, const char *fname);
int qcoh_booster_get_info(BoosterHandle handle, qcoh_booster_info *out);
/* Flattened depth-ordered layout, for inspection/tests: 8-byte nodes {uint32 value_bits;
 * uint32 meta}, see DESIGN.md "Node layout".  tree_offset has num_trees+1 entries. */
int qcoh_booster_get_flat(BoosterHandle handle, const uint32_t **nodes_xy, const uint32_t **tree_offset,
                          const int32_t **tree_depth, const int32_t **orig_id);

/* Two-level records (DESIGN.md "Two levels per gather"), for inspection/tests: 16-byte records
 * {w0, w1, w2, w3}; tree_slot[num_trees] = first record of each tree; top_xy[num_trees][16][2] = the complete
 * heap-ordered levels 0..3 that go to constant memory.  w3 = blk << blk_shift | ... (forest.hpp): blk_shift = 18
 * when the records carry the three default-direction bits (every tree < 2^14 record blocks), else 15.  Fails
 * (-1, reason in XGBGetLastError) when the booster does not qualify (> 2^17 record blocks in a tree). */
int qcoh_booster_get_duo(BoosterHandle handle, const uint32_t **rec, const uint32_t **tree_slot, const uint32_t **top_xy,
                         int64_t *num_slots);
int qcoh_booster_get_duo_info(BoosterHandle handle, int *blk_shift, int *has_default_bits);

/* Contribution tables (DESIGN.md "Contributions"), for inspection/tests; built on first use.  bins[num_bins][32][4]:
 * every root-to-leaf path as a group of consecutive lanes of one 32-lane bin, a bias lane {0, ~0, 0xFF | 1 << 8 |
 * start << 16 | len << 24, leaf value bits} then one lane per distinct feature of the path {lo_key, hi_key,
 * feat | missing_goes_here << 8 | start << 16 | len << 24, zero fraction bits}: a present value with order-preserving
 * key k follows the path iff lo_key <= k < hi_key.  tree_bin[num_trees + 1]: tree t owns bins [tree_bin[t],
 * tree_bin[t+1]).  node_mean[num_nodes]: libxgboost's node mean values by flat node index.  Fails when the booster
 * has no covers. */
int qcoh_booster_get_shap_paths(BoosterHandle handle, const uint32_t **bins, const int64_t **tree_bin,
                                const float **node_mean, int64_t *num_bins);

/* ---- device-resident predict -------------------------------------------------------- */
/* A DMatrix whose storage is allocated in HBM and filled by the caller (device pointer
 * returned by qcoh_dmatrix_device_ptr) or by qcoh_dmatrix_upload.  Call qcoh_dmatrix_seal
 * after filling: it runs the missing / inf scan XGDMatrixCreateFromMat would have run. */
int qcoh_dmatrix_create_device(bst_ulong nrow, bst_ulong ncol, float missing, DMatrixHandle *out);
int qcoh_dmatrix_device_ptr(DMatrixHandle handle, float **out_dev);
int qcoh_dmatrix_upload(DMatrixHandle handle, const float *host_rows, bst_ulong row0, bst_ulong nrows);
int qcoh_dmatrix_seal(DMatrixHandle handle);
/* The device form of a sealed matrix (what the predict kernels read): order-preserving integer keys in
 * feature-major tiles of 256 rows, Xt[tile][1 + col][256] uint32; word-row 0 of a tile is its row order (rows without
 * a missing entry first; original row index | has_missing << 8) (DESIGN.md "Data layout"); for inspection / tests. */
int qcoh_dmatrix_tiles_ptr(DMatrixHandle handle, const uint32_t **out_dev, uint64_t *num_tiles);

/* Export transform fused into the predict kernel's epilogue (OH_GridCompMod.F90:369,1569):
 * out = scale * 10**pred when exp10 != 0, else the raw prediction. */
typedef struct {
  int exp10;      /* 1: apply 10.0**x (OH_GridCompMod.F90:369) */
  float scale;    /* OHscale (OH_GridCompMod.F90:1569); 1.0 = none */
} qcoh_epilogue;
/* Predict into a DEVICE buffer (nrow floats, or nrow*ntree for option_mask 2).  No host copy.
 * epi may be NULL.  Asynchronous on the library stream; qcoh_device_synchronize() to wait. */
int qcoh_booster_predict_device(BoosterHandle handle, DMatrixHandle dmat, int option_mask,
                                unsigned ntree_limit, const qcoh_epilogue *epi, float *out_dev);
/* Per-feature contributions into a DEVICE buffer of nrow * (num_feature + 1) floats, row-major, last column the
 * bias (XGBoosterPredictFromDMatrix type 2, or type 3 when approximate != 0; ntree_limit 0 = all trees).
 * Asynchronous on the library stream; qcoh_device_synchronize() to wait. */
int qcoh_booster_predict_contribs_device(BoosterHandle handle, DMatrixHandle dmat, int approximate,
                                         unsigned ntree_limit, float *out_dev);
/* SHAP interaction values into a DEVICE buffer of nrow * (num_feature + 1)^2 floats, out[row][i][j] row-major, row i
 * the conditioning feature, index num_feature the bias (libxgboost's pred_interactions, PredictInteractionContributions:
 * type 4, or type 5 when approximate != 0; ntree_limit 0 = all trees).  Every row of M sums to the row's contribution,
 * M[F][F] is the contributions' bias, and the bias row and column are otherwise 0.  Exact values take about 57
 * conditioned TreeSHAP passes per row: explain a slab of rows at a time.  Asynchronous on the library stream;
 * qcoh_device_synchronize() to wait. */
int qcoh_booster_predict_interactions_device(BoosterHandle handle, DMatrixHandle dmat, int approximate,
                                             unsigned ntree_limit, float *out_dev);
/* Library settings of the calling thread; values are integers.  Any other name fails with "unknown parameter".
 *   duo         0: predict on the 8-byte nodes only.  Any other value (default -1): on the two-level records
 *               whenever the booster's records and the matrix allow it.
 *   speculate   1 (default): XGDMatrixCreateFromMat also predicts with the last-loaded booster, pipelined with
 *               the copy; 0: it does not.
 *   chunk_rows  rows per copy chunk of XGDMatrixCreateFromMat, rounded up to a multiple of 256 (at most 2^19 from
 *               pageable memory); <= 0 restores the default 2^21. */
int qcoh_set_param(const char *name, const char *value);
/* How many kernels the library has launched since load (for bench.py's gpu_launches). */
uint64_t qcoh_launch_count(void);
/* Which kernel family served a prediction — what the parity tests assert.  Families: "duo" (two-level records),
 * "nodes8" (8-byte depth-ordered nodes), each with the suffixes "_missing" (matrix with missing entries) and
 * "_leaf" (option_mask = 2), e.g. "duo_missing_leaf"; "soa_duo" / "soa_nodes8" (fused Run1); "seal_tiles";
 * "shap" (exact contributions) with its slice reduction "shap_reduce", and "shap_approx" (approximate contributions);
 * "shap_inter" (exact interaction values, after a "shap" launch for the same rows) with "shap_inter_reduce", and
 * "shap_inter_expand" (approximate interaction values, after a "shap_approx" launch).
 * qcoh_kernel_launches counts launches of one family since load; qcoh_last_predict_kernel names the family of the
 * last XGBoosterPredict-side launch ("" before the first). */
uint64_t qcoh_kernel_launches(const char *family);
const char *qcoh_last_predict_kernel(void);

/* ---- fused Run1 (feature assembly -> predict -> export transform) -------------------- */
typedef void *qcoh_oh_handle;

/* Static configuration: OH_GridComp state + MAPL constants (OH_GridCompMod.F90:48-80,547-567;
 * MAPL constants are external to the reference and therefore passed in, not hard-coded). */
typedef struct {
  int ncol;                 /* local columns im*jm, i fastest */
  int km;                   /* levels */
  float mapl_epsilon, mapl_avogad, mapl_runiv, mapl_radians_to_degrees, mapl_degrees_to_radians;
  float ohscale;            /* OH_instance_OH.rc:42 */
  int compute_once_per_day; /* OH_instance_OH.rc:38; dynamic_k_range = !this (:1561) */
  float tropp_min;          /* 4000 Pa (:1563) */
  float missing;            /* -999.0 (:213) */
} qcoh_oh_config;

/* Per-step inputs.  Every pointer may be HOST or DEVICE memory (detected per pointer); host
 * fields are copied to resident HBM buffers, device fields are used in place.  Layout: 3-D
 * centre fields [km][ncol], edge fields (PLE, ZLE) [km+1][ncol], 2-D fields [ncol] — the
 * Fortran (im,jm,km) arrays as they lie in memory. */
typedef struct {
  int nymd;                 /* yyyymmdd, for JulianDay (:1481) */
  int need_to_call_boost;   /* :1189-1193; 0 => reuse the persistent OH_ML (:76-78) */
  /* current model state, :1233-1236 */
  const float *T_MOD, *Q_MOD, *PLE_MOD, *TROPP;
  /* values handed to boost, selected per OH_data_source by the caller (:1326-1436,1493-1540) */
  const float *T_BST, *Q_BST, *PLE_BST, *ZLE_BST;
  const float *TAUCLW, *TAUCLI, *FCLD, *CH4, *CO;
  const float *SCA[7];      /* BC OC BR DU SU SS NI scattering coefficients at wavelength_index */
  const float *NO2, *O3, *ISOP, *ACET, *C2H6, *C3H8, *PRPE, *ALK4, *MP, *H2O2, *CH2O;
  const float *GMITO3, *GMITTO3, *ALBUV, *LATS, *LONS;
  const float *OH_CLIM;     /* oh_OH (default OH above the tropopause, :1548,1584) */
  /* optional inputs of the build-defined diagnostic (not in the reference; SURVEY.md 0.3) */
  const float *AREA;        /* [ncol] m2, may be NULL */
} qcoh_run1_in;

/* Outputs; NULL = not wanted.  HOST or DEVICE pointers. */
typedef struct {
  float *OH;        /* [km][ncol] molec/cm3 — internal state OH (:1595) */
  float *OH_boost;  /* [km][ncol] mol/mol — export OH_boost (:1571-1572) */
  float *NDWET;     /* [km][ncol] — export DIAG_NDWET (:1598-1599) */
  float *X;         /* [ncol*ksub][27] assembled feature matrix (debug / parity) */
  float *pred;      /* [ncol*ksub] raw booster output (debug / parity) */
  /* SURVEY.md 8(f)4 — what the consumers of OH need next (the parent re-exports OH for the CH4 / CO
   * chemistry, QuickChem_GridCompMod.F90:184-185; comment OH_GridCompMod.F90:1590-1591).  Build-defined,
   * not in the reference: first-order loss frequencies [km][ncol] in 1/s from the final OH (molec/cm3),
   *   LOSS_CH4 = 2.45e-12 exp(-1775 / T_MOD) * OH        (JPL 19-5, OH + CH4)
   *   LOSS_CO  = 1.5e-13 (1 + 0.6 PL_MOD / 101325) * OH  (OH + CO, pressure-dependent form) */
  float *LOSS_CH4, *LOSS_CO;
  int k1;           /* out: first predicted level, 1-based (k2 = km), :300-301 */
  /* build-defined diagnostic, local partial sums (float64): sum(OH*w), sum(w),
   * sum(nCH4*V), sum(k(T)*OH*nCH4*V); valid when AREA != NULL */
  double diag[4];
} qcoh_run1_out;

int qcoh_oh_create(BoosterHandle booster, const qcoh_oh_config *cfg, qcoh_oh_handle *out);
int qcoh_oh_run1(qcoh_oh_handle h, const qcoh_run1_in *in, qcoh_run1_out *out);
int qcoh_oh_free(qcoh_oh_handle h);
/* Replace the booster a fused-Run1 handle predicts with (27 features required).  The persistent OH_ML of
 * the previous boost step stays valid.  The booster must outlive the handle. */
int qcoh_oh_set_booster(qcoh_oh_handle h, BoosterHandle booster);
int qcoh_oh_get_booster(qcoh_oh_handle h, BoosterHandle *out);

/* ---- monthly model files (SURVEY.md 0.5 / 8(f)3) -------------------------------------- */
/* The reference expands `XGBoostFile: ..._M%m2.model` (OH_instance_OH.rc:20) with fill_grads_template on
 * every Run1 (OH_GridCompMod.F90:1187) but its SAVE'd booster is loaded once (:182,209,242-271), so a
 * month roll-over keeps predicting with the start month's model.  libqcoh keeps that behaviour unless the
 * host opts in with the three calls below.
 *
 * GrADS-style expansion of the tokens %y4 %y2 %m1 %m2 %mc %Mc %MC %d1 %d2 %h1 %h2 %n2 %j3 (%% = '%');
 * nymd = yyyymmdd, nhms = hhmmss.  Fails on an unknown token or when `cap` (including the NUL) is too small. */
int qcoh_expand_template(const char *pattern, int nymd, int nhms, char *out, size_t cap);
/* Per-thread (= per GPU) cache of parsed + uploaded boosters keyed by file name: the first request for a name loads
 * it, later ones return the same handle.  Handles belong to the cache (XGBoosterFree on one fails); a month
 * of the production forest is ~30 MB of HBM (both node layouts), so all twelve stay resident. */
int qcoh_model_cache_get(const char *fname, BoosterHandle *out);
int qcoh_model_cache_size(void);
/* Frees every cached booster; handles obtained from the cache (and fused-Run1 handles using them) die. */
int qcoh_model_cache_clear(void);
/* expand + cache_get + qcoh_oh_set_booster in one call: what a patched Run1 calls before a boost step when
 * `reload_model_on_month_change` is on.  *changed (may be NULL) is set to 1 when the booster was switched. */
int qcoh_oh_select_model(qcoh_oh_handle h, const char *pattern, int nymd, int nhms, int *changed);
/* Diagnostic exports (OH_GridCompMod.F90:1602-1735, OH_StateSpecs.rc:41-73): copy one derived field out of HBM.
 * name (case-sensitive, the DIAG_ suffix of the reference's export).  Of the LAST BOOST step, 3-D [km][ncol]:
 * "TAUCLWDN" "TAUCLIDN" "TAUCLIUP" "TAUCLWUP" "AODUP" "AODDN" "AOD" "PL" (bb%PL = PL_BST, from the PLE handed to
 * boost, Pa, :1488,:1666) "OH_boost"; 2-D [ncol]: "LAT" "SZA" "stratO3".  Of the CURRENT step (the reference
 * exports DIAG_NDWET on every alarmed step, :1598-1599): "NDWET", and "PL_MOD" (not a reference export).
 * out may be host or device memory. */
int qcoh_oh_get_diag(qcoh_oh_handle h, const char *name, float *out);
/* The noon SZA (OH_GridCompMod.F90:401-466) is cached per day of year and grid (addresses, size and a hash of a
 * strided sample of LATS / LONS).  A host that rewrites its coordinate arrays in place calls this to force a
 * recomputation at the next boost step. */
int qcoh_oh_invalidate_sza(qcoh_oh_handle h);

/* ---- Run1 control: the host-side decisions around the fused call -------------------- */
/* OH_data_source (OH_GridCompMod.F90:31-33, rc key `OH_data_source`, OH_instance_OH.rc:24). */
enum { QCOH_PRECOMPUTED = 1, QCOH_ONLINE_INST = 2, QCOH_ONLINE_AVG24 = 3 };
/* "PRECOMPUTED" / "ONLINE_INST" / "ONLINE_AVG24" -> 1 / 2 / 3 (:551-553); -1 for anything else. */
int qcoh_data_source_from_name(const char *token);
/* :1189-1193 — qcoh_run1_in.need_to_call_boost: with compute_once_per_day only the step at hhmmss == 0 boosts. */
int qcoh_need_to_call_boost(int compute_once_per_day, int nhms);
/* :1307-1320 — the 24-hour-average spin-up switch: ONLINE_AVG24 and T_avg24(1,1,1) == 0.0. */
int qcoh_use_inst_values(int data_source, float t_avg24_first);
/* Which import feeds a boost-state field (:1326-1548).  field: "T" "Q" "PLE" "ZLE" "TAUCLW" "TAUCLI" "CH4" "CO"
 * "FCLD" and "BCSCACOEF".."NISCACOEF" follow OH_data_source ("oh_X" / "X" / "X_avg24", or "X" during spin-up);
 * the climatological ones ("NO2" .. "CH2O", "ALBUV", "GMITO3", "GMITTO3", "OH") are always "oh_X"; "T_MOD" "Q_MOD"
 * "PLE_MOD" "TROPP" are the current model state "T" "Q" "PLE" "TROPP".  *is_4d (may be NULL) = 1 when the import
 * carries a wavelength axis (online scattering coefficients, sliced at wavelength_index, :1456-1465). */
int qcoh_import_name(const char *field, int data_source, int use_inst_values, char *out, size_t cap, int *is_4d);

/* ---- host mirror of the reference driver -------------------------------------------- */
/* C mirror of `predict_OH_with_XGB` (OH_GridCompMod.F90:123-398): same arguments in the same
 * order, arrays as Fortran lays them out; bb = the 27 OH_BOOST_INPUT_DATA pointers (:82-114) in
 * feature order, is2d[f] != 0 for the (i,j) members.  Goes ONLY through the eleven XGBoost-named
 * symbols above — it is what the unmodified Fortran does, restated in C for hosts without a
 * Fortran compiler — and keeps the booster in static storage like the reference's SAVE. */
int qcoh_predict_OH_with_XGB(const char *xgb_fname, int icount, int jcount, int kcount,
                             int dynamic_k_range, float tropp_min, const float *pl, const float *tropp,
                             const float *const bb[27], const int is2d[27], float *OH_ML);
/* Drop the static booster of the mirror (tests). */
void qcoh_predict_OH_reset(void);
/* on != 0: the mirror calls XGBoosterLoadModel again whenever xgb_fname differs from the file its static
 * booster was loaded from (fixes SURVEY.md 0.5); default 0 = the reference's load-once behaviour. */
void qcoh_predict_OH_reload_on_file_change(int on);

/* ---- the one collective: all-reduce of the diagnostic partial sums over NCCL ------------- */
/* One process per GPU.  Rank 0 obtains a 128-byte id and hands it to the others (MPI_Bcast in a MAPL host);
 * every rank then joins.  libnccl.so.2 is dlopen'ed on first use (no link-time dependency).  The data path
 * needs none of this: cells shard with no halo (SURVEY.md 8e). */
int qcoh_comm_get_unique_id(char id[128]);
int qcoh_comm_init(int nranks, int rank, const char id[128]);
/* In-place sum over all ranks of n float64 values in host memory (qcoh_run1_out.diag: n = 4). */
int qcoh_comm_allreduce_sum_f64(double *values, int n);
int qcoh_comm_destroy(void);

/* ---- sharding across GPUs (SURVEY.md 8e) -------------------------------------------- */
/* Contiguous, near-equal split of `ncol_global` columns over `nranks`; no halo. */
int qcoh_partition_columns(int64_t ncol_global, int nranks, int rank, int64_t *col0, int64_t *ncol_local);

#ifdef __cplusplus
}
#endif
#endif /* QCOH_H */
