// capi_oh.cpp — the fused, device-resident Run1 of the qcoh_* extension (include/qcoh.h, group 2):
// what a patched OH_GridCompMod Run1 calls instead of PREP_FOR_BOOST ... OH = (OH*NDWET)*1e-6
// (/root/reference/OH_GridComp/OH_GridCompMod.F90:1232-1599).
#include "context.hpp"

using namespace qcoh;

namespace {

// JulianDay / leap_year — OH_GridCompMod.F90:1905-1971
bool is_leap(int ny) { return ny >= 0 && ((ny % 100 == 0 && ny % 400 == 0) || (ny % 4 == 0 && ny % 100 != 0)); }
int julian_day(int nymd) {
  static const int days[12] = {31, 28, 31, 30, 31, 30, 31, 31, 30, 31, 30, 31};
  const int ny = nymd / 10000, mm = (nymd % 10000) / 100;
  int ds = nymd % 100;
  if (nymd < 0 || mm < 1 || mm > 12 || ds < 1 || ds > ((mm == 2 && is_leap(ny)) ? 29 : days[mm - 1]))
    throw Error("qcoh_oh_run1: nymd = " + std::to_string(nymd) + " is not a yyyymmdd date");
  for (int m = 1; m < mm; ++m) ds += (m == 2 && is_leap(ny)) ? 29 : days[m - 1];
  return ds;
}

// computeSolarZenithAngle_LocalNoon — OH_GridCompMod.F90:401-466.  Evaluated on the HOST with
// the C library's float32 sin/asin/cos/acos: that is what the compiled Fortran calls, and the
// GPU's libdevice versions differ from it in the last bit (a 1-ulp SZA change can flip a leaf).
// It is a 2-D field that only changes with the day of year, so it is cached per (jday, grid).
void noon_sza_range(int jday, const float *lat, const float *lon, int i0, int i1, float r2d, float d2r, float *out) {
  const float sindec = 0.3978f * sinf(0.9863f * ((float)jday - 80.0f) * d2r);
  const float cosdec = cosf(asinf(sindec));
  for (int i = i0; i < i1; ++i) {
    const float sinlat = sinf(lat[i]);
    const float coslat = cosf(asinf(sinlat));
    float mylon = lon[i] * r2d;
    if (mylon > 180.0f) mylon = mylon - 360.0f;
    if (mylon < -180.0f) mylon = mylon + 360.0f;
    const float tau = 12.0f + (mylon / -180.0f) * 12.0f;
    const float loct = ((tau * 15.0f) - 180.0f) * d2r + lon[i];
    float cosz = cosdec * coslat * cosf(loct) + sindec * sinlat;
    cosz = fminf(1.0f, cosz);
    cosz = fmaxf(-1.0f, cosz);
    out[i] = acosf(cosz) * r2d;
  }
}

void noon_sza(int jday, const float *lat, const float *lon, int n, float r2d, float d2r, float *out) {
  unsigned nt = std::thread::hardware_concurrency();
  if (nt == 0) nt = 1;
  if (nt > 64) nt = 64;
  if ((unsigned)n < nt * 1024) nt = 1;
  std::vector<std::thread> th;
  for (unsigned t = 0; t < nt; ++t) {
    const int i0 = (int)((int64_t)n * t / nt), i1 = (int)((int64_t)n * (t + 1) / nt);
    th.emplace_back(noon_sza_range, jday, lat, lon, i0, i1, r2d, d2r, out);
  }
  for (auto &t : th) t.join();
}

struct Oh {
  uint32_t magic = kOhMagic;
  Booster *booster = nullptr;
  qcoh_oh_config cfg;
  // resident copies of host-provided inputs: one slot per pointer-sized word of qcoh_run1_in (SLOT)
  DevBuf<float> in[sizeof(qcoh_run1_in) / sizeof(const float *)];
  DevBuf<float> PL_MOD, NDWET, sums[6], aod, pl_bst, OH_ML, OH, OH_boost, X, pred, sza, lat_deg, so3, loss_ch4, loss_co;
  DevBuf<uint32_t> Xt;
  DevBuf<int> ctl;
  DevBuf<double> diag;
  PinBuf<float> h_sza, h_lat, h_lon, h_probe;
  // noon-SZA cache key: day of year, the grid's size and addresses, and a hash of a strided sample of LATS / LONS
  // (a host that re-uses its buffers for another grid gets a new SZA; qcoh_oh_invalidate_sza forces one)
  int sza_jday = -1;
  size_t sza_n = 0;
  const float *sza_lat_key = nullptr, *sza_lon_key = nullptr;
  uint64_t sza_hash = 0;
  bool oh_ml_valid = false;
  ~Oh() {
    if (booster) --booster->oh_refs;
  }
};

constexpr int kProbe = 2048;
// FNV-1a over a strided sample of both coordinate arrays (host or device memory)
uint64_t grid_probe_hash(Oh *o, const float *lat, const float *lon, size_t n) {
  const size_t stride = (n + kProbe - 1) / kProbe, cnt = (n + stride - 1) / stride;  // cnt <= kProbe
  float *h = o->h_probe.need(2 * (size_t)kProbe + 2);
  CU(cudaMemcpy2DAsync(h, sizeof(float), lat, stride * sizeof(float), sizeof(float), cnt, cudaMemcpyDefault, g.stream));
  CU(cudaMemcpy2DAsync(h + cnt, sizeof(float), lon, stride * sizeof(float), sizeof(float), cnt, cudaMemcpyDefault, g.stream));
  CU(cudaMemcpyAsync(h + 2 * cnt, lat + (n - 1), sizeof(float), cudaMemcpyDefault, g.stream));
  CU(cudaMemcpyAsync(h + 2 * cnt + 1, lon + (n - 1), sizeof(float), cudaMemcpyDefault, g.stream));
  CU(cudaStreamSynchronize(g.stream));
  uint64_t x = 1469598103934665603ull;
  const unsigned char *b = (const unsigned char *)h;
  for (size_t i = 0; i < (2 * cnt + 2) * sizeof(float); ++i) x = (x ^ b[i]) * 1099511628211ull;
  return x;
}

Oh *O(qcoh_oh_handle h) {
  Oh *o = (Oh *)h;
  if (!o || !is_live(h) || o->magic != kOhMagic) throw Error("Invalid OH handle");
  return o;
}

void bind_booster(Oh *o, Booster *b) {
  if (o->booster == b) return;
  if (o->booster) --o->booster->oh_refs;
  o->booster = b;
  ++b->oh_refs;
}

// host pointer -> resident device copy; device pointer -> used in place
const float *resident(Oh *o, size_t slot, const float *p, size_t n, const char *name) {
  if (!p) throw Error(std::string("qcoh_oh_run1: input field ") + name + " is NULL");
  if (is_device_ptr(p)) return p;
  float *d = o->in[slot].need(n);
  CU(cudaMemcpyAsync(d, p, n * 4, cudaMemcpyHostToDevice, g.stream));
  return d;
}

void deliver(float *user, const float *dev, size_t n) {
  if (!user) return;
  CU(cudaMemcpyAsync(user, dev, n * 4, is_device_ptr(user) ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, g.stream));
}

}  // namespace

// The resident buffer of input field F is the one at F's position in qcoh_run1_in: the order in which qcoh_oh_run1
// reads its inputs does not matter, and skipped inputs leave the others where they are.
#define SLOT(F) (offsetof(qcoh_run1_in, F) / sizeof(const float *))
#define RESIDENT(F, n) resident(o, SLOT(F), in->F, n, #F)

extern "C" {

int qcoh_oh_create(BoosterHandle booster, const qcoh_oh_config *cfg, qcoh_oh_handle *out) {
  API_BEGIN
  Booster *b = B(booster);
  if (!cfg || !out) throw Error("qcoh_oh_create: NULL argument");
  if (cfg->ncol <= 0 || cfg->km <= 0) throw Error("qcoh_oh_create: ncol and km must be positive");
  if (!b->loaded) throw Error("Booster has no model: call XGBoosterLoadModel first");
  if (b->host.num_feature != 27)
    throw Error("OH_GridComp packs exactly 27 features (OH_GridCompMod.F90:228); the booster has " + std::to_string(b->host.num_feature));
  ensure_device();
  upload(b);
  std::unique_ptr<Oh> o(new Oh());
  bind_booster(o.get(), b);
  o->cfg = *cfg;
  const size_t n3 = (size_t)cfg->ncol * cfg->km;
  o->OH_ML.need(n3);
  CU(cudaMemsetAsync(o->OH_ML.p, 0, n3 * 4, g.stream));
  g_live_handles.insert(o.get());
  *out = o.release();
  API_END
}

int qcoh_oh_set_booster(qcoh_oh_handle h, BoosterHandle booster) {
  API_BEGIN
  Oh *o = O(h);
  Booster *b = B(booster);
  if (!b->loaded) throw Error("Booster has no model: call XGBoosterLoadModel first");
  if (b->host.num_feature != 27)
    throw Error("OH_GridComp packs exactly 27 features (OH_GridCompMod.F90:228); the booster has " + std::to_string(b->host.num_feature));
  ensure_device();
  upload(b);
  bind_booster(o, b);
  API_END
}

int qcoh_oh_get_booster(qcoh_oh_handle h, BoosterHandle *out) {
  API_BEGIN
  if (!out) throw Error("qcoh_oh_get_booster: out is NULL");
  *out = O(h)->booster;
  API_END
}

int qcoh_oh_get_diag(qcoh_oh_handle h, const char *name, float *out) {
  API_BEGIN
  Oh *o = O(h);
  if (!name || !out) throw Error("qcoh_oh_get_diag: NULL argument");
  if (!o->oh_ml_valid) throw Error("qcoh_oh_get_diag: no boost step has run yet");
  const size_t n2 = (size_t)o->cfg.ncol, n3 = n2 * o->cfg.km;
  const std::string s(name);
  const float *src = nullptr;
  size_t n = n3;
  static const char *sum_names[6] = {"TAUCLWDN", "TAUCLIDN", "TAUCLIUP", "TAUCLWUP", "AODUP", "AODDN"};
  for (int i = 0; i < 6; ++i)
    if (s == sum_names[i]) src = o->sums[i].p;
  if (s == "PL") src = o->pl_bst.p;      // bb%PL = PL_BST, from the PLE handed to boost (:1488, :1666)
  if (s == "AOD") src = o->aod.p;        // :1690
  if (s == "PL_MOD") src = o->PL_MOD.p;  // current step (not a reference export)
  if (s == "NDWET") src = o->NDWET.p;    // NDWET_MOD of the CURRENT step, as DIAG_NDWET (:1598-1599)
  if (s == "OH_boost") src = o->OH_ML.p;
  if (s == "LAT") src = o->lat_deg.p, n = n2;
  if (s == "SZA") src = o->sza.p, n = n2;
  if (s == "stratO3") src = o->so3.p, n = n2;
  if (!src) throw Error("qcoh_oh_get_diag: unknown or unavailable field '" + s + "'");
  deliver(out, src, n);
  CU(cudaStreamSynchronize(g.stream));
  API_END
}

int qcoh_oh_free(qcoh_oh_handle h) {
  API_BEGIN
  Oh *o = O(h);
  if (g.ready) CU(cudaStreamSynchronize(g.stream));
  o->magic = 0;
  g_live_handles.erase(o);
  delete o;
  API_END
}

int qcoh_oh_invalidate_sza(qcoh_oh_handle h) {
  API_BEGIN
  O(h)->sza_jday = -1;
  API_END
}

int qcoh_oh_run1(qcoh_oh_handle h, const qcoh_run1_in *in, qcoh_run1_out *out) {
  API_BEGIN
  Oh *o = O(h);
  if (!in || !out) throw Error("qcoh_oh_run1: NULL argument");
  if (!out->OH) throw Error("qcoh_oh_run1: out->OH is required");
  ensure_device();
  const qcoh_oh_config &c = o->cfg;
  const int nc = c.ncol, km = c.km;
  const size_t n2 = (size_t)nc, n3 = (size_t)nc * km, ne = (size_t)nc * (km + 1);
  Run1Dev r{};
  r.ncol = nc, r.km = km;
  r.eps = c.mapl_epsilon, r.avogad = c.mapl_avogad, r.runiv = c.mapl_runiv, r.r2d = c.mapl_radians_to_degrees;
  r.ohscale = c.ohscale, r.tropp_min = c.tropp_min, r.missing = c.missing;
  r.dynamic_k = c.compute_once_per_day ? 0 : 1;  // :1561
  r.T_MOD = RESIDENT(T_MOD, n3);
  r.Q_MOD = RESIDENT(Q_MOD, n3);
  r.PLE_MOD = RESIDENT(PLE_MOD, ne);
  r.TROPP = RESIDENT(TROPP, n2);
  r.OH_CLIM = RESIDENT(OH_CLIM, n3);
  const bool boost = in->need_to_call_boost != 0;
  if (!boost && !o->oh_ml_valid) throw Error("qcoh_oh_run1: need_to_call_boost = 0 before any boost call (OH_ML is undefined)");
  const bool want_diag = in->AREA != nullptr;
  if (boost || want_diag) {
    r.ZLE_BST = RESIDENT(ZLE_BST, ne);
    r.CH4 = RESIDENT(CH4, n3);
  }
  Run1Features feat{};
  if (boost) {
    // aliasing (ONLINE_INST hands the same arrays as model state and boost input) is preserved: identical host
    // pointers are uploaded once (PLE here, T and Q in the feature table)
    r.PLE_BST = in->PLE_BST == in->PLE_MOD ? r.PLE_MOD : RESIDENT(PLE_BST, ne);
    r.TAUCLW = RESIDENT(TAUCLW, n3);
    r.TAUCLI = RESIDENT(TAUCLI, n3);
    for (int i = 0; i < 7; ++i) r.SCA[i] = resident(o, SLOT(SCA) + i, in->SCA[i], n3, ("SCA[" + std::to_string(i) + "]").c_str());
    r.GMITO3 = RESIDENT(GMITO3, n2);
    r.GMITTO3 = RESIDENT(GMITTO3, n2);
    r.LATS = RESIDENT(LATS, n2);
    if (!in->LONS) throw Error("qcoh_oh_run1: input field LONS is NULL");
    // noon SZA (host libm, cached per day and grid)
    const int jday = julian_day(in->nymd);
    const uint64_t probe = grid_probe_hash(o, in->LATS, in->LONS, n2);
    if (jday != o->sza_jday || in->LATS != o->sza_lat_key || in->LONS != o->sza_lon_key || n2 != o->sza_n || probe != o->sza_hash) {
      float *hl = o->h_lat.need(n2), *hn = o->h_lon.need(n2), *hs = o->h_sza.need(n2);
      CU(cudaMemcpyAsync(hl, in->LATS, n2 * 4, cudaMemcpyDefault, g.stream));
      CU(cudaMemcpyAsync(hn, in->LONS, n2 * 4, cudaMemcpyDefault, g.stream));
      CU(cudaStreamSynchronize(g.stream));
      noon_sza(jday, hl, hn, nc, c.mapl_radians_to_degrees, c.mapl_degrees_to_radians, hs);
      CU(cudaMemcpyAsync(o->sza.need(n2), hs, n2 * 4, cudaMemcpyHostToDevice, g.stream));
      o->sza_jday = jday, o->sza_lat_key = in->LATS, o->sza_lon_key = in->LONS, o->sza_n = n2, o->sza_hash = probe;
    }
    for (int i = 0; i < 6; ++i) r.sums[i] = o->sums[i].need(n3);
    r.lat_deg = o->lat_deg.need(n2), r.so3 = o->so3.need(n2);
    // The 27 features of predict_OH_with_XGB, in its order (OH_GridCompMod.F90:303-345): the fused predict and the
    // matrix pack both read them from this table.
    feat.src2[0] = r.lat_deg;  // LATS * radToDeg (:1444), written by oh_sums
    feat.ple = r.PLE_BST;      // feature 1: PL_BST / 100 (:314), computed by run1_feature
    feat.src3[2] = in->T_BST == in->T_MOD ? r.T_MOD : RESIDENT(T_BST, n3);
    feat.src3[3] = RESIDENT(NO2, n3);
    feat.src3[4] = RESIDENT(O3, n3);
    feat.src3[5] = r.CH4;
    feat.src3[6] = RESIDENT(CO, n3);
    feat.src3[7] = RESIDENT(ISOP, n3);
    feat.src3[8] = RESIDENT(ACET, n3);
    feat.src3[9] = RESIDENT(C2H6, n3);
    feat.src3[10] = RESIDENT(C3H8, n3);
    feat.src3[11] = RESIDENT(PRPE, n3);
    feat.src3[12] = RESIDENT(ALK4, n3);
    feat.src3[13] = RESIDENT(MP, n3);
    feat.src3[14] = RESIDENT(H2O2, n3);
    for (int i = 0; i < 4; ++i) feat.src3[15 + i] = r.sums[i];  // TAUCLWDN TAUCLIDN TAUCLIUP TAUCLWUP
    feat.src3[19] = RESIDENT(FCLD, n3);
    feat.src3[20] = in->Q_BST == in->Q_MOD ? r.Q_MOD : RESIDENT(Q_BST, n3);
    feat.src2[21] = r.so3;     // GMITO3 - GMITTO3 (:1446), written by oh_sums
    feat.src2[22] = RESIDENT(ALBUV, n2);
    feat.src3[23] = r.sums[4];  // AODUP
    feat.src3[24] = r.sums[5];  // AODDN
    feat.src3[25] = RESIDENT(CH2O, n3);
    feat.src2[26] = o->sza.p;  // noon SZA
  }
  if (want_diag) r.AREA = RESIDENT(AREA, n2);
  r.PL_MOD = o->PL_MOD.need(n3), r.NDWET = o->NDWET.need(n3);
  r.OH_ML = o->OH_ML.p, r.OH = o->OH.need(n3), r.OH_boost = o->OH_boost.need(n3);
  r.LOSS_CH4 = out->LOSS_CH4 ? o->loss_ch4.need(n3) : nullptr;
  r.LOSS_CO = out->LOSS_CO ? o->loss_co.need(n3) : nullptr;
  r.ctl = o->ctl.need(3);
  r.diag = o->diag.need(4);
  CU(cudaMemsetAsync(r.ctl, 0, 3 * sizeof(int), g.stream));
  CU(launch_oh_state(r, g.stream));
  out->k1 = 0;
  bool check_inf_after = false;
  if (boost) {
    int ctl[2];
    CU(cudaMemcpyAsync(ctl, r.ctl, sizeof ctl, cudaMemcpyDeviceToHost, g.stream));
    CU(cudaStreamSynchronize(g.stream));
    if (!r.dynamic_k && ctl[1] != 0) throw Error("OH Prediction: Minimum tropopause pressure is not low enough!");  // :288
    const int ksub = ctl[0];
    const int k1 = km - ksub + 1;  // :300
    out->k1 = k1;
    const uint64_t npred = (uint64_t)nc * ksub, e0 = (uint64_t)(k1 - 1) * nc;
    r.aod = o->aod.need(n3), r.pl_bst = o->pl_bst.need(n3);
    CU(launch_oh_sums(r, g.stream));
    B(o->booster);  // the handle holds a reference (XGBoosterFree refuses while it does); checked all the same
    upload(o->booster);
    CU(cudaMemsetAsync(r.OH_ML, 0, n3 * 4, g.stream));  // self%OH_ML = 0.0 (:1559)
    const int ntree = o->booster->dev.ntree;
    const bool too_many_trees = ntree > kRangeTrees;  // ranged launches need the matrix form
    if (npred && !out->X && !too_many_trees) {
      // fused: pack (:303-345) + create (:347) + predict (:356) + 10**x (:369) * OHscale (:1569) in one
      // kernel reading the SoA fields; the [N x 27] matrix is never formed
      SoaArgs a;
      a.feat = feat, a.ncol = nc, a.e0 = e0, a.nrow = npred, a.missing = c.missing;
      a.ntree_used = ntree, a.exp10 = 1, a.scale = c.ohscale;
      a.out = r.OH_ML + e0;
      a.pred = out->pred ? o->pred.need(npred) : nullptr;
      a.flags = r.ctl + 2;
      CU(launch_predict_soa(o->booster->dev, hold(o->booster, 0, ntree), a, g.stream));
      if (out->pred) deliver(out->pred, a.pred, npred);
      check_inf_after = true;
    } else if (npred) {
      // debug / parity path: materialise xx_carr so that it can be handed back (out->X)
      float *X = o->X.need(npred * 27);
      CU(launch_oh_pack(feat, e0, nc, npred, X, g.stream));
      // XGDMatrixCreateFromMat (:347): scan + key tiles
      uint32_t *Xt = o->Xt.need(tile_words(npred, 27));
      CU(launch_seal_tiles(X, npred, 27, c.missing, Xt, r.ctl + 2, g.stream));
      int flags = 0;
      CU(cudaMemcpyAsync(&flags, r.ctl + 2, sizeof(int), cudaMemcpyDeviceToHost, g.stream));
      CU(cudaStreamSynchronize(g.stream));
      if ((flags & 2) && !std::isinf(c.missing)) throw Error("Check failed: valid: Input data contains `inf` or `nan`");
      PredictArgs a;
      a.Xt = Xt, a.nrow = npred, a.ncol = 27, a.has_missing = flags & 1, a.pred_leaf = 0;
      a.tree_begin = 0, a.tree_end = ntree, a.out_stride = a.tree_end;
      a.exp10 = 1, a.scale = c.ohscale;
      a.out = r.OH_ML + e0;
      launch_predict_chunked(o->booster, a, g.stream);
      if (out->pred) {
        a.exp10 = 0, a.scale = 1.f, a.out = o->pred.need(npred);
        launch_predict_chunked(o->booster, a, g.stream);
        deliver(out->pred, a.out, npred);
      }
      if (out->X) deliver(out->X, X, npred * 27);
    }
    o->oh_ml_valid = true;
  }
  CU(launch_oh_finalize(r, g.stream));
  if (want_diag) {
    CU(cudaMemsetAsync(r.diag, 0, 4 * sizeof(double), g.stream));
    CU(launch_oh_diag(r, g.stream));
    CU(cudaMemcpyAsync(out->diag, r.diag, 4 * sizeof(double), cudaMemcpyDeviceToHost, g.stream));
  }
  deliver(out->OH, r.OH, n3);
  deliver(out->OH_boost, r.OH_boost, n3);
  deliver(out->NDWET, r.NDWET, n3);
  deliver(out->LOSS_CH4, r.LOSS_CH4, n3);
  deliver(out->LOSS_CO, r.LOSS_CO, n3);
  int inf_flags = 0;
  if (check_inf_after) CU(cudaMemcpyAsync(&inf_flags, r.ctl + 2, sizeof(int), cudaMemcpyDeviceToHost, g.stream));
  CU(cudaStreamSynchronize(g.stream));
  if ((inf_flags & 2) && !std::isinf(c.missing)) {
    o->oh_ml_valid = false;
    throw Error("Check failed: valid: Input data contains `inf` or `nan`");
  }
  API_END
}

}  // extern "C"
