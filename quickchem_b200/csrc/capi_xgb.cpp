// capi_xgb.cpp — group (1) of include/qcoh.h: the eleven XGBoost-named symbols the reference's
// xgb_fortran_api.F90 binds, plus the device / booster / DMatrix utilities of the qcoh_* extension.
// Everything numerical is a kernel launch (kernels.cu); there is no CPU compute path.
#include "context.hpp"

#include <condition_variable>
#include <mutex>
#ifdef __linux__
#include <sched.h>
#endif
#if defined(__x86_64__)
#include <emmintrin.h>
#endif

using namespace qcoh;

namespace qcoh {
// n elements of device memory p as a 1-D linear texture
template <class T>
static cudaTextureObject_t linear_texture(T *p, size_t n) {
  cudaResourceDesc rd;
  memset(&rd, 0, sizeof rd);
  rd.resType = cudaResourceTypeLinear;
  rd.res.linear.devPtr = p;
  rd.res.linear.desc = cudaCreateChannelDesc<T>();
  rd.res.linear.sizeInBytes = n * sizeof(T);
  cudaTextureDesc td;
  memset(&td, 0, sizeof td);
  td.readMode = cudaReadModeElementType;
  cudaTextureObject_t t = 0;
  CU(cudaCreateTextureObject(&t, &rd, &td, nullptr));
  return t;
}

void upload(Booster *b) {
  if (b->uploaded) return;
  if (!b->loaded) throw Error("Booster has no model: call XGBoosterLoadModel first");
  ensure_device();
  const FlatForest &f = b->flat;
  const size_t nn = (size_t)f.num_nodes();
  {
    // device copy: an internal node's x word becomes -key(threshold) mod 2^32 (kernels.cu "Order-
    // preserving integer keys"); leaves keep the float bits of their value
    std::vector<uint32_t> dev_nodes(f.nodes_xy);
    for (size_t i = 0; i < nn; ++i) {
      if ((dev_nodes[2 * i + 1] & kMetaRelMask) == 0) continue;
      float thr;
      memcpy(&thr, &dev_nodes[2 * i], 4);
      if (std::isnan(thr)) throw Error("split threshold is NaN (node " + std::to_string(i) + ")");
      dev_nodes[2 * i] = neg_threshold_key(thr);  // key >= 0x007FFFFF (-inf), never 0
    }
    CU(cudaMemcpy(b->d_nodes.need(nn), dev_nodes.data(), nn * 8, cudaMemcpyHostToDevice));
    b->dev_nodes_host = std::move(dev_nodes);
  }
  CU(cudaMemcpy(b->d_off.need(f.tree_offset.size()), f.tree_offset.data(), f.tree_offset.size() * 4, cudaMemcpyHostToDevice));
  {
    // device form: max leaf depth | min leaf depth << 8 (a tree whose shallowest leaf is below the levels
    // held in constant memory needs no leaf handling there)
    std::vector<int32_t> dd(f.tree_depth.size());
    for (size_t i = 0; i < dd.size(); ++i) {
      if (f.tree_depth[i] > 255) throw Error("tree " + std::to_string(i) + " is deeper than 255 levels");
      dd[i] = f.tree_depth[i] | (std::min(f.tree_min_leaf_depth[i], 255) << 8);
    }
    CU(cudaMemcpy(b->d_depth.need(dd.size()), dd.data(), dd.size() * 4, cudaMemcpyHostToDevice));
  }
  CU(cudaMemcpy(b->d_orig.need(nn), f.orig_id.data(), nn * 4, cudaMemcpyHostToDevice));
  if (b->dev.tex) cudaDestroyTextureObject(b->dev.tex);
  if (b->dev.tex4) cudaDestroyTextureObject(b->dev.tex4);
  b->dev = DeviceForest();
  b->dev.nodes = b->d_nodes.p, b->dev.tree_offset = b->d_off.p, b->dev.tree_depth = b->d_depth.p, b->dev.orig_id = b->d_orig.p;
  b->dev.ntree = (int32_t)b->host.trees.size();
  b->dev.nfeat = (int32_t)b->host.num_feature;
  b->dev.base_score = b->host.base_score;
  if (nn > 0 && nn < ((size_t)1 << 27)) b->dev.tex = linear_texture(b->d_nodes.p, nn);
  // two-level records, when every tree qualifies
  if (b->duo.ok && b->duo.num_slots() > 0 && b->duo.num_slots() < ((int64_t)1 << 27)) {
    const size_t ns = (size_t)b->duo.num_slots();
    CU(cudaMemcpy(b->d_recs.need(ns), b->duo.rec.data(), ns * 16, cudaMemcpyHostToDevice));
    b->dev.tex4 = linear_texture(b->d_recs.p, ns);
    b->dev.recs = b->d_recs.p;
    b->dev.duo_has_dl = b->duo.has_default_bits ? 1 : 0;
    b->dev.duo_shallow = (int64_t)ns * 16 < kShallowRecBytesPerTree * std::max<int64_t>(1, b->dev.ntree) ? 1 : 0;
    b->dev.duo_blk_mul = 1u << (32 - b->duo.blk_shift);
  }
  b->uploaded = true;
}

// The constant-memory tables of tree tops exist once per device (one __constant__ bank per loaded module and
// device), and a device is driven by exactly one host thread (context.hpp), so what they hold is tracked per
// thread: one window of <= kConstTreesMax trees of one booster version, in one of two layouts — the first levels
// of the depth-ordered nodes (walk_group), or the complete heap-ordered tops of the two-level records
// (walk_group_duo) when the booster has records and a node texture and `duo` is not 0.
static thread_local struct {
  uint64_t owner = 0;  // Booster::version of the trees the window holds, 0 = none
  ConstWindow w;
} g_const;

ConstWindow hold(Booster *b, int tree0, int ntree) {
  if (ntree <= 0 || ntree > kConstTreesMax || tree0 + ntree > b->dev.ntree) return {};
  // The table holds a window of up to kConstTreesMax trees: the aligned window around the request when the request
  // fits in it (so that ranges of one forest and calls with different ntree_limit share an upload), else one that
  // starts at the request.
  int w0 = tree0 - tree0 % kConstTreesMax;
  if (tree0 + ntree > w0 + kConstTreesMax) w0 = tree0;
  const int n = std::min(b->dev.ntree - w0, kConstTreesMax);
  auto held = [&](TopLayout l) { return g_const.owner == b->version && g_const.w.holds(l, tree0, tree0 + ntree); };
  // stream-ordered re-fill; a failed upload leaves the table unowned and the launch runs without it
  auto fill = [&](TopLayout l) {
    g_const.owner = 0;
    const cudaError_t e = l == TopLayout::kRecordTops
                              ? upload_const_duo(b->duo.top_xy.data() + (size_t)w0 * (2u << kDuoTop), b->duo.tree_slot.data() + w0, n, g.stream)
                              : upload_const_top(b->dev_nodes_host.data(), b->flat.tree_offset.data() + w0, n, g.stream);
    if (e != cudaSuccess) {
      (void)cudaGetLastError();
      return false;
    }
    g_const.owner = b->version, g_const.w = ConstWindow{l, w0, n};
    return true;
  };
  const bool records = b->dev.recs != nullptr && b->dev.tex != 0 && g.duo != 0;
  if (records && (held(TopLayout::kRecordTops) || fill(TopLayout::kRecordTops))) return g_const.w;
  if (held(TopLayout::kNodeTops) || fill(TopLayout::kNodeTops)) return g_const.w;
  return {};
}

// One prediction = one launch per range of kRangeTrees trees (kernels.hpp; the tables hold kConstTreesMax and are
// re-filled, stream-ordered, when a range leaves them) and the float32 partial sum travels through `out`, so the sum
// order — tree 0, 1, 2, ... — and with it every bit of the result is the same as in a single launch.
// launch(window, range args) launches one range: launch_predict on key tiles, launch_predict_dense on a dense array.
template <class Launch>
static void predict_ranges(Booster *b, const PredictArgs &a, cudaStream_t s, Launch &&launch) {
  const int t_end = a.tree_end;
  if (a.nrow == 0) return;
  if (t_end <= 0) {  // a booster without trees predicts its base score
    if (!a.pred_leaf) {
      float v = b->host.base_score;
      if (a.exp10) v = (float)exp10((double)v) * a.scale;
      CU(launch_fill(a.out, a.nrow, v, s));
    }
    return;
  }
  for (int t0 = 0; t0 < t_end; t0 += kRangeTrees) {
    const int n = std::min(kRangeTrees, t_end - t0);
    const ConstWindow w = hold(b, t0, n);
    PredictArgs c = a;
    c.tree_begin = t0, c.tree_end = t0 + n;
    c.first = t0 == 0, c.last = t0 + n == t_end;
    CU(launch(w, c));
  }
}

void launch_predict_chunked(Booster *b, PredictArgs a, cudaStream_t s) {
  predict_ranges(b, a, s, [&](const ConstWindow &w, const PredictArgs &c) { return launch_predict(b->dev, w, c, s); });
}

static void seal(DMatrix *d) {
  ensure_device();
  int *fl = d->flags.need(1);
  CU(cudaMemsetAsync(fl, 0, sizeof(int), g.stream));
  if (g_spare_Xt.cap >= tile_words(d->nrow, d->ncol) && g_spare_Xt.p && !d->Xt.p) d->Xt.swap(g_spare_Xt);
  CU(launch_seal_tiles(d->X.p, d->nrow, (int)d->ncol, d->missing, d->Xt.need(tile_words(d->nrow, d->ncol)), fl, g.stream));
  CU(cudaMemcpyAsync(&d->hflags, fl, sizeof(int), cudaMemcpyDeviceToHost, g.stream));
  CU(cudaStreamSynchronize(g.stream));
  d->sealed = true;
  // xgboost src/data/data.cc SparsePage::Push: a finite `missing` with inf data is an error
  if (d->hflags & 2) throw Error("Check failed: valid: Input data contains `inf` or `nan`");
}

static unsigned trees_used(const Booster *b, unsigned ntree_limit) {
  const unsigned nt = (unsigned)b->host.trees.size();
  return (ntree_limit == 0 || ntree_limit > nt) ? nt : ntree_limit;
}

static void predict_into(Booster *b, DMatrix *d, int option_mask, unsigned ntree_limit, const qcoh_epilogue *epi, float *out_dev) {
  upload(b);
  if (!d->sealed) seal(d);
  if (option_mask & ~3) throw Error("option_mask " + std::to_string(option_mask) + ": only 0 (value), 1 (margin) and 2 (leaf index) are supported");
  if (d->ncol > b->host.num_feature)
    throw Error("Check failed: Number of columns does not match number of features in booster. Columns: " +
                std::to_string(d->ncol) + " Features: " + std::to_string(b->host.num_feature));
  PredictArgs a;
  a.Xt = d->Xt.p, a.nrow = d->nrow, a.ncol = (int32_t)d->ncol;
  a.has_missing = ((d->hflags & 1) || d->ncol < b->host.num_feature) ? 1 : 0;
  a.pred_leaf = (option_mask & 2) ? 1 : 0;
  a.tree_begin = 0, a.tree_end = (int32_t)trees_used(b, ntree_limit), a.out_stride = a.tree_end;
  a.exp10 = epi ? epi->exp10 : 0;
  a.scale = epi ? epi->scale : 1.f;
  a.out = out_dev;
  launch_predict_chunked(b, a, g.stream);
}

const ShapForest &shap_tables(Booster *b) {
  if (!b->loaded) throw Error("Booster has no model: call XGBoosterLoadModel first");
  if (!b->shap.ok) b->shap = build_shap(b->host, b->flat);
  return b->shap;
}

// The contribution tables of the booster in HBM, for a sealed matrix of at most num_feature columns.  The path bins
// and node means go to HBM at the first call (not at load: prediction alone never needs them).
static const ShapForest &shap_on_device(Booster *b, DMatrix *d) {
  const ShapForest &s = shap_tables(b);
  upload(b);
  if (!d->sealed) seal(d);
  const uint32_t nf = b->host.num_feature;
  if (d->ncol > nf)
    throw Error("Check failed: Number of columns does not match number of features in booster. Columns: " +
                std::to_string(d->ncol) + " Features: " + std::to_string(nf));
  if (!b->shap_uploaded) {
    const size_t nb = (size_t)s.num_bins(), nn = s.mean.size();
    CU(cudaMemcpy(b->d_shap_bins.need(nb * 32), s.bins.data(), nb * 32 * sizeof(uint4), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(b->d_shap_mean.need(nn), s.mean.data(), nn * sizeof(float), cudaMemcpyHostToDevice));
    b->shap_uploaded = true;
  }
  return s;
}

// Per-feature contributions into a device buffer [nrow][num_feature + 1], asynchronous on the library stream.
static void contribs_into(Booster *b, DMatrix *d, bool approximate, unsigned ntree_limit, float *out_dev) {
  const ShapForest &s = shap_on_device(b, d);
  const uint32_t nf = b->host.num_feature;
  const int nt = (int)trees_used(b, ntree_limit);
  ContribArgs a;
  a.ncol = (int32_t)d->ncol, a.nfeat = (int32_t)nf;
  a.bias = shap_bias(s, b->host, b->flat, nt);
  if (approximate) {
    a.Xt = d->Xt.p, a.nrow = d->nrow, a.out = out_dev;
    CU(launch_shap_approx(b->dev, b->d_shap_mean.p, nt, a, g.stream));
    return;
  }
  const int64_t nb = s.tree_bin[(size_t)nt];
  const int ns = (int)std::min<int64_t>(kShapSlices, nb);
  double *part = b->d_shap_part.need((size_t)ns * (size_t)std::min<uint64_t>(kShapChunkRows, d->nrow) * nf);
  for (uint64_t r0 = 0; r0 < d->nrow; r0 += kShapChunkRows) {
    ContribArgs c = a;
    c.Xt = d->Xt.p + tile_offset_words(r0, d->ncol), c.nrow = std::min<uint64_t>(kShapChunkRows, d->nrow - r0);
    c.out = out_dev + r0 * (nf + 1);
    CU(launch_shap(b->d_shap_bins.p, nb, ns, c, part, g.stream));
    CU(launch_shap_reduce(part, ns, c, g.stream));
  }
}

// SHAP interaction values into a device buffer [nrow][num_feature + 1][num_feature + 1], asynchronous on the library
// stream.  Exact: per chunk of kInterChunkRows rows, the contribution slices (phi) and the conditioned paths of every
// feature, reduced together.  The per-feature bin lists are built and go to HBM at the first interactions call.
static void interactions_into(Booster *b, DMatrix *d, bool approximate, unsigned ntree_limit, float *out_dev) {
  const ShapForest &s = shap_on_device(b, d);
  const uint32_t nf = b->host.num_feature;
  if (d->nrow && !out_dev) throw Error("qcoh_booster_predict_interactions_device: NULL output buffer");
  const int nt = (int)trees_used(b, ntree_limit);
  ContribArgs a;
  a.ncol = (int32_t)d->ncol, a.nfeat = (int32_t)nf;
  a.bias = shap_bias(s, b->host, b->flat, nt);
  if (approximate) {
    float *phi = b->d_inter_phi.need((size_t)d->nrow * (nf + 1));
    a.Xt = d->Xt.p, a.nrow = d->nrow, a.out = phi;
    CU(launch_shap_approx(b->dev, b->d_shap_mean.p, nt, a, g.stream));
    a.out = out_dev;
    CU(launch_shap_inter_expand(phi, a, g.stream));
    return;
  }
  if (!b->inter_uploaded) {
    if (s.feat_off.empty()) build_shap_by_feature(b->shap, nf);
    CU(cudaMemcpy(b->d_inter_off.need(s.feat_off.size()), s.feat_off.data(), s.feat_off.size() * sizeof(int64_t),
                  cudaMemcpyHostToDevice));
    CU(cudaMemcpy(b->d_inter_bins.need(s.feat_bins.size()), s.feat_bins.data(), s.feat_bins.size() * sizeof(uint32_t),
                  cudaMemcpyHostToDevice));
    b->inter_uploaded = true;
  }
  const int64_t nb = s.tree_bin[(size_t)nt];
  const int ns = (int)std::min<int64_t>(kShapSlices, nb);
  const size_t rows = (size_t)std::min<uint64_t>(kInterChunkRows, d->nrow), nc = (size_t)nf + 1;
  double *shap_part = b->d_shap_part.need((size_t)ns * rows * nf);
  double *part = b->d_inter_part.need((size_t)nf * kInterSlices * rows * nf);
  for (uint64_t r0 = 0; r0 < d->nrow; r0 += kInterChunkRows) {
    ContribArgs c = a;
    c.Xt = d->Xt.p + tile_offset_words(r0, d->ncol), c.nrow = std::min<uint64_t>(kInterChunkRows, d->nrow - r0);
    c.out = out_dev + r0 * nc * nc;
    CU(launch_shap(b->d_shap_bins.p, nb, ns, c, shap_part, g.stream));
    CU(launch_shap_inter(b->d_shap_bins.p, b->d_inter_off.p, b->d_inter_bins.p, nb, c, part, g.stream));
    CU(launch_shap_inter_reduce(part, shap_part, ns, c, g.stream));
  }
}

static cudaEvent_t chunk_event(size_t i) {
  while (g.chunk_events.size() <= i) {
    cudaEvent_t e;
    CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    g.chunk_events.push_back(e);
  }
  return g.chunk_events[i];
}

static void drain() {
  cudaStreamSynchronize(g.copy_stream);
  cudaStreamSynchronize(g.stream);
  cudaStreamSynchronize(g.d2h_stream);
}

static bool is_pinned_host(const void *p) {
  cudaPointerAttributes a;
  cudaError_t e = cudaPointerGetAttributes(&a, p);
  if (e != cudaSuccess) {
    (void)cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeHost;
}

// Multi-threaded copy (pageable host -> pinned staging) on a persistent pool: a Fortran ALLOCATE gives pageable
// memory (xx_carr, OH_GridCompMod.F90:306), and one core's memcpy (~10 GB/s) is far below PCIe 5 x16.  The
// workers are created once and parked on a condition variable; the calling thread does not copy — it issues the
// CUDA work of the previous chunk while the workers stage the next one.  Threads: the cores this process may use
// divided by the ranks sharing the node.
// Copy into the pinned staging ring with non-temporal stores: a plain memcpy reads every destination line before
// overwriting it (read-for-ownership), i.e. 3 transfers per byte where the staging copy needs 2, and the staging
// data is only ever read back by the DMA engine.  QCOH_COPY_NT=0 selects memcpy.
static void stream_copy(char *dst, const char *src, size_t n) {
  size_t i = 0;
#if defined(__x86_64__)
  static const bool nt = [] {
    const char *e = getenv("QCOH_COPY_NT");
    return !e || atoi(e) != 0;
  }();
  if (nt && (((uintptr_t)dst) & 15u) == 0u) {
    for (; i + 64 <= n; i += 64) {
      const __m128i a = _mm_loadu_si128((const __m128i *)(src + i)), b = _mm_loadu_si128((const __m128i *)(src + i + 16));
      const __m128i c = _mm_loadu_si128((const __m128i *)(src + i + 32)), d = _mm_loadu_si128((const __m128i *)(src + i + 48));
      _mm_stream_si128((__m128i *)(dst + i), a);
      _mm_stream_si128((__m128i *)(dst + i + 16), b);
      _mm_stream_si128((__m128i *)(dst + i + 32), c);
      _mm_stream_si128((__m128i *)(dst + i + 48), d);
    }
    _mm_sfence();
  }
#endif
  if (i < n) memcpy(dst + i, src + i, n - i);
}

class CopyPool {
 public:
  static CopyPool &get() {
    static CopyPool p;
    return p;
  }
  // start copying on the workers and return; wait() blocks until that copy is complete.  One copy at a time per
  // process (threads driving different GPUs take turns: begin() holds the pool until wait()).
  void begin(void *dst, const void *src, size_t bytes) {
    callers_.lock();
    if (workers_.empty() || bytes < ((size_t)4 << 20)) {
      stream_copy((char *)dst, (const char *)src, bytes);
      inline_done_ = true;
      return;
    }
    inline_done_ = false;
    const unsigned nt = (unsigned)workers_.size();
    {
      std::lock_guard<std::mutex> lk(m_);
      dst_ = (char *)dst, src_ = (const char *)src, bytes_ = bytes, per_ = (bytes / nt + 4095) / 4096 * 4096;
      pending_ = nt;
      ++generation_;
    }
    cv_.notify_all();
  }
  void wait() {
    if (!inline_done_) {
      std::unique_lock<std::mutex> lk(m_);
      done_.wait(lk, [&] { return pending_ == 0; });
    }
    callers_.unlock();
  }
  unsigned threads() const { return (unsigned)workers_.size(); }

 private:
  CopyPool() {
    unsigned cores = std::thread::hardware_concurrency();
#ifdef __linux__
    cpu_set_t set;
    if (sched_getaffinity(0, sizeof set, &set) == 0) cores = (unsigned)CPU_COUNT(&set);
#endif
    if (cores == 0) cores = 1;
    unsigned share = 1;
    if (const char *lw = getenv("LOCAL_WORLD_SIZE")) share = (unsigned)std::max(1, atoi(lw));
    unsigned nt = std::max(1u, std::min(32u, cores / share));
    if (const char *e = getenv("QCOH_COPY_THREADS")) nt = (unsigned)std::max(1, atoi(e));
    for (unsigned t = 0; t < nt; ++t) workers_.emplace_back([this, t] { run(t); });
  }
  ~CopyPool() {
    {
      std::lock_guard<std::mutex> lk(m_);
      stop_ = true;
    }
    cv_.notify_all();
    for (auto &w : workers_) w.join();
  }
  void part(unsigned t) {
    const size_t o = (size_t)t * per_;
    if (o < bytes_) stream_copy(dst_ + o, src_ + o, std::min(per_, bytes_ - o));
  }
  void run(unsigned t) {
    uint64_t seen = 0;
    for (;;) {
      {
        std::unique_lock<std::mutex> lk(m_);
        cv_.wait(lk, [&] { return stop_ || generation_ != seen; });
        if (stop_) return;
        seen = generation_;
      }
      part(t);
      std::lock_guard<std::mutex> lk(m_);
      if (--pending_ == 0) done_.notify_one();
    }
  }
  std::vector<std::thread> workers_;
  std::mutex m_, callers_;
  std::condition_variable cv_, done_;
  char *dst_ = nullptr;
  const char *src_ = nullptr;
  size_t bytes_ = 0, per_ = 0;
  unsigned pending_ = 0;
  uint64_t generation_ = 0;
  bool stop_ = false, inline_done_ = false;
};
constexpr int kStageSlots = 3;
static thread_local PinBuf<float> g_stage[kStageSlots];
static thread_local cudaEvent_t g_stage_free[kStageSlots] = {nullptr, nullptr, nullptr};

// XGDMatrixCreateFromMat from HOST memory, pipelined: the matrix is cut into row chunks; while chunk
// c+1 crosses PCIe, chunk c is scanned (missing / inf) and — since the reference keeps exactly one
// booster per process and always predicts with option_mask = 0, ntree_limit = 0 right after creating
// the matrix (OH_GridCompMod.F90:347-356) — already predicted with that booster, and its results
// stream back into a pinned buffer.  XGBoosterPredict then finds the answer ready if it is called
// with that booster and those options; any other call takes the ordinary path.  Pageable host
// memory (what a Fortran ALLOCATE gives) is staged through a ring of pinned buffers by a threaded
// memcpy so that the DMA engine never waits on the driver's own bounce buffer.  The caller's buffer
// is fully consumed before this returns.
//   copy_stream : H2D(c) -> seal(c): scan + key tiles -> flag D2H(c)      g.stream : predict(c)      d2h_stream : result D2H(c)
static uint64_t chunk_rows(bool pinned) { return pinned ? g.chunk_rows : std::min<uint64_t>(g.chunk_rows, 1ull << 19); }

// The chunked copy of a row-major host matrix into HBM, shared by XGDMatrixCreateFromMat and XGBoosterPredictFromDense:
// rows [0, nrow) of `data` go to X in chunks of cr rows (a multiple of 256) on g.copy_stream.  Pinned memory goes by
// direct DMA, every copy queued up front; pageable memory is staged through the ring of pinned slots by the copy pool,
// which stages chunk c + 1 while this thread queues the CUDA work of chunk c.  landed(c, r0, nr) queues, after H2D(c),
// the work that reads chunk c; process(c) is the host side of chunk c, called in chunk order (two chunks behind on
// pageable memory).  Returns when every chunk has been copied: the caller's buffer may go.
template <class Landed, class Process>
static void copy_chunks(const float *data, uint64_t nrow, uint64_t ncol, bool pinned, uint64_t cr, float *X, Landed &&landed,
                        Process &&process) {
  const size_t nchunk = (size_t)((nrow + cr - 1) / cr);
  if (!pinned)
    for (int s = 0; s < kStageSlots; ++s)
      if (!g_stage_free[s]) CU(cudaEventCreateWithFlags(&g_stage_free[s], cudaEventDisableTiming));
  // pageable source: stage_begin(c) starts the workers on chunk c (into ring slot c % 3, once its previous H2D has
  // drained), stage_end() waits for them; issue(c) queues H2D(c) and what reads chunk c
  auto stage_begin = [&](size_t c) {
    const uint64_t r0 = c * cr, nr = std::min(cr, nrow - r0);
    const int s = (int)(c % kStageSlots);
    float *st = g_stage[s].need(cr * ncol);
    if (c >= (size_t)kStageSlots) CU(cudaEventSynchronize(g_stage_free[s]));
    CopyPool::get().begin(st, data + r0 * ncol, nr * ncol * sizeof(float));
  };
  auto issue = [&](size_t c) {
    const uint64_t r0 = c * cr, nr = std::min(cr, nrow - r0);
    const size_t bytes = nr * ncol * sizeof(float);
    if (!pinned) {
      const int s = (int)(c % kStageSlots);
      CU(cudaMemcpyAsync(X + r0 * ncol, g_stage[s].p, bytes, cudaMemcpyHostToDevice, g.copy_stream));
      CU(cudaEventRecord(g_stage_free[s], g.copy_stream));
    } else {
      CU(cudaMemcpyAsync(X + r0 * ncol, data + r0 * ncol, bytes, cudaMemcpyHostToDevice, g.copy_stream));
    }
    landed(c, r0, nr);
  };
  if (pinned) {  // every copy can be queued up front
    for (size_t c = 0; c < nchunk; ++c) issue(c);
    for (size_t c = 0; c < nchunk; ++c) process(c);
  } else {  // the workers stage chunk c + 1 while this thread queues the CUDA work of chunk c and processes chunk c - 2
    struct PoolGuard {  // an exception between begin() and wait() must not leave the pool locked
      bool busy = false;
      ~PoolGuard() {
        if (busy) CopyPool::get().wait();
      }
    } pool;
    if (nchunk) stage_begin(0), pool.busy = true;
    for (size_t c = 0; c < nchunk; ++c) {
      CopyPool::get().wait(), pool.busy = false;
      if (c + 1 < nchunk) stage_begin(c + 1), pool.busy = true;
      issue(c);
      if (c >= 2) process(c - 2);
    }
    for (size_t c = nchunk >= 2 ? nchunk - 2 : 0; c < nchunk; ++c) process(c);
  }
  CU(cudaStreamSynchronize(g.copy_stream));  // the borrowed host buffer has been read completely
}

static void create_pipelined(DMatrix *d, const float *data, Booster *b) {
  const uint64_t nrow = d->nrow, ncol = d->ncol;
  const bool pinned = is_pinned_host(data);
  const uint64_t cr = chunk_rows(pinned);
  const size_t nchunk = (size_t)((nrow + cr - 1) / cr);
  float *X = d->X.p;
  if (g_spare_Xt.cap >= tile_words(nrow, ncol) && g_spare_Xt.p && !d->Xt.p) d->Xt.swap(g_spare_Xt);
  uint32_t *Xt = d->Xt.need(tile_words(nrow, ncol));
  const bool spec = b != nullptr;
  float *sdev = nullptr, *shost = nullptr;
  if (spec) {
    upload(b);
    if (g_spare_spec.cap >= nrow && g_spare_spec.p) d->spec_dev.swap(g_spare_spec);
    sdev = d->spec_dev.need(nrow);
    if (g_spare_pin.cap >= nrow && g_spare_pin.p) d->spec_host.swap(g_spare_pin);
    shost = d->spec_host.need(nrow);
  }
  int *fl = g_chunk_flags.need(nchunk);
  int *hfl = g_h_chunk_flags.need(nchunk);
  CU(cudaMemsetAsync(fl, 0, nchunk * sizeof(int), g.copy_stream));
  int flags = 0;
  // H2D(c) -> seal(c): scan + key tiles -> flag D2H(c) on the copy stream
  auto landed = [&](size_t c, uint64_t r0, uint64_t nr) {
    // chunks start on tile boundaries (chunk_rows is a multiple of 256)
    CU(launch_seal_tiles(X + r0 * ncol, nr, (int)ncol, d->missing, Xt + tile_offset_words(r0, ncol), fl + c, g.copy_stream));
    CU(cudaMemcpyAsync(hfl + c, fl + c, sizeof(int), cudaMemcpyDeviceToHost, g.copy_stream));
    CU(cudaEventRecord(chunk_event(2 * c), g.copy_stream));
  };
  auto process = [&](size_t c) {
    const uint64_t r0 = c * cr, nr = std::min(cr, nrow - r0);
    CU(cudaEventSynchronize(chunk_event(2 * c)));
    flags |= hfl[c];
    if (hfl[c] & 2) {
      drain();
      throw Error("Check failed: valid: Input data contains `inf` or `nan`");
    }
    if (!spec) return;
    PredictArgs a;
    a.Xt = Xt + tile_offset_words(r0, ncol), a.nrow = nr, a.ncol = (int32_t)ncol;
    a.has_missing = ((hfl[c] & 1) || ncol < b->host.num_feature) ? 1 : 0;
    a.tree_begin = 0, a.tree_end = (int32_t)b->host.trees.size(), a.out_stride = a.tree_end;
    a.out = sdev + r0;
    launch_predict_chunked(b, a, g.stream);
    CU(cudaEventRecord(chunk_event(2 * c + 1), g.stream));
    CU(cudaStreamWaitEvent(g.d2h_stream, chunk_event(2 * c + 1), 0));
    CU(cudaMemcpyAsync(shost + r0, sdev + r0, nr * sizeof(float), cudaMemcpyDeviceToHost, g.d2h_stream));
  };
  copy_chunks(data, nrow, ncol, pinned, cr, X, landed, process);
  d->hflags = flags;
  d->sealed = true;
  if (spec) d->spec_booster = b, d->spec_version = b->version, d->spec_ready = true;
}

static thread_local cudaEvent_t g_input_ready = nullptr;

// XGBoosterPredictFromDense / XGBoosterPredictFromCudaArray (libxgboost 1.6.0 Learner::InplacePredict, value and
// margin): predict_dense_kernel builds the key tiles from the caller's array in shared memory.  A device array is read
// where it is, with its strides; a host array is copied chunk by chunk (copy_chunks) and each chunk predicted as it
// lands.  Returns the float32 margins, in the booster's device buffer (on_device) or its pinned host buffer; both stay
// valid until the next predict or free on that booster.  Every refusal comes before any device work.
static const float *predict_inplace(const char *caller, bool cuda_array, BoosterHandle handle, const char *values,
                                    const char *config, DMatrixHandle m, const bst_ulong **out_shape, bst_ulong *out_dim) {
  const std::string pre = std::string(caller) + ": ";
  Booster *b = B(handle);
  if (!out_shape || !out_dim) throw Error(pre + "NULL output argument");
  if (!b->loaded) throw Error("Booster has no model: call XGBoosterLoadModel first");
  const ArrayInterface ai = parse_array_interface(values, caller);
  const PredictConfig c = parse_predict_config(config, caller, true);
  if (m) throw Error(pre + "the proxy DMatrix must be NULL (inplace prediction takes no base margin)");
  if (c.type != 0 && c.type != 1)
    throw Error(pre + "prediction type " + std::to_string(c.type) + " is not supported inplace (0 value, 1 margin)");
  if (c.iteration_begin < 0 || c.iteration_end < 0) throw Error(pre + "negative iteration range");
  if (c.iteration_begin != 0) throw Error(pre + "iteration_begin = " + std::to_string(c.iteration_begin) + " is not supported (only 0)");
  if (ai.ncol > b->host.num_feature)
    throw Error("Check failed: Number of columns does not match number of features in booster. Columns: " +
                std::to_string(ai.ncol) + " Features: " + std::to_string(b->host.num_feature));
  if (ai.ncol > kMaxMatrixCols)
    throw Error(pre + std::to_string(ai.ncol) + " columns; libqcoh's tile form holds at most " + std::to_string(kMaxMatrixCols));
  const uint64_t nrow = ai.nrow, ncol = ai.ncol;
  const bool empty = nrow * ncol == 0;
  // the pointer query binds the CUDA runtime to this thread's device first; with no device visible every address is host memory
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) == cudaSuccess && ndev > 0) ensure_device();
  else (void)cudaGetLastError();
  const float *data = reinterpret_cast<const float *>((uintptr_t)ai.addr);
  const bool on_device = !empty && is_device_ptr(data);
  if (cuda_array && !empty && !on_device) throw Error(pre + "the array is in host memory (XGBoosterPredictFromDense takes host arrays)");
  if (!empty && !on_device && (ai.col_bytes != 4 || ai.row_bytes != (int64_t)(4 * ncol)))
    throw Error(pre + "a host array must be C-contiguous: strides [" + std::to_string(4 * ncol) + ", 4] or null, got [" +
                std::to_string(ai.row_bytes) + ", " + std::to_string(ai.col_bytes) + "]");
  ensure_device();
  upload(b);
  const unsigned limit = (unsigned)std::min<int64_t>(c.iteration_end, (int64_t)UINT32_MAX);
  float *dv = b->d_result.need(nrow);
  int *fl = g_chunk_flags.need(1);
  int *hfl = g_h_chunk_flags.need(1);
  CU(cudaMemsetAsync(fl, 0, sizeof(int), g.stream));
  PredictArgs a;
  a.nrow = nrow, a.ncol = (int32_t)ncol;
  a.tree_begin = 0, a.tree_end = (int32_t)trees_used(b, limit);
  a.out = dv;
  DenseArgs da;
  da.missing = c.missing, da.flags = fl;
  auto predict = [&](const PredictArgs &pa, const DenseArgs &d) {
    predict_ranges(b, pa, g.stream, [&](const ConstWindow &w, const PredictArgs &r) { return launch_predict_dense(b->dev, w, r, d, g.stream); });
  };
  if (on_device || empty) {
    if (ai.has_stream) {  // the work queued on the caller's stream before this call has written the array
      const cudaStream_t cs = ai.stream == 1 ? cudaStreamLegacy : ai.stream == 2 ? cudaStreamPerThread : (cudaStream_t)(uintptr_t)ai.stream;
      if (!g_input_ready) CU(cudaEventCreateWithFlags(&g_input_ready, cudaEventDisableTiming));
      CU(cudaEventRecord(g_input_ready, cs));
      CU(cudaStreamWaitEvent(g.stream, g_input_ready, 0));
    }
    da.X = data, da.row_stride = ai.row_bytes / 4, da.col_stride = ai.col_bytes / 4;
    predict(a, da);
  } else {
    // the chunks land in the spare matrix buffer of XGDMatrixFree, which is given back afterwards
    DevBuf<float> X;
    if (g_spare_X.cap >= nrow * ncol) X.swap(g_spare_X);
    X.need(nrow * ncol);
    const bool pinned = is_pinned_host(data);
    copy_chunks(data, nrow, ncol, pinned, chunk_rows(pinned), X.p, [&](size_t ci, uint64_t r0, uint64_t nr) {
      CU(cudaEventRecord(chunk_event(ci), g.copy_stream));
      CU(cudaStreamWaitEvent(g.stream, chunk_event(ci), 0));
      PredictArgs pa = a;
      pa.nrow = nr, pa.out = dv + r0;
      DenseArgs d = da;
      d.X = X.p + r0 * ncol, d.row_stride = (int64_t)ncol, d.col_stride = 1;
      predict(pa, d);
    }, [](size_t) {});
    CU(cudaStreamSynchronize(g.stream));  // the chunk buffer is read before it goes back to the pool
    if (X.cap > g_spare_X.cap) X.swap(g_spare_X);
  }
  CU(cudaMemcpyAsync(hfl, fl, sizeof(int), cudaMemcpyDeviceToHost, g.stream));
  float *out = dv;
  if (!cuda_array) {
    out = b->h_result.need(nrow);
    CU(cudaMemcpyAsync(out, dv, nrow * sizeof(float), cudaMemcpyDeviceToHost, g.stream));
  }
  CU(cudaStreamSynchronize(g.stream));
  // xgboost src/data/data.cc SparsePage::Push: a finite `missing` with inf data is an error (the kernel's flag)
  if (*hfl & 2) throw Error("Check failed: valid: Input data contains `inf` or `nan`");
  b->h_shape = c.strict_shape ? std::vector<bst_ulong>{nrow, 1} : std::vector<bst_ulong>{nrow};
  *out_shape = b->h_shape.data();
  *out_dim = (bst_ulong)b->h_shape.size();
  return out;
}

}  // namespace qcoh

// =====================================================================================
// (1) xgb_fortran_api boundary
// =====================================================================================
extern "C" {

const char *XGBGetLastError(void) { return g_err.c_str(); }
__attribute__((visibility("hidden"))) void qcoh_internal_set_error(const char *msg) { g_err = msg ? msg : ""; }

int XGBoosterCreate(const DMatrixHandle dmats[], bst_ulong len, BoosterHandle *out) {
  API_BEGIN
  // The reference passes a DMatrix handle by value here with len = 0 (OH_GridCompMod.F90:255-256):
  // dmats must not be dereferenced.  Cached matrices are a training concept; ignored for len > 0.
  (void)dmats, (void)len;
  if (!out) throw Error("XGBoosterCreate: out is NULL");
  Booster *b = new Booster();
  g_live_handles.insert(b);
  *out = b;
  API_END
}

int XGBoosterFree(BoosterHandle handle) {
  API_BEGIN
  Booster *b = B(handle);
  if (b->cache_owned) throw Error("XGBoosterFree: this booster belongs to the model cache (qcoh_model_cache_clear frees it)");
  if (b->oh_refs > 0)
    throw Error("XGBoosterFree: " + std::to_string(b->oh_refs) + " fused-Run1 handle(s) still predict with this booster (qcoh_oh_free / qcoh_oh_set_booster first)");
  if (g_last_booster == b) g_last_booster = nullptr;
  if (g.ready) drain();
  b->magic = 0;
  g_live_handles.erase(b);
  delete b;
  API_END
}

int qcoh_booster_parse(BoosterHandle handle, const char *fname) {
  API_BEGIN
  Booster *b = B(handle);
  if (!fname) throw Error("model file name is NULL");
  if (b->cache_owned) throw Error("this booster belongs to the model cache and cannot be reloaded");
  // a reload replaces the device forest in place: nothing may still be reading it
  if (b->uploaded && g.ready) CU(cudaStreamSynchronize(g.stream));
  HostForest hf = load_model_file(fname);
  FlatForest ff = flatten(hf);
  DuoForest df = build_duo(ff, hf.num_feature);
  b->host = std::move(hf), b->flat = std::move(ff), b->duo = std::move(df);
  b->shap = ShapForest(), b->shap_uploaded = false, b->inter_uploaded = false;
  b->loaded = true, b->uploaded = false;
  b->version = ++g_version_counter;
  API_END
}

int XGBoosterLoadModel(BoosterHandle handle, const char *fname) {
  if (qcoh_booster_parse(handle, fname) != 0) return -1;
  API_BEGIN
  upload(B(handle));
  g_last_booster = B(handle);
  API_END
}

int XGBoosterSaveModel(BoosterHandle handle, const char *fname) {
  API_BEGIN
  Booster *b = B(handle);
  if (!b->loaded) throw Error("Booster has no model to save");
  save_model_file(b->host, fname);
  API_END
}

int XGDMatrixCreateFromMat(const float *data, bst_ulong nrow, bst_ulong ncol, float missing, DMatrixHandle *out) {
  API_BEGIN
  if (!out) throw Error("XGDMatrixCreateFromMat: out is NULL");
  if (!data && nrow && ncol) throw Error("XGDMatrixCreateFromMat: data is NULL");
  if (ncol > kMaxMatrixCols) throw Error("XGDMatrixCreateFromMat: " + std::to_string(ncol) + " columns; libqcoh's tile form holds at most " + std::to_string(kMaxMatrixCols));
  ensure_device();
  std::unique_ptr<DMatrix> d(new DMatrix());
  d->nrow = nrow, d->ncol = ncol, d->missing = missing;
  const size_t n = (size_t)nrow * ncol;
  if (g_spare_X.cap >= n && g_spare_X.p) d->X.swap(g_spare_X);
  d->X.need(n);
  // borrowed for this call only (the reference deallocates xx_carr right after predict,
  // OH_GridCompMod.F90:383): the data is in HBM when this returns.
  if (n && !is_device_ptr(data)) {
    Booster *b = g.speculate ? g_last_booster : nullptr;
    if (b && !(b->loaded && ncol <= b->host.num_feature)) b = nullptr;
    create_pipelined(d.get(), data, b);
  } else {
    if (n) {
      CU(cudaMemcpyAsync(d->X.p, data, n * sizeof(float), cudaMemcpyDeviceToDevice, g.stream));
      CU(cudaStreamSynchronize(g.stream));
    }
    seal(d.get());
  }
  g_live_handles.insert(d.get());
  *out = d.release();
  API_END
}

int XGDMatrixFree(DMatrixHandle handle) {
  API_BEGIN
  DMatrix *d = D(handle);
  // The freed buffers are pooled, not cudaFree'd (which would have synchronised): nothing may still be reading
  // them — neither the pipelined create nor an asynchronous qcoh_booster_predict_device on the compute stream.
  if (g.ready) drain();
  d->magic = 0;
  if (d->X.cap > g_spare_X.cap) d->X.swap(g_spare_X);
  if (d->Xt.cap > g_spare_Xt.cap) d->Xt.swap(g_spare_Xt);
  if (d->spec_host.cap > g_spare_pin.cap) d->spec_host.swap(g_spare_pin);
  if (d->spec_dev.cap > g_spare_spec.cap) d->spec_dev.swap(g_spare_spec);
  g_live_handles.erase(d);
  delete d;
  API_END
}

int XGDMatrixNumRow(DMatrixHandle handle, bst_ulong *out) {
  API_BEGIN
  *out = D(handle)->nrow;
  API_END
}

int XGDMatrixNumCol(DMatrixHandle handle, bst_ulong *out) {
  API_BEGIN
  *out = D(handle)->ncol;
  API_END
}

int XGBoosterPredict(BoosterHandle handle, DMatrixHandle dmat, int option_mask, unsigned ntree_limit, int training,
                     bst_ulong *out_len, const float **out_result) {
  API_BEGIN
  (void)training;  // inference only; the reference passes 0 (OH_GridCompMod.F90:235)
  Booster *b = B(handle);
  DMatrix *d = D(dmat);
  if (!out_len || !out_result) throw Error("XGBoosterPredict: NULL output argument");
  if (!b->loaded) throw Error("Booster has no model: call XGBoosterLoadModel first");
  const size_t n = (size_t)d->nrow * ((option_mask & 2) ? trees_used(b, ntree_limit) : 1);
  ensure_device();
  g_last_booster = b;
  if (d->spec_ready && d->spec_booster == b && d->spec_version == b->version && (option_mask & ~1) == 0 &&
      trees_used(b, ntree_limit) == b->host.trees.size()) {
    // already predicted while the matrix was crossing PCIe: adopt the pinned result buffer
    CU(cudaStreamSynchronize(g.d2h_stream));
    b->h_result.swap(d->spec_host);
    d->spec_ready = false;
    *out_len = n;
    *out_result = b->h_result.p;
    return 0;
  }
  float *dv = b->d_result.need(n);
  float *hv = b->h_result.need(n);
  predict_into(b, d, option_mask, ntree_limit, nullptr, dv);
  CU(cudaMemcpyAsync(hv, dv, n * sizeof(float), cudaMemcpyDeviceToHost, g.stream));
  CU(cudaStreamSynchronize(g.stream));
  *out_len = n;
  *out_result = hv;
  API_END
}

// libxgboost 1.6.0's JSON-configured predict (src/c_api/c_api.cc).  Types 0 / 1 / 6 run the kernels of
// XGBoosterPredict (option_mask 0 / 1 / 2); 2 and 3 are the per-feature contributions.
int XGBoosterPredictFromDMatrix(BoosterHandle handle, DMatrixHandle dmat, const char *config, const bst_ulong **out_shape,
                                bst_ulong *out_dim, const float **out_result) {
  API_BEGIN
  Booster *b = B(handle);
  if (!out_shape || !out_dim || !out_result) throw Error("XGBoosterPredictFromDMatrix: NULL output argument");
  if (!b->loaded) throw Error("Booster has no model: call XGBoosterLoadModel first");
  const PredictConfig c = parse_predict_config(config);
  const std::string ty = std::to_string(c.type);
  if (c.type == 4 || c.type == 5)
    throw Error("XGBoosterPredictFromDMatrix: type " + ty + " (SHAP interaction values) is not supported; 2 and 3 give per-feature contributions, and "
                "qcoh_booster_predict_interactions_device computes interaction values");
  const bool contribs = c.type == 2 || c.type == 3;
  if (!contribs && c.type != 0 && c.type != 1 && c.type != 6)
    throw Error("XGBoosterPredictFromDMatrix: unknown prediction type " + ty + " (0 value, 1 margin, 2 / 3 contributions, 6 leaf)");
  if (c.iteration_begin < 0 || c.iteration_end < 0) throw Error("XGBoosterPredictFromDMatrix: negative iteration range");
  if (contribs && c.iteration_begin != 0)
    throw Error("XGBoosterPredictFromDMatrix: contributions support only iteration_begin = 0 (predict from iteration 0 to "
                "iteration_end; slice the model instead)");
  if (c.iteration_begin != 0)
    throw Error("XGBoosterPredictFromDMatrix: iteration_begin = " + std::to_string(c.iteration_begin) + " is not supported (only 0)");
  if (contribs) (void)shap_tables(b);  // a booster without covers fails here, before any device work
  ensure_device();
  DMatrix *d = D(dmat);
  const unsigned limit = (unsigned)std::min<int64_t>(c.iteration_end, (int64_t)UINT32_MAX);
  const bst_ulong nrow = d->nrow, nt = trees_used(b, limit), nf = b->host.num_feature;
  std::vector<bst_ulong> shape;
  size_t n;
  if (contribs) {
    n = (size_t)nrow * (nf + 1);
    shape = c.strict_shape ? std::vector<bst_ulong>{nrow, 1, nf + 1} : std::vector<bst_ulong>{nrow, nf + 1};
  } else if (c.type == 6) {
    n = (size_t)nrow * nt;
    shape = c.strict_shape ? std::vector<bst_ulong>{nrow, nt, 1, 1} : std::vector<bst_ulong>{nrow, nt};
  } else {
    n = (size_t)nrow;
    shape = c.strict_shape ? std::vector<bst_ulong>{nrow, 1} : std::vector<bst_ulong>{nrow};
  }
  g_last_booster = b;
  float *dv = b->d_result.need(n);
  float *hv = b->h_result.need(n);
  if (contribs)
    contribs_into(b, d, c.type == 3, limit, dv);
  else
    predict_into(b, d, c.type == 6 ? 2 : c.type, limit, nullptr, dv);
  CU(cudaMemcpyAsync(hv, dv, n * sizeof(float), cudaMemcpyDeviceToHost, g.stream));
  CU(cudaStreamSynchronize(g.stream));
  b->h_shape = std::move(shape);
  *out_shape = b->h_shape.data();
  *out_dim = (bst_ulong)b->h_shape.size();
  *out_result = hv;
  API_END
}

// libxgboost 1.6.0's inplace predicts (src/c_api/c_api.cc), what xgboost's Python Booster.inplace_predict calls
int XGBoosterPredictFromDense(BoosterHandle handle, const char *values, const char *config, DMatrixHandle m,
                              const bst_ulong **out_shape, bst_ulong *out_dim, const float **out_result) {
  API_BEGIN
  if (!out_result) throw Error("XGBoosterPredictFromDense: NULL output argument");
  *out_result = predict_inplace("XGBoosterPredictFromDense", false, handle, values, config, m, out_shape, out_dim);
  API_END
}

int XGBoosterPredictFromCudaArray(BoosterHandle handle, const char *values, const char *config, DMatrixHandle m,
                                  const bst_ulong **out_shape, bst_ulong *out_dim, const float **out_result) {
  API_BEGIN
  if (!out_result) throw Error("XGBoosterPredictFromCudaArray: NULL output argument");
  *out_result = predict_inplace("XGBoosterPredictFromCudaArray", true, handle, values, config, m, out_shape, out_dim);
  API_END
}

// Dense container written by XGDMatrixSaveBinary: "QCDM" u32 version, u64 nrow, u64 ncol, f32 missing, data.
int XGDMatrixSaveBinary(DMatrixHandle handle, const char *fname, int silent) {
  API_BEGIN
  (void)silent;
  DMatrix *d = D(handle);
  const size_t n = (size_t)d->nrow * d->ncol;
  std::vector<float> h(n);
  if (n) {
    ensure_device();
    CU(cudaMemcpy(h.data(), d->X.p, n * 4, cudaMemcpyDeviceToHost));
  }
  FILE *fp = fopen(fname, "wb");
  if (!fp) throw Error(std::string("Opening ") + fname + " for writing failed");
  uint32_t ver = 1;
  uint64_t nr = d->nrow, nc = d->ncol;
  bool ok = fwrite("QCDM", 1, 4, fp) == 4 && fwrite(&ver, 4, 1, fp) == 1 && fwrite(&nr, 8, 1, fp) == 1 &&
            fwrite(&nc, 8, 1, fp) == 1 && fwrite(&d->missing, 4, 1, fp) == 1 && fwrite(h.data(), 4, n, fp) == n;
  fclose(fp);
  if (!ok) throw Error(std::string("Short write on ") + fname);
  API_END
}

// Text inputs libxgboost's XGDMatrixCreateFromFile also takes: libsvm ("label idx:val idx:val ...", the
// default) and csv ("<path>?format=csv[&label_column=N]").  Entries a libsvm row does not list are missing;
// the label column is parsed and dropped (prediction does not use it).
static void parse_text_matrix(const std::string &uri, std::vector<float> &h, uint64_t &nr, uint64_t &nc) {
  std::string path = uri, query;
  const size_t q = uri.find('?');
  if (q != std::string::npos) path = uri.substr(0, q), query = uri.substr(q + 1);
  const bool csv = query.find("format=csv") != std::string::npos;
  long label_col = -1;
  const size_t lc = query.find("label_column=");
  if (lc != std::string::npos) label_col = strtol(query.c_str() + lc + 13, nullptr, 10);
  FILE *fp = fopen(path.c_str(), "rb");
  if (!fp) throw Error("Opening " + path + " failed");
  std::string text;
  char buf[1 << 16];
  size_t n;
  while ((n = fread(buf, 1, sizeof buf, fp)) > 0) text.append(buf, n);
  fclose(fp);
  std::vector<std::vector<std::pair<uint64_t, float>>> rows;
  uint64_t maxcol = 0;
  size_t pos = 0;
  while (pos < text.size()) {
    size_t eol = text.find('\n', pos);
    if (eol == std::string::npos) eol = text.size();
    std::string line = text.substr(pos, eol - pos);
    pos = eol + 1;
    if (!line.empty() && line.back() == '\r') line.pop_back();
    if (line.find_first_not_of(" \t") == std::string::npos) continue;
    std::vector<std::pair<uint64_t, float>> row;
    const char *p = line.c_str();
    if (csv) {
      long col = 0;
      uint64_t out_col = 0;
      while (true) {
        char *e = nullptr;
        const float v = strtof(p, &e);
        const bool empty = e == p;
        if (col != label_col) {
          if (!empty) row.emplace_back(out_col, v);
          ++out_col;
        }
        p = e;
        while (*p == ' ') ++p;
        if (*p != ',') break;
        ++p, ++col;
      }
      maxcol = std::max<uint64_t>(maxcol, out_col);
    } else {
      char *e = nullptr;
      (void)strtof(p, &e);  // label
      if (e == p) throw Error(path + ": not a libqcoh dense matrix file, and not libsvm text either");
      p = e;
      while (*p) {
        while (*p == ' ' || *p == '\t') ++p;
        if (!*p || *p == '#') break;
        const uint64_t idx = strtoull(p, &e, 10);
        if (e == p || *e != ':') throw Error(path + ": malformed libsvm entry");
        p = e + 1;
        const float v = strtof(p, &e);
        if (e == p) throw Error(path + ": malformed libsvm value");
        p = e;
        row.emplace_back(idx, v);
        maxcol = std::max<uint64_t>(maxcol, idx + 1);
      }
    }
    rows.push_back(std::move(row));
  }
  nr = rows.size(), nc = maxcol;
  h.assign((size_t)nr * nc, NAN);
  for (uint64_t r = 0; r < nr; ++r)
    for (auto &kv : rows[r]) h[(size_t)r * nc + kv.first] = kv.second;
}

int XGDMatrixCreateFromFile(const char *fname, int silent, DMatrixHandle *out) {
  (void)silent;
  std::vector<float> h;
  uint64_t nr = 0, nc = 0;
  float missing = NAN;
  try {
    if (!fname) throw Error("XGDMatrixCreateFromFile: fname is NULL");
    const std::string uri(fname);
    bool binary = false;
    if (uri.find('?') == std::string::npos) {
      FILE *fp = fopen(fname, "rb");
      if (!fp) throw Error(std::string("Opening ") + fname + " failed");
      char magic[4];
      uint32_t ver = 0;
      binary = fread(magic, 1, 4, fp) == 4 && !memcmp(magic, "QCDM", 4);
      if (binary) {
        bool ok = fread(&ver, 4, 1, fp) == 1 && ver == 1 && fread(&nr, 8, 1, fp) == 1 && fread(&nc, 8, 1, fp) == 1 &&
                  fread(&missing, 4, 1, fp) == 1;
        if (ok) {
          h.resize((size_t)nr * nc);
          ok = fread(h.data(), 4, h.size(), fp) == h.size();
        }
        if (!ok) {
          fclose(fp);
          throw Error(std::string(fname) + ": truncated libqcoh dense matrix file");
        }
      }
      fclose(fp);
    }
    // XGBoost's own binary DMatrix container is not read; anything else is tried as libsvm / csv text
    if (!binary) parse_text_matrix(uri, h, nr, nc);
  } catch (const std::exception &e) {
    g_err = e.what();
    return -1;
  }
  return XGDMatrixCreateFromMat(h.data(), nr, nc, missing, out);
}

// =====================================================================================
// (2) qcoh_* extension
// =====================================================================================
const char *qcoh_version(void) { return "libqcoh 0.2 (sm_100a)"; }

int qcoh_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    (void)cudaGetLastError();
    return 0;
  }
  return n;
}

int qcoh_set_device(int device) {
  API_BEGIN
  if (g.ready && g.device != device) throw Error("qcoh_set_device: the library is already bound to device " + std::to_string(g.device));
  requested_device = device;
  ensure_device();
  API_END
}

int qcoh_host_alloc(size_t bytes, void **out) {
  API_BEGIN
  ensure_device();
  CU(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault));
  API_END
}
int qcoh_host_free(void *p) {
  API_BEGIN
  CU(cudaFreeHost(p));
  API_END
}
int qcoh_device_alloc(size_t bytes, void **out) {
  API_BEGIN
  ensure_device();
  CU(cudaMalloc(out, bytes ? bytes : 1));
  API_END
}
int qcoh_device_free(void *p) {
  API_BEGIN
  CU(cudaFree(p));
  API_END
}
int qcoh_memcpy_h2d(void *dst, const void *src, size_t bytes) {
  API_BEGIN
  ensure_device();
  CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, g.stream));
  CU(cudaStreamSynchronize(g.stream));
  API_END
}
int qcoh_memcpy_d2h(void *dst, const void *src, size_t bytes) {
  API_BEGIN
  ensure_device();
  CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, g.stream));
  CU(cudaStreamSynchronize(g.stream));
  API_END
}
int qcoh_device_synchronize(void) {
  API_BEGIN
  ensure_device();
  CU(cudaStreamSynchronize(g.stream));
  API_END
}
int qcoh_timer_start(void) {
  API_BEGIN
  ensure_device();
  CU(cudaEventRecord(g.ev0, g.stream));
  API_END
}
int qcoh_timer_stop(float *ms) {
  API_BEGIN
  ensure_device();
  CU(cudaEventRecord(g.ev1, g.stream));
  CU(cudaEventSynchronize(g.ev1));
  CU(cudaEventElapsedTime(ms, g.ev0, g.ev1));
  API_END
}
int qcoh_flush_l2(void) {
  API_BEGIN
  ensure_device();
  if (!g.flush) {
    g.flush_bytes = (size_t)256 << 20;  // 2x the 126 MB L2
    CU(cudaMalloc(&g.flush, g.flush_bytes));
  }
  CU(cudaMemsetAsync(g.flush, 0, g.flush_bytes, g.stream));
  API_END
}

int qcoh_set_param(const char *name, const char *value) {
  API_BEGIN
  if (!name || !value) throw Error("qcoh_set_param: NULL argument");
  const int v = atoi(value);
  std::string n(name);
  if (n == "duo") g.duo = v;
  else if (n == "speculate") g.speculate = v;
  else if (n == "chunk_rows") g.chunk_rows = v > 0 ? ((uint64_t)v + 255) / 256 * 256 : (1ull << 21);
  else throw Error("qcoh_set_param: unknown parameter '" + n + "'");
  API_END
}

uint64_t qcoh_launch_count(void) { return launch_count(); }
uint64_t qcoh_kernel_launches(const char *family) { return family ? kernel_launches(family) : 0; }
const char *qcoh_last_predict_kernel(void) { return last_predict_kernel(); }

int qcoh_booster_get_info(BoosterHandle handle, qcoh_booster_info *out) {
  API_BEGIN
  Booster *b = B(handle);
  if (!b->loaded) throw Error("Booster has no model");
  out->num_trees = (int32_t)b->host.trees.size();
  out->num_feature = (int32_t)b->host.num_feature;
  out->max_depth = b->flat.max_depth;
  out->num_nodes = b->flat.num_nodes();
  out->base_score = b->host.base_score;
  out->format = (int32_t)b->host.format;
  for (int i = 0; i < 3; ++i) out->version[i] = b->host.version[i];
  API_END
}

int qcoh_booster_get_flat(BoosterHandle handle, const uint32_t **nodes_xy, const uint32_t **tree_offset,
                          const int32_t **tree_depth, const int32_t **orig_id) {
  API_BEGIN
  Booster *b = B(handle);
  if (!b->loaded) throw Error("Booster has no model");
  if (nodes_xy) *nodes_xy = b->flat.nodes_xy.data();
  if (tree_offset) *tree_offset = b->flat.tree_offset.data();
  if (tree_depth) *tree_depth = b->flat.tree_depth.data();
  if (orig_id) *orig_id = b->flat.orig_id.data();
  API_END
}

int qcoh_booster_get_duo(BoosterHandle handle, const uint32_t **rec, const uint32_t **tree_slot, const uint32_t **top_xy,
                         int64_t *num_slots) {
  API_BEGIN
  Booster *b = B(handle);
  if (!b->loaded) throw Error("Booster has no model");
  if (!b->duo.ok) throw Error("two-level records are not available for this booster: " + b->duo.why);
  if (rec) *rec = b->duo.rec.data();
  if (tree_slot) *tree_slot = b->duo.tree_slot.data();
  if (top_xy) *top_xy = b->duo.top_xy.data();
  if (num_slots) *num_slots = b->duo.num_slots();
  API_END
}

int qcoh_booster_get_duo_info(BoosterHandle handle, int *blk_shift, int *has_default_bits) {
  API_BEGIN
  Booster *b = B(handle);
  if (!b->loaded) throw Error("Booster has no model");
  if (!b->duo.ok) throw Error("two-level records are not available for this booster: " + b->duo.why);
  if (blk_shift) *blk_shift = b->duo.blk_shift;
  if (has_default_bits) *has_default_bits = b->duo.has_default_bits ? 1 : 0;
  API_END
}

int qcoh_dmatrix_create_device(bst_ulong nrow, bst_ulong ncol, float missing, DMatrixHandle *out) {
  API_BEGIN
  if (ncol > kMaxMatrixCols) throw Error("qcoh_dmatrix_create_device: " + std::to_string(ncol) + " columns; libqcoh's tile form holds at most " + std::to_string(kMaxMatrixCols));
  ensure_device();
  std::unique_ptr<DMatrix> d(new DMatrix());
  d->nrow = nrow, d->ncol = ncol, d->missing = missing;
  d->X.need((size_t)nrow * ncol);
  g_live_handles.insert(d.get());
  *out = d.release();
  API_END
}
int qcoh_dmatrix_device_ptr(DMatrixHandle handle, float **out_dev) {
  API_BEGIN
  *out_dev = D(handle)->X.p;
  API_END
}
int qcoh_dmatrix_upload(DMatrixHandle handle, const float *host_rows, bst_ulong row0, bst_ulong nrows) {
  API_BEGIN
  DMatrix *d = D(handle);
  if (row0 + nrows > d->nrow) throw Error("qcoh_dmatrix_upload: row range out of bounds");
  CU(cudaMemcpyAsync(d->X.p + (size_t)row0 * d->ncol, host_rows, (size_t)nrows * d->ncol * 4,
                     is_device_ptr(host_rows) ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, g.stream));
  CU(cudaStreamSynchronize(g.stream));
  d->sealed = false;
  API_END
}
int qcoh_dmatrix_seal(DMatrixHandle handle) {
  API_BEGIN
  seal(D(handle));
  API_END
}
int qcoh_dmatrix_tiles_ptr(DMatrixHandle handle, const uint32_t **out_dev, uint64_t *num_tiles) {
  API_BEGIN
  DMatrix *d = D(handle);
  if (!d->sealed) seal(d);
  if (out_dev) *out_dev = d->Xt.p;
  if (num_tiles) *num_tiles = tile_count(d->nrow);
  API_END
}

int qcoh_booster_predict_device(BoosterHandle handle, DMatrixHandle dmat, int option_mask, unsigned ntree_limit,
                                const qcoh_epilogue *epi, float *out_dev) {
  API_BEGIN
  predict_into(B(handle), D(dmat), option_mask, ntree_limit, epi, out_dev);
  API_END
}

int qcoh_booster_predict_contribs_device(BoosterHandle handle, DMatrixHandle dmat, int approximate, unsigned ntree_limit,
                                         float *out_dev) {
  API_BEGIN
  contribs_into(B(handle), D(dmat), approximate != 0, ntree_limit, out_dev);
  API_END
}

int qcoh_booster_predict_interactions_device(BoosterHandle handle, DMatrixHandle dmat, int approximate, unsigned ntree_limit,
                                             float *out_dev) {
  API_BEGIN
  Booster *b = B(handle);
  (void)shap_tables(b);  // a booster without covers fails here, before any device work
  ensure_device();
  interactions_into(b, D(dmat), approximate != 0, ntree_limit, out_dev);
  API_END
}

int qcoh_booster_get_shap_paths(BoosterHandle handle, const uint32_t **bins, const int64_t **tree_bin, const float **node_mean,
                                int64_t *num_bins) {
  API_BEGIN
  const ShapForest &s = shap_tables(B(handle));
  if (bins) *bins = s.bins.data();
  if (tree_bin) *tree_bin = s.tree_bin.data();
  if (node_mean) *node_mean = s.mean.data();
  if (num_bins) *num_bins = s.num_bins();
  API_END
}

int qcoh_partition_columns(int64_t ncol_global, int nranks, int rank, int64_t *col0, int64_t *ncol_local) {
  API_BEGIN
  if (nranks <= 0 || rank < 0 || rank >= nranks || ncol_global < 0) throw Error("qcoh_partition_columns: bad arguments");
  const int64_t q = ncol_global / nranks, r = ncol_global % nranks;
  // the first r ranks own one extra column; contiguous ranges, no halo (SURVEY.md 8e)
  *col0 = q * rank + (rank < r ? rank : r);
  *ncol_local = q + (rank < r ? 1 : 0);
  API_END
}

}  // extern "C"
