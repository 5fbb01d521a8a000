// context.hpp — shared plumbing of libqcoh's C ABI translation units: error channel, device context,
// owning buffers, handle types.  Internal; nothing here is exported.
#pragma once
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>  // header-only; a no-op unless a profiler is attached

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <thread>
#include <unordered_set>
#include <utility>
#include <vector>

#include "../../include/qcoh.h"
#include "forest.hpp"
#include "kernels.hpp"

namespace qcoh {

inline thread_local std::string g_err;

struct Error : std::runtime_error {
  using std::runtime_error::runtime_error;
};

#define CU(call)                                                                                      \
  do {                                                                                                \
    cudaError_t e__ = (call);                                                                         \
    if (e__ != cudaSuccess)                                                                           \
      throw Error(std::string("CUDA error in " #call ": ") + cudaGetErrorName(e__) + " — " +          \
                  cudaGetErrorString(e__));                                                           \
  } while (0)

// every C ABI entry point is an NVTX range named after the function (visible in Nsight Systems / ncu)
struct NvtxRange {
  explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};
#define API_BEGIN        \
  NvtxRange nvtx__(__func__); \
  try {
#define API_END                      \
  }                                  \
  catch (const std::exception &e) {  \
    g_err = e.what();                \
    return -1;                       \
  }                                  \
  catch (...) {                      \
    g_err = "unknown error";         \
    return -1;                       \
  }                                  \
  return 0;

// ---- device context ---------------------------------------------------------------
// Thread model (SURVEY.md 8e: "one process per GPU" and "one process, one host thread per device" are both
// supported): ALL mutable library state — the device context below, the buffer pools, the constant-table
// window, the live-handle set, the model cache, the mirror's SAVE'd booster, the NCCL communicator — is
// thread_local.  A host thread is one "rank": it binds to one GPU (qcoh_set_device / $LOCAL_RANK) and owns the
// handles it creates; a handle is not valid in another thread.  One thread per device: the constant-memory tables
// are per device, so a second thread binding to a device that already has an owner is refused.
struct Ctx {
  bool ready = false;
  int device = -1;
  cudaStream_t stream = nullptr;       // compute (and everything ordered with it)
  cudaStream_t copy_stream = nullptr;  // H2D of matrix chunks
  cudaStream_t d2h_stream = nullptr;   // D2H of result chunks
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  std::vector<cudaEvent_t> chunk_events;
  int duo = -1;                        // two-level records when the booster qualifies; 0 = 8-byte nodes only
  int speculate = 1;                   // pipeline prediction into XGDMatrixCreateFromMat
  uint64_t chunk_rows = 1ull << 21;
  void *flush = nullptr;
  size_t flush_bytes = 0;
};
inline thread_local Ctx g;

inline thread_local int requested_device = -1;

// device -> the thread that owns it (process-wide; the only shared mutable state besides the copy pool)
inline std::mutex g_device_owner_mutex;
inline std::thread::id g_device_owner[64];
inline bool g_device_owned[64] = {false};
struct DeviceLease {  // released when the owning thread ends
  int device = -1;
  ~DeviceLease() {
    if (device >= 0) {
      std::lock_guard<std::mutex> lk(g_device_owner_mutex);
      g_device_owned[device] = false;
    }
  }
};
inline thread_local DeviceLease g_device_lease;

inline void ensure_device() {
  if (g.ready) return;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    (void)cudaGetLastError();
    throw Error(std::string("libqcoh: no CUDA device is visible (") + (e == cudaSuccess ? "device count 0" : cudaGetErrorString(e)) +
                "); the OH path runs on the GPU only, there is no CPU fallback");
  }
  int dev = requested_device;
  if (dev < 0) {
    const char *lr = getenv("LOCAL_RANK");
    dev = lr ? atoi(lr) % n : 0;
  }
  if (dev >= n) throw Error("libqcoh: device " + std::to_string(dev) + " requested but only " + std::to_string(n) + " visible");
  if (dev < 64) {
    std::lock_guard<std::mutex> lk(g_device_owner_mutex);
    if (g_device_owned[dev] && g_device_owner[dev] != std::this_thread::get_id())
      throw Error("libqcoh: device " + std::to_string(dev) + " is already driven by another host thread of this process (one thread per GPU)");
    g_device_owned[dev] = true, g_device_owner[dev] = std::this_thread::get_id();
    g_device_lease.device = dev;
  }
  CU(cudaSetDevice(dev));
  cudaDeviceProp p;
  CU(cudaGetDeviceProperties(&p, dev));
  if (p.major < 10)
    throw Error(std::string("libqcoh is built for sm_100a (B200); device '") + p.name + "' is sm_" + std::to_string(p.major) +
                std::to_string(p.minor));
  CU(cudaStreamCreateWithFlags(&g.stream, cudaStreamNonBlocking));
  CU(cudaStreamCreateWithFlags(&g.copy_stream, cudaStreamNonBlocking));
  CU(cudaStreamCreateWithFlags(&g.d2h_stream, cudaStreamNonBlocking));
  CU(cudaEventCreate(&g.ev0));
  CU(cudaEventCreate(&g.ev1));
  g.device = dev;
  g.ready = true;
}

template <class T>
struct DevBuf {
  T *p = nullptr;
  size_t cap = 0;  // elements
  T *need(size_t n) {
    if (n > cap) {
      if (p) cudaFree(p);
      p = nullptr, cap = 0;
      CU(cudaMalloc((void **)&p, (n ? n : 1) * sizeof(T)));
      cap = n;
    }
    return p;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr, cap = 0;
  }
  void swap(DevBuf &o) {
    std::swap(p, o.p);
    std::swap(cap, o.cap);
  }
  DevBuf() = default;
  DevBuf(const DevBuf &) = delete;
  DevBuf &operator=(const DevBuf &) = delete;
  ~DevBuf() { release(); }
};

template <class T>
struct PinBuf {
  T *p = nullptr;
  size_t cap = 0;
  T *need(size_t n) {
    if (n > cap) {
      if (p) cudaFreeHost(p);
      p = nullptr, cap = 0;
      CU(cudaHostAlloc((void **)&p, (n ? n : 1) * sizeof(T), cudaHostAllocDefault));
      cap = n;
    }
    return p;
  }
  void swap(PinBuf &o) {
    std::swap(p, o.p);
    std::swap(cap, o.cap);
  }
  PinBuf() = default;
  PinBuf(const PinBuf &) = delete;
  PinBuf &operator=(const PinBuf &) = delete;
  ~PinBuf() {
    if (p) cudaFreeHost(p);
  }
};

inline bool is_device_ptr(const void *p) {
  cudaPointerAttributes a;
  cudaError_t e = cudaPointerGetAttributes(&a, p);
  if (e != cudaSuccess) {
    (void)cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// ---- handles ------------------------------------------------------------------------
constexpr uint32_t kBoosterMagic = 0x51434253;  // 'QCBS'
constexpr uint32_t kDMatrixMagic = 0x5143444d;  // 'QCDM'
constexpr uint32_t kOhMagic = 0x51434f48;       // 'QCOH'

// Live handles: a freed handle is recognised by its absence here, not by reading freed memory.
inline thread_local std::unordered_set<const void *> g_live_handles;
inline bool is_live(const void *h) { return h && g_live_handles.count(h) != 0; }

struct Booster {
  uint32_t magic = kBoosterMagic;
  int oh_refs = 0;       // fused-Run1 handles predicting with this booster: it cannot be freed while > 0
  uint64_t version = 0;  // changes with every (re)load
  bool loaded = false, uploaded = false;
  bool cache_owned = false;  // lives in the model cache (model_cache.cpp): not the caller's to free or reload
  HostForest host;
  FlatForest flat;
  std::vector<uint32_t> dev_nodes_host;  // the device form of the nodes (keys), kept for the constant-top table
  DeviceForest dev;
  DuoForest duo;            // two-level records (forest.hpp); built with the model, ok == false if it does not qualify
  DevBuf<uint4> d_recs;
  DevBuf<uint2> d_nodes;
  DevBuf<uint32_t> d_off;
  DevBuf<int32_t> d_depth, d_orig;
  DevBuf<float> d_result;
  PinBuf<float> h_result;
  std::vector<bst_ulong> h_shape;  // XGBoosterPredictFromDMatrix's out_shape
  // contributions (forest.hpp ShapForest): built on the host and uploaded at the first contributions call
  ShapForest shap;
  bool shap_uploaded = false;
  DevBuf<uint4> d_shap_bins;
  DevBuf<float> d_shap_mean;
  DevBuf<double> d_shap_part;  // float64 partial sums of the bin slices, [kShapSlices][kShapChunkRows][nfeat]
  // interactions: the per-feature bin lists (ShapForest::feat_off / feat_bins), uploaded at the first interactions call
  bool inter_uploaded = false;
  DevBuf<int64_t> d_inter_off;
  DevBuf<uint32_t> d_inter_bins;
  DevBuf<double> d_inter_part;  // [nfeat][kInterSlices][kInterChunkRows][nfeat]
  DevBuf<float> d_inter_phi;    // approximate: the Saabas contributions [nrow][nfeat + 1] that go on the diagonal
  Booster() = default;
  Booster(const Booster &) = delete;
  Booster &operator=(const Booster &) = delete;
  ~Booster() {
    if (dev.tex) cudaDestroyTextureObject(dev.tex);
    if (dev.tex4) cudaDestroyTextureObject(dev.tex4);
  }
};

struct DMatrix {
  uint32_t magic = kDMatrixMagic;
  uint64_t nrow = 0, ncol = 0;
  float missing = NAN;
  DevBuf<float> X;       // row-major floats as handed in (XGDMatrixSaveBinary, qcoh_dmatrix_device_ptr)
  DevBuf<uint32_t> Xt;   // the device form the kernels read: key tiles (kernels.hpp), built by seal
  DevBuf<int> flags;
  int hflags = 1;  // bit0 has-missing, bit1 has-inf; conservative until sealed
  bool sealed = false;
  // prediction pipelined into XGDMatrixCreateFromMat (see create_pipelined)
  const void *spec_booster = nullptr;
  uint64_t spec_version = 0;
  bool spec_ready = false;
  DevBuf<float> spec_dev;
  PinBuf<float> spec_host;
};

// XGDMatrixFree keeps the largest freed matrix buffer for the next XGDMatrixCreateFromMat: the
// reference creates and frees a same-sized DMatrix on every call (OH_GridCompMod.F90:347,377) and
// cudaMalloc / cudaFree of multi-GB buffers would otherwise dominate the step.
inline thread_local DevBuf<float> g_spare_X;
inline thread_local DevBuf<uint32_t> g_spare_Xt;
inline thread_local PinBuf<float> g_spare_pin;
inline thread_local DevBuf<float> g_spare_spec;
inline thread_local DevBuf<int> g_chunk_flags;
inline thread_local PinBuf<int> g_h_chunk_flags;
inline thread_local Booster *g_last_booster = nullptr;  // the process's booster (the reference keeps exactly one, SAVE :182)
inline thread_local uint64_t g_version_counter = 0;

inline Booster *B(BoosterHandle h) {
  Booster *b = (Booster *)h;
  if (!b || !is_live(h) || b->magic != kBoosterMagic) throw Error("Invalid booster handle");
  return b;
}
inline DMatrix *D(DMatrixHandle h) {
  DMatrix *d = (DMatrix *)h;
  if (!d || !is_live(h) || d->magic != kDMatrixMagic) throw Error("Invalid DMatrix handle");
  return d;
}

// capi_xgb.cpp
void upload(Booster *b);
// make the constant-memory tables of tree tops hold trees [tree0, tree0 + ntree) of this booster, uploading them if
// they do not yet, and return what the tables hold (see capi_xgb.cpp)
ConstWindow hold(Booster *b, int tree0, int ntree);
// one prediction = one launch per range of kRangeTrees trees (capi_xgb.cpp)
void launch_predict_chunked(Booster *b, PredictArgs a, cudaStream_t s);
// the booster's ShapForest, built on first use (host only; throws when the booster has no covers)
const ShapForest &shap_tables(Booster *b);

}  // namespace qcoh
