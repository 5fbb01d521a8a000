// kernels.cu — hand-written sm_100a kernels of the OH hot path.
//
//   K3  seal_tiles_kernel     the missing / inf scan of XGDMatrixCreateFromMat (OH_GridCompMod.F90:347) fused with
//                             the conversion of the row-major float matrix into the DMatrix's device form:
//                             feature-major tiles of order-preserving integer keys
//   K2  predict_tiles_kernel  tree-ensemble traversal, replaces libxgboost's CPUPredictor behind XGBoosterPredict
//                             (reference call site :356) with the export transform 10**x * OHscale (:369,:1569) fused
//                             as epilogue; sums / leaf indices, clean matrices / missing entries; tiles arrive by TMA.
//                             Its walk policy picks the node layout and the launch shape: DuoWalk on the two-level
//                             16-byte records (one gather per two tree levels), NodesWalk on the 8-byte depth-ordered
//                             nodes (boosters the records do not hold)
//       predict_soa_kernel    K2 with the tile assembled straight from the Run1 SoA fields (run1_feature, which
//                             oh_pack reads the features with too)
//       predict_dense_kernel  K2 with the tile assembled from a caller's strided float array (inplace prediction)
//   K6  shap_paths / shap_reduce / shap_approx   per-feature contributions (exact TreeSHAP, approximate Saabas)
//       shap_inter / shap_inter_reduce / shap_inter_expand   SHAP interaction values (conditioned TreeSHAP)
//   K1  oh_state / oh_sums / oh_pack    Run1 feature assembly (:1240-1257, :1441-1488, :303-345)
//   K5  oh_finalize           troposphere mask + unit conversion (:1579-1595)
//   K4  oh_diag               build-defined mass-weighted mean OH / CH4 lifetime partial sums
//
// Numerics: compiled with -fmad=false and written with explicit round-to-nearest intrinsics where
// the Fortran evaluation order matters, so every float32 feature is bit-identical to the CPU
// evaluation.  No tensor cores: tree traversal is not a dense contraction.
#include "kernels.hpp"

#include <cfloat>
#include <cmath>
#include <cstring>
#include <vector>

#include "forest.hpp"

namespace qcoh {

static thread_local uint64_t g_launches = 0;
uint64_t launch_count() { return g_launches; }

#define QC_LAUNCHED() (++g_launches, cudaGetLastError())

// launches per kernel family: what the parity tests assert ("this launch was served by the two-level kernel").  The
// predict families are ordered base, _missing, _leaf, _missing_leaf: base + has_missing + 2 * pred_leaf.
namespace {
enum Family {
  kDuo, kNodes8 = kDuo + 4, kSoaDuo = kNodes8 + 4, kSoaNodes8, kSealTiles, kShap, kShapReduce, kShapApprox, kDenseDuo, kDenseNodes8,
  kShapInter, kShapInterReduce, kShapInterExpand, kFamilies
};
const char *const kFamilyName[kFamilies] = {"duo", "duo_missing", "duo_leaf", "duo_missing_leaf", "nodes8", "nodes8_missing",
                                            "nodes8_leaf", "nodes8_missing_leaf", "soa_duo", "soa_nodes8", "seal_tiles",
                                            "shap", "shap_reduce", "shap_approx", "dense_duo", "dense_nodes8",
                                            "shap_inter", "shap_inter_reduce", "shap_inter_expand"};
thread_local uint64_t g_family[kFamilies];
thread_local const char *g_last_predict = "";
void count_family(int f) { ++g_family[f]; }
// the predict and contribution launches also record the family that served the last of them
void count_predict(int f) { ++g_family[f], g_last_predict = kFamilyName[f]; }
}  // namespace
uint64_t kernel_launches(const char *family) {
  for (int i = 0; i < kFamilies; ++i)
    if (!strcmp(kFamilyName[i], family)) return g_family[i];
  return 0;
}
const char *last_predict_kernel() { return g_last_predict; }

__global__ void fill_kernel(float *p, uint64_t n, float v) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) p[i] = v;
}
cudaError_t launch_fill(float *p, uint64_t n, float v, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  int blocks = (int)((n + 255) / 256 < 148 * 16 ? (n + 255) / 256 : 148 * 16);
  fill_kernel<<<blocks, 256, 0, s>>>(p, n, v);
  return QC_LAUNCHED();
}

// =====================================================================================
// Keys, tiles, constant tables
// =====================================================================================
// One thread = one row (grid cell).  A CTA's 256 rows sit in shared memory TRANSPOSED, skey[f][tid]:
// whatever feature each lane asks for, lane L always hits bank L — the data-dependent feature fetch is
// bank-conflict-free by construction.  The tile holds order-preserving integer keys of the values
// (below); slot `nfeat` of every row holds key 0: leaves are encoded with feat = nfeat, so the compare
// never says "right" there — no leaf test inside the descent.  Missing entries (NaN or == missing) are
// key 0xFFFFFFFF.
//
// XGBoost semantics restated (xgboost 1.6.0 src/predictor/predict_fn.h GetNextNode,
// src/predictor/cpu_predictor.cc PredictByAllTrees): missing -> default child, else
// left + !(fvalue < split_cond); out = base_score, then += leaf value tree by tree in float32.
constexpr int kBlock = kTileRows;  // rows (= threads) per CTA
constexpr int kStride = kTileRows; // feature stride of the transposed tile, in keys (1 KB: the PRMT address trick)
static_assert(kStride * 4 == 1024, "the address arithmetic of the walks assumes a 1 KB feature stride");

// Order-preserving integer keys: key(v) = bits ^ (sign ? 0xFFFFFFFF : 0x80000000) of the value with -0.0
// folded into +0.0, which is monotone: a < b  <=>  key(a) < key(b) (unsigned) for all non-NaN floats, and
// key(-0) == key(+0) like the float compare.  An internal node stores x = -key(threshold) (mod 2^32;
// key(thr) is never 0), so
//     !(v < thr)  <=>  key(thr) <= key(v)  <=>  x + key(v) >= 2^32
// which is the carry of x + key(v): `add.cc` + `addc` fold the compare into the index update in two
// instructions and no predicate.  Missing is key 0xFFFFFFFF (above +inf: it carries against every
// threshold, and the walks that may see it test for it explicitly and take the default child).
constexpr uint32_t kKeyMissing = 0xFFFFFFFFu;
__device__ __forceinline__ uint32_t float_key(float v) {
  const uint32_t b = __float_as_uint(__fadd_rn(v, 0.0f));  // -0.0 + 0.0 = +0.0
  return b ^ ((uint32_t)((int32_t)b >> 31) | 0x80000000u);
}
// idx + rel + carry(x + kv)
__device__ __forceinline__ uint32_t step_index(uint32_t idx, uint32_t rel, uint32_t x, uint32_t kv) {
  asm("{\n\t.reg .u32 t;\n\tadd.cc.u32 t, %2, %3;\n\taddc.u32 %0, %0, %1;\n\t}" : "+r"(idx) : "r"(rel), "r"(x), "r"(kv));
  return idx;
}
__device__ __forceinline__ uint32_t add_carry_out(uint32_t a, uint32_t b) {
  uint32_t c;
  asm("{\n\t.reg .u32 t;\n\tadd.cc.u32 t, %1, %2;\n\taddc.u32 %0, 0, 0;\n\t}" : "=r"(c) : "r"(a), "r"(b));
  return c;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t saddr) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(saddr));
  return v;
}

// Top of every tree in constant memory: constant loads go through the constant cache, not the LSU / TEX
// data pipes; lanes of a warp mostly agree at those levels, so the per-address serialisation of divergent
// constant loads stays short.  The table belongs to one booster (and one range of its trees) at a time:
//   8-byte-node walk: the first 2^CTOP - 1 nodes of a tree in breadth-first order = its levels 0..CTOP-1
//   two-level records: DuoForest::top_xy (complete heap-ordered tops) + c_duo_base, the global index of each
//                      tree's first record (the block pointers are tree-relative)
constexpr int kConstTopNodes = kConstTreesMax << kDuoTop;  // 61 440 B of the 64 KB constant bank
__constant__ uint2 c_top[kConstTopNodes];
__constant__ uint32_t c_duo_base[kConstTreesMax];

cudaError_t upload_const_top(const uint32_t *dev_nodes_xy, const uint32_t *tree_offset, int ntree, cudaStream_t s) {
  constexpr int stride = 1 << kDuoTop;
  if (ntree > kConstTreesMax) return cudaErrorInvalidValue;
  std::vector<uint2> host((size_t)ntree * stride);
  for (int t = 0; t < ntree; ++t) {
    const uint32_t n0 = tree_offset[t], n1 = tree_offset[t + 1];
    for (int i = 0; i < stride; ++i) {
      const uint32_t n = n0 + (uint32_t)i;
      host[t * stride + i] = n < n1 ? make_uint2(dev_nodes_xy[2 * n], dev_nodes_xy[2 * n + 1]) : make_uint2(0u, 0u);
    }
  }
  // pageable source: the call returns once the data is staged, so the local buffer may go
  return cudaMemcpyToSymbolAsync(c_top, host.data(), sizeof(uint2) * (size_t)ntree * stride, 0, cudaMemcpyHostToDevice, s);
}

cudaError_t upload_const_duo(const uint32_t *top_xy, const uint32_t *tree_slot, int ntree, cudaStream_t s) {
  if (ntree > kConstTreesMax) return cudaErrorInvalidValue;
  cudaError_t e = cudaMemcpyToSymbolAsync(c_top, top_xy, sizeof(uint2) * ((size_t)ntree << kDuoTop), 0, cudaMemcpyHostToDevice, s);
  if (e != cudaSuccess) return e;
  return cudaMemcpyToSymbolAsync(c_duo_base, tree_slot, sizeof(uint32_t) * (size_t)ntree, 0, cudaMemcpyHostToDevice, s);
}

// ---- TMA (bulk async copy) + mbarrier helpers: global -> shared without the LSU ------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(bar),
      "r"(parity)
      : "memory");
}

// The tile loop shared by the predict kernels.  A CTA walks tiles blockIdx.x, + gridDim.x, ...; the grid is one
// CTA per tile, and the resident CTAs of an SM overlap each other's loads.  A tile arrives with one bulk copy (TMA,
// cp.async.bulk completing on an mbarrier — SASS UBLKCP + SYNCS) of ncol KB of keys in their final layout: no LSU
// instruction, no register, no arithmetic between HBM and the walk.  One thread issues the copy and polls the
// mbarrier, the CTA then passes a barrier (256 threads polling one word showed up as shared-memory bank-conflict
// wavefronts on the LSU data pipe, profiles/README.md v4).
struct TilePipe {
  uint32_t smem0, bar0, tile_bytes, src_skip, dst_skip;
  const uint32_t *Xt;
  uint64_t ntile, tile, tile_stride;
  uint32_t it;
  __device__ __forceinline__ void issue(uint64_t t) const {
    mbar_expect_tx(bar0, tile_bytes);
    if (tile_bytes) bulk_g2s(smem0 + dst_skip, Xt + t * tile_stride + src_skip, tile_bytes, bar0);
  }
  // The buffer is [row order | nfeat feature slots | key-0 slot], 1 KB each.  Slots the matrix does not have are
  // missing (xgboost FVec::Fill leaves them flagged); the last slot is the key-0 slot leaves point at.  Both are
  // written once: the bulk copies only touch the order slot (with_order) and slots 0..ncol-1.
  __device__ __forceinline__ void begin(uint32_t *smem, unsigned long long *bar, const PredictArgs &a, int nfeat, bool with_order, int tid) {
    smem0 = (uint32_t)__cvta_generic_to_shared(smem), bar0 = (uint32_t)__cvta_generic_to_shared(bar);
    tile_stride = (uint64_t)(a.ncol + 1) * kStride;
    tile_bytes = (uint32_t)(a.ncol + (with_order ? 1 : 0)) * kStride * 4u;
    src_skip = with_order ? 0u : (uint32_t)kStride, dst_skip = with_order ? 0u : (uint32_t)kStride * 4u;
    Xt = a.Xt, ntile = (a.nrow + kTileRows - 1) / kTileRows, tile = blockIdx.x, it = 0;
    uint32_t *k = smem + kStride;
    for (int c = a.ncol; c < nfeat; ++c) k[c * kStride + tid] = kKeyMissing;
    k[nfeat * kStride + tid] = 0u;
    if (tid == 0) {
      mbar_init(bar0, 1);
      mbar_init_fence();
    }
    __syncthreads();
    if (tid == 0 && tile < ntile) issue(tile);
  }
  __device__ __forceinline__ bool more() const { return tile < ntile; }
  // returns the shared address of the buffer (its row-order slot; the feature slots follow 1 KB later)
  __device__ __forceinline__ uint32_t acquire(int tid) {
    if (tid == 0) mbar_wait(bar0, it & 1u);
    __syncthreads();
    return smem0;
  }
  __device__ __forceinline__ void release(int tid) {
    // every thread is done with the buffer before it is refilled
    if (tile + gridDim.x < ntile) {
      __syncthreads();
      if (tid == 0) issue(tile + gridDim.x);
    }
    tile += gridDim.x, ++it;
  }
};

// =====================================================================================
// K3 — seal: row-major float matrix -> key tiles, with the missing / inf scan
// =====================================================================================
__global__ void __launch_bounds__(kTileRows) seal_tiles_kernel(const float *__restrict__ X, uint64_t nrow, int ncol, float missing,
                                                               int check_inf, uint32_t *__restrict__ Xt, int *flags) {
  extern __shared__ __align__(16) float srows[];  // [256][ld] row-major, ld odd: the per-thread row reads are conflict-free
  __shared__ int warp_clean[kTileRows / 32];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int ld = ncol | 1;
  const uint64_t r0 = (uint64_t)blockIdx.x * kTileRows;
  const uint64_t left = nrow - r0;
  const int nr = left < (uint64_t)kTileRows ? (int)left : kTileRows;
  const float *__restrict__ src = X + r0 * (uint64_t)ncol;
  const int n = nr * ncol;
  if (ld == ncol) {  // the tile's rows are one contiguous run of X: flat, coalesced copy
    if ((((uintptr_t)src) & 15u) == 0u) {
      const float4 *s4 = reinterpret_cast<const float4 *>(src);
      float4 *d4 = reinterpret_cast<float4 *>(srows);
      for (int i = tid; i < (n >> 2); i += kTileRows) d4[i] = __ldg(s4 + i);
      for (int i = (n & ~3) + tid; i < n; i += kTileRows) srows[i] = __ldg(src + i);
    } else {
      for (int i = tid; i < n; i += kTileRows) srows[i] = __ldg(src + i);
    }
  } else {
    for (int i = tid; i < n; i += kTileRows) srows[(i / ncol) * ld + (i % ncol)] = __ldg(src + i);
  }
  __syncthreads();
  // pass 1: does my row hold a missing entry?  (rows past the end of the matrix count as clean; never stored)
  int fl = 0;
  if (tid < nr) {
    for (int c = 0; c < ncol; ++c) {
      const float x = srows[tid * ld + c];
      if (x != x || x == missing) fl |= 1;
      if (check_inf && isinf(x)) fl |= 2;
    }
  }
  // row order: clean rows first, rows with a missing entry last, both in their original order (stable)
  const unsigned clean_mask = __ballot_sync(0xffffffffu, !(fl & 1));
  if (lane == 0) warp_clean[wid] = __popc(clean_mask);
  __syncthreads();
  int clean_before = 0, clean_total = 0;
#pragma unroll
  for (int w = 0; w < kTileRows / 32; ++w) {
    const int cw = warp_clean[w];
    clean_total += cw;
    if (w < wid) clean_before += cw;
  }
  const int my_clean_rank = clean_before + __popc(clean_mask & ((1u << lane) - 1u));
  const int pos = (fl & 1) ? clean_total + (tid - my_clean_rank) : my_clean_rank;
  uint32_t *__restrict__ tile = Xt + (size_t)blockIdx.x * (size_t)(ncol + 1) * kTileRows;
  tile[pos] = (uint32_t)tid | ((uint32_t)(fl & 1) << 8);
  // pass 2: my row's keys, column by column, to my position (1 KB per column; coalesced where the order is the identity)
  uint32_t *__restrict__ dst = tile + kTileRows + pos;
  for (int c = 0; c < ncol; ++c) {
    uint32_t k = 0u;
    if (tid < nr) {
      const float x = srows[tid * ld + c];
      k = (x != x || x == missing) ? kKeyMissing : float_key(x);
    }
    dst[(size_t)c * kTileRows] = k;
  }
  fl = __reduce_or_sync(0xffffffffu, fl);
  if (lane == 0 && fl) atomicOr(flags, fl);
}

cudaError_t launch_seal_tiles(const float *X, uint64_t nrow, int ncol, float missing, uint32_t *Xt, int *flags, cudaStream_t s) {
  if (nrow == 0) return cudaSuccess;
  const uint64_t ntile = tile_count(nrow);
  if (ntile > 0x7fffffffull) return cudaErrorInvalidConfiguration;
  const size_t smem = (size_t)kTileRows * (size_t)(ncol | 1) * sizeof(float);
  cudaError_t e = cudaFuncSetAttribute(seal_tiles_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  // xgboost src/data/data.cc: `!std::isinf(missing) && std::isinf(value)` invalidates the input
  seal_tiles_kernel<<<(unsigned)ntile, kTileRows, smem, s>>>(X, nrow, ncol, missing, std::isinf(missing) ? 0 : 1, Xt, flags);
  count_family(kSealTiles);
  return QC_LAUNCHED();
}

// =====================================================================================
// Walk on the 8-byte depth-ordered nodes
// =====================================================================================
// TEXMODE is a bit mask over the ILP trees in flight: tree j fetches its nodes through the texture pipe
// (tex1Dfetch on the same buffer) if bit j is set, through the LSU (LDG) otherwise.  ctree0: the first tree
// the constant table holds.
template <int ILP, bool HAS_MISSING, int TEXMODE = 0, int CTOP = 0>
__device__ __forceinline__ void walk_group(const uint2 *__restrict__ nodes, cudaTextureObject_t tex, const uint32_t *__restrict__ toff,
                                           const int32_t *__restrict__ tdepth, int t, int ctree0, uint32_t my_saddr,
                                           uint32_t (&idx)[ILP], uint32_t (&xbits)[ILP]) {
  int depth = 0, minleaf = 255;  // tdepth[] = deepest leaf | shallowest leaf << 8
  uint2 nd[ILP];
  uint32_t rel[ILP];
#pragma unroll
  for (int j = 0; j < ILP; ++j) {
    idx[j] = __ldg(toff + t + j);
    const int dd = __ldg(tdepth + t + j);
    depth = max(depth, dd & 0xFF);
    minleaf = min(minleaf, dd >> 8);
    nd[j] = make_uint2(0u, 0u);
    rel[j] = 1u;
  }
  // depth + 1 fetches per tree: the last one reads the leaf itself, whose x word is the leaf value.
  // A lane that has reached its leaf (rel == 0) parks: it stops fetching — it would otherwise re-read its
  // own leaf line at every remaining level, and at the deep levels those are up to 32 different
  // lines per warp request; the L1TEX data pipe is the bound of this kernel (DESIGN.md).  The
  // fetch is predicated, so nd[j] keeps the leaf node and no per-level copy of the value is needed.
  auto visit = [&](int j) {
    // shared address of skey[feat][tid] = my_saddr + feat * 1024: the top byte of the meta word
    // is feat * 4, so moving it to byte 1 (one PRMT) gives feat * 1024
    static_assert(kMetaFeatShift == 26, "address trick assumes feat in the top 6 bits");
    const uint32_t kv = lds_u32(my_saddr + __byte_perm(nd[j].y, 0u, 0x4434));
    rel[j] = nd[j].y & kMetaRelMask;
    if (HAS_MISSING && kv == kKeyMissing)  // default child: left = idx + rel, right = left + 1
      idx[j] += rel[j] + ((nd[j].y & kMetaDefaultLeftBit) ? 0u : (rel[j] != 0u ? 1u : 0u));
    else
      idx[j] = step_index(idx[j], rel[j], nd[j].x, kv);
  };
  if (CTOP > 0) {
    uint32_t cbase[ILP];  // index of this tree's table row minus its first node
#pragma unroll
    for (int j = 0; j < ILP; ++j) cbase[j] = ((uint32_t)(t + j - ctree0) << CTOP) - idx[j];
    if (minleaf >= CTOP) {
      // no leaf above level CTOP in any of these trees (the usual case for deep trees): every lane walks
      // all CTOP levels — no park predicate, no branches
#pragma unroll
      for (int d = 0; d < CTOP; ++d) {
#pragma unroll
        for (int j = 0; j < ILP; ++j) {
          nd[j] = c_top[cbase[j] + idx[j]];
          visit(j);
        }
      }
    } else {
#pragma unroll
      for (int d = 0; d < CTOP; ++d) {
        if (d <= depth) {
#pragma unroll
          for (int j = 0; j < ILP; ++j) {
            if (rel[j] != 0u) {
              nd[j] = c_top[cbase[j] + idx[j]];
              visit(j);
            }
            asm volatile("" : "+r"(rel[j]));
          }
        }
      }
    }
  }
  auto fetch = [&](int j) {
    if ((TEXMODE >> j) & 1)
      nd[j] = tex1Dfetch<uint2>(tex, (int)idx[j]);
    else
      nd[j] = __ldg(nodes + idx[j]);
  };
  for (int d = CTOP; d < depth; ++d) {
#pragma unroll
    for (int j = 0; j < ILP; ++j) {
      if (rel[j] != 0u) {
        fetch(j);
        visit(j);
      }
      // keep "still walking" in the rel register only (one ISETP per level instead of predicate shuffling)
      asm volatile("" : "+r"(rel[j]));
    }
  }
  // level `depth` holds only leaves: the last fetch reads the leaf a lane stands on — its value is all that is needed
  if (depth >= CTOP) {
#pragma unroll
    for (int j = 0; j < ILP; ++j)
      if (rel[j] != 0u) fetch(j);
  }
#pragma unroll
  for (int j = 0; j < ILP; ++j) xbits[j] = nd[j].x;
}

// all trees [t0, t1) on the 8-byte nodes, in tree order; emit(t, value bits, node index)
template <int ILP, bool HAS_MISSING, int TEXMODE, int CTOP, class Emit>
__device__ __forceinline__ void forest_walk(const DeviceForest &f, uint32_t my, int ctree0, int t0, int t1, Emit &&emit) {
  int t = t0;
  for (; t + ILP <= t1; t += ILP) {
    uint32_t idx[ILP], xb[ILP];
    walk_group<ILP, HAS_MISSING, TEXMODE, CTOP>(f.nodes, f.tex, f.tree_offset, f.tree_depth, t, ctree0, my, idx, xb);
#pragma unroll
    for (int j = 0; j < ILP; ++j) emit(t + j, xb[j], idx[j]);
  }
  for (; t < t1; ++t) {
    uint32_t idx[1], xb[1];
    walk_group<1, HAS_MISSING, 0, 0>(f.nodes, f.tex, f.tree_offset, f.tree_depth, t, 0, my, idx, xb);
    emit(t, xb[0], idx[0]);
  }
}

// =====================================================================================
// Walk on the two-level records (forest.hpp DuoForest)
// =====================================================================================
// Levels 0..3 come from constant memory as complete heap-ordered tops (entry i, children 2i and 2i + 1: no
// branch, no predicate); from level 4 on one 16-byte record {root, left, right thresholds; features; block
// pointer} decides two levels, and the four possible successors are contiguous.  Against the 8-byte nodes
// this halves the dependent gathers of a walk and takes ~40 % of the distinct lines per warp request off the
// L1TEX data pipes (tools/replay_two_level_records.py).
// HAS_MISSING: a missing entry (key 0xFFFFFFFF) takes the node's default child (bits 17..15 of w3 / bit 0 of a
// top entry's y word); the records carry those bits when DeviceForest::duo_has_dl.
template <int ILP, int TEXMODE, bool HAS_MISSING>
__device__ __forceinline__ void walk_group_duo(const uint4 *__restrict__ recs, cudaTextureObject_t tex4,
                                               const int32_t *__restrict__ tdepth, uint32_t blk_mul, int t, int ctree0, uint32_t my_saddr,
                                               uint32_t (&xbits)[ILP], uint32_t (&ids)[ILP]) {
  constexpr int CTOP = kDuoTop;
  int depth = CTOP - 1;  // at least one record (a shallower tree ends in the terminal records of its padded leaves)
  uint32_t idx[ILP];
#pragma unroll
  for (int j = 0; j < ILP; ++j) {
    depth = max(depth, __ldg(tdepth + t + j) & 0xFF);
    idx[j] = 1u;  // heap position in the complete top: children of i are 2i and 2i + 1
  }
  const int tl = t - ctree0;  // row of the constant tables
#pragma unroll
  for (int d = 0; d < CTOP; ++d) {
#pragma unroll
    for (int j = 0; j < ILP; ++j) {
      const uint2 nd = c_top[((uint32_t)(tl + j) << CTOP) + idx[j]];
      const uint32_t kv = lds_u32(my_saddr + __byte_perm(nd.y, 0u, 0x4434));
      if (HAS_MISSING) {
        uint32_t right = add_carry_out(nd.x, kv);
        if (kv == kKeyMissing) right = (nd.y & kTopDefaultLeftBit) ^ 1u;
        idx[j] = 2u * idx[j] + right;
      } else {
        idx[j] = step_index(idx[j], idx[j], nd.x, kv);  // 2i + right
      }
    }
  }
  uint4 r[ILP];
  uint32_t walking[ILP];
#pragma unroll
  for (int j = 0; j < ILP; ++j) {
    idx[j] += c_duo_base[tl + j] - (1u << CTOP);  // heap position 16..31 -> record index
    r[j] = make_uint4(0u, 0u, 0u, 0u);
    walking[j] = 1u;
  }
  // the terminal record of a leaf at depth D is rooted at depth D (D even) or D + 1 (D odd).  Only the
  // gather is predicated (a lane that has reached its terminal record stops fetching and keeps it); the
  // arithmetic below runs unconditionally, phase by phase across the ILP trees, so that the trees'
  // dependent chains interleave: on a terminal record (w3 == 0) it reads feature 0 and leaves walking at 0.
  auto gather = [&](int j) {
    if (walking[j] != 0u) {
      if ((TEXMODE >> j) & 1)
        r[j] = tex1Dfetch<uint4>(tex4, (int)idx[j]);
      else
        r[j] = __ldg(recs + idx[j]);
    }
  };
  // Records rooted at the deepest level a walk of these trees can reach (depth, or depth + 1 for an odd depth) are
  // all terminal: the last iteration is the gather alone — its arithmetic would only confirm w3 == 0.  For the
  // depth-18 booster that is one eighth of the record arithmetic and of its feature fetches; for a depth-6 forest half.
  int d = CTOP;
  for (; d + 2 <= depth + 1; d += 2) {
#pragma unroll
    for (int j = 0; j < ILP; ++j) gather(j);
    uint32_t kv0[ILP], kv[ILP], right1[ILP];
#pragma unroll
    for (int j = 0; j < ILP; ++j) {
      // skey[feat(root)][tid]: feat is the low 5 bits of w3; one AND + one multiply-add
      uint32_t sa;
      asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(sa) : "r"(r[j].w & 31u), "r"((uint32_t)(kStride * 4)), "r"(my_saddr));
      kv0[j] = lds_u32(sa);
    }
#pragma unroll
    for (int j = 0; j < ILP; ++j) {
      right1[j] = add_carry_out(r[j].x, kv0[j]);
      if (HAS_MISSING && kv0[j] == kKeyMissing) right1[j] = (r[j].w & kDuoDlRoot) ? 0u : 1u;
      // feat(left) sits at bits 14..10 — already feat * 1024 —, feat(right) at 9..5
      const uint32_t ms = right1[j] ? (r[j].w << 5) : r[j].w;
      kv[j] = lds_u32(my_saddr + (ms & (31u << 10)));
    }
#pragma unroll
    for (int j = 0; j < ILP; ++j) {
      const uint32_t xs = right1[j] ? r[j].z : r[j].y;
      // blk = w3 >> blk_shift as a multiply-high: the FMA pipe has room, the ALU pipe (SEL / LOP3 / IADD3) does not
      uint32_t blk;
      asm("mul.hi.u32 %0, %1, %2;" : "=r"(blk) : "r"(r[j].w), "r"(blk_mul));
      if (HAS_MISSING) {
        uint32_t right2 = add_carry_out(xs, kv[j]);
        // a leaf child compares the key-0 slot: never missing.  Default bit of the child that was taken.
        if (kv[j] == kKeyMissing) right2 = (r[j].w & (right1[j] ? kDuoDlRight : kDuoDlLeft)) ? 0u : 1u;
        const uint32_t half = 2u * blk + right1[j];
        idx[j] = c_duo_base[tl + j] + 2u * half + right2;
      } else {
        // next record = base + blk * 4 + 2 * right1 + right2
        // half = 2 * blk + right1, the carry of the root compare folded into a multiply-add (FMA pipe again)
        uint32_t half;
        asm("{\n\t.reg .u32 t;\n\tadd.cc.u32 t, %1, %2;\n\tmadc.lo.u32 %0, %3, 2, 0;\n\t}" : "=r"(half) : "r"(r[j].x), "r"(kv0[j]), "r"(blk));
        idx[j] = step_index(c_duo_base[tl + j] + half, half, xs, kv[j]);
      }
      walking[j] = blk;  // 0: this was a terminal record, r[j].x is the leaf value
      asm volatile("" : "+r"(walking[j]));
    }
  }
#pragma unroll
  for (int j = 0; j < ILP; ++j) gather(j);
#pragma unroll
  for (int j = 0; j < ILP; ++j) xbits[j] = r[j].x, ids[j] = r[j].y;
}

// all trees [t0, t1) on the two-level records: ILP-wide groups, then half-width groups (one LSU tree, the rest on
// the texture pipe), then one by one — always in tree order (float32 sum order is part of parity).
// emit(t, leaf value bits, XGBoost node id of the leaf)
template <int ILP, int TEXMODE, bool HAS_MISSING, class Emit>
__device__ __forceinline__ void forest_walk_duo(const DeviceForest &f, uint32_t my, int ctree0, int t0, int t1, Emit &&emit) {
  int t = t0;
  for (; t + ILP <= t1; t += ILP) {
    uint32_t xb[ILP], id[ILP];
    walk_group_duo<ILP, TEXMODE, HAS_MISSING>(f.recs, f.tex4, f.tree_depth, f.duo_blk_mul, t, ctree0, my, xb, id);
#pragma unroll
    for (int j = 0; j < ILP; ++j) emit(t + j, xb[j], id[j]);
  }
  constexpr int H = ILP / 2;
  if (H >= 2) {
    for (; t + H <= t1; t += H) {
      uint32_t xb[H > 0 ? H : 1], id[H > 0 ? H : 1];
      walk_group_duo<(H > 0 ? H : 1), ((1 << H) - 2), HAS_MISSING>(f.recs, f.tex4, f.tree_depth, f.duo_blk_mul, t, ctree0, my, xb, id);
#pragma unroll
      for (int j = 0; j < H; ++j) emit(t + j, xb[j], id[j]);
    }
  }
  for (; t < t1; ++t) {
    uint32_t xb[1], id[1];
    walk_group_duo<1, 0, HAS_MISSING>(f.recs, f.tex4, f.tree_depth, f.duo_blk_mul, t, ctree0, my, xb, id);
    emit(t, xb[0], id[0]);
  }
}

// ---- walk policies: which walk a launch runs, and its launch shape ------------------------------------------
// run<HAS_MISSING, PRED_LEAF>(f, my, ctree0, t0, t1, emit) walks trees [t0, t1) of one row in tree order and calls
// emit(t, leaf value bits, XGBoost node id of the leaf); the node id is looked up only when PRED_LEAF.
// walks_missing(f): whether a row with missing entries may take this walk.
template <int ILP, int TEXMASK, int MINB>
struct DuoWalk {
  static constexpr int kMinBlocks = MINB, kFamily = kDuo;
  __device__ static bool walks_missing(const DeviceForest &f) { return f.duo_has_dl != 0; }
  template <bool HAS_MISSING, bool PRED_LEAF, class Emit>
  __device__ __forceinline__ static void run(const DeviceForest &f, uint32_t my, int ctree0, int t0, int t1, Emit &&emit) {
    forest_walk_duo<ILP, TEXMASK, HAS_MISSING>(f, my, ctree0, t0, t1, emit);
  }
};
template <int ILP, int TEXMASK, int CTOP, int MINB>
struct NodesWalk {
  static constexpr int kMinBlocks = MINB, kFamily = kNodes8;
  __device__ static bool walks_missing(const DeviceForest &) { return true; }
  template <bool HAS_MISSING, bool PRED_LEAF, class Emit>
  __device__ __forceinline__ static void run(const DeviceForest &f, uint32_t my, int ctree0, int t0, int t1, Emit &&emit) {
    forest_walk<ILP, HAS_MISSING, TEXMASK, CTOP>(f, my, ctree0, t0, t1, [&](int t, uint32_t xb, uint32_t idx) {
      emit(t, xb, PRED_LEAF ? (uint32_t)__ldg(f.orig_id + idx) : 0u);
    });
  }
};

// The launch shapes (B200; measurements in profiles/README.md):
//   two-level records, default ("two-level records"): 6 trees in flight, 4 of them (mask 0x36) gathering through the
//     texture pipe, 5 resident CTAs per SM — LSU and TEX data pipes, ALU and issue slots all end up at 76-86 % busy
//   two-level records, shallow (kernels.hpp kShallowRecBytesPerTree): 4 trees in flight, 6 resident CTAs
//   8-byte nodes: 4 trees in flight, 6 resident CTAs; levels 0..3 of every tree from constant memory when the table
//     holds them; below that trees 1 and 3 of each group fetch their nodes through the texture pipe and trees 0 and 2
//     through the LSU (mask 0xA), or all through the LSU when the booster has no node texture
using RecordsWalk = DuoWalk<6, 0x36, 5>;
using RecordsShallowWalk = DuoWalk<4, 0xA, 6>;
using NodesTableWalk = NodesWalk<4, 0xA, kDuoTop, 6>;
using NodesTexWalk = NodesWalk<4, 0xA, 0, 6>;
using NodesLsuWalk = NodesWalk<4, 0, 0, 6>;

__device__ __forceinline__ float export_transform(float acc, int exp10_on, float scale) {
  if (!exp10_on) return acc;
  // OH_ML = 10.0 ** pred (OH_GridCompMod.F90:369), then OH_ML * OHscale (:1569): two float32
  // roundings.  10**x is evaluated in float64 and rounded once (SURVEY.md hard part 7).
  const float p = (float)exp10((double)acc);
  return __fmul_rn(p, scale);
}

// what a row does with its leaves: float32 sum in tree order (+ export transform on the last launch of a
// chunked forest), or the leaf's XGBoost node id per tree (option_mask = 2)
template <bool PRED_LEAF, class Walk>
__device__ __forceinline__ void row_result(const DeviceForest &f, const PredictArgs &a, uint64_t row, bool live, Walk &&walk) {
  if (PRED_LEAF) {
    float *o = a.out + row * (uint64_t)a.out_stride;
    walk([&](int t, uint32_t, uint32_t id) {
      if (live) o[t] = (float)id;
    });
  } else {
    float acc = f.base_score;
    if (!a.first && live) acc = a.out[row];
    walk([&](int, uint32_t xb, uint32_t) { acc = __fadd_rn(acc, __uint_as_float(xb)); });
    if (live) a.out[row] = a.last ? export_transform(acc, a.exp10, a.scale) : acc;
  }
}

// A launch on a matrix with missing entries reads the tile's row order (kernels.hpp): thread tid walks the row at
// position tid — clean rows first — and a warp whose 32 rows are all clean takes the walk without the
// default-direction test.  Returns the row's index in the matrix; `hm` = this warp needs the test.
template <bool HAS_MISSING>
__device__ __forceinline__ uint64_t tile_row(uint32_t buf, uint64_t tile, int tid, bool absent_columns, bool &hm) {
  uint32_t orig = (uint32_t)tid;
  hm = false;
  if (HAS_MISSING) {
    const uint32_t p = lds_u32(buf + 4u * (uint32_t)tid);
    orig = p & 0xFFu;
    hm = __any_sync(0xffffffffu, (p >> 8) & 1u) || absent_columns;
  }
  return tile * kTileRows + orig;
}

template <class Walk, bool HAS_MISSING, bool PRED_LEAF>
__global__ void __launch_bounds__(kBlock, Walk::kMinBlocks) predict_tiles_kernel(DeviceForest f, PredictArgs a) {
  extern __shared__ __align__(128) uint32_t skey[];
  __shared__ __align__(8) unsigned long long bars[1];
  const int tid = threadIdx.x;
  TilePipe pipe;
  pipe.begin(skey, bars, a, f.nfeat, HAS_MISSING, tid);
  while (pipe.more()) {
    const uint32_t buf = pipe.acquire(tid);
    const uint32_t my = buf + 4u * (uint32_t)(kStride + tid);
    bool hm;
    const uint64_t row = tile_row<HAS_MISSING>(buf, pipe.tile, tid, a.ncol < f.nfeat, hm);
    row_result<PRED_LEAF>(f, a, row, row < a.nrow, [&](auto &&emit) {
      if (HAS_MISSING && hm)
        Walk::template run<true, PRED_LEAF>(f, my, a.ctree0, a.tree_begin, a.tree_end, emit);
      else
        Walk::template run<false, PRED_LEAF>(f, my, a.ctree0, a.tree_begin, a.tree_end, emit);
    });
    pipe.release(tid);
  }
}

// Feature ft of cell e in column c, as predict_OH_with_XGB packs it (:303-345): what the fused predict puts in its
// tiles and oh_pack_kernel in the matrix.
__device__ __forceinline__ float run1_feature(const Run1Features &x, int ft, size_t e, int c, int ncol) {
  if (ft == 1)  // PL_BST = (PLE(k-1) + PLE(k)) * 0.5 (:1488), / 100.0 as a true divide (:314)
    return __fdiv_rn(__fmul_rn(__fadd_rn(__ldg(x.ple + e), __ldg(x.ple + e + ncol)), 0.5f), 100.0f);
  return x.src3[ft] ? __ldg(x.src3[ft] + e) : __ldg(x.src2[ft] + c);
}

// ---- fused Run1 variant: the tile is assembled straight from the SoA feature fields ------------------
// (OH_GridCompMod.F90:303-345 pack + :347 create + :356 predict + :369,:1569 transform in one kernel).
// Row m of the slab is cell e = e0 + m; per feature the CTA's 256 cells are contiguous in the source
// field, so every load is coalesced and lands directly in the transposed tile — the [N x 27] matrix is
// never formed, and no transposition is needed.  Whether a tile holds missing entries is decided per
// tile (block-wide OR) and selects the walk specialisation at run time; +-inf raises the error flag.
// Walk serves the tiles, and the tiles with missing entries too when it walks_missing(); MissingWalk serves those
// otherwise (the two-level records without the default bits).
template <class Walk, class MissingWalk>
__global__ void __launch_bounds__(kBlock, Walk::kMinBlocks) predict_soa_kernel(DeviceForest f, SoaArgs a) {
  extern __shared__ __align__(128) uint32_t skey[];
  const int tid = threadIdx.x;
  constexpr int B = kBlock;
  const uint64_t m = (uint64_t)blockIdx.x * B + tid;
  const bool live = m < a.nrow;
  int flags = 0;
  if (live) {
    const size_t e = a.e0 + m;
    const int c = (int)(m % (uint64_t)a.ncol);
    const bool chk_inf = !isinf(a.missing);
#pragma unroll
    for (int ft = 0; ft < 27; ++ft) {
      const float x = run1_feature(a.feat, ft, e, c, a.ncol);
      uint32_t k = float_key(x);
      if (x != x || x == a.missing) k = kKeyMissing, flags |= 1;
      if (chk_inf && isinf(x)) flags |= 2;
      skey[ft * kStride + tid] = k;
    }
  } else {
#pragma unroll
    for (int ft = 0; ft < 27; ++ft) skey[ft * kStride + tid] = 0u;
  }
  skey[27 * kStride + tid] = 0u;  // the slot leaves point at (nfeat == 27 is checked by the host)
  // __syncthreads_or returns a truth value, not the bitwise OR: one vote per flag
  const bool tile_missing = __syncthreads_or(flags & 1) != 0;
  if (__syncthreads_or(flags & 2) != 0) {
    if (tid == 0) atomicOr(a.flags, 2);
  }
  if (!live) return;
  const uint32_t my = (uint32_t)__cvta_generic_to_shared(skey + tid);
  float acc = f.base_score;
  auto add = [&](int, uint32_t xb, uint32_t) { acc = __fadd_rn(acc, __uint_as_float(xb)); };
  if (!tile_missing || Walk::walks_missing(f)) {
    if (tile_missing)
      Walk::template run<true, false>(f, my, a.ctree0, 0, a.ntree_used, add);
    else
      Walk::template run<false, false>(f, my, a.ctree0, 0, a.ntree_used, add);
  } else {
    MissingWalk::template run<true, false>(f, my, a.ctree0, 0, a.ntree_used, add);
  }
  if (a.pred) a.pred[m] = acc;
  a.out[m] = export_transform(acc, a.exp10, a.scale);
}

// ---- inplace variant: the tile is assembled straight from a caller's dense float array ------------------------
// (XGBoosterPredictFromDense / XGBoosterPredictFromCudaArray).  The same tile as predict_tiles_kernel walks — feature
// slots of 1 KB, absent columns missing, the key-0 slot last — built in shared memory from the strided array, so no
// copy of the array and no key tiles go to HBM.  Rows keep their order: a warp takes the default-direction walk when
// one of its 32 rows holds a missing entry, and MissingWalk serves it when Walk cannot walk missing entries.  Ranges
// of trees are separate launches (the partial sum travels through `out` as in predict_tiles_kernel); each one
// reassembles the tile.
template <class Walk, class MissingWalk>
__global__ void __launch_bounds__(kBlock, Walk::kMinBlocks) predict_dense_kernel(DeviceForest f, PredictArgs a, DenseArgs d) {
  extern __shared__ __align__(128) uint32_t skey[];
  const int tid = threadIdx.x, ncol = a.ncol;
  const uint64_t r0 = (uint64_t)blockIdx.x * kBlock;
  const uint64_t left = a.nrow - r0;
  const int nr = left < (uint64_t)kBlock ? (int)left : kBlock;
  const bool live = tid < nr;
  const bool chk_inf = !isinf(d.missing);
  int flags = 0;
  auto key = [&](float x) {
    if (chk_inf && isinf(x)) flags |= 2;
    if (x != x || x == d.missing) {
      flags |= 1;
      return kKeyMissing;
    }
    return float_key(x);
  };
  if (d.col_stride == 1 && d.row_stride == ncol) {
    // contiguous rows: one flat coalesced copy into a row-major staging area of odd stride (conflict-free per-thread
    // row reads, as in seal_tiles_kernel) that aliases the key slots; each thread lifts its row through registers
    float *stage = reinterpret_cast<float *>(skey);
    const int ld = ncol | 1, n = nr * ncol;
    const float *__restrict__ src = d.X + r0 * (uint64_t)ncol;
    if (ld == ncol && (((uintptr_t)src) & 15u) == 0u) {
      const float4 *s4 = reinterpret_cast<const float4 *>(src);
      float4 *d4 = reinterpret_cast<float4 *>(stage);
      for (int i = tid; i < (n >> 2); i += kBlock) d4[i] = __ldg(s4 + i);
      for (int i = (n & ~3) + tid; i < n; i += kBlock) stage[i] = __ldg(src + i);
    } else if (ld == ncol) {
      for (int i = tid; i < n; i += kBlock) stage[i] = __ldg(src + i);
    } else {
      for (int i = tid; i < n; i += kBlock) stage[(i / ncol) * ld + (i % ncol)] = __ldg(src + i);
    }
    __syncthreads();
    uint32_t k[kMaxFeatures];
#pragma unroll
    for (int c = 0; c < (int)kMaxFeatures; ++c)
      if (c < ncol) k[c] = live ? key(stage[tid * ld + c]) : 0u;
    __syncthreads();
#pragma unroll
    for (int c = 0; c < (int)kMaxFeatures; ++c)
      if (c < ncol) skey[c * kStride + tid] = k[c];
  } else {
    // any other strides: element by element; a feature-major array is coalesced per feature
    const float *__restrict__ src = d.X + (r0 + (uint64_t)tid) * d.row_stride;
    for (int c = 0; c < ncol; ++c) skey[c * kStride + tid] = live ? key(__ldg(src + (int64_t)c * d.col_stride)) : 0u;
  }
  for (int c = ncol; c < f.nfeat; ++c) skey[c * kStride + tid] = kKeyMissing;
  skey[f.nfeat * kStride + tid] = 0u;
  // __syncthreads_or returns a truth value, not the bitwise OR: one vote for the inf flag
  if (__syncthreads_or(flags & 2) != 0) {
    if (tid == 0) atomicOr(d.flags, 2);
  }
  const bool hm = __any_sync(0xffffffffu, flags & 1) || ncol < f.nfeat;
  if (!live) return;
  const uint32_t my = (uint32_t)__cvta_generic_to_shared(skey + tid);
  row_result<false>(f, a, r0 + (uint64_t)tid, true, [&](auto &&emit) {
    if (!hm)
      Walk::template run<false, false>(f, my, a.ctree0, a.tree_begin, a.tree_end, emit);
    else if (Walk::walks_missing(f))
      Walk::template run<true, false>(f, my, a.ctree0, a.tree_begin, a.tree_end, emit);
    else
      MissingWalk::template run<true, false>(f, my, a.ctree0, a.tree_begin, a.tree_end, emit);
  });
}

// The layout rule of the predict launches: the two-level records when the window holds the record tops of trees
// [t0, t1) and the rows have no missing entries or the records carry the default bits; otherwise the 8-byte nodes,
// with the table when the window holds their node tops, and through the LSU alone when there is no node texture.
enum class Layout { kRecords, kNodesTable, kNodesTex, kNodesLsu };
static Layout layout(const DeviceForest &f, const ConstWindow &w, int t0, int t1, bool has_missing) {
  if (w.holds(TopLayout::kRecordTops, t0, t1) && (!has_missing || f.duo_has_dl)) return Layout::kRecords;
  if (f.tex == 0) return Layout::kNodesLsu;
  return w.holds(TopLayout::kNodeTops, t0, t1) ? Layout::kNodesTable : Layout::kNodesTex;
}

cudaError_t launch_predict_soa(const DeviceForest &f, const ConstWindow &w, const SoaArgs &args, cudaStream_t s) {
  if (args.nrow == 0) return cudaSuccess;
  if (f.nfeat != 27) return cudaErrorInvalidValue;
  const size_t smem = (size_t)kStride * 28 * sizeof(float);
  const uint64_t nblk = (args.nrow + kBlock - 1) / kBlock;
  if (nblk > 0x7fffffffull) return cudaErrorInvalidConfiguration;
  SoaArgs a = args;
  a.ctree0 = w.tree0;
  // whether a tile has missing entries is known only in the kernel: the layout is that of clean rows, and the
  // kernel sends a tile with missing entries the records cannot walk to the 8-byte nodes without the table
  const Layout l = layout(f, w, 0, a.ntree_used, false);
  auto k = predict_soa_kernel<RecordsWalk, NodesTexWalk>;
  if (l == Layout::kNodesTable) k = predict_soa_kernel<NodesTableWalk, NodesTableWalk>;
  if (l == Layout::kNodesTex) k = predict_soa_kernel<NodesTexWalk, NodesTexWalk>;
  if (l == Layout::kNodesLsu) k = predict_soa_kernel<NodesLsuWalk, NodesLsuWalk>;
  cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  k<<<dim3((unsigned)nblk), kBlock, smem, s>>>(f, a);
  count_family(l == Layout::kRecords ? kSoaDuo : kSoaNodes8);
  return QC_LAUNCHED();
}

cudaError_t launch_predict_dense(const DeviceForest &f, const ConstWindow &w, const PredictArgs &args, const DenseArgs &d, cudaStream_t s) {
  if (args.nrow == 0 || args.tree_end <= args.tree_begin) return cudaSuccess;
  if (args.ncol > f.nfeat || f.nfeat > (int)kMaxFeatures || args.pred_leaf) return cudaErrorInvalidValue;
  // the key slots 0..nfeat; the row-major staging area of the contiguous loader ((ncol | 1) KB) fits in them
  const size_t smem = (size_t)kStride * (size_t)(f.nfeat + 1) * sizeof(uint32_t);
  const uint64_t grid = tile_count(args.nrow);
  if (grid > 0x7fffffffull) return cudaErrorInvalidConfiguration;
  PredictArgs a = args;
  a.ctree0 = w.tree0;
  // as in launch_predict_soa: the layout of clean rows; the kernel sends a warp with missing entries the records cannot
  // walk to the 8-byte nodes without the table
  const Layout l = layout(f, w, a.tree_begin, a.tree_end, false);
  auto k = predict_dense_kernel<RecordsWalk, NodesTexWalk>;
  if (f.duo_shallow) k = predict_dense_kernel<RecordsShallowWalk, NodesTexWalk>;
  if (l == Layout::kNodesTable) k = predict_dense_kernel<NodesTableWalk, NodesTableWalk>;
  if (l == Layout::kNodesTex) k = predict_dense_kernel<NodesTexWalk, NodesTexWalk>;
  if (l == Layout::kNodesLsu) k = predict_dense_kernel<NodesLsuWalk, NodesLsuWalk>;
  cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  k<<<dim3((unsigned)grid), kBlock, smem, s>>>(f, a, d);
  count_predict(l == Layout::kRecords ? kDenseDuo : kDenseNodes8);
  return QC_LAUNCHED();
}

// ---- launches ------------------------------------------------------------------------------------------
static thread_local int g_sm_count = 0;
static int sm_count() {
  if (g_sm_count == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&g_sm_count, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || g_sm_count <= 0) g_sm_count = 148;
  }
  return g_sm_count;
}

// one CTA per tile
template <class K>
static cudaError_t launch_tiles(K k, const DeviceForest &f, const PredictArgs &a, cudaStream_t s) {
  const size_t smem = (size_t)kStride * (size_t)(f.nfeat + 2) * sizeof(uint32_t);
  const uint64_t grid = tile_count(a.nrow);
  if (grid > 0x7fffffffull) return cudaErrorInvalidConfiguration;
  cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  k<<<dim3((unsigned)grid), kBlock, smem, s>>>(f, a);
  return QC_LAUNCHED();
}

// HM / PL chosen at run time
template <class Walk>
static cudaError_t launch_walk(const DeviceForest &f, const PredictArgs &a, cudaStream_t s) {
  const bool hm = a.has_missing != 0, pl = a.pred_leaf != 0;
  count_predict(Walk::kFamily + hm + 2 * pl);
  if (hm && pl) return launch_tiles(predict_tiles_kernel<Walk, true, true>, f, a, s);
  if (hm) return launch_tiles(predict_tiles_kernel<Walk, true, false>, f, a, s);
  if (pl) return launch_tiles(predict_tiles_kernel<Walk, false, true>, f, a, s);
  return launch_tiles(predict_tiles_kernel<Walk, false, false>, f, a, s);
}

cudaError_t launch_predict(const DeviceForest &f, const ConstWindow &w, const PredictArgs &args, cudaStream_t s) {
  if (args.nrow == 0 || args.tree_end <= args.tree_begin) return cudaSuccess;
  if (args.ncol > f.nfeat || f.nfeat > (int)kMaxFeatures) return cudaErrorInvalidValue;
  PredictArgs a = args;
  a.ctree0 = w.tree0;
  switch (layout(f, w, a.tree_begin, a.tree_end, a.has_missing != 0)) {
    case Layout::kRecords: return f.duo_shallow ? launch_walk<RecordsShallowWalk>(f, a, s) : launch_walk<RecordsWalk>(f, a, s);
    case Layout::kNodesTable: return launch_walk<NodesTableWalk>(f, a, s);
    case Layout::kNodesTex: return launch_walk<NodesTexWalk>(f, a, s);
    case Layout::kNodesLsu: break;
  }
  return launch_walk<NodesLsuWalk>(f, a, s);
}

// =====================================================================================
// K6 — per-feature contributions (libxgboost 1.6.0 cpu_predictor PredictContribution)
// =====================================================================================
// Exact: path-dependent TreeSHAP in the path-parallel form of GPUTreeShap (Mitchell, Frank, Holmes 2022).  A
// path's elements sit on consecutive lanes of a 32-lane bin (forest.hpp ShapForest); for one row a lane evaluates
// its element's one fraction (one key range test, or the missing flag), the lanes of a path run ExtendPath with
// shuffles, then every lane unwinds its own element (UnwoundPathSum) and adds w * (one - zero) * leaf to its
// feature.  float64 throughout; a row's sum over the bins of one slice is a float64 in shared memory.
//   grid = (tiles, slices): a CTA takes one 256-row key tile (TMA, like the predict kernels) and one slice of the
//   bins; each warp owns 32 tile positions and walks the slice's bins in order, row by row.  Paths of one bin add
//   into a row's accumulator group by group, so the float64 sums have a fixed order.
constexpr unsigned kFull = 0xffffffffu;

__device__ __forceinline__ int shap_region_words(int nf) {
  const int ast = nf | 1;
  return max(2 * kTileRows * ast, kTileRows * (nf + 2));
}

__global__ void __launch_bounds__(kTileRows, 2) shap_paths_kernel(const uint4 *__restrict__ bins, int64_t nbins, int nslices,
                                                                  ContribArgs a, double *__restrict__ part) {
  extern __shared__ __align__(128) uint32_t smem[];
  __shared__ __align__(8) unsigned long long bars[1];
  __shared__ double s_inv[34];  // 1 / k
  const int nf = a.nfeat, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int ast = nf | 1, kst = nf | 1;  // odd row strides: the lanes of a warp read / add distinct features of one row
  double *acc = reinterpret_cast<double *>(smem);    // [256][ast] by tile position; the TMA buffer aliases its start
  uint32_t *keys = smem + shap_region_words(nf);     // [256][kst] keys by tile position
  uint32_t *order = keys + kTileRows * kst;          // [256] the tile's row order
  PredictArgs pa;
  pa.Xt = a.Xt, pa.nrow = a.nrow, pa.ncol = a.ncol;
  TilePipe pipe;
  pipe.begin(smem, bars, pa, nf, true, tid);
  if (tid < 34) s_inv[tid] = tid ? 1.0 / (double)tid : 0.0;
  (void)pipe.acquire(tid);
  order[tid] = smem[tid];
  for (int c = 0; c < nf; ++c) keys[tid * kst + c] = smem[(1 + c) * kStride + tid];
  __syncthreads();
  for (int i = tid; i < kTileRows * ast; i += kTileRows) acc[i] = 0.0;
  __syncthreads();
  const uint64_t tile = blockIdx.x;
  const int64_t b0 = nbins * (int64_t)blockIdx.y / nslices, b1 = nbins * (int64_t)(blockIdx.y + 1) / nslices;
  for (int64_t b = b0; b < b1; ++b) {
    const uint4 e = __ldg(bins + b * 32 + lane);
    const uint32_t feat = e.z & 0xFFu, g0 = (e.z >> 16) & 31u, len = e.z >> 24;
    const int j = lane - (int)g0, D = (int)len - 1;  // my place in my path, and the path's unique depth
    const bool elem = feat != kShapNoFeature && j >= 1;
    const bool miss_here = (e.z >> 8) & 1u;
    const float zf = __uint_as_float(e.w);
    const double z = elem ? (double)zf : 1.0;
    const double v = (double)__shfl_sync(kFull, zf, (int)g0);  // leaf value, from the path's bias lane
    const int maxlen = (int)__reduce_max_sync(kFull, len);
    const double invz = 1.0 / z, d1 = (double)(D + 1), inv_d1 = s_inv[D + 1 > 0 ? D + 1 : 0];
    const unsigned starts = __ballot_sync(kFull, len > 0 && j == 0);
    const int ngroups = __popc(starts), my_group = __popc(starts & ((1u << g0) - 1u));
    for (int r = warp * 32; r < warp * 32 + 32; ++r) {
      const uint32_t orig = order[r] & 0xFFu;
      if (tile * kTileRows + orig >= a.nrow) continue;  // warp-uniform
      bool one = true;
      if (elem) {
        const uint32_t k = keys[r * kst + feat];
        one = k == kKeyMissing ? miss_here : (e.x <= k && k < e.y);
      }
      const float zo = one ? zf : -zf;  // (one, zero) of my element in one word: zero fractions are > 0
      // ExtendPath, element by element: pw[j] <- zero_i * pw[j] * (i - j) / (i + 1) + one_i * pw[j - 1] * j / (i + 1)
      double pw = j == 0 ? 1.0 : 0.0;
      for (int i = 1; i < maxlen; ++i) {
        const float zi = __shfl_sync(kFull, zo, (int)(g0 + i) & 31);
        const double left = __shfl_up_sync(kFull, pw, 1);
        if (i <= D) {
          const double inv = s_inv[i + 1];
          pw = (double)fabsf(zi) * pw * (double)max(i - j, 0) * inv + (zi > 0.f ? left : 0.0) * (double)j * inv;
        }
      }
      // UnwoundPathSum of my element
      double next = __shfl_sync(kFull, pw, (int)(g0 + (D > 0 ? D : 0)) & 31), total = 0.0;
      for (int i = maxlen - 2; i >= 0; --i) {
        const double pwi = __shfl_sync(kFull, pw, (int)(g0 + min(i, D > 0 ? D : 0)) & 31);
        if (i < D) {
          if (one) {
            const double tmp = next * d1 * s_inv[i + 1];
            total += tmp;
            next = pwi - tmp * z * (double)(D - i) * inv_d1;
          } else {
            total += pwi * invz * d1 * s_inv[D - i];
          }
        }
      }
      const double c = total * ((one ? 1.0 : 0.0) - z) * v;
      double *arow = acc + r * ast;
      for (int g = 0; g < ngroups; ++g) {  // paths of the bin in order: a feature may recur across paths
        if (elem && my_group == g) arow[feat] += c;
        __syncwarp();
      }
    }
  }
  __syncthreads();
  for (int i = tid; i < kTileRows * nf; i += kTileRows) {
    const int p = i / nf, f = i - p * nf;
    const uint64_t row = tile * kTileRows + (order[p] & 0xFFu);
    if (row < a.nrow) part[((uint64_t)blockIdx.y * a.nrow + row) * (uint64_t)nf + f] = acc[p * ast + f];
  }
}

__global__ void __launch_bounds__(256) shap_reduce_kernel(const double *__restrict__ part, int nslices, ContribArgs a) {
  const int nf = a.nfeat;
  const uint64_t n = a.nrow * (uint64_t)(nf + 1), stride = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const uint64_t row = i / (uint64_t)(nf + 1);
    const int f = (int)(i - row * (uint64_t)(nf + 1));
    float v = a.bias;
    if (f < nf) {
      double s = 0.0;
      for (int k = 0; k < nslices; ++k) s += part[((uint64_t)k * a.nrow + row) * (uint64_t)nf + f];
      v = (float)s;
    }
    a.out[i] = v;
  }
}

// dynamic shared memory of shap_paths_kernel and shap_inter_kernel: shap_region_words, then keys and row order
static size_t shap_smem_bytes(int nf) {
  const int kst = nf | 1, ast = nf | 1;
  return 4 * ((size_t)std::max(2 * kTileRows * ast, kTileRows * (nf + 2)) + (size_t)kTileRows * kst + kTileRows);
}

cudaError_t launch_shap(const uint4 *bins, int64_t nbins, int nslices, const ContribArgs &a, double *part, cudaStream_t s) {
  if (a.nrow == 0 || nbins <= 0 || nslices <= 0) return cudaSuccess;
  if (a.nrow > kShapChunkRows || a.ncol > a.nfeat || a.nfeat > (int)kMaxFeatures) return cudaErrorInvalidValue;
  const size_t smem = shap_smem_bytes(a.nfeat);
  cudaError_t e = cudaFuncSetAttribute(shap_paths_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  shap_paths_kernel<<<dim3((unsigned)tile_count(a.nrow), (unsigned)nslices), kTileRows, smem, s>>>(bins, nbins, nslices, a, part);
  count_predict(kShap);
  return QC_LAUNCHED();
}

cudaError_t launch_shap_reduce(const double *part, int nslices, const ContribArgs &a, cudaStream_t s) {
  if (a.nrow == 0) return cudaSuccess;
  const uint64_t n = a.nrow * (uint64_t)(a.nfeat + 1);
  const int blocks = (int)std::min<uint64_t>((n + 255) / 256, (uint64_t)sm_count() * 16);
  shap_reduce_kernel<<<blocks, 256, 0, s>>>(part, nslices, a);
  count_family(kShapReduce);
  return QC_LAUNCHED();
}

// Approximate (Saabas): one thread per row walks each tree on the 8-byte nodes and adds mean(next) - mean(node) to
// the split feature — float32, in libxgboost's order: a per-tree vector (tp, only the features the path touched,
// tracked in a bit mask) is added into the row's accumulator after every tree.  Both are feature-major [f][row]
// in shared memory: thread t always hits bank t % 32, like skey.
__global__ void __launch_bounds__(kBlock, 2) shap_approx_kernel(DeviceForest f, const float *__restrict__ mean, int ntree, ContribArgs a) {
  extern __shared__ __align__(128) uint32_t skey[];
  __shared__ __align__(8) unsigned long long bars[1];
  const int tid = threadIdx.x, nf = a.nfeat;
  float *acc = reinterpret_cast<float *>(skey + (nf + 2) * kStride);  // [nf][256]
  float *tp = acc + nf * kStride;                                     // [nf][256]
  PredictArgs pa;
  pa.Xt = a.Xt, pa.nrow = a.nrow, pa.ncol = a.ncol;
  TilePipe pipe;
  pipe.begin(skey, bars, pa, nf, true, tid);
  for (int c = 0; c < nf; ++c) acc[c * kStride + tid] = 0.f;
  const uint32_t buf = pipe.acquire(tid);
  const uint32_t my = buf + 4u * (uint32_t)(kStride + tid);
  const uint64_t row = pipe.tile * kTileRows + (lds_u32(buf + 4u * (uint32_t)tid) & 0xFFu);
  if (row >= a.nrow) return;
  for (int t = 0; t < ntree; ++t) {
    uint32_t idx = __ldg(f.tree_offset + t);
    uint2 nd = __ldg(f.nodes + idx);
    float node_value = __ldg(mean + idx);
    uint32_t mask = 0u, last = 0u, rel = nd.y & kMetaRelMask;
    while (rel != 0u) {
      const uint32_t ft = nd.y >> kMetaFeatShift;
      const uint32_t kv = lds_u32(my + ft * 1024u);
      if (kv == kKeyMissing)
        idx += rel + ((nd.y & kMetaDefaultLeftBit) ? 0u : 1u);
      else
        idx = step_index(idx, rel, nd.x, kv);
      const float nv = __ldg(mean + idx);
      float *p = tp + ft * kStride + tid;
      *p = __fadd_rn((mask >> ft) & 1u ? *p : 0.f, __fsub_rn(nv, node_value));
      mask |= 1u << ft, last = ft, node_value = nv;
      nd = __ldg(f.nodes + idx);
      rel = nd.y & kMetaRelMask;
    }
    if (mask) {
      float *p = tp + last * kStride + tid;
      *p = __fadd_rn(*p, __fsub_rn(__uint_as_float(nd.x), node_value));  // leaf - mean(leaf): libxgboost adds it too
      while (mask) {
        const int c = __ffs(mask) - 1;
        mask &= mask - 1u;
        acc[c * kStride + tid] = __fadd_rn(acc[c * kStride + tid], tp[c * kStride + tid]);
      }
    }
  }
  float *o = a.out + row * (uint64_t)(nf + 1);
  for (int c = 0; c < nf; ++c) o[c] = acc[c * kStride + tid];
  o[nf] = a.bias;
}

cudaError_t launch_shap_approx(const DeviceForest &f, const float *mean, int ntree, const ContribArgs &a, cudaStream_t s) {
  if (a.nrow == 0) return cudaSuccess;
  if (a.ncol > a.nfeat || a.nfeat != f.nfeat || a.nfeat > (int)kMaxFeatures) return cudaErrorInvalidValue;
  const uint64_t ntile = tile_count(a.nrow);
  if (ntile > 0x7fffffffull) return cudaErrorInvalidConfiguration;
  const size_t smem = (size_t)kStride * 4 * (size_t)(a.nfeat + 2 + 2 * a.nfeat);
  cudaError_t e = cudaFuncSetAttribute(shap_approx_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  shap_approx_kernel<<<(unsigned)ntile, kBlock, smem, s>>>(f, mean, ntree, a);
  count_predict(kShapApprox);
  return QC_LAUNCHED();
}

// SHAP interaction values (libxgboost 1.6.0 PredictInteractionContributions).  libxgboost runs TreeShap conditioned
// on feature c: c is never extended into the unique path, and at c's splits the cold branch gets condition fraction
// 0 (c on) or each branch its cover ratio (c off).  On a path P with leaf v, where c's merged element has the one
// fraction o_c and the zero fraction z_c, (on - off) / 2 adds to M[c][f_i], for every other element i,
//     1/2 (o_c - z_c) W_i(P \ c) (o_i - z_i) v
// with W_i(P \ c) the UnwoundPathSum of i in P extended without c (unique depth D - 1).  shap_inter_kernel is
// shap_paths_kernel over the bins of c's list, with c's lane left out: the lanes of the path without c are addressed
// through lane_of(p), so nothing is divided by o_c or z_c.  It accumulates (o_c - z_c) W_i (o_i - z_i) v; the reduce
// halves the slice sums.  grid = (tiles, kInterSlices, nfeat): blockIdx.z is c.
__global__ void __launch_bounds__(kTileRows, 2) shap_inter_kernel(const uint4 *__restrict__ bins, const int64_t *__restrict__ feat_off,
                                                                  const uint32_t *__restrict__ feat_bins, int64_t nbins,
                                                                  ContribArgs a, double *__restrict__ part) {
  extern __shared__ __align__(128) uint32_t smem[];
  __shared__ __align__(8) unsigned long long bars[1];
  __shared__ double s_inv[34];  // 1 / k
  __shared__ int64_t s_list[2];  // this CTA's range of c's list
  const int nf = a.nfeat, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t cf = blockIdx.z;
  const int ast = nf | 1, kst = nf | 1;
  double *acc = reinterpret_cast<double *>(smem);    // [256][ast] by tile position; the TMA buffer aliases its start
  uint32_t *keys = smem + shap_region_words(nf);     // [256][kst] keys by tile position
  uint32_t *order = keys + kTileRows * kst;          // [256] the tile's row order
  PredictArgs pa;
  pa.Xt = a.Xt, pa.nrow = a.nrow, pa.ncol = a.ncol;
  TilePipe pipe;
  pipe.begin(smem, bars, pa, nf, true, tid);
  if (tid < 34) s_inv[tid] = tid ? 1.0 / (double)tid : 0.0;
  if (tid == 0) {  // c's bins among the first nbins are a prefix of its ascending list; this CTA takes one slice of it
    const int64_t l0 = feat_off[cf];
    int64_t lo = l0, hi = feat_off[cf + 1];
    while (lo < hi) {
      const int64_t m = (lo + hi) >> 1;
      if ((int64_t)feat_bins[m] < nbins) lo = m + 1;
      else hi = m;
    }
    s_list[0] = l0 + (lo - l0) * (int64_t)blockIdx.y / kInterSlices;
    s_list[1] = l0 + (lo - l0) * (int64_t)(blockIdx.y + 1) / kInterSlices;
  }
  (void)pipe.acquire(tid);
  order[tid] = smem[tid];
  for (int c = 0; c < nf; ++c) keys[tid * kst + c] = smem[(1 + c) * kStride + tid];
  __syncthreads();
  for (int i = tid; i < kTileRows * ast; i += kTileRows) acc[i] = 0.0;
  __syncthreads();
  const uint64_t tile = blockIdx.x;
  const int64_t q0 = s_list[0], q1 = s_list[1];
  for (int64_t q = q0; q < q1; ++q) {
    const uint4 e = __ldg(bins + (int64_t)__ldg(feat_bins + q) * 32 + lane);
    const uint32_t feat = e.z & 0xFFu, g0 = (e.z >> 16) & 31u, len = e.z >> 24;
    const int j = lane - (int)g0;  // my place in my path
    const bool elem = feat != kShapNoFeature && j >= 1, is_c = elem && feat == cf;
    const bool miss_here = (e.z >> 8) & 1u;
    const float zf = __uint_as_float(e.w);
    const double z = elem ? (double)zf : 1.0;
    const double v = (double)__shfl_sync(kFull, zf, (int)g0);  // leaf value, from the path's bias lane
    const unsigned c_lanes = __ballot_sync(kFull, is_c) & (unsigned)(((1ull << len) - 1ull) << g0);
    const bool has_c = c_lanes != 0u;
    const int pc = has_c ? __ffs(c_lanes) - 1 - (int)g0 : 0;  // c's place in my path
    const int Dr = has_c && !is_c ? (int)len - 2 : -1;        // unique depth of my path without c; -1: lane idle
    const int jr = j < pc ? j : j - 1;                         // my place in the path without c
    const bool adds = elem && Dr >= 0;
    auto lane_of = [&](int p) { return ((int)g0 + p + (p >= pc ? 1 : 0)) & 31; };  // lane of place p without c
    const int left = jr >= 1 ? lane_of(jr - 1) : lane, top = lane_of(Dr > 0 ? Dr : 0), c_lane = ((int)g0 + pc) & 31;
    const int maxlen = (int)__reduce_max_sync(kFull, has_c ? len - 1u : 0u);  // lanes of the longest path without c
    const double invz = 1.0 / z, d1 = (double)(Dr + 1), inv_d1 = s_inv[Dr + 1 > 0 ? Dr + 1 : 0];
    const unsigned starts = __ballot_sync(kFull, has_c && j == 0);  // the paths that contain c, in lane order
    for (int r = warp * 32; r < warp * 32 + 32; ++r) {
      const uint32_t orig = order[r] & 0xFFu;
      if (tile * kTileRows + orig >= a.nrow) continue;  // warp-uniform
      bool one = true;
      if (elem) {
        const uint32_t k = keys[r * kst + feat];
        one = k == kKeyMissing ? miss_here : (e.x <= k && k < e.y);
      }
      const float zo = one ? zf : -zf;  // (one, zero) of my element in one word: zero fractions are > 0
      const float zc = __shfl_sync(kFull, zo, c_lane);
      // ExtendPath over the elements other than c
      double pw = jr == 0 ? 1.0 : 0.0;
      for (int i = 1; i < maxlen; ++i) {
        const float zi = __shfl_sync(kFull, zo, lane_of(i));
        const double l = __shfl_sync(kFull, pw, left);
        if (i <= Dr) {
          const double inv = s_inv[i + 1];
          pw = (double)fabsf(zi) * pw * (double)max(i - jr, 0) * inv + (zi > 0.f ? l : 0.0) * (double)jr * inv;
        }
      }
      // UnwoundPathSum of my element in the path without c
      double next = __shfl_sync(kFull, pw, top), total = 0.0;
      for (int i = maxlen - 2; i >= 0; --i) {
        const double pwi = __shfl_sync(kFull, pw, lane_of(min(i, Dr > 0 ? Dr : 0)));
        if (i < Dr) {
          if (one) {
            const double tmp = next * d1 * s_inv[i + 1];
            total += tmp;
            next = pwi - tmp * z * (double)(Dr - i) * inv_d1;
          } else {
            total += pwi * invz * d1 * s_inv[Dr - i];
          }
        }
      }
      const double t = total * ((one ? 1.0 : 0.0) - z) * v * ((zc > 0.f ? 1.0 : 0.0) - (double)fabsf(zc));
      double *arow = acc + r * ast;
      for (unsigned g = starts; g; g &= g - 1u) {  // paths of the bin in order: a feature may recur across paths
        if (adds && (int)g0 == __ffs(g) - 1) arow[feat] += t;
        __syncwarp();
      }
    }
  }
  __syncthreads();
  double *out = part + ((uint64_t)cf * kInterSlices + blockIdx.y) * a.nrow * (uint64_t)nf;
  for (int i = tid; i < kTileRows * nf; i += kTileRows) {
    const int p = i / nf, f = i - p * nf;
    const uint64_t row = tile * kTileRows + (order[p] & 0xFFu);
    if (row < a.nrow) out[row * (uint64_t)nf + f] = acc[p * ast + f];
  }
}

// One thread per (row, conditioning feature): a row of M.  Off-diagonal: half the slice sums, added in slice order;
// diagonal: phi_c (the contribution slices, in slice order) minus the off-diagonal sum of the row, in float64; bias
// row: 0 and the contributions' bias.  Each output is rounded once.
__global__ void __launch_bounds__(256) shap_inter_reduce_kernel(const double *__restrict__ part, const double *__restrict__ shap_part,
                                                                int shap_slices, ContribArgs a) {
  const int nf = a.nfeat, nc = nf + 1;
  const uint64_t n = a.nrow * (uint64_t)nc, stride = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const uint64_t row = i / (uint64_t)nc;
    const int c = (int)(i - row * (uint64_t)nc);
    float *o = a.out + i * (uint64_t)nc;
    if (c == nf) {
      for (int k = 0; k < nf; ++k) o[k] = 0.f;
      o[nf] = a.bias;
      continue;
    }
    double rs = 0.0;
    for (int k = 0; k < nf; ++k) {
      if (k == c) continue;
      double s = 0.0;
      for (int sl = 0; sl < kInterSlices; ++sl) s += part[(((uint64_t)c * kInterSlices + sl) * a.nrow + row) * (uint64_t)nf + k];
      s *= 0.5;
      o[k] = (float)s;
      rs += s;
    }
    double phi = 0.0;
    for (int sl = 0; sl < shap_slices; ++sl) phi += shap_part[((uint64_t)sl * a.nrow + row) * (uint64_t)nf + c];
    o[c] = (float)(phi - rs);
    o[nf] = 0.f;
  }
}

// Approximate: libxgboost's loop with on == off gives +0 off the diagonal and 0 + phi_i on it.
__global__ void __launch_bounds__(256) shap_inter_expand_kernel(const float *__restrict__ contribs, ContribArgs a) {
  const uint64_t nc = (uint64_t)a.nfeat + 1, n = a.nrow * nc * nc, stride = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const uint64_t row = i / (nc * nc), rem = i - row * nc * nc, c = rem / nc, k = rem - c * nc;
    a.out[i] = k == c ? __fadd_rn(0.f, contribs[row * nc + c]) : 0.f;
  }
}

cudaError_t launch_shap_inter(const uint4 *bins, const int64_t *feat_off, const uint32_t *feat_bins, int64_t nbins,
                              const ContribArgs &a, double *part, cudaStream_t s) {
  if (a.nrow == 0 || a.nfeat == 0) return cudaSuccess;
  if (a.nrow > kInterChunkRows || a.ncol > a.nfeat || a.nfeat > (int)kMaxFeatures) return cudaErrorInvalidValue;
  const size_t smem = shap_smem_bytes(a.nfeat);
  cudaError_t e = cudaFuncSetAttribute(shap_inter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const dim3 grid((unsigned)tile_count(a.nrow), (unsigned)kInterSlices, (unsigned)a.nfeat);
  shap_inter_kernel<<<grid, kTileRows, smem, s>>>(bins, feat_off, feat_bins, nbins, a, part);
  count_predict(kShapInter);
  return QC_LAUNCHED();
}

cudaError_t launch_shap_inter_reduce(const double *part, const double *shap_part, int shap_slices, const ContribArgs &a,
                                     cudaStream_t s) {
  if (a.nrow == 0) return cudaSuccess;
  const uint64_t n = a.nrow * (uint64_t)(a.nfeat + 1);
  const int blocks = (int)std::min<uint64_t>((n + 255) / 256, (uint64_t)sm_count() * 16);
  shap_inter_reduce_kernel<<<blocks, 256, 0, s>>>(part, shap_part, shap_slices, a);
  count_family(kShapInterReduce);
  return QC_LAUNCHED();
}

cudaError_t launch_shap_inter_expand(const float *contribs, const ContribArgs &a, cudaStream_t s) {
  if (a.nrow == 0) return cudaSuccess;
  const uint64_t n = a.nrow * (uint64_t)(a.nfeat + 1) * (uint64_t)(a.nfeat + 1);
  const int blocks = (int)std::min<uint64_t>((n + 255) / 256, (uint64_t)sm_count() * 16);
  shap_inter_expand_kernel<<<blocks, 256, 0, s>>>(contribs, a);
  count_family(kShapInterExpand);
  return QC_LAUNCHED();
}

// =====================================================================================
// K1 — Run1 feature assembly
// =====================================================================================
// oh_state: PL_MOD, NDWET (OH_GridCompMod.F90:1247-1257) and the level-slab count (:275-298).
// One thread per column, coalesced across columns at every level.
__global__ void __launch_bounds__(128) oh_state_kernel(Run1Dev r) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  int cnt = 0, bad = 0;
  if (c < r.ncol) {
    const float tropp = r.TROPP[c];
    const float cmp = r.dynamic_k ? tropp : r.tropp_min;
    if (!r.dynamic_k && tropp <= r.tropp_min) bad = 1;  // :287
    float ple_up = r.PLE_MOD[c];
    for (int k = 0; k < r.km; ++k) {
      const size_t e = (size_t)k * r.ncol + c;
      const float ple_dn = r.PLE_MOD[e + r.ncol];
      const float pl = __fmul_rn(__fadd_rn(ple_up, ple_dn), 0.5f);  // :1247
      const float q = r.Q_MOD[e];
      // TV = T * (1 + Q/eps) / (1 + Q), left to right (:1250)
      const float tv = __fdiv_rn(__fmul_rn(r.T_MOD[e], __fadd_rn(1.0f, __fdiv_rn(q, r.eps))), __fadd_rn(1.0f, q));
      r.PL_MOD[e] = pl;
      r.NDWET[e] = __fdiv_rn(__fmul_rn(r.avogad, pl), __fmul_rn(r.runiv, tv));  // :1257
      cnt += pl > cmp;
      ple_up = ple_dn;
    }
  }
  cnt = __reduce_max_sync(0xffffffffu, cnt);
  bad = __reduce_add_sync(0xffffffffu, bad);
  if ((threadIdx.x & 31) == 0) {
    atomicMax(&r.ctl[0], cnt);
    if (bad) atomicAdd(&r.ctl[1], bad);
  }
}

cudaError_t launch_oh_state(const Run1Dev &r, cudaStream_t s) {
  oh_state_kernel<<<(r.ncol + 127) / 128, 128, 0, s>>>(r);
  return QC_LAUNCHED();
}

// oh_sums: aod (:1451-1466) and the six vertical sums (:1468-1478).  Every SUM(x(:,:,a:b),3)
// restarts at its first level and adds downward, so the DN sums are NOT a suffix scan: level k
// needs its own forward chain x(k) + x(k+1) + ... (SURVEY.md hard part 6).  One thread per
// column keeps KB chains per field in registers and sweeps the column once per block of KB
// levels; the UP sums are a running prefix.  aod and PL_BST are kept (DIAG_AOD, DIAG_PL).
// (Tried: parking the column's TAUCLW / TAUCLI / aod in shared memory for the second pass — 108 KB per 128-column CTA
// leaves 8 warps per SM and the streaming first pass then starves: the fused Run1 step grew from 43.3 to 44.2 ms at
// C360.  The sweeps of the second pass hit L2.)
constexpr int KB = 8;
__global__ void __launch_bounds__(128) oh_sums_kernel(Run1Dev r) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= r.ncol) return;
  const int nc = r.ncol, km = r.km;
  float *__restrict__ aod = r.aod;
  float *wdn = r.sums[0], *idn = r.sums[1], *iup = r.sums[2], *wup = r.sums[3], *aup = r.sums[4], *adn = r.sums[5];
  if (r.lat_deg) r.lat_deg[c] = __fmul_rn(r.LATS[c], r.r2d);         // latarr (:1444)
  if (r.so3) r.so3[c] = __fadd_rn(r.GMITO3[c], -r.GMITTO3[c]);       // stratO3 (:1446)
  // pass 1: aod and the UP prefixes
  float s_iup = 0.f, s_wup = 0.f, s_aup = 0.f;
  float z_up = r.ZLE_BST[c];
  float p_up = r.PLE_BST[c];
  for (int k = 0; k < km; ++k) {
    const size_t e = (size_t)k * nc + c;
    const float z_dn = r.ZLE_BST[e + nc];
    const float p_dn = r.PLE_BST[e + nc];
    r.pl_bst[e] = __fmul_rn(__fadd_rn(p_up, p_dn), 0.5f);  // PL_BST (:1488): bb%PL, the DIAG_PL export (:1666)
    p_up = p_dn;
    const float thick = __fadd_rn(z_up, -z_dn);  // REAL*8 gridBoxThickness holds this float exactly
    float sc = __fadd_rn(r.SCA[0][e], r.SCA[1][e]);
    sc = __fadd_rn(sc, r.SCA[2][e]);
    sc = __fadd_rn(sc, r.SCA[3][e]);
    sc = __fadd_rn(sc, r.SCA[4][e]);
    sc = __fadd_rn(sc, r.SCA[5][e]);
    sc = __fadd_rn(sc, r.SCA[6][e]);
    // double(thick) * double(sc) is exact (24 + 24 bits), so rounding it to REAL equals the
    // correctly rounded float32 product
    const float a = __fmul_rn(thick, sc);
    aod[e] = a;
    s_iup = __fadd_rn(s_iup, r.TAUCLI[e]);
    s_wup = __fadd_rn(s_wup, r.TAUCLW[e]);
    s_aup = __fadd_rn(s_aup, a);
    iup[e] = s_iup, wup[e] = s_wup, aup[e] = s_aup;
    z_up = z_dn;
  }
  // pass 2: DN chains, KB start levels at a time
  for (int k0 = 0; k0 < km; k0 += KB) {
    float cw[KB], ci[KB], ca[KB];
#pragma unroll
    for (int j = 0; j < KB; ++j) cw[j] = ci[j] = ca[j] = 0.f;
    for (int kk = k0; kk < km; ++kk) {
      const size_t e = (size_t)kk * nc + c;
      const float w = r.TAUCLW[e], i = r.TAUCLI[e], a = aod[e];
#pragma unroll
      for (int j = 0; j < KB; ++j)
        if (k0 + j <= kk) {
          cw[j] = __fadd_rn(cw[j], w);
          ci[j] = __fadd_rn(ci[j], i);
          ca[j] = __fadd_rn(ca[j], a);
        }
    }
#pragma unroll
    for (int j = 0; j < KB; ++j)
      if (k0 + j < km) {
        const size_t e = (size_t)(k0 + j) * nc + c;
        wdn[e] = cw[j], idn[e] = ci[j], adn[e] = ca[j];
      }
  }
}

cudaError_t launch_oh_sums(const Run1Dev &r, cudaStream_t s) {
  oh_sums_kernel<<<(r.ncol + 127) / 128, 128, 0, s>>>(r);
  return QC_LAUNCHED();
}

// oh_pack: xx_carr(27, N) in the reference's order (OH_GridCompMod.F90:308-345): row m runs
// over k = k1..km, then column (i fastest).  A CTA packs 256 consecutive rows: per feature the
// 256 sources are contiguous (coalesced), the [256][27] tile is transposed through shared
// memory (stride 27 is odd: conflict-free) and written back as one contiguous run.  The
// missing / inf scan is seal_tiles', which reads the matrix next.
__global__ void __launch_bounds__(256) oh_pack_kernel(Run1Features x, uint64_t e0, int ncol, uint64_t npred, float *__restrict__ X) {
  __shared__ float tile[256 * 27];
  const int tid = threadIdx.x;
  const uint64_t m0 = (uint64_t)blockIdx.x * 256;
  const uint64_t m = m0 + tid;
  if (m < npred) {
    const int c = (int)(m % (uint64_t)ncol);
#pragma unroll
    for (int ft = 0; ft < 27; ++ft) tile[tid * 27 + ft] = run1_feature(x, ft, e0 + m, c, ncol);
  }
  __syncthreads();
  const uint64_t left = npred - m0;
  const int n = (int)(left < 256 ? left : 256) * 27;
  float *dst = X + m0 * 27;
  for (int i = tid; i < n; i += 256) dst[i] = tile[i];
}

cudaError_t launch_oh_pack(const Run1Features &x, uint64_t e0, int32_t ncol, uint64_t npred, float *X, cudaStream_t s) {
  if (npred == 0) return cudaSuccess;
  oh_pack_kernel<<<(unsigned)((npred + 255) / 256), 256, 0, s>>>(x, e0, ncol, npred, X);
  return QC_LAUNCHED();
}

// oh_finalize (OH_GridCompMod.F90:1579-1599): OH_boost export, troposphere mask against the
// climatological OH using the CURRENT model PL / TROPP, mol/mol -> molec/cm3; optionally the
// loss frequencies k(T)[OH] the downstream CH4 / CO chemistry needs.
__global__ void __launch_bounds__(256) oh_finalize_kernel(Run1Dev r, uint64_t n) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += stride) {
    const int c = (int)(e % (uint64_t)r.ncol);
    const float ml = r.OH_ML[e];
    if (r.OH_boost) r.OH_boost[e] = ml;
    const float oh = (r.PL_MOD[e] > r.TROPP[c]) ? ml : r.OH_CLIM[e];
    const float ohn = __fmul_rn(__fmul_rn(oh, r.NDWET[e]), 1.0e-6f);
    r.OH[e] = ohn;
    // first-order loss frequencies for the CH4 / CO consumers of OH (build-defined; qcoh.h): float64, rounded once
    if (r.LOSS_CH4) r.LOSS_CH4[e] = (float)(2.45e-12 * exp(-1775.0 / (double)r.T_MOD[e]) * (double)ohn);
    if (r.LOSS_CO) r.LOSS_CO[e] = (float)(1.5e-13 * (1.0 + 0.6 * ((double)r.PL_MOD[e] / 101325.0)) * (double)ohn);
  }
}

cudaError_t launch_oh_finalize(const Run1Dev &r, cudaStream_t s) {
  const uint64_t n = (uint64_t)r.ncol * r.km;
  int blocks = (int)((n + 255) / 256 < 148 * 16 ? (n + 255) / 256 : 148 * 16);
  oh_finalize_kernel<<<blocks, 256, 0, s>>>(r, n);
  return QC_LAUNCHED();
}

// K4 — build-defined diagnostic (not in the reference, SURVEY.md 0.3 / 8e): float64 partial sums
//   [0] sum(OH * w)   [1] sum(w)            w = dP * area / g over tropospheric cells (PL > TROPP)
//   [2] sum(nCH4 * V) [3] sum(k(T) * OH * nCH4 * V),  k = 2.45e-12 exp(-1775/T), V = area * dz
// OH in molec/cm3, nCH4 = CH4 * NDWET.  The host (or NCCL) adds the ranks' partial sums.
__global__ void __launch_bounds__(256) oh_diag_kernel(Run1Dev r, uint64_t n) {
  double s0 = 0, s1 = 0, s2 = 0, s3 = 0;
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += stride) {
    const int c = (int)(e % (uint64_t)r.ncol);
    if (r.PL_MOD[e] > r.TROPP[c]) {
      const double area = r.AREA[c];
      const double dp = (double)r.PLE_MOD[e + r.ncol] - (double)r.PLE_MOD[e];
      const double dz = (double)r.ZLE_BST[e] - (double)r.ZLE_BST[e + r.ncol];
      const double w = dp * area / 9.80665;
      const double oh = r.OH[e];
      const double nch4 = (double)r.CH4[e] * (double)r.NDWET[e];
      const double kt = 2.45e-12 * exp(-1775.0 / (double)r.T_MOD[e]);
      s0 += oh * w, s1 += w, s2 += nch4 * area * dz, s3 += kt * oh * nch4 * area * dz;
    }
  }
  __shared__ double sh[4][8];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s0 += __shfl_down_sync(0xffffffffu, s0, o);
    s1 += __shfl_down_sync(0xffffffffu, s1, o);
    s2 += __shfl_down_sync(0xffffffffu, s2, o);
    s3 += __shfl_down_sync(0xffffffffu, s3, o);
  }
  if (lane == 0) sh[0][wid] = s0, sh[1][wid] = s1, sh[2][wid] = s2, sh[3][wid] = s3;
  __syncthreads();
  if (threadIdx.x < 4) {
    double t = 0;
    for (int w = 0; w < 8; ++w) t += sh[threadIdx.x][w];
    atomicAdd(&r.diag[threadIdx.x], t);
  }
}

cudaError_t launch_oh_diag(const Run1Dev &r, cudaStream_t s) {
  const uint64_t n = (uint64_t)r.ncol * r.km;
  int blocks = (int)((n + 255) / 256 < 148 * 4 ? (n + 255) / 256 : 148 * 4);
  oh_diag_kernel<<<blocks, 256, 0, s>>>(r, n);
  return QC_LAUNCHED();
}

}  // namespace qcoh
