// ml_tma_dev.cuh -- device-side helpers and the tensor-map encoder shared by the TMA-staged kernels
// (ml_tma.cu: one height per launch; ml_tma3.cu: steric, thermosteric and halosteric heights in one pass).
#pragma once
#include <cuda.h>

#include "ml_common.cuh"
#include "ml_host.cuh"

namespace ml {
namespace tma {

constexpr int kTile = 256;                    // columns per CTA = threads per CTA
constexpr int kConsumerWarps = kTile / 32;    // 8
constexpr int kThreads = kTile;               // no dedicated producer warp, see refill_stage()

// ------------------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_1d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0) {
  asm volatile(
      "cp.async.bulk.tensor.1d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}

// A warp has finished reading a ring stage (call from lane 0, after a __syncwarp() that gathers the warp's reads).
// Returns true in the lane whose warp is the LAST of the CTA to leave the stage: that lane issues the TMA refill,
// an async-proxy write into memory the other warps have just read through the generic proxy.
//
// Default: a relaxed shared-memory counter elects the last warp.  What keeps the refill behind the reads is the
// hardware's order, not the PTX memory model: a warp's LDS and its ATOMS go through the same in-order shared-memory
// pipe (the __syncwarp() keeps the compiler from sinking a read below the atomic), the refill is issued only after
// the eighth ATOMS has RETURNED, and the copy it starts needs hundreds of nanoseconds to come back from L2 / HBM.
//
// -DML_TMA_FENCED_RELEASE builds the version that is also right by the memory model: every warp ARRIVES (release)
// on the stage's "empty" mbarrier (initialised to the number of warps); the state the arrive returns holds the
// pending count from before it, so the warp that finds 1 there is the last one, and it WAITS (acquire) on the
// phase it has just completed before it issues the refill.  All GPU tests pass with either build.  The fenced
// one is 3 % slower on the headline step (1.94-1.97 against 1.88-1.91 ms, four alternating runs,
// profiles/r02_experiments.md): a release has to wait for the thread's loads in flight, and the next level's
// volcello / rho_ref prefetch -- issued one level ahead precisely so that nobody waits for it -- is in flight
// then.  (An acq_rel atomic on the counter, MEMBAR.ALL.CTA + ATOMS, cost the thermo- / halosteric kernels 5-11 %.)
__device__ __forceinline__ bool stage_done(uint64_t* empty_bar, int* counter, int nwarps, uint32_t parity) {
#ifndef ML_TMA_FENCED_RELEASE
  (void)empty_bar;
  (void)parity;
  return (atomicAdd(counter, 1) & (nwarps - 1)) == nwarps - 1;
#else
  (void)counter;
  (void)nwarps;
  uint64_t state;
  uint32_t pending;
  asm volatile("mbarrier.arrive.shared::cta.b64 %0, [%1];" : "=l"(state) : "r"(smem_u32(empty_bar)) : "memory");
  asm volatile("mbarrier.pending_count.b64 %0, %1;" : "=r"(pending) : "l"(state));
  if (pending != 1u) return false;
  mbar_wait(empty_bar, parity);
  return true;
#endif
}

// acc += w * d unless d is NaN (xarray's skipna sum).  d comes out of fp64 arithmetic, so a
// NaN is quiet and the test is one integer compare on the high word.
__device__ __forceinline__ void fma_skipnan(double& acc, double w, double d) {
  asm("{\n\t.reg .pred p;\n\t.reg .b32 lo, hi;\n\t"
      "mov.b64 {lo, hi}, %1;\n\t"
      "add.u32 hi, hi, hi;\n\t"
      "setp.le.u32 p, hi, 0xffe00000;\n\t"
      "@p fma.rn.f64 %0, %2, %1, %0;\n\t}"
      : "+d"(acc)
      : "d"(d), "d"(w));
}

// v_ref (fp32 in this family) is prefetched one level ahead as a raw bit pattern: converting,
// testing or even MOVing the value at load time makes the warp wait for the very load it is
// trying to hide (25-30 % of all stall samples in two profiles).
__device__ __forceinline__ unsigned ld_vraw(const float* v, i64 i) { return __ldg(reinterpret_cast<const unsigned*>(v) + i); }
__device__ __forceinline__ bool vraw_isnan(unsigned w) { return (w & 0x7fffffffu) > 0x7f800000u; }
__device__ __forceinline__ double vraw_value(unsigned w) { return (double)__uint_as_float(w); }
// the same for a reference volume stored as fp64
__device__ __forceinline__ unsigned long long ld_vraw(const double* v, i64 i) {
  return __ldg(reinterpret_cast<const unsigned long long*>(v) + i);
}
__device__ __forceinline__ bool vraw_isnan(unsigned long long w) { return (w & 0x7fffffffffffffffull) > 0x7ff0000000000000ull; }
__device__ __forceinline__ double vraw_value(unsigned long long w) { return __longlong_as_double((long long)w); }
template <typename T>
struct RawBits;
template <>
struct RawBits<float> {
  typedef unsigned type;
};
template <>
struct RawBits<double> {
  typedef unsigned long long type;
};

// partial-cell thickness, derived.py:308-318 for top = 0 / bottom = None, written with plain
// compares: depth and z_i are never NaN here (deptho is NaN-filled with 0 on entry, derived.py:295)
__device__ __forceinline__ double level_dz(double depth, double ztop, double zbot) {
  const double part = depth - ztop, full = zbot - ztop;
  const double p0 = part < 0.0 ? 0.0 : part;
  return p0 < full ? p0 : full;
}
__device__ __forceinline__ bool nonzero(double x) {  // x != 0 without touching the fp64 pipe
  return ((((unsigned)__double2hiint(x)) << 1) | (unsigned)__double2loint(x)) != 0u;
}

// number of levels whose upper interface lies above the sea floor (those with dz > 0); NaN depth = land = 0
__device__ __forceinline__ int wet_levels(double depth, const double* s_zi, int nz) {
  int lo = 0, hi = nz;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (s_zi[mid] < depth) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// Column of the tile that thread `tid` integrates, given every thread's key (wet levels of column
// `tid`): a bitonic sort of the 256 (key, column) words, deepest first -- unique words, so one fixed
// order -- in registers (shuffles) and one shared-memory array.  Sorted position p goes to warp slot
// 0 1 2 3 7 6 5 4 (by depth band p / 32), so that the two warps an SM sub-partition hosts (w and
// w + 4) carry a deep and a shallow band.  Every thread of the CTA must call it.
template <int TILE>
__device__ __forceinline__ int sorted_column_t(int key, unsigned* s_key, int* s_col, int rot = 0) {
  const int tid = threadIdx.x, lane = tid & 31;
  unsigned v = ((unsigned)key << 8) | (unsigned)(TILE - 1 - tid);
  for (int k = 2; k <= TILE; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      unsigned o;
      if (j >= 32) {
        __syncthreads();
        s_key[tid] = v;
        __syncthreads();
        o = s_key[tid ^ j];
      } else {
        o = __shfl_xor_sync(0xffffffffu, v, j);
      }
      const bool lower = (tid & j) == 0, desc = (tid & k) == 0;  // final merge (k = TILE): descending
      v = (lower == desc) ? max(v, o) : min(v, o);
    }
  }
  const int band = tid >> 5;
  // 256 columns: bands to warp slots 0 1 2 3 7 6 5 4 (a deep and a shallow band per SM sub-partition);
  // 128 columns: one warp per sub-partition, bands in order
  // rot (0..3) turns the assignment round the four sub-partitions: CTAs that share an SM then put their deep
  // bands on different sub-partitions instead of all on the first one
  int slot = TILE == 256 ? (band < 4 ? band : 11 - band) : band;
  slot = (slot & ~3) | ((slot + rot) & 3);
  s_col[slot * 32 + lane] = TILE - 1 - (int)(v & 255u);
  __syncthreads();
  return s_col[tid];
}
__device__ __forceinline__ int sorted_column(int key, unsigned* s_key, int* s_col) {
  return sorted_column_t<kTile>(key, s_key, s_col);
}

// ----------------------------------------------------------------------- depth layers
// The layered modes (kLocalLayers in ml_tma.cu, kLocalLayers3 in ml_tma3.cu): level z feeds layer b with the weight
// calc_dz(top=edges[b], bottom=edges[b+1]) (derived.py:295-318) and the height of a layer is stored when the sweep
// leaves its last level.  The edges are a kernel parameter of their own (a larger Params cost the kLocal kernel four
// registers); the other modes take an empty one.
constexpr int kNoLayer = 0xffff;  // no layer touches the level
struct LayerParams {
  int nlayers;                      // eta is [nt][nlayers][ncol]
  double edges[ML_MAX_LAYERS + 1];  // increasing; the last may be +inf
};
struct NoLayers {};
__device__ __forceinline__ int layer_count(const LayerParams& L) { return L.nlayers; }
__device__ __forceinline__ int layer_count(const NoLayers&) { return 0; }
__device__ __forceinline__ double layer_edge(const LayerParams& L, int b) { return L.edges[b]; }
__device__ __forceinline__ double layer_edge(const NoLayers&, int) { return 0.0; }
// The layers that touch each level, worked out once per CTA: layer b touches level k iff z_i[k+1] > edges[b] &&
// z_i[k] < edges[b+1]; they are consecutive: lo | hi << 8, or kNoLayer.  The layers a level touches are the same
// for every column (only the bottom clip varies, and it can only zero a weight).
template <int NTHREADS, typename LP>
__device__ __forceinline__ void fill_layer_table(int* s_lay, const double* z_i, int nz, const LP& L) {
  for (int i = threadIdx.x; i < nz; i += NTHREADS) {
    const double zt = __ldg(z_i + i), zb = __ldg(z_i + i + 1);
    int lo = -1, hi = -1;
    for (int b = 0; b < layer_count(L); ++b)
      if (zb > layer_edge(L, b) && zt < layer_edge(L, b + 1)) {
        if (lo < 0) lo = b;
        hi = b;
      }
    s_lay[i] = lo < 0 ? kNoLayer : (lo | (hi << 8));
  }
}
__device__ __forceinline__ bool layer_touches(int lay, int b) { return lay != kNoLayer && (lay & 255) <= b && b <= (lay >> 8); }
// where a thread stores the heights of its column; one per output field (in == false: nothing is stored)
struct LayerOut {
  double* eta;
  double coef;
  int nt;
  i64 ncol, c;
  int t0;
  bool in, surface_wet;
};
// weight of level z in layer b: derived.py:295-318 with top = edges[b], bottom = edges[b+1] (the arithmetic of
// k_calc_dz); depth and z_i are never NaN here
template <typename LP>
__device__ __forceinline__ double layer_w(const LP& L, const double* s_zi, double depth, int z, int b) {
  return fmin(fmax(s_zi[z + 1] - layer_edge(L, b), 0.0), level_dz(fmin(depth, layer_edge(L, b + 1)), s_zi[z], s_zi[z + 1]));
}
template <typename LP>
__device__ __forceinline__ void store_height(const LayerOut& o, const LP& L, int b, int k, double a) {
  if (o.in && o.t0 + k < o.nt) o.eta[((i64)(o.t0 + k) * layer_count(L) + b) * o.ncol + o.c] = o.surface_wet ? o.coef * a : nan("");
}
// the sweep has left layer b: store its sums and start the next layer from zero
template <int TC, typename LP>
__device__ __forceinline__ void close_layer(double (&acc)[TC], bool& poisoned, const LayerOut& o, const LP& L, int b) {
#pragma unroll
  for (int k = 0; k < TC; ++k) {
    poisoned |= is_nan_q(acc[k]);
    store_height(o, L, b, k, acc[k]);
    acc[k] = 0.0;
  }
}
// level z closes layers lo .. hi - 1 and opens hi (an edge falls inside it).  acc already holds layer lo with the
// level's share of d = rho - rho_ref of step k added: store it, store the layers that lie inside the level, and
// start layer hi with its share of d
template <typename LP>
__device__ __forceinline__ void split_level(double& acc, bool& poisoned, const LayerOut& o, const LP& L, const double* s_zi,
                                            double depth, int z, int lo, int hi, bool live, int k, double d) {
  poisoned |= is_nan_q(acc);
  store_height(o, L, lo, k, acc);
  for (int b = lo + 1; b < hi; ++b) {
    const double a = (live ? layer_w(L, s_zi, depth, z, b) : 0.0) * d;
    poisoned |= is_nan_q(a);
    store_height(o, L, b, k, a);
  }
  acc = (live ? layer_w(L, s_zi, depth, z, hi) : 0.0) * d;
}

// ----------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn query_encode_fn() {
  void* p = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
      q == cudaDriverEntryPointSuccess)
    return reinterpret_cast<EncodeTiledFn>(p);
  return nullptr;
}

static EncodeTiledFn encode_fn() {
  static const EncodeTiledFn fn = query_encode_fn();  // initialised once, thread-safe
  return fn;
}

// fp32 field [nt][nz][ncol] (rank 3) or [nz][ncol] (rank 2); box = {kTile, 1, tc}
static bool make_map(CUtensorMap* map, const void* base, int rank, i64 ncol, i64 nz, i64 nt, int tc, int tile = kTile,
                     int elem_bytes = 4) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return false;
  const cuuint64_t es = (cuuint64_t)elem_bytes;
  cuuint64_t dims[3] = {(cuuint64_t)ncol, (cuuint64_t)nz, (cuuint64_t)nt};
  cuuint64_t strides[2] = {(cuuint64_t)ncol * es, (cuuint64_t)ncol * (cuuint64_t)nz * es};
  cuuint32_t box[3] = {(cuuint32_t)tile, 1, (cuuint32_t)tc};
  cuuint32_t estr[3] = {1, 1, 1};
  return fn(map, elem_bytes == 8 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT64 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, (cuuint32_t)rank, const_cast<void*>(base), dims, strides, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// A field seen as ONE row of n values (rank 1), box = {tile}: what a grid whose rows are not a multiple of 16 bytes
// can still offer a tensor map -- a box may start at any element, only base and strides are bound to 16 bytes.
static bool make_flat_map(CUtensorMap* map, const void* base, i64 n, int tile = kTile, int elem_bytes = 4) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return false;
  cuuint64_t dims[1] = {(cuuint64_t)n};
  cuuint64_t strides[1] = {0};  // unused for rank 1
  cuuint32_t box[1] = {(cuuint32_t)tile};
  cuuint32_t estr[1] = {1};
  return fn(map, elem_bytes == 8 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT64 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 1u,
            const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
            CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace tma
}  // namespace ml
