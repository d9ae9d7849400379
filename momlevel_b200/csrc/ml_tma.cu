// ml_tma.cu -- TMA-staged kernel family for the fused steric kernels (sm_100a).
//
// Layout of the work: fields are [t][z][col] fp32 (col = flattened y,x).  A CTA owns a tile
// of kTile = 256 adjacent columns and a chunk of TC time steps.  For each level ONE 3-D TMA box
// per field ({256 cols, 1 level, TC steps} = TC KB) lands in a ring of shared-memory stages
// guarded by "full" mbarriers; the warp that is last to leave a stage refills it (there is no
// producer warp).  Eight warps (one column per thread) read T,S from shared memory, evaluate
// the EOS in fp64 registers and keep the TC running column sums in registers, so
//   - every byte of T and S crosses HBM exactly once, in 1 KB contiguous rows,
//   - rho_ref / v_ref (3-D, time-invariant) are fetched once per (level, column, chunk)
//     with ordinary loads, prefetched one level ahead, and reused for TC steps; the chunks of
//     a tile run together, so only the first of them takes these rows from HBM,
//   - loads cost no registers and no issue slots in the compute warps; the depth of the
//     ring (not occupancy) hides HBM latency,
//   - out-of-range columns / time steps of edge tiles are zero-filled by the TMA unit.
// Levels at which no lane of a warp has any water (dz = 0: land, below the sea floor) are
// skipped by that warp: their terms are multiplied by dz = 0 in steric.py:163 and vanish.
// The columns of a tile are sorted by wet depth first (ML_TMA_SORT) so that dry columns share
// warps with other dry columns instead of riding along in wet ones.
//
// Eligibility: fields and volcello stored alike (fp32, or fp64 -- what the reference's own test data and any
// xarray arithmetic on model output produce -- with half as many steps per chunk), 16-byte aligned bases,
// rows a multiple of 16 bytes (TMA global strides), ncol >= kTile, no delta_rho output.  Everything else
// takes the direct family in ml_api.cu.
#include "ml_tma_dev.cuh"
#include "ml_tma.cuh"

#include <type_traits>

namespace ml {
namespace tma {

// Ring depth (levels in flight per CTA) and resident CTAs per SM, by mode.  The local modes run two
// CTAs per SM with a 4-level ring and ~120 registers per thread.  The global kernel carries no
// rho_ref / dz operands and fits 64 registers, so it runs four CTAs per SM with a 2-level ring (the
// same bytes in flight per SM): +4.5 % (profiles/r01_experiments.md).  The self-reference mode reads
// row 0 of the NEXT level while it works on this one and loses 15 % with a 2-level ring.
// A launch with S held at its reference slab (thermosteric: BC == 2) stages TC + 1 rows per level instead of 2 TC, so the
// same shared memory holds a ring twice as deep: 1.50 -> 1.44-1.47 ms on OM4p25 x 12.  Not so for the halosteric launch
// (no change) nor for the global kernel (a deeper ring costs it its fourth CTA per SM: 1.37-1.50 -> 1.54 ms);
// tools/pinned_probe.py, profiles/r02_experiments.md.
#ifndef ML_TMA_BC_STAGES
#define ML_TMA_BC_STAGES 8
#endif
__host__ __device__ constexpr int stages_of(int mode, int bc = 0, int es = 4) {
  return mode == 1 /* kGlobal */ ? 2 : ((bc == 2 && es == 4) ? ML_TMA_BC_STAGES : 4);
}
// Columns a CTA owns.  FLAT (rows of the grid are not a multiple of 16 bytes): a TMA box must START on 16 bytes in
// global memory and holds at most 256 values, so it starts at the row's address rounded down, and the CTA owns the
// 256 - (16 / size) columns that are inside the box whatever the row's misalignment (252 for fp32, 254 for fp64);
// the readers add the row's offset of 0 ... (16 / size - 1) values, the last few threads have no column.
__host__ __device__ constexpr int cols_of(int elem, bool flat) { return flat ? 256 - 16 / elem : 256; }
__host__ __device__ constexpr int ctas_per_sm_of(int mode) { return mode == 1 /* kGlobal */ ? 4 : 2; }
// Which column of the tile a thread integrates: 0 = thread i takes column i; otherwise the columns
// are ranked by wet depth across the tile first (sorted_column below).  A warp skips a level when
// none of its lanes has water there, so packing columns of similar depth (and land) into the same
// warps removes the fp64 work of dry lanes that ride along in partly wet warps -- 0.90 -> 0.58 of all
// (warp, level) pairs on the synthetic ocean.  (Ranking within residue classes mod 32 keeps the
// shared-memory reads conflict-free but only reaches 0.72 and was slower: profiles/r01_experiments.md.)
#ifndef ML_TMA_SORT
#define ML_TMA_SORT 1
#endif
// Ceiling experiments (tools/k3_sweep.sh; results are WRONG by construction, never shipped):
//   1 = compute only: the ring is filled once and re-read, nothing streams from HBM
//   2 = memory only:  every level is streamed, the arithmetic is skipped
#ifndef ML_TMA_EXPERIMENT
#define ML_TMA_EXPERIMENT 0
#endif
constexpr int kNoLayer = 0xffff;  // kLocalLayers: no layer touches the level


struct Params {
  const void* T;          // the fields themselves (the streaming path goes through the tensor maps;
  const void* S;          //  these are for the repair pass of a column that met a missing value); fp32 or fp64
  const double* rho_ref;  // kLocal: read
  double* rho_ref_out;    // kSelfRef: written (may be NULL)
  const void* v_ref;      // volcello of the reference state, stored like the fields
  const double* z_i;      // local modes
  const double* deptho;   // local modes
  const double* p_level;
  double coef;
  int nt, nz;
  int es;                 // bytes per stored value of T, S and v_ref: 4 or 8
  int flat;               // rows are not a multiple of 16 bytes: rank-1 maps, one 1-D box per row (see refill_stage)
  int t_start;            // first time step covered by this launch
  int first_is_reference; // kLocal: step 0 of the field IS the reference state -> its height is exactly zero
  unsigned nchunks;       // time chunks covered by this launch; grid = tiles * nchunks, chunk fastest
  unsigned tiles;         // column tiles
  i64 ncol;
  double* eta;            // local modes: [nt][ncol]
  double* partials;       // kGlobal: [nt][tiles];  kSelfRef: [2][tiles] = {volo, masso}
};

// kLocalLayers: the depth layers, a kernel parameter of their own (the other modes take an empty one: a larger
// Params cost the kLocal kernel four registers)
struct LayerParams {
  int nlayers;                      // eta is [nt][nlayers][ncol]
  double edges[ML_MAX_LAYERS + 1];  // increasing; the last may be +inf
};
struct NoLayers {};
__device__ __forceinline__ int layer_count(const LayerParams& L) { return L.nlayers; }
__device__ __forceinline__ int layer_count(const NoLayers&) { return 0; }
__device__ __forceinline__ double layer_edge(const LayerParams& L, int b) { return L.edges[b]; }
__device__ __forceinline__ double layer_edge(const NoLayers&, int) { return 0.0; }
// where a thread stores the heights of its column (kLocalLayers)
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

template <int MODE>
using LayersOf = typename std::conditional<MODE == 3 /* kLocalLayers */, LayerParams, NoLayers>::type;

// What a launch computes.
//   kLocal   eta from rho - rho_ref with rho_ref read from memory          (steric.py:150-166)
//   kGlobal  per-step sums of rho * v_ref                                    (steric.py:135)
//   kSelfRef kLocal for the chunk that starts at the reference step itself: rho_ref is the
//            density of row 0 of every stage, evaluated here, stored for the caller and
//            reduced into volo / masso on the way -- the reference-state pass
//            (reference.py:71-80) costs no extra read of T, S.
//   kLocalLayers  kLocal split by depth layer: level z feeds layer b with the weight
//            calc_dz(top=edges[b], bottom=edges[b+1]) (derived.py:295-318) and the height of a layer is stored
//            when the sweep leaves its last level.  One set of TC sums lives in registers: the layers a level
//            touches are the same for every column (only the bottom clip varies, and it can only zero a weight),
//            so they are worked out once per CTA, and a level feeds more than one layer only where an edge
//            falls inside it.
enum Mode { kLocal = 0, kGlobal = 1, kSelfRef = 2, kLocalLayers = 3 };

// BC: 0 = T and S both [t][z][col]; 1 = T is [z][col] (halosteric); 2 = S is [z][col] (thermosteric)
#ifdef ML_TMA_MAXNREG  // experiment builds: explicit register cap instead of the occupancy hint
#define ML_TMA_KERNEL_ATTR __maxnreg__(ML_TMA_MAXNREG)
#else
#define ML_TMA_KERNEL_ATTR __launch_bounds__(kThreads, ctas_per_sm_of(MODE))
#endif

template <typename TIn, int EOS, int TC, int BC, int MODE, bool FLAT>
__global__ void ML_TMA_KERNEL_ATTR
    k_steric_tma(const __grid_constant__ CUtensorMap mapT, const __grid_constant__ CUtensorMap mapS, const Params P,
                 const LayersOf<MODE> L) {
  constexpr bool GLOBAL = MODE == kGlobal;
  constexpr bool SELFREF = MODE == kSelfRef;
  constexpr bool LAYERS = MODE == kLocalLayers;
  constexpr bool READREF = MODE == kLocal || LAYERS;  // rho_ref is read from memory
  constexpr int kStages = stages_of(MODE, BC, (int)sizeof(TIn));
  constexpr int SORT = ML_TMA_SORT;
  constexpr int kRowsT = (BC == 1) ? 1 : TC;
  constexpr int kRowsS = (BC == 2) ? 1 : TC;
  constexpr int kPitch = kTile;                               // values between the rows of a stage = one box
  constexpr int kUnit = 16 / (int)sizeof(TIn);                // values per 16 bytes
  constexpr int kCols = cols_of((int)sizeof(TIn), FLAT);      // columns this CTA owns
  constexpr uint32_t kStageBytes = (uint32_t)(kRowsT + kRowsS) * kPitch * sizeof(TIn);
  constexpr uint32_t kStageTx = kStageBytes;
  constexpr int kStageFloats = (int)(kStageBytes / sizeof(TIn));
  constexpr int kRed = GLOBAL ? TC : 2;  // values reduced across the CTA at the end

  extern __shared__ __align__(128) unsigned char smem_raw[];
  TIn* stage_base = reinterpret_cast<TIn*>(smem_raw);
  const TIn* const gT = static_cast<const TIn*>(P.T);
  const TIn* const gS = static_cast<const TIn*>(P.S);
  const TIn* const gV = static_cast<const TIn*>(P.v_ref);
  typedef typename RawBits<TIn>::type vbits;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + (size_t)kStages * kStageBytes);
  uint64_t* empty = full + kStages;                            // [kStages] "every warp has left the stage"
  int* released = reinterpret_cast<int*>(full + 2 * kStages);  // [kStages] warps that are done with the stage
  double* red = reinterpret_cast<double*>(full + 3 * kStages);  // [kConsumerWarps][TC]
  double* s_p = red + kConsumerWarps * TC;                   // [nz]   pressure per level
  double* s_zi = s_p + P.nz;                                 // [nz+1] interfaces (local modes)
  int* s_key = reinterpret_cast<int*>(s_zi + P.nz + 1);      // [kTile] wet levels per column (SORT)
  int* s_col = s_key + kTile;                                // [kTile] column handled by each thread (SORT)
  int* s_lay = s_col + kTile;                                // [nz] kLocalLayers: layers touching the level

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // The chunks of one tile are neighbours in launch order, so they are resident together and the
  // time-invariant rows they all read (rho_ref, v_ref, a broadcast operand) come from HBM once and
  // from L2 for the others; with the tiles fastest those rows were re-read from HBM for every chunk.
  const unsigned tile = blockIdx.x / P.nchunks;
  const int c0 = (int)tile * kCols;
  const int t0 = P.t_start + (int)(blockIdx.x - tile * P.nchunks) * TC;
  const int nz = P.nz;

  // Loads level z of this CTA's tile into its stage.  Called by thread 0 for the first kStages
  // levels and afterwards by whichever warp is the LAST to finish with a stage (a shared-memory
  // counter tells): the refill is issued the moment the slot is free, without a producer warp
  // spinning on "empty" barriers and taking registers and issue slots from the math warps.
  auto refill_stage = [&](int z) {
    const int s = z % kStages;
    TIn* dT = stage_base + (size_t)s * kStageFloats;
    TIn* dS = dT + kRowsT * kPitch;
    mbar_expect_tx(full + s, kStageTx);
    if (FLAT) {
      // Rows that are not a multiple of 16 bytes (ncol % 4 != 0 for fp32): no strided tensor map can describe the
      // field, but a rank-1 map over the flat array can -- one 1-D box per row of the stage, started at the row's
      // first value rounded down to 16 bytes (a box must start aligned; flat_off() is what the readers add).
      // Columns past the end of a row hold the head of the next row (never stored), rows past the last step lie
      // beyond the map and are zero-filled.
      const i64 row0 = (i64)z * P.ncol + c0, step = (i64)nz * P.ncol;
#pragma unroll
      for (int k = 0; k < kRowsT; ++k)
        tma_load_1d(dT + k * kPitch, &mapT, full + s, (int)((row0 + (BC == 1 ? 0 : (i64)(t0 + k) * step)) & ~(i64)(kUnit - 1)));
#pragma unroll
      for (int k = 0; k < kRowsS; ++k)
        tma_load_1d(dS + k * kPitch, &mapS, full + s, (int)((row0 + (BC == 2 ? 0 : (i64)(t0 + k) * step)) & ~(i64)(kUnit - 1)));
      return;
    }
    if (BC == 1) tma_load_2d(dT, &mapT, full + s, c0, z); else tma_load_3d(dT, &mapT, full + s, c0, z, t0);
    if (BC == 2) tma_load_2d(dS, &mapS, full + s, c0, z); else tma_load_3d(dS, &mapS, full + s, c0, z, t0);
  };

  // FLAT: where the tile's first column sits inside the stage row of (level z, step t) -- the same for every thread
  // of the CTA, so this is uniform-datapath arithmetic; `fixed` marks a time-invariant operand ([z][col])
  auto flat_off = [&](int z, int t, bool fixed) -> int {
    if (!FLAT) return 0;
    return (int)(((i64)z * P.ncol + c0 + (fixed ? 0 : (i64)t * nz * P.ncol)) & (i64)(kUnit - 1));
  };

  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full + s, 1);
      mbar_init(empty + s, kConsumerWarps);
      released[s] = 0;
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    for (int z = 0; z < kStages && z < nz; ++z) refill_stage(z);
  }
  for (int i = threadIdx.x; i < P.nz; i += kThreads) s_p[i] = __ldg(P.p_level + i);
  if (!GLOBAL)
    for (int i = threadIdx.x; i <= P.nz; i += kThreads) s_zi[i] = __ldg(P.z_i + i);
  if (LAYERS) {
    // layer b touches level k iff z_i[k+1] > edges[b] && z_i[k] < edges[b+1]; the layers touching a level are
    // consecutive: lo | hi << 8, or kNoLayer
    for (int i = threadIdx.x; i < P.nz; i += kThreads) {
      const double zt = __ldg(P.z_i + i), zb = __ldg(P.z_i + i + 1);
      int lo = -1, hi = -1;
      for (int b = 0; b < layer_count(L); ++b)
        if (zb > layer_edge(L, b) && zt < layer_edge(L, b + 1)) {
          if (lo < 0) lo = b;
          hi = b;
        }
      s_lay[i] = lo < 0 ? kNoLayer : (lo | (hi << 8));
    }
  }
  __syncthreads();

  int col = tid;  // column of the tile this thread integrates
  if (SORT != 0) {
    // key = number of wet levels of the column: levels above the sea floor (local modes) or levels
    // whose reference volume is present (global mode, which has no deptho)
    const i64 cg = (i64)c0 + tid;
    const bool owned = tid < kCols && cg < P.ncol;  // (FLAT: the last few threads of a CTA have no column)
    int key = 0;
    if (GLOBAL) {
      if (owned)
        for (int z = 0; z < nz; ++z) key += vraw_isnan(ld_vraw(gV, (i64)z * P.ncol + cg)) ? 0 : 1;
    } else {
      key = wet_levels(owned ? __ldg(P.deptho + cg) : 0.0, s_zi, nz);
    }
    col = sorted_column(key, reinterpret_cast<unsigned*>(s_key), s_col);
  }

  {
    const i64 c = (i64)c0 + col;
    const bool in = col < kCols && c < P.ncol;
    const i64 cc = in ? c : (P.ncol - 1);  // clamp: edge lanes read a valid column, never store
    Eos<EOS> eos;
    double acc[TC];
#pragma unroll
    for (int k = 0; k < TC; ++k) acc[k] = 0.0;
    double vol = 0.0, mass = 0.0;  // kSelfRef
    double depth = 0.0;
    if (!GLOBAL) {
      depth = __ldg(P.deptho + cc);
      if (isnan(depth)) depth = 0.0;  // derived.py:295
    }
    // per-level operands, fetched one level ahead (raw bits, see ld_vraw)
    double rref_n = 0.0;
    vbits v_n = ld_vraw(gV, cc);
    if (READREF) rref_n = __ldg(P.rho_ref + cc);
    const bool surface_wet = !vraw_isnan(v_n);  // steric.py:166
    const bool zero_first = MODE == kLocal && P.first_is_reference != 0 && t0 == 0;
    // kLocalLayers: the layer the sums belong to, and whether a closed layer met a missing value
    int cur = 0;
    bool poisoned = false;
    // (the layered steps are free functions, not lambdas: an unused closure that holds &acc cost the kSelfRef
    // kernels four registers)
    const LayerOut out = {P.eta, P.coef, P.nt, P.ncol, c, t0, in, surface_wet};
    // kSelfRef: the reference density of level z+1 is evaluated together with the points of
    // level z (from row 0 of the next stage, inside the same unrolled block so the scheduler
    // interleaves it), stored for the caller and used one iteration later.
    double sub_n = 0.0;
    if (SELFREF) {
      mbar_wait(full + 0, 0u);
      const TIn* row = stage_base + col;
      sub_n = eos.rho_at((double)row[flat_off(0, t0, BC == 1)], (double)row[kRowsT * kPitch + flat_off(0, t0, BC == 2)], s_p[0]);  // reference.py:60-71
      if (in && P.rho_ref_out) P.rho_ref_out[c] = sub_n;
    }
    for (int z = 0; z < nz; ++z) {
      const double rref_z = SELFREF ? sub_n : rref_n;
      const vbits v_z = v_n;
      if (z + 1 < nz) {
        const i64 j = (i64)(z + 1) * P.ncol + cc;
        v_n = ld_vraw(gV, j);
        if (READREF) rref_n = __ldg(P.rho_ref + j);
      }
      // weight of this cell in the sum and the value subtracted from rho
      const bool dry = vraw_isnan(v_z);
      double w, sub;
      if (GLOBAL) {
        w = dry ? 0.0 : vraw_value(v_z);  // rho * NaN is dropped by the skipna sum (derived.py:435-438)
        sub = 0.0;
      } else {
        w = level_dz(depth, s_zi[z], s_zi[z + 1]);
        // steric.py:151-153: delta_rho is NaN (and skipped) wherever the reference volume is missing
        sub = rref_z;
        if (dry || (READREF && isnan(rref_z))) w = 0.0;
        if (LAYERS && s_lay[z] == kNoLayer) w = 0.0;  // no layer takes this level
        if (SELFREF && in && !dry) {  // volo, masso: skipna sums (derived.py:787-789, :435-438)
          const double v = vraw_value(v_z);
          vol += v;
          const double m = rref_z * v;
          if (!is_nan_q(m)) mass += m;
        }
      }
      eos.set_level(s_p[z]);
      const bool live = nonzero(w);
      if (!live) sub = 0.0;  // a dry lane adds 0 * (rho of a borrowed column - sub): keep a missing rho_ref out of it
      // kLocalLayers: close the layers that ended above this level (in every warp, wet or not); `wl` is the weight
      // of the level in its one layer, or -- where an edge falls inside the level (lo < hi) -- in layer lo
      int lo = 0, hi = 0;
      double wl = w;
      if (LAYERS && s_lay[z] != kNoLayer) {
        lo = s_lay[z] & 255;
        hi = s_lay[z] >> 8;
        for (; cur < lo; ++cur) close_layer<TC>(acc, poisoned, out, L, cur);
        wl = live ? layer_w(L, s_zi, depth, z, lo) : 0.0;
      }
      const unsigned live_lanes = __ballot_sync(0xffffffffu, live);
      // kSelfRef: row 0 of the NEXT level (clamped at the bottom level, where the value is
      // recomputed and discarded) -- wait for it up front so that the reference point and the
      // TC - 1 points below form one straight-line block
      const int zn = (z + 1 < nz) ? z + 1 : z;
      const TIn* rowN = stage_base + (size_t)(zn % kStages) * kStageFloats + col;
      const double p_next = s_p[zn];
      const int s = z % kStages;
      if (SELFREF && (ML_TMA_EXPERIMENT != 1 || zn < kStages)) mbar_wait(full + (zn % kStages), (uint32_t)(zn / kStages) & 1u);
      if (ML_TMA_EXPERIMENT != 1 || z < kStages) mbar_wait(full + s, (uint32_t)(z / kStages) & 1u);
      if (ML_TMA_EXPERIMENT != 2 && live_lanes != 0u) {
        // A lane whose cell is dry (w = 0: land, below the sea floor) holds missing values and would
        // put NaN into its sums (0 * NaN), so it evaluates the column of the warp's first wet lane
        // instead -- the same shared-memory words, a broadcast -- and adds 0 * (a finite number).
        // The sums are then plain FMAs: the four ALU instructions of a per-point NaN test were 6-10 %
        // of the thermo- / halosteric kernels.  A hole at a WET cell does reach the sums; it is
        // caught after the sweep and that column is redone with the skipna rule (repair pass below).
        const int first_wet = __shfl_sync(0xffffffffu, col, __ffs(live_lanes) - 1);  // every lane takes part
        const TIn* sT = stage_base + (size_t)s * kStageFloats + (live ? col : first_wet);
        const TIn* sS = sT + kRowsT * kPitch;
        if (SELFREF)
          sub_n = eos.rho_at((double)rowN[flat_off(zn, t0, BC == 1)], (double)rowN[kRowsT * kPitch + flat_off(zn, t0, BC == 2)], p_next);
        // a time-invariant operand is folded into the polynomial's coefficients once per level
        // (thermosteric +15 %, halosteric +16 %)
        typename Eos<EOS>::Pinned pin = {};
        if (BC == 1) pin = eos.pin_t((double)sT[flat_off(z, 0, true)]);
        if (BC == 2) pin = eos.pin_s((double)sS[flat_off(z, 0, true)]);
        double d[LAYERS ? TC : 1];  // kLocalLayers: rho - rho_ref of each step, for a level that closes layers
#pragma unroll
        for (int kk = SELFREF ? 1 : 0; kk < TC; ++kk) {  // kSelfRef: step 0 is the reference itself
          if (MODE == kLocal && kk == 0 && zero_first) continue;  // ... and so it is here, by the caller's word
          const double Tv = (double)sT[(BC == 1 ? 0 : kk) * kPitch + flat_off(z, t0 + kk, BC == 1)];
          const double Sv = (double)sS[(BC == 2 ? 0 : kk) * kPitch + flat_off(z, t0 + kk, BC == 2)];
          const double rho = BC == 1 ? eos.rho_pinned_t(pin, Sv) : (BC == 2 ? eos.rho_pinned_s(pin, Tv) : eos.rho(Tv, Sv));
          // kLocalLayers: the sum of layer lo takes the kLocal kernel's FMA in the same straight-line block (where
          // the compiler folds the subtraction of rho_ref into the EOS's last multiply), so one layer (0, inf) is
          // bit-identical to ml_steric_local, and the TC evaluations stay free to interleave
          acc[kk] = fma(LAYERS ? wl : w, GLOBAL ? rho : rho - sub, acc[kk]);
          if (LAYERS) d[LAYERS ? kk : 0] = rho - sub;
        }
        if (LAYERS && lo < hi)
#pragma unroll
          for (int kk = 0; kk < TC; ++kk) split_level(acc[kk], poisoned, out, L, s_zi, depth, z, lo, hi, live, kk, d[LAYERS ? kk : 0]);
      } else if (LAYERS && lo < hi) {
#pragma unroll
        for (int kk = 0; kk < TC; ++kk)  // a warp without water still closes its layers
          split_level(acc[kk], poisoned, out, L, s_zi, depth, z, lo, hi, live, kk, 0.0);
      } else if (SELFREF) {
        // a warp without water still owes rho_ref of the next level (reference.py:71 evaluates the
        // EOS everywhere); over land T, S are missing and so is the result -- no arithmetic needed
        const TIn tN = rowN[flat_off(zn, t0, BC == 1)], sN = rowN[kRowsT * kPitch + flat_off(zn, t0, BC == 2)];
        sub_n = nan("");
        if (__any_sync(0xffffffffu, !(isnan(tN) || isnan(sN)))) sub_n = eos.rho_at((double)tN, (double)sN, p_next);
      }
      if (LAYERS && lo < hi) cur = hi;  // layers lo .. hi - 1 are stored; the sums now belong to layer hi
      if (SELFREF && in && z + 1 < nz && P.rho_ref_out) P.rho_ref_out[(i64)(z + 1) * P.ncol + c] = sub_n;
      __syncwarp();
      if (lane == 0) {
        // the 8th warp to leave the stage refills it with the level kStages further on
        if (stage_done(empty + s, released + s, kConsumerWarps, (uint32_t)(z / kStages) & 1u) && ML_TMA_EXPERIMENT != 1 &&
            z + kStages < nz)
          refill_stage(z + kStages);
      }
    }
    if (LAYERS)
      for (; cur < layer_count(L); ++cur) close_layer<TC>(acc, poisoned, out, L, cur);  // the last layer, and those wholly below the grid: 0
    // Repair pass (rare: consistent model output has no holes at wet cells).  xarray's sum skips a
    // missing term (steric.py:163, derived.py:435-438); the sweep above does not, so a column whose
    // sums turned NaN is integrated again from global memory with the skipna rule.  kLocalLayers: every
    // layer of the column is integrated again and overwritten.
#pragma unroll
    for (int k = 0; k < TC; ++k) poisoned |= is_nan_q(acc[k]);
    if (poisoned && in) {
      for (int b = 0; b < (LAYERS ? layer_count(L) : 1); ++b) {
#pragma unroll
        for (int k = 0; k < TC; ++k) acc[k] = 0.0;
        const i64 lvl = (i64)nz * P.ncol;
        for (int z = 0; z < nz; ++z) {
          const i64 j = (i64)z * P.ncol + c;
          const vbits v = ld_vraw(gV, j);
          double w, sub = 0.0;
          if (GLOBAL) {
            w = vraw_isnan(v) ? 0.0 : vraw_value(v);
          } else if (LAYERS) {
            const int lay = s_lay[z];
            const bool touches = lay != kNoLayer && (lay & 255) <= b && b <= (lay >> 8);
            w = (vraw_isnan(v) || !touches) ? 0.0 : layer_w(L, s_zi, depth, z, b);
            sub = __ldg(P.rho_ref + j);
          } else {
            w = vraw_isnan(v) ? 0.0 : level_dz(depth, s_zi[z], s_zi[z + 1]);
            if (!SELFREF) sub = __ldg(P.rho_ref + j);
          }
          if (!nonzero(w)) continue;
          eos.set_level(s_p[z]);
          if (SELFREF)  // the reference density again, from step 0 of this column (same arithmetic as in the sweep)
            sub = eos.rho((double)__ldg(gT + j), (double)__ldg(gS + j));
          // the same evaluation as the sweep (a pinned operand folded into the coefficients), so that a repaired
          // column does not depend on how the time axis was cut into chunks
          typename Eos<EOS>::Pinned pin = {};
          if (BC == 1) pin = eos.pin_t((double)__ldg(gT + j));
          if (BC == 2) pin = eos.pin_s((double)__ldg(gS + j));
#pragma unroll
          for (int k = SELFREF ? 1 : 0; k < TC; ++k) {
            if (t0 + k >= P.nt || (k == 0 && zero_first)) continue;
            const double Tv = (double)__ldg(gT + (BC == 1 ? 0 : (i64)(t0 + k) * lvl) + j);
            const double Sv = (double)__ldg(gS + (BC == 2 ? 0 : (i64)(t0 + k) * lvl) + j);
            const double rho = BC == 1 ? eos.rho_pinned_t(pin, Sv) : (BC == 2 ? eos.rho_pinned_s(pin, Tv) : eos.rho(Tv, Sv));
            fma_skipnan(acc[k], w, GLOBAL ? rho : rho - sub);
          }
        }
        if (LAYERS)
#pragma unroll
          for (int k = 0; k < TC; ++k) store_height(out, L, b, k, acc[k]);
      }
    }
    if (!GLOBAL && !LAYERS) {
      if (in) {
#pragma unroll
        for (int k = 0; k < TC; ++k)
          if (t0 + k < P.nt) P.eta[(i64)(t0 + k) * P.ncol + c] = surface_wet ? P.coef * acc[k] : nan("");
      }
    }
    if (GLOBAL) {
#pragma unroll
      for (int k = 0; k < TC; ++k) {
        const double sacc = warp_sum(in ? acc[k] : 0.0);
        if (lane == 0) red[warp * TC + k] = sacc;
      }
    } else if (SELFREF) {
      vol = warp_sum(vol);
      mass = warp_sum(mass);
      if (lane == 0) {
        red[warp * TC + 0] = vol;
        red[warp * TC + 1] = mass;
      }
    }
  }
  if (GLOBAL || SELFREF) {
    __syncthreads();
    if (tid < kRed && (SELFREF || t0 + tid < P.nt)) {
      double sacc = 0.0;
#pragma unroll
      for (int w8 = 0; w8 < kConsumerWarps; ++w8) sacc += red[w8 * TC + tid];
      const i64 row = SELFREF ? tid : (t0 + tid);
      P.partials[row * P.tiles + tile] = sacc;
    }
  }
}

// ----------------------------------------------------------------------- host side

#ifndef ML_TMA_FLAT_TU
static bool rows_aligned(int dtype, int64_t ncol) { return ncol % (dtype == ML_F32 ? 4 : 2) == 0; }

static bool common_eligible(int dtype, int vref_dtype, const void* T, const void* S, int64_t nt, int64_t nz,
                            int64_t ncol) {
  if ((dtype != ML_F32 && dtype != ML_F64) || vref_dtype != dtype) return false;  // volcello stored like the fields
  if ((reinterpret_cast<uintptr_t>(T) | reinterpret_cast<uintptr_t>(S)) & 15u) return false;
  if (ncol < kTile || ncol > 0x7fffff00ll) return false;
  // rows that are not a multiple of 16 bytes go through rank-1 maps, whose 32-bit coordinate must reach the end of
  // the last (zero-padded) chunk
  const int64_t mtc = dtype == ML_F32 ? 12 : 6;
  if (!rows_aligned(dtype, ncol) && (double)((nt + mtc - 1) / mtc * mtc) * (double)nz * (double)ncol >= 2147483647.0) return false;
  if (nt < 1 || nz < 1 || nz > 512) return false;
  // grid.x = tiles * time chunks (chunks of at least 4 steps)
  if ((double)((ncol + kTile - 1) / kTile) * (double)((nt + 3) / 4) > 2147483647.0) return false;
  // TMA global strides must stay below 2^40 bytes
  if ((double)ncol * (double)nz * 8.0 >= 1099511627776.0) return false;
  return encode_fn() != nullptr;
}

bool local_eligible(int dtype, const void* T, const void* S, int, int, const double*, const void*, int vref_dtype,
                    int64_t nt, int64_t nz, int64_t ncol, const double*, const double* delta_rho) {
  return delta_rho == nullptr && common_eligible(dtype, vref_dtype, T, S, nt, nz, ncol);
}

bool global_eligible(int dtype, const void* T, const void* S, int, int, const void*, int vref_dtype, int64_t nt,
                     int64_t nz, int64_t ncol) {
  return common_eligible(dtype, vref_dtype, T, S, nt, nz, ncol);
}

#else
static bool rows_aligned(int dtype, int64_t ncol);
#endif

template <int TC>
inline size_t smem_bytes(int bc, int nz, int mode, int es) {
  const int kStages = stages_of(mode, bc, es);
  return (size_t)kStages * (size_t)((bc == 0 ? 2 * TC : TC + 1) * kTile * es) + 3 * kStages * sizeof(uint64_t) +
         (size_t)kConsumerWarps * TC * sizeof(double) + (size_t)(2 * nz + 1) * sizeof(double) + 2 * kTile * sizeof(int) + 128 +
         (mode == kLocalLayers ? (size_t)nz * sizeof(int) : 0);
}

template <typename TIn, int EOS, int TC, int BC, int MODE, bool FLAT>
static int launch_one(const CUtensorMap& mT, const CUtensorMap& mS, const Params& P, unsigned tiles, unsigned chunks,
                      cudaStream_t st, const LayerParams* lp) {
  auto kern = k_steric_tma<TIn, EOS, TC, BC, MODE, FLAT>;
  const size_t smem = smem_bytes<TC>(BC, P.nz, MODE, (int)sizeof(TIn));
  // opt in to > 48 KB of dynamic shared memory; the attribute is per device and per context, so it
  // is set on every launch (a host-side table lookup) rather than cached in a static
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(k_steric_tma)");
  Params Q = P;
  Q.tiles = tiles;
  Q.nchunks = chunks;
  LayersOf<MODE> L{};
  if constexpr (MODE == kLocalLayers) L = *lp;
  kern<<<tiles * chunks, kThreads, smem, st>>>(mT, mS, Q, L);
  return launched("k_steric_tma");
}

template <typename TIn, int EOS, int TC, int MODE, bool FLAT>
static int launch_bc(int bc, const CUtensorMap& mT, const CUtensorMap& mS, const Params& P, unsigned tiles,
                     unsigned chunks, cudaStream_t st, const LayerParams* lp) {
#ifdef ML_TMA_FAST_BUILD  // experiment builds: only the fp32 / Wright / 12-step / no-broadcast kernels
  if (sizeof(TIn) != 4 || EOS != 0 || TC != 12 || bc != 0) return fail(ML_ERR_MODE, "kernel not instantiated in a fast build");
  return launch_one<float, 0, 12, 0, MODE, FLAT>(mT, mS, P, tiles, chunks, st, lp);
#else
  if (bc == 0) return launch_one<TIn, EOS, TC, 0, MODE, FLAT>(mT, mS, P, tiles, chunks, st, lp);
  if (bc == 1) return launch_one<TIn, EOS, TC, 1, MODE, FLAT>(mT, mS, P, tiles, chunks, st, lp);
  return launch_one<TIn, EOS, TC, 2, MODE, FLAT>(mT, mS, P, tiles, chunks, st, lp);
#endif
}

// A launch covers `chunks` register chunks of `tc` time steps starting at `t_start`.  The time axis
// is cut into 12-step chunks plus ONE remainder chunk of the smallest width in {4, 8, 12} that holds
// what is left: rows past nt are zero-filled by the TMA unit and cost no bytes, but they do cost
// arithmetic, so a 10-step window runs as one 12-step chunk (2 idle rows), not as 8 + 8 (6 idle).
// Fields stored as fp64 take twice the shared memory per step: 6-step chunks, remainder in {4, 6}.
struct Segment {
  CUtensorMap mT, mS;
  int tc, t_start;
  unsigned chunks;
};

static unsigned tiles_of(const Params& P) {
  const int cols = cols_of(P.es, P.flat != 0);
  return (unsigned)((P.ncol + cols - 1) / cols);
}
static int main_tc(int es) { return es == 4 ? 12 : 6; }
static int remainder_tc(int steps, int es) {
  if (es == 4) return steps <= 4 ? 4 : (steps <= 8 ? 8 : 12);
  return steps <= 4 ? 4 : 6;
}

struct Plan {
  int bc;
  unsigned tiles;
  int nseg;
  Segment seg[2];
};

static int add_segment(Plan* pl, const void* T, const void* S, int t_bcast, int s_bcast, const Params& P, int tc,
                       int t_start, unsigned chunks) {
  Segment& g = pl->seg[pl->nseg++];
  g.tc = tc;
  g.t_start = t_start;
  g.chunks = chunks;
  bool okT, okS;
  if (P.flat) {
    const i64 lvl = (i64)P.nz * P.ncol;
    okT = make_flat_map(&g.mT, T, t_bcast ? lvl : lvl * P.nt, kTile, P.es);
    okS = make_flat_map(&g.mS, S, s_bcast ? lvl : lvl * P.nt, kTile, P.es);
  } else {
    okT = t_bcast ? make_map(&g.mT, T, 2, P.ncol, P.nz, 1, 1, kTile, P.es) : make_map(&g.mT, T, 3, P.ncol, P.nz, P.nt, tc, kTile, P.es);
    okS = s_bcast ? make_map(&g.mS, S, 2, P.ncol, P.nz, 1, 1, kTile, P.es) : make_map(&g.mS, S, 3, P.ncol, P.nz, P.nt, tc, kTile, P.es);
  }
  return (okT && okS) ? ML_OK : fail(ML_ERR_ALIGN, "cuTensorMapEncodeTiled rejected the field layout");
}

// segments covering the time steps [t_begin, nt)
static int make_plan(Plan* pl, const void* T, const void* S, int t_bcast, int s_bcast, const Params& P, int t_begin) {
  pl->bc = t_bcast ? 1 : (s_bcast ? 2 : 0);
  pl->tiles = tiles_of(P);
  pl->nseg = 0;
  const int mtc = main_tc(P.es);
  const int steps = P.nt - t_begin, full = steps / mtc, rest = steps % mtc;
  int rc = ML_OK;
  if (full > 0) rc = add_segment(pl, T, S, t_bcast, s_bcast, P, mtc, t_begin, (unsigned)full);
  if (rc == ML_OK && rest > 0)
    rc = add_segment(pl, T, S, t_bcast, s_bcast, P, remainder_tc(rest, P.es), t_begin + mtc * full, 1u);
  return rc;
}

template <int MODE, bool FLAT>
static int launch_segment(int eos, const Plan& pl, const Segment& g, Params P, cudaStream_t st, const LayerParams* lp) {
  P.t_start = g.t_start;
#define ML_TMA_GO(TIN, E, TCV) return launch_bc<TIN, E, TCV, MODE, FLAT>(pl.bc, g.mT, g.mS, P, pl.tiles, g.chunks, st, lp)
  if (P.es == 8) {  // fields stored as fp64
#ifndef ML_TMA_FAST_BUILD
    if (eos == ML_EOS_WRIGHT) {
      if (g.tc == 6) ML_TMA_GO(double, 0, 6);
      ML_TMA_GO(double, 0, 4);
    }
    if (g.tc == 6) ML_TMA_GO(double, 1, 6);
    ML_TMA_GO(double, 1, 4);
#else
    return fail(ML_ERR_MODE, "kernel not instantiated in a fast build");
#endif
  }
  if (eos == ML_EOS_WRIGHT) {
    if (g.tc == 12) ML_TMA_GO(float, 0, 12);
    if (g.tc == 8) ML_TMA_GO(float, 0, 8);
    ML_TMA_GO(float, 0, 4);
  }
  if (g.tc == 12) ML_TMA_GO(float, 1, 12);
  if (g.tc == 8) ML_TMA_GO(float, 1, 8);
  ML_TMA_GO(float, 1, 4);
#undef ML_TMA_GO
}

// The kernels for rows that are not a multiple of 16 bytes (rank-1 maps, FLAT = true) are compiled in their own
// translation unit (ml_tma_flat.cu includes this file with ML_TMA_FLAT_TU defined): a second set of instantiations
// next to these would double the compile time of this file, and a run-time switch inside one kernel cost the
// headline kernel a spill in its level loop.
int launch_segment_flat(int mode, int eos, const Plan& pl, const Segment& g, const Params& P, cudaStream_t st,
                        const LayerParams* lp);

#ifdef ML_TMA_FLAT_TU
int launch_segment_flat(int mode, int eos, const Plan& pl, const Segment& g, const Params& P, cudaStream_t st,
                        const LayerParams* lp) {
  if (mode == kLocal) return launch_segment<kLocal, true>(eos, pl, g, P, st, lp);
  if (mode == kLocalLayers) return launch_segment<kLocalLayers, true>(eos, pl, g, P, st, lp);
  if (mode == kGlobal) return launch_segment<kGlobal, true>(eos, pl, g, P, st, lp);
  return launch_segment<kSelfRef, true>(eos, pl, g, P, st, lp);
}
#else

template <int MODE>
static int launch_plan(int eos, const Plan& pl, const Params& P, cudaStream_t st, const LayerParams* lp = nullptr) {
  for (int i = 0; i < pl.nseg; ++i) {
    int rc = P.flat ? launch_segment_flat(MODE, eos, pl, pl.seg[i], P, st, lp)
                    : launch_segment<MODE, false>(eos, pl, pl.seg[i], P, st, lp);
    if (rc) return rc;
  }
  return ML_OK;
}

static Params base_params(const void* T, const void* S, const void* v_ref, int vref_dtype, const double* p_level,
                          int nt, int nz, int64_t ncol) {
  Params P;
  P.T = T;
  P.S = S;
  P.es = vref_dtype == ML_F64 ? 8 : 4;  // eligibility guarantees fields and volcello share a dtype
  P.flat = rows_aligned(vref_dtype, ncol) ? 0 : 1;
  P.rho_ref = nullptr;
  P.rho_ref_out = nullptr;
  P.v_ref = v_ref;
  P.z_i = nullptr;
  P.deptho = nullptr;
  P.p_level = p_level;
  P.coef = 0.0;
  P.nt = nt;
  P.nz = nz;
  P.t_start = 0;
  P.first_is_reference = 0;
  P.nchunks = 1;
  P.tiles = 0;
  P.ncol = ncol;
  P.eta = nullptr;
  P.partials = nullptr;
  return P;
}

int launch_local(int eos, int, const void* T, const void* S, int t_bcast, int s_bcast, const double* rho_ref,
                 const void* v_ref, int vref_dtype, const double* z_i, const double* deptho, const double* p_level,
                 double coef, int nt, int nz, int64_t ncol, double* eta, double*, cudaStream_t st,
                 int first_is_reference) {
  Params P = base_params(T, S, v_ref, vref_dtype, p_level, nt, nz, ncol);
  P.first_is_reference = first_is_reference;
  P.rho_ref = rho_ref;
  P.z_i = z_i;
  P.deptho = deptho;
  P.coef = coef;
  P.eta = eta;
  Plan pl;
  int rc = make_plan(&pl, T, S, t_bcast, s_bcast, P, 0);
  if (rc) return rc;
  return launch_plan<kLocal>(eos, pl, P, st);
}

int launch_local_layers(int eos, const void* T, const void* S, int t_bcast, int s_bcast, const double* rho_ref,
                        const void* v_ref, int vref_dtype, const double* z_i, const double* deptho, const double* p_level,
                        double coef, const double* edges, int nlayers, int nt, int nz, int64_t ncol, double* eta,
                        cudaStream_t st) {
  Params P = base_params(T, S, v_ref, vref_dtype, p_level, nt, nz, ncol);
  P.rho_ref = rho_ref;
  P.z_i = z_i;
  P.deptho = deptho;
  P.coef = coef;
  P.eta = eta;
  LayerParams lp;
  lp.nlayers = nlayers;
  for (int b = 0; b <= ML_MAX_LAYERS; ++b) lp.edges[b] = b <= nlayers ? edges[b] : 0.0;
  Plan pl;
  int rc = make_plan(&pl, T, S, t_bcast, s_bcast, P, 0);
  if (rc) return rc;
  return launch_plan<kLocalLayers>(eos, pl, P, st, &lp);
}

int launch_selfref(int eos, const void* T, const void* S, int t_bcast, int s_bcast, const void* v_ref, int vref_dtype,
                   const double* z_i, const double* deptho, const double* p_level, double coef, int nt, int nz,
                   int64_t ncol, double* eta, double* rho_ref, double* sums, double* partials, cudaStream_t st) {
  Params P = base_params(T, S, v_ref, vref_dtype, p_level, nt, nz, ncol);
  P.rho_ref_out = rho_ref;
  P.z_i = z_i;
  P.deptho = deptho;
  P.coef = coef;
  P.eta = eta;
  P.partials = partials;
  // the chunk that starts at the reference step: rho_ref, volo, masso and eta in one pass
  Plan first;
  first.bc = t_bcast ? 1 : (s_bcast ? 2 : 0);
  first.tiles = tiles_of(P);
  first.nseg = 0;
  const int tc0 = nt >= main_tc(P.es) ? main_tc(P.es) : remainder_tc(nt, P.es);
  int rc = add_segment(&first, T, S, t_bcast, s_bcast, P, tc0, 0, 1u);
  if (rc) return rc;
  if ((rc = launch_plan<kSelfRef>(eos, first, P, st))) return rc;
  if ((rc = reduce_rows(partials, first.tiles, sums, 2, st))) return rc;
  if (nt > tc0) {  // later chunks read the rho_ref just written (same stream: ordered)
    Plan rest;
    if ((rc = make_plan(&rest, T, S, t_bcast, s_bcast, P, tc0))) return rc;
    P.rho_ref = rho_ref;
    P.rho_ref_out = nullptr;
    rc = launch_plan<kLocal>(eos, rest, P, st);
  }
  return rc;
}

int launch_global(int eos, int, const void* T, const void* S, int t_bcast, int s_bcast, const void* v_ref,
                  int vref_dtype, const double* p_level, int nt, int nz, int64_t ncol, double* masso, double* partials,
                  cudaStream_t st) {
  Params P = base_params(T, S, v_ref, vref_dtype, p_level, nt, nz, ncol);
  P.partials = partials;
  Plan pl;
  int rc = make_plan(&pl, T, S, t_bcast, s_bcast, P, 0);
  if (rc) return rc;
  if ((rc = launch_plan<kGlobal>(eos, pl, P, st))) return rc;
  return reduce_rows(partials, pl.tiles, masso, nt, st);
}

#endif  // ML_TMA_FLAT_TU

}  // namespace tma
}  // namespace ml
