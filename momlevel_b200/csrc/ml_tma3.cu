// ml_tma3.cu -- steric, thermosteric and halosteric height from ONE pass over T and S (sm_100a).
//
// BASELINE config 2 names the three heights together; the reference computes one per call and only swaps
// which operand of the equation of state is held at its reference value (src/momlevel/steric.py:115-121):
//     steric        rho(T, S)          thermosteric  rho(T, S_ref)          halosteric  rho(T_ref, S)
// Three launches of the single-height kernel (ml_tma.cu) read T and S three times (28 GB for an OM4p25
// year where one pass needs 13 GB).  Here a CTA stages, per level, the TC time rows of T and of S plus the
// level's T_ref and S_ref rows in one shared-memory ring stage ({256 columns} x (2 TC + 2) rows, one
// mbarrier), and every thread evaluates the three densities of a point from the same two shared-memory
// words: the loads, the two fp32->fp64 conversions, the level bookkeeping and the dz / mask logic are paid
// once instead of three times, the T-only sub-polynomials of the Wright fit are shared between the steric
// and the thermosteric density by the compiler (same expressions on the same registers), and the halosteric
// one costs four fused multiply-adds once T_ref is folded into the coefficients for the level.
//
// The arithmetic of each height is the single-height kernel's, instruction for instruction
// (Eos<0>::terms / terms_pinned_s / terms_pinned_t + div_lean), so the three fields are bit-identical to
// three ml_steric_local / ml_steric_local_selfref calls; tests/test_gpu_steric.py checks that.
//
// Modes:  kLocal3    reference supplied: T_ref, S_ref [nz][ncol] fp32 staged by 2-D maps, rho_ref read
//         kSelfRef3  reference = step 0 of the fields (what steric() does by default): T_ref / S_ref are the
//                    step-0 slabs, rho_ref is evaluated per level from the staged reference row (every
//                    chunk: 17 fp64 instructions per level and column instead of an 8-byte load), and the
//                    chunk that starts at step 0 also reduces volo / masso, stores rho_ref when asked and
//                    leaves its step-0 heights at exactly zero.
//         kLocalLayers3  kLocal3 split by depth layer (ml_tma.cu, kLocalLayers): level z feeds layer b with the weight
//                    calc_dz(top=edges[b], bottom=edges[b+1]); the 3 x TC sums belong to one layer at a time and are
//                    stored ([t][layer][col] per height) when the sweep leaves the layer's last level.  A level that
//                    holds an edge (at most nlayers - 1 of them) evaluates its three densities again after the
//                    straight-line block instead of keeping 3 x TC differences live through it; the evaluation is the
//                    same, so are the bits.
// Eligibility is the single-height family's (fp32, 16-byte aligned, ncol % 4 == 0, ncol >= 256).
#include "ml_tma_dev.cuh"
#include "ml_tma.cuh"

#include <type_traits>

namespace ml {
namespace tma {

#include <stdlib.h>
// Montgomery's trick for the three reciprocals of a point (one MUFU.RCP64H seed instead of three; same fp64
// count, longer chains).  Off: the results would no longer be bit-identical to the single-height kernels.
#ifndef ML_TMA3_MONTGOMERY
#define ML_TMA3_MONTGOMERY 0
#endif

enum Mode3 { kLocal3 = 0, kSelfRef3 = 2, kLocalLayers3 = 4 };
template <int MODE>
using LayersOf3 = typename std::conditional<MODE == kLocalLayers3, LayerParams, NoLayers>::type;

struct Params3 {
  const float *T, *S;        // [nt][nz][ncol]  (repair pass; the sweep goes through the tensor maps)
  const float *Tref, *Sref;  // [nz][ncol]
  const double* rho_ref;     // kLocal3, kLocalLayers3: read
  double* rho_ref_out;       // kSelfRef3, chunk 0: written (may be NULL)
  const float* v_ref;
  const double *z_i, *deptho, *p_level;
  double coef;
  int nt, nz, t_start;
  unsigned nchunks, tiles;
  i64 ncol;
  double* eta[3];            // steric, thermosteric, halosteric: [nt][ncol] each, kLocalLayers3 [nt][nlayers][ncol]
                             // (NULL = not wanted)
  double* partials;          // kSelfRef3: [2][tiles] = {volo, masso}, written by the chunk that starts at step 0
};

// Registers: 3 x TC running sums.  TC = 12 needs ~216 registers (one CTA of 8 warps per SM, a 6-level ring);
// TC <= 8 fits the 128 of two CTAs per SM (4-level rings).
// TILE = 128 halves the CTA (one warp per SM sub-partition) and doubles the CTAs per SM: the four warps that share
// a sub-partition then come from four CTAs at unrelated depths of their sweeps, instead of a fixed deep / shallow
// pair of one CTA whose partner idles whenever its own band is dry.
__host__ __device__ constexpr int ctas_per_sm3(int tc, int tile = 256) { return (tc > 8 ? 1 : 2) * (256 / tile); }
__host__ __device__ constexpr int stages3(int tc) { return tc > 8 ? 6 : 4; }

template <int EOS, int TC, int MODE, int TILE>
__global__ void __launch_bounds__(TILE, ctas_per_sm3(TC, TILE))
    k_steric_tma3(const __grid_constant__ CUtensorMap mapT, const __grid_constant__ CUtensorMap mapS,
                  const __grid_constant__ CUtensorMap mapTr, const __grid_constant__ CUtensorMap mapSr, const Params3 P,
                  const LayersOf3<MODE> L) {
  constexpr bool SELFREF = MODE == kSelfRef3;
  constexpr bool LAYERS = MODE == kLocalLayers3;
  constexpr int kWarpsT = TILE / 32;
  constexpr int kStages = stages3(TC);
  constexpr int kRows = 2 * TC + 2;
  constexpr uint32_t kStageBytes = (uint32_t)kRows * TILE * sizeof(float);
  constexpr int kStageFloats = kRows * TILE;
  constexpr int kOffS = TC * TILE, kOffTr = 2 * TC * TILE, kOffSr = (2 * TC + 1) * TILE;

  extern __shared__ __align__(128) unsigned char smem_raw[];
  float* stage_base = reinterpret_cast<float*>(smem_raw);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + (size_t)kStages * kStageBytes);
  uint64_t* empty = full + kStages;
  int* released = reinterpret_cast<int*>(full + 2 * kStages);
  double* red = reinterpret_cast<double*>(full + 3 * kStages);  // [kWarpsT][2]
  double* s_p = red + kWarpsT * 2;
  double* s_zi = s_p + P.nz;
  int* s_key = reinterpret_cast<int*>(s_zi + P.nz + 1);
  int* s_col = s_key + TILE;
  int* s_lay = s_col + TILE;  // [nz] kLocalLayers3: layers touching the level

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const unsigned tile = blockIdx.x / P.nchunks;
  const int c0 = (int)tile * TILE;
  const int t0 = P.t_start + (int)(blockIdx.x - tile * P.nchunks) * TC;
  const int nz = P.nz;
  const bool chunk0 = SELFREF && t0 == 0;  // this CTA's chunk starts at the reference step

  auto refill_stage = [&](int z) {
    const int s = z % kStages;
    float* d = stage_base + (size_t)s * kStageFloats;
    mbar_expect_tx(full + s, kStageBytes);
    tma_load_3d(d, &mapT, full + s, c0, z, t0);
    tma_load_3d(d + kOffS, &mapS, full + s, c0, z, t0);
    tma_load_2d(d + kOffTr, &mapTr, full + s, c0, z);
    tma_load_2d(d + kOffSr, &mapSr, full + s, c0, z);
  };

  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full + s, 1);
      mbar_init(empty + s, kWarpsT);
      released[s] = 0;
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    for (int z = 0; z < kStages && z < nz; ++z) refill_stage(z);
  }
  for (int i = threadIdx.x; i < nz; i += TILE) s_p[i] = __ldg(P.p_level + i);
  for (int i = threadIdx.x; i <= nz; i += TILE) s_zi[i] = __ldg(P.z_i + i);
  if (LAYERS) fill_layer_table<TILE>(s_lay, P.z_i, nz, L);
  __syncthreads();

  // columns of the tile ranked by wet depth (see ml_tma.cu): thread i integrates the i-th deepest column
  int col;
  {
    const i64 cg = (i64)c0 + tid;
    const int key = wet_levels(cg < P.ncol ? __ldg(P.deptho + cg) : 0.0, s_zi, nz);
    // CTAs that share an SM should not all put their deepest band on the same sub-partition (2 % with two CTAs per SM)
    const int rot = (int)((blockIdx.x * 2654435761u) >> 20) & 3;
    col = sorted_column_t<TILE>(key, reinterpret_cast<unsigned*>(s_key), s_col, rot);
  }

  const i64 c = (i64)c0 + col;
  const bool in = c < P.ncol;
  const i64 cc = in ? c : (P.ncol - 1);
  Eos<EOS> eos;
  double acc[3][TC];
#pragma unroll
  for (int v = 0; v < 3; ++v)
#pragma unroll
    for (int k = 0; k < TC; ++k) acc[v][k] = 0.0;
  double vol = 0.0, mass = 0.0;
  double depth = __ldg(P.deptho + cc);
  if (isnan(depth)) depth = 0.0;  // derived.py:295
  double rref_n = 0.0;
  unsigned v_n = ld_vraw(P.v_ref, cc);
  if (!SELFREF) rref_n = __ldg(P.rho_ref + cc);
  const bool surface_wet = !vraw_isnan(v_n);  // steric.py:166
  // kLocalLayers3: the layer the sums belong to, whether a stored sum met a missing value, and where each height goes
  int cur = 0;
  bool poisoned = false;
  LayerOut out[3];
#pragma unroll
  for (int v = 0; v < 3; ++v) out[v] = {P.eta[v], P.coef, P.nt, P.ncol, c, t0, in && P.eta[v] != nullptr, surface_wet};

  for (int z = 0; z < nz; ++z) {
    const double rref_z = rref_n;
    const unsigned v_z = v_n;
#ifndef ML_TMA3_PREFETCH_LATE
    if (z + 1 < nz) {
      const i64 j = (i64)(z + 1) * P.ncol + cc;
      v_n = ld_vraw(P.v_ref, j);
      if (!SELFREF) rref_n = __ldg(P.rho_ref + j);
    }
#endif
    const bool dry = vraw_isnan(v_z);
    double w = level_dz(depth, s_zi[z], s_zi[z + 1]);
    if (dry || (!SELFREF && isnan(rref_z))) w = 0.0;  // steric.py:151-153
    if (LAYERS && s_lay[z] == kNoLayer) w = 0.0;      // no layer takes this level
    eos.set_level(s_p[z]);
    const bool live = nonzero(w);
    // kLocalLayers3: close the layers that ended above this level (in every warp, wet or not); `wl` is the weight of
    // the level in its one layer, or -- where an edge falls inside the level (lo < hi) -- in layer lo
    int lo = 0, hi = 0;
    double wl = w;
    if (LAYERS && s_lay[z] != kNoLayer) {
      lo = s_lay[z] & 255;
      hi = s_lay[z] >> 8;
      for (; cur < lo; ++cur)
#pragma unroll
        for (int v = 0; v < 3; ++v) close_layer<TC>(acc[v], poisoned, out[v], L, cur);
      wl = live ? layer_w(L, s_zi, depth, z, lo) : 0.0;
    }
    const unsigned live_lanes = __ballot_sync(0xffffffffu, live);
    const int s = z % kStages;
    const float* st = stage_base + (size_t)s * kStageFloats;
    mbar_wait(full + s, (uint32_t)(z / kStages) & 1u);
    double sub = SELFREF ? 0.0 : rref_z;
    if (live_lanes != 0u) {
      // a dry lane of a partly wet warp evaluates the column of the warp's first wet lane (a shared-memory
      // broadcast) with weight 0, so no missing value reaches the sums and they are plain FMAs (ml_tma.cu)
      const int first_wet = __shfl_sync(0xffffffffu, col, __ffs(live_lanes) - 1);
      const int src = live ? col : first_wet;
      const double Tr = (double)st[kOffTr + src], Sr = (double)st[kOffSr + src];
      if (SELFREF) {
        // reference density of this level (reference.py:60-71): the chunk that starts at the reference step owes
        // it for every column (volo / masso, rho_ref_out), the others only where they integrate
        const int own = chunk0 ? col : src;
        sub = eos.rho((double)st[kOffTr + own], (double)st[kOffSr + own]);
      }
      const typename Eos<EOS>::Pinned qs = eos.pin_s(Sr);  // thermosteric: S held at the reference slab
      const typename Eos<EOS>::Pinned qt = eos.pin_t(Tr);  // halosteric: T held at the reference slab
      const double rsub = live ? sub : 0.0;  // keep a missing rho_ref of a dry lane out of 0 * (...)
#pragma unroll
      for (int kk = 0; kk < TC; ++kk) {
        if (SELFREF && kk == 0 && chunk0) continue;  // step 0 is the reference itself: exactly zero
        const double Tv = (double)st[kk * TILE + src];
        const double Sv = (double)st[kOffS + kk * TILE + src];
        if constexpr (ML_TMA3_MONTGOMERY != 0 && EOS == 0) {
          double p1, d1, p2, d2, p3, d3;
          eos.terms_of(Tv, Sv, p1, d1);
          eos.terms_pinned_s(qs, Tv, p2, d2);
          eos.terms_pinned_t(qt, Sv, p3, d3);
          const double d12 = d1 * d2;
          const double R = rcp_lean(d12 * d3);
          const double R12 = R * d3;
          acc[0][kk] = fma(w, p1 * (R12 * d2) - rsub, acc[0][kk]);
          acc[1][kk] = fma(w, p2 * (R12 * d1) - rsub, acc[1][kk]);
          acc[2][kk] = fma(w, p3 * (R * d12) - rsub, acc[2][kk]);
        } else {
          acc[0][kk] = fma(LAYERS ? wl : w, eos.rho(Tv, Sv) - rsub, acc[0][kk]);
          acc[1][kk] = fma(LAYERS ? wl : w, eos.rho_pinned_s(qs, Tv) - rsub, acc[1][kk]);
          acc[2][kk] = fma(LAYERS ? wl : w, eos.rho_pinned_t(qt, Sv) - rsub, acc[2][kk]);
        }
      }
    } else if (chunk0) {
      // a warp without water still owes rho_ref (reference.py:71 evaluates the EOS everywhere); over land T, S
      // are missing and so is the result -- no arithmetic needed
      const float tN = st[kOffTr + col], sN = st[kOffSr + col];
      sub = nan("");
      if (__any_sync(0xffffffffu, !(isnan(tN) || isnan(sN)))) sub = eos.rho((double)tN, (double)sN);
    }
    if (chunk0 && in) {
      if (!dry) {  // volo, masso: skipna sums (derived.py:787-789, :435-438)
        const double v = vraw_value(v_z);
        vol += v;
        const double m = sub * v;
        if (!is_nan_q(m)) mass += m;
      }
      if (P.rho_ref_out) P.rho_ref_out[(i64)z * P.ncol + c] = sub;
    }
    if (LAYERS && lo < hi) {
      // an edge falls inside level z: layers lo .. hi - 1 are stored and the sums start layer hi.  The differences
      // rho - rho_ref of the level are evaluated again here, out of the straight-line block above (a layer test
      // inside it broke the folding of - rho_ref into the EOS's last multiply: other bits, 1.77x the time)
      if (live_lanes != 0u) {
        const int first_wet = __shfl_sync(0xffffffffu, col, __ffs(live_lanes) - 1);
        const int src = live ? col : first_wet;
        const typename Eos<EOS>::Pinned qs = eos.pin_s((double)st[kOffSr + src]);
        const typename Eos<EOS>::Pinned qt = eos.pin_t((double)st[kOffTr + src]);
        const double rsub = live ? sub : 0.0;
#pragma unroll
        for (int kk = 0; kk < TC; ++kk) {
          const double Tv = (double)st[kk * TILE + src];
          const double Sv = (double)st[kOffS + kk * TILE + src];
          split_level(acc[0][kk], poisoned, out[0], L, s_zi, depth, z, lo, hi, live, kk, eos.rho(Tv, Sv) - rsub);
          split_level(acc[1][kk], poisoned, out[1], L, s_zi, depth, z, lo, hi, live, kk, eos.rho_pinned_s(qs, Tv) - rsub);
          split_level(acc[2][kk], poisoned, out[2], L, s_zi, depth, z, lo, hi, live, kk, eos.rho_pinned_t(qt, Sv) - rsub);
        }
      } else {
#pragma unroll
        for (int kk = 0; kk < TC; ++kk)  // a warp without water still closes its layers
#pragma unroll
          for (int v = 0; v < 3; ++v) split_level(acc[v][kk], poisoned, out[v], L, s_zi, depth, z, lo, hi, live, kk, 0.0);
      }
      cur = hi;
    }
    __syncwarp();
    if (lane == 0 && stage_done(empty + s, released + s, kWarpsT, (uint32_t)(z / kStages) & 1u) && z + kStages < nz)
      refill_stage(z + kStages);
#ifdef ML_TMA3_PREFETCH_LATE
    if (z + 1 < nz) {  // behind the release: it then has no load of this thread to wait for
      const i64 j = (i64)(z + 1) * P.ncol + cc;
      v_n = ld_vraw(P.v_ref, j);
      if (!SELFREF) rref_n = __ldg(P.rho_ref + j);
    }
#endif
  }

  // Repair pass (rare: consistent model output has no holes at wet cells).  A hole at a wet cell turned some of the
  // column's sums into NaN; xarray's sum skips the missing term (steric.py:163), so the column is integrated again
  // from global memory with that rule -- all three heights, with the sweep's own evaluation: a height that met no
  // hole comes out as it was, and a repaired one does not depend on how the time axis was cut into chunks, so the
  // fields stay identical to the single-height kernels'.  (Kept in this simple form on purpose: repairing per height,
  // or out of line, changed the register allocation of the sweep above and cost it 4 %.)  kLocalLayers3: every layer of
  // every height of the column is integrated again and overwritten.
  if (LAYERS)
    for (; cur < layer_count(L); ++cur)  // the last layer, and those wholly below the grid: 0
#pragma unroll
      for (int v = 0; v < 3; ++v) close_layer<TC>(acc[v], poisoned, out[v], L, cur);
#pragma unroll
  for (int v = 0; v < 3; ++v)
#pragma unroll
    for (int k = 0; k < TC; ++k) poisoned |= is_nan_q(acc[v][k]);
  if (poisoned && in) {
    for (int b = 0; b < (LAYERS ? layer_count(L) : 1); ++b) {
#pragma unroll
      for (int v = 0; v < 3; ++v)
#pragma unroll
        for (int k = 0; k < TC; ++k) acc[v][k] = 0.0;
      const i64 lvl = (i64)nz * P.ncol;
      for (int z = 0; z < nz; ++z) {
        const i64 j = (i64)z * P.ncol + c;
        const unsigned v = ld_vraw(P.v_ref, j);
        double w = vraw_isnan(v) ? 0.0 : level_dz(depth, s_zi[z], s_zi[z + 1]);
        if (LAYERS) {
          const bool touches = layer_touches(s_lay[z], b);
          w = (vraw_isnan(v) || !touches) ? 0.0 : layer_w(L, s_zi, depth, z, b);
        }
        if (!nonzero(w)) continue;
        eos.set_level(s_p[z]);
        const double Tr = (double)__ldg(P.Tref + j), Sr = (double)__ldg(P.Sref + j);
        const double sub = SELFREF ? eos.rho(Tr, Sr) : __ldg(P.rho_ref + j);
        const typename Eos<EOS>::Pinned qs = eos.pin_s(Sr);
        const typename Eos<EOS>::Pinned qt = eos.pin_t(Tr);
#pragma unroll
        for (int k = 0; k < TC; ++k) {
          if (t0 + k >= P.nt || (chunk0 && k == 0)) continue;
          const double Tv = (double)__ldg(P.T + (i64)(t0 + k) * lvl + j);
          const double Sv = (double)__ldg(P.S + (i64)(t0 + k) * lvl + j);
          fma_skipnan(acc[0][k], w, eos.rho(Tv, Sv) - sub);
          fma_skipnan(acc[1][k], w, eos.rho_pinned_s(qs, Tv) - sub);
          fma_skipnan(acc[2][k], w, eos.rho_pinned_t(qt, Sv) - sub);
        }
      }
      if (LAYERS)
#pragma unroll
        for (int v = 0; v < 3; ++v)
#pragma unroll
          for (int k = 0; k < TC; ++k) store_height(out[v], L, b, k, acc[v][k]);
    }
  }
  if (in && !LAYERS) {
#pragma unroll
    for (int v = 0; v < 3; ++v) {
      if (P.eta[v] == nullptr) continue;
#pragma unroll
      for (int k = 0; k < TC; ++k)
        if (t0 + k < P.nt) P.eta[v][(i64)(t0 + k) * P.ncol + c] = surface_wet ? P.coef * acc[v][k] : nan("");
    }
  }
  if (SELFREF && chunk0) {  // uniform per CTA
    vol = warp_sum(vol);
    mass = warp_sum(mass);
    if (lane == 0) {
      red[warp * 2 + 0] = vol;
      red[warp * 2 + 1] = mass;
    }
    __syncthreads();
    if (tid < 2) {
      double sacc = 0.0;
#pragma unroll
      for (int w8 = 0; w8 < kWarpsT; ++w8) sacc += red[w8 * 2 + tid];
      P.partials[(i64)tid * P.tiles + tile] = sacc;
    }
  }
}

// ------------------------------------------------------------------ global masses from one pass
// The global branch (steric.py:134-135) of the three variants: per step the volume-weighted sums
//     M_steric = sum rho(T, S) V     M_thermo = sum rho(T, S_ref) V     M_halo = sum rho(T_ref, S) V
// with V = reference["volcello"] and skipna sums (derived.py:435-438).  The stage layout is the local kernel's
// (TC rows of T, TC rows of S, one T_ref and one S_ref row per level); there is no z_i / deptho / rho_ref, the weight
// is the reference volume of the level.  Everything that decides the bits of a mass is the single-height global kernel's
// (ml_tma.cu, kGlobal): 256-column tiles, columns ranked by the number of levels with a present volume, the dry lane
// that borrows the first wet lane's column, the per-density instructions, the repair pass and the warp / CTA reduction
// order, so each mass is bit-identical to one ml_steric_global launch with BC = 0 / 2 / 1.
//   kGlobal3         T_ref, S_ref supplied
//   kGlobalSelfRef3  T_ref, S_ref are the step-0 slabs of T, S; the chunk that starts at step 0 also reduces
//                    {volo, masso} of the reference state (reference.py:71-80) -- the reference density is not stored
enum GlobalMode3 { kGlobal3 = 1, kGlobalSelfRef3 = 3 };

struct ParamsG3 {
  const float *T, *S;        // [nt][nz][ncol]  (repair pass)
  const float *Tref, *Sref;  // [nz][ncol]
  const float* v_ref;        // [nz][ncol]
  const double* p_level;
  int nt, nz, t_start;
  unsigned nchunks, tiles;
  i64 ncol;
  double* partials;          // [3][nt][tiles] masses; kGlobalSelfRef3: then [2][tiles] = {volo, masso}
};

template <int EOS, int TC, int MODE>
__global__ void __launch_bounds__(kTile, ctas_per_sm3(TC))
    k_steric_tma3_global(const __grid_constant__ CUtensorMap mapT, const __grid_constant__ CUtensorMap mapS,
                         const __grid_constant__ CUtensorMap mapTr, const __grid_constant__ CUtensorMap mapSr,
                         const ParamsG3 P) {
  constexpr bool SELFREF = MODE == kGlobalSelfRef3;
  constexpr int kStages = stages3(TC);
  constexpr int kRows = 2 * TC + 2;
  constexpr uint32_t kStageBytes = (uint32_t)kRows * kTile * sizeof(float);
  constexpr int kStageFloats = kRows * kTile;
  constexpr int kOffS = TC * kTile, kOffTr = 2 * TC * kTile, kOffSr = (2 * TC + 1) * kTile;

  extern __shared__ __align__(128) unsigned char smem_raw[];
  float* stage_base = reinterpret_cast<float*>(smem_raw);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + (size_t)kStages * kStageBytes);
  uint64_t* empty = full + kStages;
  int* released = reinterpret_cast<int*>(full + 2 * kStages);
  double* red = reinterpret_cast<double*>(full + 3 * kStages);  // [kConsumerWarps][3 TC + 2]
  double* s_p = red + kConsumerWarps * (3 * TC + 2);
  int* s_key = reinterpret_cast<int*>(s_p + P.nz);
  int* s_col = s_key + kTile;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const unsigned tile = blockIdx.x / P.nchunks;
  const int c0 = (int)tile * kTile;
  const int t0 = P.t_start + (int)(blockIdx.x - tile * P.nchunks) * TC;
  const int nz = P.nz;
  const bool chunk0 = SELFREF && t0 == 0;  // this CTA's chunk starts at the reference step

  auto refill_stage = [&](int z) {
    const int s = z % kStages;
    float* d = stage_base + (size_t)s * kStageFloats;
    mbar_expect_tx(full + s, kStageBytes);
    tma_load_3d(d, &mapT, full + s, c0, z, t0);
    tma_load_3d(d + kOffS, &mapS, full + s, c0, z, t0);
    tma_load_2d(d + kOffTr, &mapTr, full + s, c0, z);
    tma_load_2d(d + kOffSr, &mapSr, full + s, c0, z);
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
  for (int i = threadIdx.x; i < nz; i += kTile) s_p[i] = __ldg(P.p_level + i);
  __syncthreads();

  // the single-height global kernel's column order: ranked by the number of levels whose reference volume is present
  int col;
  {
    const i64 cg = (i64)c0 + tid;
    int key = 0;
    if (cg < P.ncol)
      for (int z = 0; z < nz; ++z) key += vraw_isnan(ld_vraw(P.v_ref, (i64)z * P.ncol + cg)) ? 0 : 1;
    col = sorted_column(key, reinterpret_cast<unsigned*>(s_key), s_col);
  }

  const i64 c = (i64)c0 + col;
  const bool in = c < P.ncol;
  const i64 cc = in ? c : (P.ncol - 1);
  Eos<EOS> eos;
  double acc[3][TC];
#pragma unroll
  for (int v = 0; v < 3; ++v)
#pragma unroll
    for (int k = 0; k < TC; ++k) acc[v][k] = 0.0;
  double vol = 0.0, mass = 0.0;
  unsigned v_n = ld_vraw(P.v_ref, cc);

  for (int z = 0; z < nz; ++z) {
    const unsigned v_z = v_n;
    if (z + 1 < nz) v_n = ld_vraw(P.v_ref, (i64)(z + 1) * P.ncol + cc);
    const bool dry = vraw_isnan(v_z);
    const double w = dry ? 0.0 : vraw_value(v_z);  // rho * NaN is dropped by the skipna sum (derived.py:435-438)
    eos.set_level(s_p[z]);
    const bool live = nonzero(w);
    const unsigned live_lanes = __ballot_sync(0xffffffffu, live);
    const int s = z % kStages;
    const float* st = stage_base + (size_t)s * kStageFloats;
    mbar_wait(full + s, (uint32_t)(z / kStages) & 1u);
    if (live_lanes != 0u) {
      const int first_wet = __shfl_sync(0xffffffffu, col, __ffs(live_lanes) - 1);
      const int src = live ? col : first_wet;
      const typename Eos<EOS>::Pinned qs = eos.pin_s((double)st[kOffSr + src]);  // thermosteric: S held at S_ref
      const typename Eos<EOS>::Pinned qt = eos.pin_t((double)st[kOffTr + src]);  // halosteric: T held at T_ref
#pragma unroll
      for (int kk = 0; kk < TC; ++kk) {
        const double Tv = (double)st[kk * kTile + src];
        const double Sv = (double)st[kOffS + kk * kTile + src];
        acc[0][kk] = fma(w, eos.rho(Tv, Sv), acc[0][kk]);
        acc[1][kk] = fma(w, eos.rho_pinned_s(qs, Tv), acc[1][kk]);
        acc[2][kk] = fma(w, eos.rho_pinned_t(qt, Sv), acc[2][kk]);
      }
    }
    if (chunk0 && in && !dry) {  // volo, masso of the reference state: skipna sums (derived.py:787-789, :435-438)
      const double r = eos.rho((double)st[kOffTr + col], (double)st[kOffSr + col]);  // reference.py:71
      vol += w;
      const double m = r * w;
      if (!is_nan_q(m)) mass += m;
    }
    __syncwarp();
    if (lane == 0 && stage_done(empty + s, released + s, kConsumerWarps, (uint32_t)(z / kStages) & 1u) && z + kStages < nz)
      refill_stage(z + kStages);
  }

  // Repair pass (ml_tma.cu): a column whose sums met a hole at a wet cell is summed again from global memory with the
  // skipna rule.  A mass that met no hole comes out as it was (same FMAs in the same order), so repairing the three
  // together keeps each of them identical to its single-height launch.
  bool poisoned = false;
#pragma unroll
  for (int v = 0; v < 3; ++v)
#pragma unroll
    for (int k = 0; k < TC; ++k) poisoned |= is_nan_q(acc[v][k]);
  if (poisoned && in) {
#pragma unroll
    for (int v = 0; v < 3; ++v)
#pragma unroll
      for (int k = 0; k < TC; ++k) acc[v][k] = 0.0;
    const i64 lvl = (i64)nz * P.ncol;
    for (int z = 0; z < nz; ++z) {
      const i64 j = (i64)z * P.ncol + c;
      const unsigned vr = ld_vraw(P.v_ref, j);
      const double w = vraw_isnan(vr) ? 0.0 : vraw_value(vr);
      if (!nonzero(w)) continue;
      eos.set_level(s_p[z]);
      const typename Eos<EOS>::Pinned qs = eos.pin_s((double)__ldg(P.Sref + j));
      const typename Eos<EOS>::Pinned qt = eos.pin_t((double)__ldg(P.Tref + j));
#pragma unroll
      for (int k = 0; k < TC; ++k) {
        if (t0 + k >= P.nt) continue;
        const double Tv = (double)__ldg(P.T + (i64)(t0 + k) * lvl + j);
        const double Sv = (double)__ldg(P.S + (i64)(t0 + k) * lvl + j);
        fma_skipnan(acc[0][k], w, eos.rho(Tv, Sv));
        fma_skipnan(acc[1][k], w, eos.rho_pinned_s(qs, Tv));
        fma_skipnan(acc[2][k], w, eos.rho_pinned_t(qt, Sv));
      }
    }
  }

  // warp sums, then the CTA's warps in order (the single-height kernel's order per mass)
  constexpr int kRed = 3 * TC + 2;
#pragma unroll
  for (int v = 0; v < 3; ++v)
#pragma unroll
    for (int k = 0; k < TC; ++k) {
      const double sacc = warp_sum(in ? acc[v][k] : 0.0);
      if (lane == 0) red[warp * kRed + v * TC + k] = sacc;
    }
  if (chunk0) {  // uniform per CTA
    vol = warp_sum(vol);
    mass = warp_sum(mass);
    if (lane == 0) {
      red[warp * kRed + 3 * TC] = vol;
      red[warp * kRed + 3 * TC + 1] = mass;
    }
  }
  __syncthreads();
  if (tid < 3 * TC) {
    const int v = tid / TC, k = tid - v * TC;
    if (t0 + k < P.nt) {
      double sacc = 0.0;
#pragma unroll
      for (int w8 = 0; w8 < kConsumerWarps; ++w8) sacc += red[w8 * kRed + tid];
      P.partials[((i64)v * P.nt + t0 + k) * P.tiles + tile] = sacc;
    }
  } else if (chunk0 && tid < 3 * TC + 2) {
    double sacc = 0.0;
#pragma unroll
    for (int w8 = 0; w8 < kConsumerWarps; ++w8) sacc += red[w8 * kRed + tid];
    P.partials[((i64)3 * P.nt + (tid - 3 * TC)) * P.tiles + tile] = sacc;
  }
}

// ----------------------------------------------------------------------- host side
template <int TC, int TILE>
static size_t smem_bytes3(int nz, bool layers) {
  return (size_t)stages3(TC) * (size_t)((2 * TC + 2) * TILE * 4) + 3 * stages3(TC) * sizeof(uint64_t) +
         (size_t)(TILE / 32) * 2 * sizeof(double) + (size_t)(2 * nz + 1) * sizeof(double) + 2 * TILE * sizeof(int) + 128 +
         (layers ? (size_t)nz * sizeof(int) : 0);
}

template <int EOS, int TC, int MODE, int TILE>
static int launch_one3(const CUtensorMap maps[4], const Params3& P, unsigned tiles, unsigned chunks, cudaStream_t st,
                       const LayerParams* lp) {
  auto kern = k_steric_tma3<EOS, TC, MODE, TILE>;
  const size_t smem = smem_bytes3<TC, TILE>(P.nz, MODE == kLocalLayers3);
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(k_steric_tma3)");
  Params3 Q = P;
  Q.tiles = tiles;
  Q.nchunks = chunks;
  LayersOf3<MODE> L{};
  if constexpr (MODE == kLocalLayers3) L = *lp;
  kern<<<tiles * chunks, TILE, smem, st>>>(maps[0], maps[1], maps[2], maps[3], Q, L);
  return launched("k_steric_tma3");
}

// chunk widths of a launch sequence: whole main-width chunks, then one remainder chunk of the smallest width
// in {4, 6, 8, 12} that holds what is left (rows past nt are zero-filled by the TMA unit and cost arithmetic only).
// The main width can be overridden for experiments (ML_TMA3_TC = 4 | 6 | 8 | 12 in the environment).
// Measured on OM4p25 x 12 (profiles/r02_experiments.md): 12-step chunks, one CTA per SM: 4.13 ms; 6-step chunks, two
// CTAs per SM: 4.27-4.36 ms (the per-level stage release weighs twice as much); three single-height launches: 4.79 ms.
#ifndef ML_TMA3_TC
#define ML_TMA3_TC 12
#endif
// columns per CTA: 256 or 128 (ML_TMA3_TILE in the environment, or 100 added to the value given to
// ml_set_variants_chunk, e.g. 106 = 128-column tiles with 6-step chunks)
#ifndef ML_TMA3_TILE
#define ML_TMA3_TILE 256
#endif
static int tile3() {
  static const int from_env = [] {
    const char* v = getenv("ML_TMA3_TILE");
    const int n = v ? atoi(v) : ML_TMA3_TILE;
    return n == 128 ? 128 : (n == 256 ? 256 : ML_TMA3_TILE);
  }();
  const int t = tls().variants_chunk;
  if (t >= 200) return 256;
  return t >= 100 ? 128 : from_env;
}
static int main_tc3() {
  static const int from_env = [] {
    const char* v = getenv("ML_TMA3_TC");
    const int n = v ? atoi(v) : ML_TMA3_TC;
    return (n == 4 || n == 6 || n == 8 || n == 12) ? n : ML_TMA3_TC;
  }();
  const int t = tls().variants_chunk % 100;  // ml_set_variants_chunk
  return (t == 4 || t == 6 || t == 8 || t == 12) ? t : from_env;
}
// kLocalLayers3 carries the 3 x TC sums of kLocal3 plus the layer bookkeeping; only the widths that compile without
// spills are instantiated: 4, 6 and 12 (the Wright kernel spills at 8 under the 128-register cap of two CTAs per SM;
// ptxas, sm_100a: profiles/r05_ptxas_registers.txt).  Main width measured on OM4p25 x 12, one B200 at 1000 W
// (profiles/r05_layers_variants.json, medians): 6-step chunks, two CTAs per SM: 5.42 ms; 4-step: 6.01 ms; 12-step, one
// CTA per SM (222 registers): 6.78 ms.  ml_set_variants_chunk / ML_TMA3_TC select among the instantiated ones.
__host__ __device__ constexpr bool has_tc3(int mode, int tc) { return mode != kLocalLayers3 || tc != 8; }
#ifndef ML_TMA3L_TC
#define ML_TMA3L_TC 6
#endif
static int main_tc_layers3() {
  const int t = main_tc3();
  const bool asked = tls().variants_chunk % 100 != 0 || getenv("ML_TMA3_TC") != nullptr;
  return asked && has_tc3(kLocalLayers3, t) ? t : ML_TMA3L_TC;
}

template <int MODE, int TILE>
static int launch_span3(int eos, const void* T, const void* S, const void* Tr, const void* Sr, Params3 P, int t_begin,
                        int t_end, int tc, cudaStream_t st, const LayerParams* lp) {
  // one launch: chunks of `tc` steps covering [t_begin, t_end)
  CUtensorMap maps[4];
  const bool ok = make_map(&maps[0], T, 3, P.ncol, P.nz, P.nt, tc, TILE) && make_map(&maps[1], S, 3, P.ncol, P.nz, P.nt, tc, TILE) &&
                  make_map(&maps[2], Tr, 2, P.ncol, P.nz, 1, 1, TILE) && make_map(&maps[3], Sr, 2, P.ncol, P.nz, 1, 1, TILE);
  if (!ok) return fail(ML_ERR_ALIGN, "cuTensorMapEncodeTiled rejected the field layout");
  P.t_start = t_begin;
  const unsigned tiles = (unsigned)((P.ncol + TILE - 1) / TILE);
  const unsigned chunks = (unsigned)((t_end - t_begin + tc - 1) / tc);
#define ML_TMA3_GO(E, TCV) \
  if constexpr (has_tc3(MODE, TCV)) return launch_one3<E, TCV, MODE, TILE>(maps, P, tiles, chunks, st, lp)
  if (eos == ML_EOS_WRIGHT) {
    if (tc == 12) ML_TMA3_GO(0, 12);
    if (tc == 8) ML_TMA3_GO(0, 8);
    if (tc == 6) ML_TMA3_GO(0, 6);
    if (tc == 4) ML_TMA3_GO(0, 4);
  } else {
    if (tc == 12) ML_TMA3_GO(1, 12);
    if (tc == 8) ML_TMA3_GO(1, 8);
    if (tc == 6) ML_TMA3_GO(1, 6);
    if (tc == 4) ML_TMA3_GO(1, 4);
  }
#undef ML_TMA3_GO
  return fail(ML_ERR_MODE, "no %d-step chunk kernel for this mode", tc);
}

template <int MODE, int TILE>
static int launch_all3(int eos, const void* T, const void* S, const void* Tr, const void* Sr, const Params3& P,
                       cudaStream_t st, const LayerParams* lp = nullptr) {
  const int main_tc = MODE == kLocalLayers3 ? main_tc_layers3() : main_tc3();
  const int full = P.nt / main_tc, rest = P.nt % main_tc;
  int rc = ML_OK;
  if (full > 0) rc = launch_span3<MODE, TILE>(eos, T, S, Tr, Sr, P, 0, full * main_tc, main_tc, st, lp);
  if (rc == ML_OK && rest > 0) {
    int tc = 12;
    for (const int w : {8, 6, 4})
      if (w >= rest && has_tc3(MODE, w)) tc = w;
    rc = launch_span3<MODE, TILE>(eos, T, S, Tr, Sr, P, full * main_tc, P.nt, tc, st, lp);
  }
  return rc;
}

bool variants_eligible(int dtype, const void* T, const void* S, const void* Tr, const void* Sr, int vref_dtype,
                       int64_t nt, int64_t nz, int64_t ncol) {
  if (dtype != ML_F32 || vref_dtype != ML_F32 || ncol % 4 != 0) return false;  // fp32 rows of whole 16-byte units only
  if ((reinterpret_cast<uintptr_t>(Tr) | reinterpret_cast<uintptr_t>(Sr)) & 15u) return false;
  return local_eligible(dtype, T, S, 0, 0, nullptr, nullptr, vref_dtype, nt, nz, ncol, nullptr, nullptr);
}

int launch_variants(int eos, const void* T, const void* S, const void* T_ref, const void* S_ref, const double* rho_ref,
                    const void* v_ref, const double* z_i, const double* deptho, const double* p_level, double coef, int nt,
                    int nz, int64_t ncol, double* eta_steric, double* eta_thermo, double* eta_halo, double* rho_ref_out,
                    double* sums, double* partials, cudaStream_t st) {
  Params3 P;
  P.T = static_cast<const float*>(T);
  P.S = static_cast<const float*>(S);
  P.Tref = static_cast<const float*>(T_ref);
  P.Sref = static_cast<const float*>(S_ref);
  P.rho_ref = rho_ref;
  P.rho_ref_out = rho_ref_out;
  P.v_ref = static_cast<const float*>(v_ref);
  P.z_i = z_i;
  P.deptho = deptho;
  P.p_level = p_level;
  P.coef = coef;
  P.nt = nt;
  P.nz = nz;
  P.t_start = 0;
  P.nchunks = 1;
  P.tiles = 0;
  P.ncol = ncol;
  P.eta[0] = eta_steric;
  P.eta[1] = eta_thermo;
  P.eta[2] = eta_halo;
  P.partials = partials;
  const int tile = tile3();
  if (rho_ref != nullptr)
    return tile == 128 ? launch_all3<kLocal3, 128>(eos, T, S, T_ref, S_ref, P, st)
                       : launch_all3<kLocal3, 256>(eos, T, S, T_ref, S_ref, P, st);
  // reference = step 0 of the fields: T_ref / S_ref are the step-0 slabs
  int rc = tile == 128 ? launch_all3<kSelfRef3, 128>(eos, T, S, T_ref, S_ref, P, st)
                       : launch_all3<kSelfRef3, 256>(eos, T, S, T_ref, S_ref, P, st);
  if (rc) return rc;
  return reduce_rows(partials, (ncol + tile - 1) / tile, sums, 2, st);
}

int launch_local_layers_variants(int eos, const void* T, const void* S, const void* T_ref, const void* S_ref,
                                 const double* rho_ref, const void* v_ref, const double* z_i, const double* deptho,
                                 const double* p_level, double coef, const double* edges, int nlayers, int nt, int nz,
                                 int64_t ncol, double* eta_steric, double* eta_thermo, double* eta_halo, cudaStream_t st) {
  Params3 P;
  P.T = static_cast<const float*>(T);
  P.S = static_cast<const float*>(S);
  P.Tref = static_cast<const float*>(T_ref);
  P.Sref = static_cast<const float*>(S_ref);
  P.rho_ref = rho_ref;
  P.rho_ref_out = nullptr;
  P.v_ref = static_cast<const float*>(v_ref);
  P.z_i = z_i;
  P.deptho = deptho;
  P.p_level = p_level;
  P.coef = coef;
  P.nt = nt;
  P.nz = nz;
  P.t_start = 0;
  P.nchunks = 1;
  P.tiles = 0;
  P.ncol = ncol;
  P.eta[0] = eta_steric;
  P.eta[1] = eta_thermo;
  P.eta[2] = eta_halo;
  P.partials = nullptr;
  LayerParams lp;
  lp.nlayers = nlayers;
  for (int b = 0; b <= ML_MAX_LAYERS; ++b) lp.edges[b] = b <= nlayers ? edges[b] : 0.0;
  return launch_all3<kLocalLayers3, kTile>(eos, T, S, T_ref, S_ref, P, st, &lp);
}

// global masses: 256-column tiles whatever ML_TMA3_TILE says (the column order inside a tile decides the bits)
template <int TC>
static size_t smem_bytes_g3(int nz) {
  return (size_t)stages3(TC) * (size_t)((2 * TC + 2) * kTile * 4) + 3 * stages3(TC) * sizeof(uint64_t) +
         (size_t)kConsumerWarps * (3 * TC + 2) * sizeof(double) + (size_t)nz * sizeof(double) + 2 * kTile * sizeof(int) + 128;
}

template <int EOS, int TC, int MODE>
static int launch_one_g3(const CUtensorMap maps[4], const ParamsG3& P, unsigned tiles, unsigned chunks, cudaStream_t st) {
  auto kern = k_steric_tma3_global<EOS, TC, MODE>;
  const size_t smem = smem_bytes_g3<TC>(P.nz);
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(k_steric_tma3_global)");
  ParamsG3 Q = P;
  Q.tiles = tiles;
  Q.nchunks = chunks;
  kern<<<tiles * chunks, kTile, smem, st>>>(maps[0], maps[1], maps[2], maps[3], Q);
  return launched("k_steric_tma3_global");
}

template <int MODE>
static int launch_span_g3(int eos, ParamsG3 P, int t_begin, int t_end, int tc, cudaStream_t st) {
  CUtensorMap maps[4];
  const bool ok = make_map(&maps[0], P.T, 3, P.ncol, P.nz, P.nt, tc) && make_map(&maps[1], P.S, 3, P.ncol, P.nz, P.nt, tc) &&
                  make_map(&maps[2], P.Tref, 2, P.ncol, P.nz, 1, 1) && make_map(&maps[3], P.Sref, 2, P.ncol, P.nz, 1, 1);
  if (!ok) return fail(ML_ERR_ALIGN, "cuTensorMapEncodeTiled rejected the field layout");
  P.t_start = t_begin;
  const unsigned tiles = (unsigned)((P.ncol + kTile - 1) / kTile);
  const unsigned chunks = (unsigned)((t_end - t_begin + tc - 1) / tc);
#define ML_TMA3G_GO(E, TCV) return launch_one_g3<E, TCV, MODE>(maps, P, tiles, chunks, st)
  if (eos == ML_EOS_WRIGHT) {
    if (tc == 12) ML_TMA3G_GO(0, 12);
    if (tc == 8) ML_TMA3G_GO(0, 8);
    if (tc == 6) ML_TMA3G_GO(0, 6);
    ML_TMA3G_GO(0, 4);
  }
  if (tc == 12) ML_TMA3G_GO(1, 12);
  if (tc == 8) ML_TMA3G_GO(1, 8);
  if (tc == 6) ML_TMA3G_GO(1, 6);
  ML_TMA3G_GO(1, 4);
#undef ML_TMA3G_GO
}

template <int MODE>
static int launch_all_g3(int eos, const ParamsG3& P, cudaStream_t st) {
  const int main_tc = main_tc3();
  const int full = P.nt / main_tc, rest = P.nt % main_tc;
  int rc = ML_OK;
  if (full > 0) rc = launch_span_g3<MODE>(eos, P, 0, full * main_tc, main_tc, st);
  if (rc == ML_OK && rest > 0) {
    const int tc = rest <= 4 ? 4 : (rest <= 6 ? 6 : (rest <= 8 ? 8 : 12));
    rc = launch_span_g3<MODE>(eos, P, full * main_tc, P.nt, tc, st);
  }
  return rc;
}

size_t global_variants_partials(int64_t nt, int64_t ncol) {
  return (size_t)(3 * nt + 2) * (size_t)((ncol + kTile - 1) / kTile) * sizeof(double);
}

int launch_global_variants(int eos, const void* T, const void* S, const void* T_ref, const void* S_ref, const void* v_ref,
                           const double* p_level, int nt, int nz, int64_t ncol, double* masso_steric,
                           double* masso_thermo, double* masso_halo, double* sums, double* partials, cudaStream_t st) {
  ParamsG3 P;
  P.T = static_cast<const float*>(T);
  P.S = static_cast<const float*>(S);
  P.Tref = static_cast<const float*>(T_ref);
  P.Sref = static_cast<const float*>(S_ref);
  P.v_ref = static_cast<const float*>(v_ref);
  P.p_level = p_level;
  P.nt = nt;
  P.nz = nz;
  P.t_start = 0;
  P.nchunks = 1;
  P.tiles = 0;
  P.ncol = ncol;
  P.partials = partials;
  int rc = sums != nullptr ? launch_all_g3<kGlobalSelfRef3>(eos, P, st) : launch_all_g3<kGlobal3>(eos, P, st);
  if (rc) return rc;
  const int64_t tiles = (ncol + kTile - 1) / kTile;
  double* outs[3] = {masso_steric, masso_thermo, masso_halo};
  for (int v = 0; v < 3; ++v)
    if (outs[v] != nullptr && (rc = reduce_rows(partials + (size_t)v * nt * tiles, tiles, outs[v], nt, st))) return rc;
  if (sums != nullptr) rc = reduce_rows(partials + (size_t)3 * nt * tiles, tiles, sums, 2, st);
  return rc;
}

}  // namespace tma
}  // namespace ml
