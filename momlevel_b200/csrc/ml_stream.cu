// ml_stream.cu -- the elementwise operators as streaming kernels over a shared-memory ring (sm_100a).
//
// eos.wright.density / eos.linear.density applied over a field (src/momlevel/derived.py:624-630),
// spice.flament.spice (src/momlevel/spice/flament.py:78-90) and the reference-state pass
// (src/momlevel/reference.py:71-80) read 8-12 bytes and write 8 bytes per point around 18-30 fp64
// instructions.  With plain loads a thread holds its operands in registers while they are in flight, and
// the ~50-60 registers of the evaluation leave room for ~1000 threads per SM: too few bytes in flight to
// cover HBM latency at 6.5 TB/s, so those kernels sat at 0.66-0.82 of the copy bandwidth.  Here a
// persistent CTA streams its tiles through a 4-stage ring filled by 1-D bulk copies
// (cp.async.bulk.shared::cluster.global, one mbarrier per stage): loads cost no registers and no issue
// slots, ~128 KB per SM are in flight whatever the occupancy, the math reads 128-bit words from shared
// memory and results leave as 256-bit streaming stores.
//
// Layout: the operands are rows of `ncol` points (a level of one time step; a flat array is one row); a tile
// is kTile consecutive points of one row.  Rows must start 16-byte aligned in every operand
// (ncol % 4 == 0 and aligned bases); anything else takes the plain kernels in ml_api.cu.
#include "ml_tma_dev.cuh"

#include "ml_stream.cuh"

namespace ml {
namespace stream {

// experiment knobs (tools/ab_stream.sh): ring depth, CTAs per SM of the map kernel, cache hint of the result stores
#ifndef ML_STREAM_STAGES
#define ML_STREAM_STAGES 4
#endif
#ifndef ML_STREAM_CTAS
#define ML_STREAM_CTAS 3
#endif
#ifndef ML_STREAM_ST
#define ML_STREAM_ST 0
#endif
constexpr int kTile = 2048;     // points per tile: 8 KB per fp32 operand
constexpr int kStages = ML_STREAM_STAGES;
constexpr int kThreads = 256;   // two quads of a tile per thread
constexpr int kWarps = kThreads / 32;

__device__ __forceinline__ void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   tma::smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(tma::smem_u32(bar))
               : "memory");
}
// four results of a quad leave as ONE 256-bit store (sm_100: STG.256): a lane writes a whole 32-byte sector and a
// warp 1 KB in a row; two 128-bit stores per lane would each write half of every sector they touch
__device__ __forceinline__ void st4(double* p, double a, double b, double c, double d) {
#if ML_STREAM_ST == 1
  asm volatile("st.global.cs.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(p), "d"(a), "d"(b), "d"(c), "d"(d) : "memory");
#elif ML_STREAM_ST == 2
  asm volatile("st.global.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(p), "d"(a), "d"(b), "d"(c), "d"(d) : "memory");
#else
  asm volatile("st.global.L1::no_allocate.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(p), "d"(a), "d"(b), "d"(c), "d"(d)
               : "memory");
#endif
}
// A warp is done with a stage: true in lane 0 of the warp that is the LAST of the CTA to leave it (that lane
// refills the stage); tma::stage_done orders every warp's reads of the stage before the refill.
__device__ __forceinline__ bool last_to_leave(uint64_t* empty_bar, int* counter, uint32_t parity) {
  __syncwarp();
  if ((threadIdx.x & 31) != 0) return false;
  return tma::stage_done(empty_bar, counter, kWarps, parity);
}

struct Geom {
  i64 ncol;           // points per row
  i64 ntiles;         // rows * tiles_per_row
  int tiles_per_row;
  int nz;             // rows per outer (time) index: row = t * nz + z
};

// Ring of kStages stages of NIN fp32 operand tiles.  Everybody waits on the stage's mbarrier; the warp that is the
// last to leave a stage refills it (no producer warp, no CTA-wide barrier in the loop).
template <int NIN>
struct Ring {
  float* base;
  uint64_t *full, *empty;
  int* released;  // [kStages] warps that have left the stage (mod kWarps)
  __device__ __forceinline__ float* stage(int s, int k) const { return base + ((size_t)s * NIN + k) * kTile; }
  __device__ __forceinline__ void init(unsigned char* smem) {
    base = reinterpret_cast<float*>(smem);
    full = reinterpret_cast<uint64_t*>(smem + (size_t)kStages * NIN * kTile * sizeof(float));
    empty = full + kStages;
    released = reinterpret_cast<int*>(full + 2 * kStages);
    if (threadIdx.x == 0) {
#pragma unroll
      for (int s = 0; s < kStages; ++s) {
        tma::mbar_init(full + s, 1);
        tma::mbar_init(empty + s, kWarps);
        released[s] = 0;
      }
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
  }
};
template <int NIN>
constexpr size_t ring_bytes() {
  return (size_t)kStages * NIN * kTile * sizeof(float) + kStages * (2 * sizeof(uint64_t) + sizeof(int)) + 64;
}

// ------------------------------------------------------------------------------ spice / density
// OP 0: Flament spiciness (T, S).  OP 1: density of EOS (T, S, p per row: scalar or per level).
template <int OP, int EOS>
__global__ void __launch_bounds__(kThreads, ML_STREAM_CTAS)
    k_stream_map(const float* __restrict__ T, const float* __restrict__ S, i64 t_stride, i64 s_stride,
                 const double* __restrict__ p, int pmode, Geom g, double* __restrict__ out) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  Ring<2> ring;
  ring.init(smem_raw);
  const int tid = threadIdx.x;
  auto issue = [&](i64 tile, int s) {
    const i64 row = tile / g.tiles_per_row;
    const i64 col0 = (tile - row * g.tiles_per_row) * kTile;
    const i64 t = row / g.nz, z = row - t * g.nz;
    const i64 len = g.ncol - col0 < kTile ? g.ncol - col0 : kTile;
    const uint32_t bytes = (uint32_t)len * 4u;
    tma::mbar_expect_tx(ring.full + s, 2 * bytes);
    bulk_load(ring.stage(s, 0), T + t * t_stride + z * g.ncol + col0, bytes, ring.full + s);
    bulk_load(ring.stage(s, 1), S + t * s_stride + z * g.ncol + col0, bytes, ring.full + s);
  };
  __syncthreads();
  if (tid == 0)
    for (int s = 0; s < kStages; ++s) {
      const i64 tile = (i64)blockIdx.x + (i64)s * gridDim.x;
      if (tile < g.ntiles) issue(tile, s);
    }
  Eos<EOS> eos;
  int it = 0;
  for (i64 tile = blockIdx.x; tile < g.ntiles; tile += gridDim.x, ++it) {
    const int s = it % kStages;
    const i64 row = tile / g.tiles_per_row;
    const i64 col0 = (tile - row * g.tiles_per_row) * kTile;
    const i64 len = g.ncol - col0 < kTile ? g.ncol - col0 : kTile;
    if (OP == 1) {
      const i64 z = row % g.nz;
      eos.set_level(pmode == ML_P_SCALAR ? __ldg(p) : (pmode == ML_P_PER_LEVEL ? __ldg(p + z) : 0.0));
    }
    double* o = out + row * g.ncol + col0;
    tma::mbar_wait(ring.full + s, (uint32_t)(it / kStages) & 1u);
    const float4* sT = reinterpret_cast<const float4*>(ring.stage(s, 0));
    const float4* sS = reinterpret_cast<const float4*>(ring.stage(s, 1));
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int q = tid + h * kThreads;
      if (4 * q < len) {
        const float4 a = sT[q], b = sS[q];
        double r0, r1, r2, r3;
        if (OP == 0) {
          r0 = flament_spice((double)a.x, (double)b.x);
          r1 = flament_spice((double)a.y, (double)b.y);
          r2 = flament_spice((double)a.z, (double)b.z);
          r3 = flament_spice((double)a.w, (double)b.w);
        } else {
          r0 = eos.rho_checked((double)a.x, (double)b.x);
          r1 = eos.rho_checked((double)a.y, (double)b.y);
          r2 = eos.rho_checked((double)a.z, (double)b.z);
          r3 = eos.rho_checked((double)a.w, (double)b.w);
        }
        st4(o + 4 * q, r0, r1, r2, r3);
      }
    }
    if (last_to_leave(ring.empty + s, ring.released + s, (uint32_t)(it / kStages) & 1u)) {
      const i64 next = tile + (i64)kStages * gridDim.x;
      if (next < g.ntiles) issue(next, s);
    }
  }
}

// ------------------------------------------------------------------------------ reference state
// rho_ref = rho(T0, S0, p_z) everywhere, volo = nansum(V0), masso = nansum(rho_ref * V0)
// (reference.py:71-80, derived.py:787-789, :435-438).  Block partials: [2][gridDim.x], fixed order.
template <int EOS>
__global__ void __launch_bounds__(kThreads, 2)
    k_stream_refstate(const float* __restrict__ T0, const float* __restrict__ S0, const float* __restrict__ V0,
                      const double* __restrict__ p_level, Geom g, double* __restrict__ rho_ref,
                      double* __restrict__ partials) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ double sm[kWarps];
  Ring<3> ring;
  ring.init(smem_raw);
  const int tid = threadIdx.x;
  auto issue = [&](i64 tile, int s) {
    const i64 row = tile / g.tiles_per_row;
    const i64 col0 = (tile - row * g.tiles_per_row) * kTile;
    const i64 len = g.ncol - col0 < kTile ? g.ncol - col0 : kTile;
    const uint32_t bytes = (uint32_t)len * 4u;
    const i64 off = row * g.ncol + col0;
    tma::mbar_expect_tx(ring.full + s, 3 * bytes);
    bulk_load(ring.stage(s, 0), T0 + off, bytes, ring.full + s);
    bulk_load(ring.stage(s, 1), S0 + off, bytes, ring.full + s);
    bulk_load(ring.stage(s, 2), V0 + off, bytes, ring.full + s);
  };
  __syncthreads();
  if (tid == 0)
    for (int s = 0; s < kStages; ++s) {
      const i64 tile = (i64)blockIdx.x + (i64)s * gridDim.x;
      if (tile < g.ntiles) issue(tile, s);
    }
  Eos<EOS> eos;
  double vol = 0.0, mass = 0.0;
  int it = 0;
  for (i64 tile = blockIdx.x; tile < g.ntiles; tile += gridDim.x, ++it) {
    const int s = it % kStages;
    const i64 row = tile / g.tiles_per_row;
    const i64 col0 = (tile - row * g.tiles_per_row) * kTile;
    const i64 len = g.ncol - col0 < kTile ? g.ncol - col0 : kTile;
    eos.set_level(__ldg(p_level + row));
    double* o = rho_ref + row * g.ncol + col0;
    tma::mbar_wait(ring.full + s, (uint32_t)(it / kStages) & 1u);
    const float4* sT = reinterpret_cast<const float4*>(ring.stage(s, 0));
    const float4* sS = reinterpret_cast<const float4*>(ring.stage(s, 1));
    const float4* sV = reinterpret_cast<const float4*>(ring.stage(s, 2));
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int q = tid + h * kThreads;
      if (4 * q < len) {
        const float4 a = sT[q], b = sS[q], v = sV[q];
        const float vv[4] = {v.x, v.y, v.z, v.w};
        double r[4];
        r[0] = eos.rho((double)a.x, (double)b.x);
        r[1] = eos.rho((double)a.y, (double)b.y);
        r[2] = eos.rho((double)a.z, (double)b.z);
        r[3] = eos.rho((double)a.w, (double)b.w);
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (!isnan(vv[j])) {
            vol += (double)vv[j];
            const double m = r[j] * (double)vv[j];
            if (!is_nan_q(m)) mass += m;
          }
        st4(o + 4 * q, r[0], r[1], r[2], r[3]);
      }
    }
    if (last_to_leave(ring.empty + s, ring.released + s, (uint32_t)(it / kStages) & 1u)) {
      const i64 next = tile + (i64)kStages * gridDim.x;
      if (next < g.ntiles) issue(next, s);
    }
  }
  vol = block_sum<kWarps>(vol, sm);
  mass = block_sum<kWarps>(mass, sm);
  if (tid == 0) {
    partials[blockIdx.x] = vol;
    partials[(i64)gridDim.x + blockIdx.x] = mass;
  }
}

// ------------------------------------------------------------------------------ density anomaly
// delta_rho[t][z][col] = V_ref notnull ? rho(T, S, p_z) - rho_ref : NaN (steric.py:151-153).  A CTA owns (level,
// column segment) pairs; rho_ref and the volume mask of a pair are read once into registers and reused for every
// time step, whose T and S tiles stream through the ring (the sequence runs on across pair boundaries, so the ring
// never drains).
template <int EOS, typename TV>
__global__ void __launch_bounds__(kThreads, 2)
    k_stream_delta_rho(const float* __restrict__ T, const float* __restrict__ S, i64 t_stride, i64 s_stride,
                       const double* __restrict__ rho_ref, const TV* __restrict__ v_ref,
                       const double* __restrict__ p_level, int nt, Geom g, double* __restrict__ out) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  Ring<2> ring;
  ring.init(smem_raw);
  const int tid = threadIdx.x;
  const i64 npairs = g.ntiles;                         // (level, segment) pairs; g.nz rows
  const i64 mine = npairs > (i64)blockIdx.x ? (npairs - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  const i64 nseq = mine * nt;                          // tiles this CTA streams, time fastest
  auto issue = [&](i64 q, int s) {
    const i64 pair = (i64)blockIdx.x + (q / nt) * gridDim.x;
    const int t = (int)(q % nt);
    const i64 row = pair / g.tiles_per_row;            // level
    const i64 col0 = (pair - row * g.tiles_per_row) * kTile;
    const i64 len = g.ncol - col0 < kTile ? g.ncol - col0 : kTile;
    const uint32_t bytes = (uint32_t)len * 4u;
    const i64 off = row * g.ncol + col0;
    tma::mbar_expect_tx(ring.full + s, 2 * bytes);
    bulk_load(ring.stage(s, 0), T + (i64)t * t_stride + off, bytes, ring.full + s);
    bulk_load(ring.stage(s, 1), S + (i64)t * s_stride + off, bytes, ring.full + s);
  };
  __syncthreads();
  if (tid == 0)
    for (int s = 0; s < kStages && s < nseq; ++s) issue(s, s);
  Eos<EOS> eos;
  const i64 lvl = (i64)g.nz * g.ncol;
  i64 q = 0;
  for (i64 i = 0; i < mine; ++i) {
    const i64 pair = (i64)blockIdx.x + i * gridDim.x;
    const i64 row = pair / g.tiles_per_row;
    const i64 col0 = (pair - row * g.tiles_per_row) * kTile;
    const i64 len = g.ncol - col0 < kTile ? g.ncol - col0 : kTile;
    const i64 off = row * g.ncol + col0;
    eos.set_level(__ldg(p_level + row));
    double ref[2][4];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int qd = tid + h * kThreads;
#pragma unroll
      for (int j = 0; j < 4; ++j) ref[h][j] = nan("");
      if (4 * qd < len) {
        const double2 a = __ldg(reinterpret_cast<const double2*>(rho_ref + off + 4 * qd));
        const double2 b = __ldg(reinterpret_cast<const double2*>(rho_ref + off + 4 * qd) + 1);
        const double r4[4] = {a.x, a.y, b.x, b.y};
#pragma unroll
        for (int j = 0; j < 4; ++j) ref[h][j] = isnan(__ldg(v_ref + off + 4 * qd + j)) ? nan("") : r4[j];
      }
    }
    for (int t = 0; t < nt; ++t, ++q) {
      const int s = (int)(q % kStages);
      tma::mbar_wait(ring.full + s, (uint32_t)(q / kStages) & 1u);
      const float4* sT = reinterpret_cast<const float4*>(ring.stage(s, 0));
      const float4* sS = reinterpret_cast<const float4*>(ring.stage(s, 1));
      double* o = out + (i64)t * lvl + off;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int qd = tid + h * kThreads;
        if (4 * qd < len) {
          const float4 a = sT[qd], b = sS[qd];
          st4(o + 4 * qd, eos.rho((double)a.x, (double)b.x) - ref[h][0], eos.rho((double)a.y, (double)b.y) - ref[h][1],
              eos.rho((double)a.z, (double)b.z) - ref[h][2], eos.rho((double)a.w, (double)b.w) - ref[h][3]);
        }
      }
      if (last_to_leave(ring.empty + s, ring.released + s, (uint32_t)(q / kStages) & 1u)) {
        const i64 next = q + kStages;
        if (next < nseq) issue(next, s);
      }
    }
  }
}

// ------------------------------------------------------------------------------ level profile
// The area-weighted steric / thermosteric / halosteric height change of each level (ml_steric_local_profile):
// partials[v][t * nz + z][seg * kWarps + warp] = sum over the warp's points of cw * (rho_v - rho_ref), skipna, with
// cw = coef * m * w * dz (profile_weight).  The (level, segment) ownership and time-fastest sequence of
// k_stream_delta_rho: per pair, rho_ref (NaN where the reference volume is missing), cw and the reference slabs the
// variants hold fixed stay in registers.  Per streamed step a thread sums its 8 points in a fixed order, the warp
// sums by shuffle and lane 0 stores the warp's partial: no CTA-wide barrier in the loop, and a partial's slot depends
// on the point's position only, so the sums do not depend on the grid.  VM: bit 0 steric (T, S), bit 1 thermosteric
// (T, S_ref), bit 2 halosteric (T_ref, S) (steric.py:115-121); only the operands the variants read are staged.
// REG (ml_steric_local_region_profile): one partial per region, partials[v][r][t * nz + z][seg * kWarps + warp].
// At the setup of a pair a thread packs the region index of its 8 points into 4-bit fields of one register (0xF: no
// region) and the warp ORs the regions its points touch into a mask fixed for the pair; the shared memory is full, so
// the codes stay in registers.  Per step the warp walks the set bits of that mask in ascending order and in
// iteration r each thread sums, in the order above, only its points of region r: every density is evaluated once,
// and a warp whose points all lie in one region sums exactly as without regions.  Lane 0 stores region r's
// partial; lane r stores 0 for a region the warp does not touch, so every slot is written on every step.
// ZON (ml_steric_local_zonal_profile): one partial row per grid row.  A work item is a (level z, row j, kTile-column
// sub-tile s) triple: the geometry above on a grid of nz * ny rows of nx columns (g.ncol = nx, g.nz = nz * ny,
// row = z * ny + j), so the field offsets, the thread -> point map, the per-item state, the order of the sums and the
// slot formula are those of a call on row j alone: partials[v][((t * nz + z) * ny + j) * nsub * kWarps + s * kWarps +
// warp].  Only the level (pressure, interfaces) and the column of the (y, x) plane (deptho, weights, surface mask) are
// read through z and j * nx + col.  So row j's partials are bit-identical to ml_steric_local_profile on row j sliced
// out alone, and every slot is written on every step, a warp without points storing its 0.
constexpr size_t kProfileRing = ring_bytes<2>();  // the per-point state follows the ring
struct ProfileOut {
  double* part[3];  // per variant, [nregions][nt * nz][tiles_per_row * kWarps]; NULL for a variant not asked for
  const int8_t* region;  // REG: [ncol] region index of each column, one in [0, nregions) or none
  int nregions;
  int ny;  // ZON: grid rows per level
};

template <int EOS, int VM, bool ZON, bool REG>
__global__ void __launch_bounds__(kThreads, 2)
    k_stream_profile(const float* __restrict__ T, const float* __restrict__ S, const float* __restrict__ T_ref,
                     const float* __restrict__ S_ref, const double* __restrict__ rho_ref, const void* __restrict__ v_ref,
                     int v_f32, const double* __restrict__ z_i, const double* __restrict__ deptho,
                     const double* __restrict__ weights, const double* __restrict__ p_level, double coef, int nt, Geom g,
                     ProfileOut out) {
  constexpr bool kT = (VM & 3) != 0, kS = (VM & 5) != 0;  // which of T, S the ring carries
  extern __shared__ __align__(128) unsigned char smem_raw[];
  Ring<2> ring;
  ring.init(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // per-pair state of a thread's 8 points, [point][thread]: only the owning thread reads its slots, so no barrier
  double* const ref = reinterpret_cast<double*>(smem_raw + kProfileRing) + tid;
  double* const cw = ref + 8 * kThreads;
  // the reference slabs the variants hold fixed
  float* const tref = reinterpret_cast<float*>(smem_raw + kProfileRing + 16 * kThreads * sizeof(double)) + tid;
  float* const sref = tref + 8 * kThreads;
  const i64 npairs = g.ntiles;
  const i64 mine = npairs > (i64)blockIdx.x ? (npairs - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  const i64 nseq = mine * nt;
  const i64 lvl = (i64)g.nz * g.ncol;
  const i64 nblk = (i64)g.tiles_per_row * kWarps;
  auto issue = [&](i64 q, int s) {
    const i64 pair = (i64)blockIdx.x + (q / nt) * gridDim.x;
    const int t = (int)(q % nt);
    const i64 row = pair / g.tiles_per_row;
    const i64 col0 = (pair - row * g.tiles_per_row) * kTile;
    const i64 len = g.ncol - col0 < kTile ? g.ncol - col0 : kTile;
    const uint32_t bytes = (uint32_t)len * 4u;
    const i64 off = (i64)t * lvl + row * g.ncol + col0;
    tma::mbar_expect_tx(ring.full + s, (kT + kS) * bytes);
    if (kT) bulk_load(ring.stage(s, 0), T + off, bytes, ring.full + s);
    if (kS) bulk_load(ring.stage(s, 1), S + off, bytes, ring.full + s);
  };
  __syncthreads();
  if (tid == 0)
    for (int s = 0; s < kStages && s < nseq; ++s) issue(s, s);
  Eos<EOS> eos;
  i64 q = 0;
  for (i64 i = 0; i < mine; ++i) {
    const i64 pair = (i64)blockIdx.x + i * gridDim.x;
    const i64 row = pair / g.tiles_per_row;
    const i64 seg = pair - row * g.tiles_per_row;
    const i64 col0 = seg * kTile;
    const i64 len = g.ncol - col0 < kTile ? g.ncol - col0 : kTile;
    const i64 off = row * g.ncol + col0;
    i64 lev = row, cplane = col0;  // the level, and the first column of the item in the (y, x) plane
    if constexpr (ZON) {
      lev = row / out.ny;
      cplane = (row - lev * out.ny) * g.ncol + col0;
    }
    eos.set_level(__ldg(p_level + lev));
    const double ztop = __ldg(z_i + lev), zbot = __ldg(z_i + lev + 1);
    uint32_t rbits = 0, wmask = 0;  // REG: the 4-bit region index of each point; the regions the warp touches
    if constexpr (REG) {
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const i64 p = 4 * (tid + (k >> 2) * kThreads) + (k & 3);
        const uint32_t r = p < len ? region_nibble(out.region, col0 + p, out.nregions) : 0xFu;
        rbits |= r << (4 * k);
        wmask |= r < 0xFu ? 1u << r : 0u;
      }
      wmask = __reduce_or_sync(0xffffffffu, wmask);
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int qd = tid + h * kThreads;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        ref[(4 * h + j) * kThreads] = nan("");
        cw[(4 * h + j) * kThreads] = 0.0;
        tref[(4 * h + j) * kThreads] = sref[(4 * h + j) * kThreads] = 0.0f;
      }
      if (4 * qd < len) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const i64 c = cplane + 4 * qd + j;
          const bool wet = v_f32 ? !isnan(__ldg(reinterpret_cast<const float*>(v_ref) + off + 4 * qd + j))
                                 : !isnan(__ldg(reinterpret_cast<const double*>(v_ref) + off + 4 * qd + j));
          const bool top = v_f32 ? !isnan(__ldg(reinterpret_cast<const float*>(v_ref) + c))
                                 : !isnan(__ldg(reinterpret_cast<const double*>(v_ref) + c));
          double depth = __ldg(deptho + c);
          if (isnan(depth)) depth = 0.0;  // derived.py:295
          ref[(4 * h + j) * kThreads] = wet ? __ldg(rho_ref + off + 4 * qd + j) : nan("");
          cw[(4 * h + j) * kThreads] = profile_weight(top, __ldg(weights + c), clipped_dz(depth, ztop, zbot), coef);
          if (VM & 4) tref[(4 * h + j) * kThreads] = __ldg(T_ref + off + 4 * qd + j);
          if (VM & 2) sref[(4 * h + j) * kThreads] = __ldg(S_ref + off + 4 * qd + j);
        }
      }
    }
    for (int t = 0; t < nt; ++t, ++q) {
      const int s = (int)(q % kStages);
      tma::mbar_wait(ring.full + s, (uint32_t)(q / kStages) & 1u);
      const float4* sT = reinterpret_cast<const float4*>(ring.stage(s, 0));
      const float4* sS = reinterpret_cast<const float4*>(ring.stage(s, 1));
      const i64 slot = ((i64)t * g.nz + row) * nblk + seg * kWarps + warp;
      const i64 rstride = (i64)nt * g.nz * nblk;  // REG: from one region's partials to the next
      double acc[3];
      // without REG one iteration over every point; with REG one per region the warp touches
      for (uint32_t todo = REG ? wmask : 1u; todo != 0; todo &= todo - 1) {
        const uint32_t r = __ffs(todo) - 1;
        acc[0] = acc[1] = acc[2] = 0.0;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int qd = tid + h * kThreads;
          if (4 * qd < len) {
            float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
            if (kT) a = sT[qd];
            if (kS) b = sS[qd];
            const float ta[4] = {a.x, a.y, a.z, a.w}, sa[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              if (REG && ((rbits >> (4 * (4 * h + j))) & 0xFu) != r) continue;
              if (VM & 1) acc[0] = profile_add(acc[0], cw[(4 * h + j) * kThreads], eos.rho((double)ta[j], (double)sa[j]), ref[(4 * h + j) * kThreads]);
              if (VM & 2) acc[1] = profile_add(acc[1], cw[(4 * h + j) * kThreads], eos.rho((double)ta[j], (double)sref[(4 * h + j) * kThreads]), ref[(4 * h + j) * kThreads]);
              if (VM & 4) acc[2] = profile_add(acc[2], cw[(4 * h + j) * kThreads], eos.rho((double)tref[(4 * h + j) * kThreads], (double)sa[j]), ref[(4 * h + j) * kThreads]);
            }
          }
        }
        if constexpr (REG) {
#pragma unroll
          for (int v = 0; v < 3; ++v)
            if (VM & (1 << v)) {
              const double w = warp_sum(acc[v]);
              if (lane == 0) out.part[v][r * rstride + slot] = w;
            }
        }
      }
      if (last_to_leave(ring.empty + s, ring.released + s, (uint32_t)(q / kStages) & 1u)) {
        const i64 next = q + kStages;
        if (next < nseq) issue(next, s);
      }
      if constexpr (REG) {
        if (lane < out.nregions && ((wmask >> lane) & 1u) == 0) {
#pragma unroll
          for (int v = 0; v < 3; ++v)
            if (VM & (1 << v)) out.part[v][lane * rstride + slot] = 0.0;
        }
      } else {
#pragma unroll
        for (int v = 0; v < 3; ++v)
          if (VM & (1 << v)) {
            const double w = warp_sum(acc[v]);
            if (lane == 0) out.part[v][slot] = w;
          }
      }
    }
  }
}

// ----------------------------------------------------------------------- host side
static Geom geometry(i64 nrows, int nz, i64 ncol) {
  Geom g;
  g.ncol = ncol;
  g.tiles_per_row = (int)((ncol + kTile - 1) / kTile);
  g.ntiles = nrows * g.tiles_per_row;
  g.nz = nz;
  return g;
}

static unsigned persistent_grid(i64 ntiles, int ctas_per_sm) {
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const i64 want = (i64)ctas_per_sm * sms;
  return (unsigned)(ntiles < want ? ntiles : want);
}

bool eligible(const void* a, const void* b, const void* c, const void* out, i64 ncol) {
  const uintptr_t bits = reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(c);
  // fp32 rows start on 16 bytes (bulk copies), fp64 result rows on 32 (256-bit stores)
  return (bits & 15u) == 0 && (reinterpret_cast<uintptr_t>(out) & 31u) == 0 && ncol % 4 == 0 && ncol >= 4 &&
         ncol / kTile < 0x7fffffff;
}

template <typename K>
static int opt_in(K kern, size_t smem) {
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  return e == cudaSuccess ? ML_OK : cuda_fail(e, "cudaFuncSetAttribute(k_stream)");
}

int launch_spice(const float* T, const float* S, i64 n, double* out, cudaStream_t st) {
  const Geom g = geometry(1, 1, n);
  auto kern = k_stream_map<0, 0>;
  if (int rc = opt_in(kern, ring_bytes<2>())) return rc;
  kern<<<persistent_grid(g.ntiles, ML_STREAM_CTAS), kThreads, ring_bytes<2>(), st>>>(T, S, 0, 0, nullptr, 0, g, out);
  return launched("k_stream_map(spice)");
}

int launch_density(int eos, const float* T, const float* S, i64 t_stride, i64 s_stride, const double* p, int pmode,
                   i64 nrows, int nz, i64 ncol, double* out, cudaStream_t st) {
  const Geom g = geometry(nrows, nz, ncol);
  const unsigned grid = persistent_grid(g.ntiles, ML_STREAM_CTAS);
  if (eos == ML_EOS_WRIGHT) {
    auto kern = k_stream_map<1, 0>;
    if (int rc = opt_in(kern, ring_bytes<2>())) return rc;
    kern<<<grid, kThreads, ring_bytes<2>(), st>>>(T, S, t_stride, s_stride, p, pmode, g, out);
  } else {
    auto kern = k_stream_map<1, 1>;
    if (int rc = opt_in(kern, ring_bytes<2>())) return rc;
    kern<<<grid, kThreads, ring_bytes<2>(), st>>>(T, S, t_stride, s_stride, p, pmode, g, out);
  }
  return launched("k_stream_map(density)");
}

int refstate_blocks(i64 nz, i64 ncol) {
  const Geom g = geometry(nz, (int)nz, ncol);
  return (int)persistent_grid(g.ntiles, 2);
}

int launch_refstate(int eos, const float* T0, const float* S0, const float* V0, const double* p_level, i64 nz, i64 ncol,
                    double* rho_ref, double* partials, cudaStream_t st) {
  const Geom g = geometry(nz, (int)nz, ncol);
  const unsigned grid = persistent_grid(g.ntiles, 2);
  if (eos == ML_EOS_WRIGHT) {
    auto kern = k_stream_refstate<0>;
    if (int rc = opt_in(kern, ring_bytes<3>())) return rc;
    kern<<<grid, kThreads, ring_bytes<3>(), st>>>(T0, S0, V0, p_level, g, rho_ref, partials);
  } else {
    auto kern = k_stream_refstate<1>;
    if (int rc = opt_in(kern, ring_bytes<3>())) return rc;
    kern<<<grid, kThreads, ring_bytes<3>(), st>>>(T0, S0, V0, p_level, g, rho_ref, partials);
  }
  return launched("k_stream_refstate");
}

int launch_delta_rho(int eos, const float* T, const float* S, i64 t_stride, i64 s_stride, const double* rho_ref,
                     const void* v_ref, int v_f32, const double* p_level, int nt, i64 nz, i64 ncol, double* out,
                     cudaStream_t st) {
  const Geom g = geometry(nz, (int)nz, ncol);
  const unsigned grid = persistent_grid(g.ntiles, 2);
#define ML_STREAM_DRHO(E, TV)                                                                                     \
  do {                                                                                                            \
    auto kern = k_stream_delta_rho<E, TV>;                                                                        \
    if (int rc = opt_in(kern, ring_bytes<2>())) return rc;                                                        \
    kern<<<grid, kThreads, ring_bytes<2>(), st>>>(T, S, t_stride, s_stride, rho_ref, (const TV*)v_ref, p_level, nt, g, out); \
  } while (0)
  if (eos == ML_EOS_WRIGHT) {
    if (v_f32) ML_STREAM_DRHO(0, float); else ML_STREAM_DRHO(0, double);
  } else {
    if (v_f32) ML_STREAM_DRHO(1, float); else ML_STREAM_DRHO(1, double);
  }
#undef ML_STREAM_DRHO
  return launched("k_stream_delta_rho");
}

constexpr size_t profile_smem_bytes() { return kProfileRing + 2 * kTile * (sizeof(double) + sizeof(float)); }

int profile_slots(i64 ncol) { return (int)((ncol + kTile - 1) / kTile) * kWarps; }

template <int EOS, int VM, bool ZON, bool REG>
static int launch_profile_vm(const float* T, const float* S, const float* T_ref, const float* S_ref,
                             const double* rho_ref, const void* v_ref, int v_f32, const double* z_i,
                             const double* deptho, const double* weights, const double* p_level, double coef, int nt,
                             const Geom& g, const ProfileOut& out, cudaStream_t st) {
  auto kern = k_stream_profile<EOS, VM, ZON, REG>;
  if (int rc = opt_in(kern, profile_smem_bytes())) return rc;
  kern<<<persistent_grid(g.ntiles, 2), kThreads, profile_smem_bytes(), st>>>(T, S, T_ref, S_ref, rho_ref, v_ref, v_f32, z_i,
                                                                         deptho, weights, p_level, coef, nt, g, out);
  return launched("k_stream_profile");
}

template <int EOS>
static int launch_profile_eos(int vm, const float* T, const float* S, const float* T_ref, const float* S_ref,
                              const double* rho_ref, const void* v_ref, int v_f32, const double* z_i,
                              const double* deptho, const double* weights, const double* p_level, double coef, int nt,
                              const Geom& g, const ProfileOut& out, cudaStream_t st) {
#define ML_STREAM_PROF(VM)                                                                                               \
  case VM:                                                                                                               \
    return out.region ? launch_profile_vm<EOS, VM, false, true>(T, S, T_ref, S_ref, rho_ref, v_ref, v_f32, z_i,         \
                                                                deptho, weights, p_level, coef, nt, g, out, st)         \
           : out.ny   ? launch_profile_vm<EOS, VM, true, false>(T, S, T_ref, S_ref, rho_ref, v_ref, v_f32, z_i,         \
                                                                deptho, weights, p_level, coef, nt, g, out, st)         \
                      : launch_profile_vm<EOS, VM, false, false>(T, S, T_ref, S_ref, rho_ref, v_ref, v_f32, z_i,        \
                                                                 deptho, weights, p_level, coef, nt, g, out, st)
  switch (vm) {
    ML_STREAM_PROF(1);
    ML_STREAM_PROF(2);
    ML_STREAM_PROF(3);
    ML_STREAM_PROF(4);
    ML_STREAM_PROF(5);
    ML_STREAM_PROF(6);
    ML_STREAM_PROF(7);
  }
#undef ML_STREAM_PROF
  return fail(ML_ERR_MODE, "variant mask %d", vm);
}

int launch_profile(int eos, int vm, const float* T, const float* S, const float* T_ref, const float* S_ref,
                   const double* rho_ref, const void* v_ref, int v_f32, const double* z_i, const double* deptho,
                   const double* weights, const double* p_level, double coef, int nt, i64 nz, i64 ncol,
                   double* const part[3], const int8_t* region, int nregions, int ny, cudaStream_t st) {
  const i64 rows = ny ? nz * ny : nz;  // ZON: nz * ny rows of ncol = nx columns
  const Geom g = geometry(rows, (int)rows, ncol);
  const ProfileOut out = {{part[0], part[1], part[2]}, region, nregions, ny};
  if (eos == ML_EOS_WRIGHT)
    return launch_profile_eos<0>(vm, T, S, T_ref, S_ref, rho_ref, v_ref, v_f32, z_i, deptho, weights, p_level, coef, nt, g, out, st);
  return launch_profile_eos<1>(vm, T, S, T_ref, S_ref, rho_ref, v_ref, v_f32, z_i, deptho, weights, p_level, coef, nt, g, out, st);
}

}  // namespace stream
}  // namespace ml
