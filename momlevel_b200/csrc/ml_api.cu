// ml_api.cu -- C ABI entry points of libmomlevel_b200 and the "direct" kernel family.
//
// The direct kernels read global memory straight into registers with coalesced loads, one
// water column per thread, and accept any extent and alignment.  They are the path for
// small or ragged grids (the reference's 5x5x5 test dataset) and the correctness baseline
// for the TMA-staged kernels in ml_tma.cu, which the entry points prefer when the grid
// meets TMA's 16-byte stride rule.
//
// Loop order (both families): a thread owns one column; z is the outer serial loop and a
// chunk of TC time steps the inner one, so rho_ref / v_ref / dz are fetched once per
// (level, column) and reused for TC steps, and the column sum never leaves registers.
#include "ml_common.cuh"
#include "ml_host.cuh"
#include "ml_stream.cuh"
#include "ml_tma.cuh"

namespace ml {

ThreadState& tls() {
  static thread_local ThreadState s = {{0}, ML_PATH_NONE, 0, 0};
  return s;
}

constexpr int kBlock = 256;
constexpr int kWarps = kBlock / 32;
constexpr int kTC = 12;  // time steps per register chunk of the direct kernels
constexpr int kPNone = 3;  // internal pressure mode: operand absent

__device__ __forceinline__ bool vref_wet(const void* v, int v_f32, i64 i) {
  return v_f32 ? !isnan(__ldg(reinterpret_cast<const float*>(v) + i))
               : !isnan(__ldg(reinterpret_cast<const double*>(v) + i));
}
__device__ __forceinline__ double vref_val(const void* v, int v_f32, i64 i) {
  return v_f32 ? (double)__ldg(reinterpret_cast<const float*>(v) + i)
               : __ldg(reinterpret_cast<const double*>(v) + i);
}

// 128-bit streaming loads / stores of four consecutive values (every byte is touched once).
__device__ __forceinline__ void ld4(const float* p, double v[4]) {
  float4 f;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(f.x), "=f"(f.y), "=f"(f.z), "=f"(f.w) : "l"(p));
  v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w;
}
__device__ __forceinline__ void ld4(const double* p, double v[4]) {
  asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0, %1}, [%2];" : "=d"(v[0]), "=d"(v[1]) : "l"(p));
  asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0, %1}, [%2];" : "=d"(v[2]), "=d"(v[3]) : "l"(p + 2));
}
__device__ __forceinline__ void st4(double* p, const double v[4]) {
  asm volatile("st.global.L1::no_allocate.v2.f64 [%0], {%1, %2};" ::"l"(p), "d"(v[0]), "d"(v[1]) : "memory");
  asm volatile("st.global.L1::no_allocate.v2.f64 [%0], {%1, %2};" ::"l"(p + 2), "d"(v[2]), "d"(v[3]) : "memory");
}

// ------------------------------------------------------------------ K1: elementwise EOS
template <typename TIn, int EOS, int FUNC>
__global__ void __launch_bounds__(kBlock) k_eos_eval(const TIn* __restrict__ T, const TIn* __restrict__ S,
                                                     i64 t_stride, i64 s_stride, const double* __restrict__ p,
                                                     int pmode, i64 nrows, int nz, i64 ncol,
                                                     double* __restrict__ out) {
  const i64 c = (i64)blockIdx.x * kBlock + threadIdx.x;
  if (c >= ncol) return;
  for (i64 row = blockIdx.y; row < nrows; row += gridDim.y) {
    const i64 t = row / nz;
    const int z = (int)(row - t * nz);
    const i64 o = row * ncol + c;
    double pv = 0.0;  // kPNone: the linear EOS takes no pressure (linear.py:26)
    if (pmode == ML_P_SCALAR) pv = __ldg(p);
    else if (pmode == ML_P_PER_LEVEL) pv = __ldg(p + z);
    else if (pmode == ML_P_FULL) pv = __ldg(p + o);
    const double Tv = ldf(T + t * t_stride + (i64)z * ncol + c);
    const double Sv = ldf(S + t * s_stride + (i64)z * ncol + c);
    out[o] = eos_func<EOS, FUNC>(Tv, Sv, pv);
  }
}

// Vectorised K1: a thread owns four adjacent columns and walks the rows assigned to its block.
// Needs ncol % 4 == 0 and 16-byte aligned bases (rows then stay aligned).
template <typename TIn, int EOS, int FUNC>
__global__ void __launch_bounds__(kBlock) k_eos_eval_vec(const TIn* __restrict__ T, const TIn* __restrict__ S,
                                                         i64 t_stride, i64 s_stride, const double* __restrict__ p,
                                                         int pmode, i64 nrows, int nz, i64 ncol,
                                                         double* __restrict__ out) {
  const i64 c = 4 * ((i64)blockIdx.x * kBlock + threadIdx.x);
  if (c >= ncol) return;
  for (i64 row = blockIdx.y; row < nrows; row += gridDim.y) {
    const i64 t = row / nz;
    const int z = (int)(row - t * nz);
    const i64 o = row * ncol + c;
    double tv[4], sv[4], pv[4], r[4];
    ld4(T + t * t_stride + (i64)z * ncol + c, tv);
    ld4(S + t * s_stride + (i64)z * ncol + c, sv);
    if (pmode == ML_P_FULL) {
      ld4(p + o, pv);
    } else {
      const double p1 = pmode == ML_P_SCALAR ? __ldg(p) : (pmode == ML_P_PER_LEVEL ? __ldg(p + z) : 0.0);
      pv[0] = pv[1] = pv[2] = pv[3] = p1;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) r[j] = eos_func<EOS, FUNC>(tv[j], sv[j], pv[j]);
    st4(out + o, r);
  }
}

// ------------------------------------------------------------------ K1b: density anomaly
// delta_rho[t][z][col] = V_ref notnull ? rho(T,S,p_z) - rho_ref : NaN   (steric.py:151-153).
// One level per trip of blockIdx.y; rho_ref / v_ref are read once per (level, column) and reused
// for every time step.  VEC = 4 adjacent columns per thread with 128-bit accesses, or 1.
// ANNUAL: out[year][z][col] = sum_m w_m d_m / sum_m w_m over the 12 steps of each year, NaNs skipped
// and the weights renormalised per cell (xarray's weighted(...).mean, util.py:84-87) -- the 4-D
// monthly anomaly is never stored.
template <typename TIn, int EOS, int VEC, bool ANNUAL>
__global__ void __launch_bounds__(kBlock) k_delta_rho(const TIn* __restrict__ T, const TIn* __restrict__ S,
                                                      i64 t_stride, i64 s_stride,
                                                      const double* __restrict__ rho_ref,
                                                      const void* __restrict__ v_ref, int v_f32,
                                                      const double* __restrict__ p_level,
                                                      const double* __restrict__ p_col,
                                                      const double* __restrict__ weights, int nt, int nz, i64 ncol,
                                                      double* __restrict__ out) {
  const i64 c = VEC * ((i64)blockIdx.x * kBlock + threadIdx.x);
  if (c >= ncol) return;
  Eos<EOS> eos;
  const double pc = (VEC == 1 && p_col != nullptr) ? __ldg(p_col + c) : 0.0;  // a 2-D patm (steric.py:96); VEC = 1 then
  for (int z = blockIdx.y; z < nz; z += gridDim.y) {
    const i64 i = (i64)z * ncol + c;
    eos.set_level(__ldg(p_level + z) + pc);
    double ref[VEC];
    if (VEC == 4) {
      ld4(rho_ref + i, ref);
    } else {
      ref[0] = __ldg(rho_ref + i);
    }
#pragma unroll
    for (int j = 0; j < VEC; ++j)
      if (!vref_wet(v_ref, v_f32, i + j)) ref[j] = nan("");
    double num[VEC], den[VEC];
#pragma unroll
    for (int j = 0; j < VEC; ++j) num[j] = den[j] = 0.0;
    for (int t = 0; t < nt; ++t) {
      double tv[VEC], sv[VEC], r[VEC];
      if (VEC == 4) {
        ld4(T + t * t_stride + i, tv);
        ld4(S + t * s_stride + i, sv);
      } else {
        tv[0] = ldf(T + t * t_stride + i);
        sv[0] = ldf(S + t * s_stride + i);
      }
#pragma unroll
      for (int j = 0; j < VEC; ++j) r[j] = eos.rho(tv[j], sv[j]) - ref[j];
      if (ANNUAL) {
        const double w = __ldg(weights + t);
#pragma unroll
        for (int j = 0; j < VEC; ++j)
          if (!is_nan_q(r[j])) {
            num[j] = fma(w, r[j], num[j]);
            den[j] += w;
          }
        if (t % 12 != 11) continue;
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
          r[j] = num[j] / den[j];  // 0/0 = NaN where every month is missing
          num[j] = den[j] = 0.0;
        }
      }
      double* o = out + ((i64)(ANNUAL ? t / 12 : t) * nz + z) * ncol + c;
      if (VEC == 4) {
        st4(o, r);
      } else {
        o[0] = r[0];
      }
    }
  }
}

// ---------------------------------------------------------------------------- K5: spice
template <typename TIn>
__global__ void __launch_bounds__(kBlock) k_spice(const TIn* __restrict__ T, const TIn* __restrict__ S, i64 n,
                                                  double* __restrict__ out) {
  const i64 stride = (i64)gridDim.x * kBlock;
  for (i64 i = (i64)blockIdx.x * kBlock + threadIdx.x; i < n; i += stride)
    out[i] = flament_spice(ldf(T + i), ldf(S + i));
}

// Vectorised variant (helpers ld4 / st4 above): four consecutive points per thread.
template <typename TIn>
__global__ void __launch_bounds__(kBlock) k_spice_vec(const TIn* __restrict__ T, const TIn* __restrict__ S, i64 n4,
                                                      double* __restrict__ out) {
  const i64 stride = (i64)gridDim.x * kBlock;
  for (i64 q = (i64)blockIdx.x * kBlock + threadIdx.x; q < n4; q += stride) {
    double t[4], s[4], r[4];
    ld4(T + 4 * q, t);
    ld4(S + 4 * q, s);
#pragma unroll
    for (int j = 0; j < 4; ++j) r[j] = flament_spice(t[j], s[j]);
    st4(out + 4 * q, r);
  }
}

// ------------------------------------------------------------------------------- K6: dz
__global__ void __launch_bounds__(kBlock) k_calc_dz(const double* __restrict__ z_i, const double* __restrict__ deptho,
                                                    double top, double bottom, int has_bottom, int fraction,
                                                    int nz, i64 ncol, double* __restrict__ out) {
  const i64 c = (i64)blockIdx.x * kBlock + threadIdx.x;
  if (c >= ncol) return;
  double depth = __ldg(deptho + c);
  if (isnan(depth)) depth = 0.0;                  // derived.py:295
  if (has_bottom) depth = fmin(depth, bottom);    // derived.py:298
  for (int z = blockIdx.y; z < nz; z += gridDim.y) {
    const double ztop = __ldg(z_i + z), zbot = __ldg(z_i + z + 1);
    const double full = zbot - ztop;
    double r = fmin(fmax(depth - ztop, 0.0), full);  // derived.py:308-313
    r = fmin(fmax(zbot - top, 0.0), r);              // derived.py:316-318
    if (fraction) {                                  // derived.py:320-323
      const double num = r == 0.0 ? nan("") : r;
      const double den = full == 0.0 ? nan("") : full;
      r = num / den;
    }
    out[(i64)z * ncol + c] = r;
  }
}

// ------------------------------------------------------- K7: volume / mass sums of given fields
// partials[row][block] = skipna sum over the block's share of a[row][i] * w[i] (w absent: of a[row][i]):
// derived.calc_volo (derived.py:787-789: volcello.sum()) and derived.calc_masso on a density field that already
// exists (derived.py:435-438: (rho * volcello).sum() per time step) without the rho * volcello temporary.
template <typename TA, typename TW>
__global__ void __launch_bounds__(kBlock) k_weighted_nansum(const TA* __restrict__ a, const TW* __restrict__ w, i64 n,
                                                            double* __restrict__ partials /* [rows][gridDim.x] */) {
  __shared__ double sm[kWarps];
  const TA* row = a + (i64)blockIdx.y * n;
  double acc = 0.0;
  for (i64 i = (i64)blockIdx.x * kBlock + threadIdx.x; i < n; i += (i64)gridDim.x * kBlock) {
    const double x = ldf(row + i);
    const double p = w != nullptr ? x * ldf(w + i) : x;
    if (!isnan(p)) acc += p;
  }
  acc = block_sum<kWarps>(acc, sm);
  if (threadIdx.x == 0) partials[(i64)blockIdx.y * gridDim.x + blockIdx.x] = acc;
}

// ------------------------------------------------------- fixed-order second reduce stage
// out[row] = sum_b partials[row][b]; one block per row, each thread a strided serial sum.
__global__ void __launch_bounds__(kBlock) k_reduce_rows(const double* __restrict__ partials, i64 nblk,
                                                        double* __restrict__ out) {
  __shared__ double sm[kWarps];
  const double* row = partials + (i64)blockIdx.x * nblk;
  double a = 0.0;
  for (i64 b = threadIdx.x; b < nblk; b += kBlock) a += row[b];
  a = block_sum<kWarps>(a, sm);
  if (threadIdx.x == 0) out[blockIdx.x] = a;
}

// ------------------------------------------------------------------ K2: reference state
template <typename TIn, int EOS>
__global__ void __launch_bounds__(kBlock) k_reference_state(const TIn* __restrict__ T0, const TIn* __restrict__ S0,
                                                            const void* __restrict__ V0, int v_f32,
                                                            const double* __restrict__ p_level,
                                                            const double* __restrict__ p_col,
                                                            int nz, i64 ncol, double* __restrict__ rho_ref,
                                                            double* __restrict__ partials /* [2][gridDim.x] */) {
  __shared__ double sm[kWarps];
  const i64 c = (i64)blockIdx.x * kBlock + threadIdx.x;
  double vol = 0.0, mass = 0.0;
  Eos<EOS> eos;
  if (c < ncol) {
    const double pc = p_col != nullptr ? __ldg(p_col + c) : 0.0;  // a 2-D patm: pres = z_l * 1e4 + patm (reference.py:54)
    for (int z = 0; z < nz; ++z) {
      const i64 i = (i64)z * ncol + c;
      eos.set_level(__ldg(p_level + z) + pc);
      const double rho = eos.rho(ldf(T0 + i), ldf(S0 + i));
      const double v = vref_val(V0, v_f32, i);
      rho_ref[i] = rho;
      if (!isnan(v)) {  // nansum (derived.py:787-789, :435-438)
        vol += v;
        const double m = rho * v;
        if (!is_nan_q(m)) mass += m;
      }
    }
  }
  vol = block_sum<kWarps>(vol, sm);
  mass = block_sum<kWarps>(mass, sm);
  if (threadIdx.x == 0) {
    partials[blockIdx.x] = vol;
    partials[(i64)gridDim.x + blockIdx.x] = mass;
  }
}

// Vectorised K2: one level per blockIdx.y, four adjacent columns per thread, 128-bit accesses.
// Block partials are laid out [2][gridDim.y * gridDim.x] for k_reduce_rows.
template <typename TIn, int EOS>
__global__ void __launch_bounds__(kBlock) k_reference_state_vec(const TIn* __restrict__ T0, const TIn* __restrict__ S0,
                                                                const TIn* __restrict__ V0,
                                                                const double* __restrict__ p_level, i64 ncol,
                                                                double* __restrict__ rho_ref,
                                                                double* __restrict__ partials) {
  __shared__ double sm[kWarps];
  const int z = blockIdx.y;
  const i64 nq = ncol / 4, base = (i64)z * ncol;
  Eos<EOS> eos;
  eos.set_level(__ldg(p_level + z));
  double vol = 0.0, mass = 0.0;
  const i64 stride = (i64)gridDim.x * kBlock;
  for (i64 q0 = (i64)blockIdx.x * kBlock + threadIdx.x; q0 < nq; q0 += 2 * stride) {
    // two quads per trip: all six loads are issued before any arithmetic
    const bool two = q0 + stride < nq;
    const i64 q1 = two ? q0 + stride : q0;
    double ta[4], sa[4], va[4], ra[4], tb[4], sb[4], vb[4], rb[4];
    ld4(T0 + base + 4 * q0, ta);
    ld4(S0 + base + 4 * q0, sa);
    ld4(V0 + base + 4 * q0, va);
    ld4(T0 + base + 4 * q1, tb);
    ld4(S0 + base + 4 * q1, sb);
    ld4(V0 + base + 4 * q1, vb);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      ra[j] = eos.rho(ta[j], sa[j]);
      rb[j] = eos.rho(tb[j], sb[j]);
      if (!isnan(va[j])) {  // nansum (derived.py:787-789, :435-438)
        vol += va[j];
        const double m = ra[j] * va[j];
        if (!is_nan_q(m)) mass += m;
      }
      if (two && !isnan(vb[j])) {
        vol += vb[j];
        const double m = rb[j] * vb[j];
        if (!is_nan_q(m)) mass += m;
      }
    }
    st4(rho_ref + base + 4 * q0, ra);
    if (two) st4(rho_ref + base + 4 * q1, rb);
  }
  vol = block_sum<kWarps>(vol, sm);
  mass = block_sum<kWarps>(mass, sm);
  if (threadIdx.x == 0) {
    const i64 nblk = (i64)gridDim.x * gridDim.y, b = (i64)blockIdx.y * gridDim.x + blockIdx.x;
    partials[b] = vol;
    partials[nblk + b] = mass;
  }
}

// ------------------------------------------------------------- K3 direct: local steric
// Layer edges of ml_steric_local_layers, passed by value.
struct LayerEdges {
  int n;                           // layers
  double e[ML_MAX_LAYERS + 1];     // increasing; the last may be +inf
};

// LAYERS: the height split by depth layer (ml_steric_local_layers), eta [nt][nlayers][ncol]; level z feeds layer b
// with calc_dz(top=e[b], bottom=e[b+1]) (derived.py:295-318) and a layer is stored when the sweep leaves it.
template <typename TIn, int EOS, bool WRITE_DRHO, bool LAYERS = false>
__global__ void __launch_bounds__(kBlock)
    k_steric_local_direct(const TIn* __restrict__ T, const TIn* __restrict__ S, i64 t_stride, i64 s_stride,
                          const double* __restrict__ rho_ref, const void* __restrict__ v_ref, int v_f32,
                          const double* __restrict__ z_i, const double* __restrict__ deptho,
                          const double* __restrict__ p_level, const double* __restrict__ p_col, double coef, int nt,
                          int nz, i64 ncol, double* __restrict__ eta, double* __restrict__ drho,
                          const LayerEdges L = LayerEdges()) {
  const i64 c = (i64)blockIdx.x * kBlock + threadIdx.x;
  if (c >= ncol) return;
  const int t0 = blockIdx.y * kTC;
  const i64 lvl = ncol;  // elements per level

  double depth = __ldg(deptho + c);
  if (isnan(depth)) depth = 0.0;  // derived.py:295
  const bool surface_wet = vref_wet(v_ref, v_f32, c);  // steric.py:166

  double acc[kTC];
#pragma unroll
  for (int k = 0; k < kTC; ++k) acc[k] = 0.0;
  Eos<EOS> eos;
  const double pc = p_col != nullptr ? __ldg(p_col + c) : 0.0;  // a 2-D patm (steric.py:96)
  int cur = 0;  // LAYERS: the layer the sums belong to
  auto store_layer = [&](int b, int k, double a) {
    if (t0 + k < nt) eta[((i64)(t0 + k) * L.n + b) * ncol + c] = surface_wet ? coef * a : nan("");
  };
  auto close_layer = [&](int b) {
#pragma unroll
    for (int k = 0; k < kTC; ++k) {
      store_layer(b, k, acc[k]);
      acc[k] = 0.0;
    }
  };

  for (int z = 0; z < nz; ++z) {
    const i64 i = (i64)z * lvl + c;
    const double ztop = __ldg(z_i + z), zbot = __ldg(z_i + z + 1);
    const double dz = clipped_dz(depth, ztop, zbot);
    // LAYERS: layers lo .. hi touch this level (z_i[z+1] > e[b] && z_i[z] < e[b+1]); a level no layer touches
    // adds nothing.  Layers that ended above it are stored first.
    int lo = -1, hi = -1;
    if (LAYERS) {
      for (int b = 0; b < L.n; ++b)
        if (zbot > L.e[b] && ztop < L.e[b + 1]) {
          if (lo < 0) lo = b;
          hi = b;
        }
      if (lo < 0) continue;
      for (; cur < lo; ++cur) close_layer(cur);
    }
    auto layer_w = [&](int b) { return fmin(fmax(zbot - L.e[b], 0.0), clipped_dz(fmin(depth, L.e[b + 1]), ztop, zbot)); };
    const double wl = LAYERS ? layer_w(lo) : dz;
    // steric.py:151-153: delta_rho is NaN wherever the reference volume is missing
    const double rref = vref_wet(v_ref, v_f32, i) ? __ldg(rho_ref + i) : nan("");
    eos.set_level(__ldg(p_level + z) + pc);
    // all loads of the chunk first (time index clamped: a short last chunk re-reads the
    // final step instead of branching), then the arithmetic
    TIn tv[kTC], sv[kTC];
#pragma unroll
    for (int k = 0; k < kTC; ++k) {
      const i64 t = min(t0 + k, nt - 1);
      tv[k] = __ldg(T + t * t_stride + i);
      sv[k] = __ldg(S + t * s_stride + i);
    }
#pragma unroll
    for (int k = 0; k < kTC; ++k) {
      const double d = eos.rho((double)tv[k], (double)sv[k]) - rref;
      if (WRITE_DRHO) {
        if (t0 + k < nt) drho[((i64)(t0 + k) * nz + z) * lvl + c] = d;
      }
      if (LAYERS && lo < hi) {
        // the level closes layers lo .. hi - 1 and opens hi
        const bool skip = is_nan_q(d);
        store_layer(lo, k, skip ? acc[k] : fma(wl, d, acc[k]));
        for (int b = lo + 1; b < hi; ++b) store_layer(b, k, skip ? 0.0 : layer_w(b) * d);
        acc[k] = skip ? 0.0 : layer_w(hi) * d;
      } else if (!is_nan_q(d)) {
        acc[k] = fma(wl, d, acc[k]);  // skipna sum, steric.py:163
      }
    }
    if (LAYERS && lo < hi) cur = hi;  // layers lo .. hi - 1 are stored; the sums now belong to layer hi
  }
  if (LAYERS) {
    for (; cur < L.n; ++cur) close_layer(cur);  // the last layer, and those wholly below the grid: 0
    return;
  }
#pragma unroll
  for (int k = 0; k < kTC; ++k) {
    const int t = t0 + k;
    if (t < nt) eta[(i64)t * ncol + c] = surface_wet ? coef * acc[k] : nan("");
  }
}

// ------------------------------------------------------------ K4 direct: global steric
template <typename TIn, int EOS>
__global__ void __launch_bounds__(kBlock)
    k_steric_global_direct(const TIn* __restrict__ T, const TIn* __restrict__ S, i64 t_stride, i64 s_stride,
                           const void* __restrict__ v_ref, int v_f32, const double* __restrict__ p_level,
                           const double* __restrict__ p_col, int nt, int nz, i64 ncol,
                           double* __restrict__ partials /* [nt][gridDim.x] */) {
  __shared__ double sm[kWarps];
  const i64 c = (i64)blockIdx.x * kBlock + threadIdx.x;
  const int t0 = blockIdx.y * kTC;
  double acc[kTC];
#pragma unroll
  for (int k = 0; k < kTC; ++k) acc[k] = 0.0;
  Eos<EOS> eos;
  if (c < ncol) {
    const double pc = p_col != nullptr ? __ldg(p_col + c) : 0.0;  // a 2-D patm (steric.py:96)
    for (int z = 0; z < nz; ++z) {
      const i64 i = (i64)z * ncol + c;
      const double v = vref_val(v_ref, v_f32, i);
      if (isnan(v)) continue;  // rho*NaN is dropped by the skipna sum (derived.py:435-438)
      eos.set_level(__ldg(p_level + z) + pc);
      TIn tv[kTC], sv[kTC];
#pragma unroll
      for (int k = 0; k < kTC; ++k) {
        const i64 t = min(t0 + k, nt - 1);
        tv[k] = __ldg(T + t * t_stride + i);
        sv[k] = __ldg(S + t * s_stride + i);
      }
#pragma unroll
      for (int k = 0; k < kTC; ++k) {
        const double rho = eos.rho((double)tv[k], (double)sv[k]);
        if (!is_nan_q(rho)) acc[k] = fma(rho, v, acc[k]);
      }
    }
  }
#pragma unroll
  for (int k = 0; k < kTC; ++k) {
    const int t = t0 + k;
    if (t < nt) {  // uniform across the block
      const double s = block_sum<kWarps>(acc[k], sm);
      if (threadIdx.x == 0) partials[(i64)t * gridDim.x + blockIdx.x] = s;
    }
  }
}

// --------------------------------------------------------------------------- dispatch
inline i64 cdiv(i64 a, i64 b) { return (a + b - 1) / b; }

// the plain-load kernels only: asked for (ml_set_force_direct(1)) or needed because a per-column pressure offset
// is set (ml_set_column_pressure), which the ring-staged families do not carry
inline bool direct_only() { return tls().force_direct == 1 || tls().p_col != nullptr; }

// every entry point that evaluates the EOS per column checks the offset's length against its own ncol
inline int check_column_pressure(int64_t ncol) {
  if (tls().p_col != nullptr && tls().p_col_n != ncol)
    return fail(ML_ERR_SHAPE, "column pressure set for %lld columns, call has %lld", (long long)tls().p_col_n, (long long)ncol);
  return ML_OK;
}

inline int check_common(int eos, int dtype) {
  if (eos != ML_EOS_WRIGHT && eos != ML_EOS_LINEAR) return fail(ML_ERR_EOS, "unknown equation of state id %d", eos);
  if (dtype != ML_F32 && dtype != ML_F64) return fail(ML_ERR_DTYPE, "unknown dtype id %d", dtype);
  return ML_OK;
}

inline int check_bcast(int t_bcast, int s_bcast) {
  if (t_bcast && s_bcast) return fail(ML_ERR_MODE, "T and S cannot both be broadcast over time");
  return ML_OK;
}

template <int EOS, int FUNC>
int launch_eos(int dtype, const void* T, const void* S, i64 ts, i64 ss, const double* p, int pmode, i64 nrows, int nz,
               i64 ncol, double* out, cudaStream_t st) {
  const uintptr_t bits = reinterpret_cast<uintptr_t>(T) | reinterpret_cast<uintptr_t>(S) | reinterpret_cast<uintptr_t>(out) |
                         (pmode == ML_P_FULL ? reinterpret_cast<uintptr_t>(p) : 0);
  // fp32 fields, density, a pressure per row: the ring-staged streaming kernel (ml_stream.cu)
  if (FUNC == 0 && dtype == ML_F32 && pmode != ML_P_FULL && direct_only() == false && stream::eligible(T, S, nullptr, out, ncol) &&
      ts % 4 == 0 && ss % 4 == 0 && nz > 0)
    return stream::launch_density(EOS == 0 ? ML_EOS_WRIGHT : ML_EOS_LINEAR, (const float*)T, (const float*)S, ts, ss, p,
                                  pmode, nrows, nz, ncol, out, st);
  if (ncol % 4 == 0 && (bits & 15u) == 0) {
    // ~16 resident blocks per SM; each block walks its share of the rows
    const i64 gx = cdiv(ncol / 4, kBlock);
    i64 gy = cdiv(148 * 16, gx);
    gy = gy < 1 ? 1 : (gy > nrows ? nrows : gy);
    dim3 grid((unsigned)gx, (unsigned)(gy < 65535 ? gy : 65535));
    if (dtype == ML_F32)
      k_eos_eval_vec<float, EOS, FUNC><<<grid, kBlock, 0, st>>>((const float*)T, (const float*)S, ts, ss, p, pmode, nrows, nz, ncol, out);
    else
      k_eos_eval_vec<double, EOS, FUNC><<<grid, kBlock, 0, st>>>((const double*)T, (const double*)S, ts, ss, p, pmode, nrows, nz, ncol, out);
    return launched("k_eos_eval_vec");
  }
  dim3 grid((unsigned)cdiv(ncol, kBlock), (unsigned)(nrows < 65535 ? nrows : 65535));
  if (dtype == ML_F32)
    k_eos_eval<float, EOS, FUNC><<<grid, kBlock, 0, st>>>((const float*)T, (const float*)S, ts, ss, p, pmode, nrows, nz, ncol, out);
  else
    k_eos_eval<double, EOS, FUNC><<<grid, kBlock, 0, st>>>((const double*)T, (const double*)S, ts, ss, p, pmode, nrows, nz, ncol, out);
  return launched("k_eos_eval");
}

template <int EOS>
int launch_eos_func(int func, int dtype, const void* T, const void* S, i64 ts, i64 ss, const double* p, int pmode,
                    i64 nrows, int nz, i64 ncol, double* out, cudaStream_t st) {
  switch (func) {
    case ML_FUNC_DENSITY: return launch_eos<EOS, 0>(dtype, T, S, ts, ss, p, pmode, nrows, nz, ncol, out, st);
    case ML_FUNC_DRHO_DTEMP: return launch_eos<EOS, 1>(dtype, T, S, ts, ss, p, pmode, nrows, nz, ncol, out, st);
    case ML_FUNC_DRHO_DSAL: return launch_eos<EOS, 2>(dtype, T, S, ts, ss, p, pmode, nrows, nz, ncol, out, st);
    case ML_FUNC_ALPHA: return launch_eos<EOS, 3>(dtype, T, S, ts, ss, p, pmode, nrows, nz, ncol, out, st);
    case ML_FUNC_BETA: return launch_eos<EOS, 4>(dtype, T, S, ts, ss, p, pmode, nrows, nz, ncol, out, st);
  }
  return fail(ML_ERR_EOS, "unknown eos function id %d", func);
}

template <typename TIn, int EOS>
int launch_local_direct(const void* T, const void* S, i64 ts, i64 ss, const double* rho_ref, const void* v_ref,
                        int v_f32, const double* z_i, const double* deptho, const double* p_level, double coef, int nt,
                        int nz, i64 ncol, double* eta, double* drho, cudaStream_t st) {
  dim3 grid((unsigned)cdiv(ncol, kBlock), (unsigned)cdiv(nt, kTC));
  if (drho)
    k_steric_local_direct<TIn, EOS, true><<<grid, kBlock, 0, st>>>((const TIn*)T, (const TIn*)S, ts, ss, rho_ref, v_ref, v_f32, z_i, deptho, p_level, tls().p_col, coef, nt, nz, ncol, eta, drho);
  else
    k_steric_local_direct<TIn, EOS, false><<<grid, kBlock, 0, st>>>((const TIn*)T, (const TIn*)S, ts, ss, rho_ref, v_ref, v_f32, z_i, deptho, p_level, tls().p_col, coef, nt, nz, ncol, eta, drho);
  return launched("k_steric_local_direct");
}

template <typename TIn, int EOS>
int launch_layers_direct(const void* T, const void* S, i64 ts, i64 ss, const double* rho_ref, const void* v_ref,
                         int v_f32, const double* z_i, const double* deptho, const double* p_level, double coef, int nt,
                         int nz, i64 ncol, double* eta, const LayerEdges& L, cudaStream_t st) {
  dim3 grid((unsigned)cdiv(ncol, kBlock), (unsigned)cdiv(nt, kTC));
  k_steric_local_direct<TIn, EOS, false, true><<<grid, kBlock, 0, st>>>((const TIn*)T, (const TIn*)S, ts, ss, rho_ref, v_ref, v_f32, z_i, deptho, p_level, tls().p_col, coef, nt, nz, ncol, eta, nullptr, L);
  return launched("k_steric_local_direct");
}

template <typename TIn, int EOS>
int launch_global_direct(const void* T, const void* S, i64 ts, i64 ss, const void* v_ref, int v_f32,
                         const double* p_level, int nt, int nz, i64 ncol, double* masso, double* partials,
                         cudaStream_t st) {
  const i64 nblk = cdiv(ncol, kBlock);
  dim3 grid((unsigned)nblk, (unsigned)cdiv(nt, kTC));
  k_steric_global_direct<TIn, EOS><<<grid, kBlock, 0, st>>>((const TIn*)T, (const TIn*)S, ts, ss, v_ref, v_f32, p_level, tls().p_col, nt, nz, ncol, partials);
  int rc = launched("k_steric_global_direct");
  if (rc) return rc;
  k_reduce_rows<<<nt, kBlock, 0, st>>>(partials, nblk, masso);
  return launched("k_reduce_rows");
}

namespace tma {
int reduce_rows(const double* partials, int64_t nblk, double* out, int nrows, cudaStream_t st) {
  k_reduce_rows<<<nrows, kBlock, 0, st>>>(partials, nblk, out);
  return launched("k_reduce_rows");
}
}  // namespace tma

}  // namespace ml

using namespace ml;

// depth layers of the layered entry points: 1 <= nlayers <= ML_MAX_LAYERS, edges strictly increasing values >= 0, only
// the last may be +inf
static int check_layers(const double* edges, int nlayers) {
  if (nlayers < 1 || nlayers > ML_MAX_LAYERS)
    return fail(ML_ERR_SHAPE, "nlayers=%d: between 1 and %d depth layers", nlayers, ML_MAX_LAYERS);
  for (int b = 0; b <= nlayers; ++b) {
    const double e = edges[b];
    if (isnan(e) || e < 0.0 || (isinf(e) && b != nlayers) || (b > 0 && !(e > edges[b - 1])))
      return fail(ML_ERR_SHAPE, "layer edges must be strictly increasing values >= 0, only the last may be +inf; "
                                "edges[%d] = %g", b, e);
  }
  return ML_OK;
}

extern "C" {

int ml_version(void) { return ML_ABI_VERSION; }
const char* ml_last_error(void) { return tls().err; }
int ml_last_path(void) { return tls().last_path; }
int64_t ml_launch_count(void) { return tls().launches; }
int ml_set_force_direct(int on) {
  const int prev = tls().force_direct;
  tls().force_direct = on == 2 ? 2 : (on ? 1 : 0);
  return prev;
}

int ml_set_column_pressure(const double* p_col, int64_t ncol) {
  if (p_col != nullptr && ncol <= 0) return fail(ML_ERR_SHAPE, "column pressure needs ncol > 0, got %lld", (long long)ncol);
  tls().p_col = p_col;
  tls().p_col_n = p_col ? ncol : 0;
  return ML_OK;
}

int ml_set_variants_chunk(int tc) {
  const int prev = tls().variants_chunk;
  const int w = tc % 100;  // + 100: 128-column tiles, + 200: 256-column tiles (experiments)
  tls().variants_chunk = (tc >= 0 && tc < 300 && (w == 0 || w == 4 || w == 6 || w == 8 || w == 12)) ? tc : 0;
  return prev;
}

size_t ml_workspace_bytes(int64_t nt, int64_t nz, int64_t ncol) {
  if (nt < 2) nt = 2;  // reference_state needs two rows
  if (nz < 1) nz = 1;
  // per-row block partials: ceil(ncol/256) (direct family) or fewer (TMA family); the vectorised
  // reference-state kernel keeps up to 512 blocks per level for each of its two sums
  const int64_t nblk = cdiv(ncol > 0 ? ncol : 1, 128);
  const int64_t ref = 2 * nz * 512;
  return (size_t)(nt * nblk > ref ? nt * nblk : ref) * sizeof(double) + 256;
}

int ml_eos_eval(int eos, int func, int dtype, const void* T, const void* S, int t_bcast, int s_bcast, const double* p,
                int pmode, int64_t nouter, int64_t nz, int64_t ncol, double* out, void* stream) {
  int rc = check_common(eos, dtype);
  if (rc) return rc;
  if ((rc = check_bcast(t_bcast, s_bcast))) return rc;
  ML_REQUIRE_PTR(T);
  ML_REQUIRE_PTR(S);
  ML_REQUIRE_PTR(out);
  if (pmode != ML_P_SCALAR && pmode != ML_P_PER_LEVEL && pmode != ML_P_FULL)
    return fail(ML_ERR_MODE, "unknown pressure mode %d", pmode);
  if (eos == ML_EOS_WRIGHT) ML_REQUIRE_PTR(p);
  if (nouter < 0 || nz <= 0 || ncol < 0 || nz > INT32_MAX) return fail(ML_ERR_SHAPE, "bad extents nouter=%lld nz=%lld ncol=%lld", (long long)nouter, (long long)nz, (long long)ncol);
  ML_REQUIRE_ALIGNED(T, elem_size(dtype));
  ML_REQUIRE_ALIGNED(S, elem_size(dtype));
  ML_REQUIRE_ALIGNED(out, 8);
  if (nouter == 0 || ncol == 0) return ML_OK;  // empty input, nothing to launch
  const i64 lvl = nz * ncol;
  const i64 ts = t_bcast ? 0 : lvl, ss = s_bcast ? 0 : lvl;
  cudaStream_t st = (cudaStream_t)stream;
  if (p == nullptr) pmode = kPNone;  // linear EOS ignores pressure (linear.py:26)
  if (eos == ML_EOS_WRIGHT) return launch_eos_func<0>(func, dtype, T, S, ts, ss, p, pmode, nouter * nz, (int)nz, ncol, out, st);
  return launch_eos_func<1>(func, dtype, T, S, ts, ss, p, pmode, nouter * nz, (int)nz, ncol, out, st);
}

int ml_flament_spice(int dtype, const void* T, const void* S, int64_t n, double* out, void* stream) {
  if (dtype != ML_F32 && dtype != ML_F64) return fail(ML_ERR_DTYPE, "unknown dtype id %d", dtype);
  if (n < 0) return fail(ML_ERR_SHAPE, "n=%lld", (long long)n);
  if (n == 0) return ML_OK;
  ML_REQUIRE_PTR(T);
  ML_REQUIRE_PTR(S);
  ML_REQUIRE_PTR(out);
  ML_REQUIRE_ALIGNED(T, elem_size(dtype));
  ML_REQUIRE_ALIGNED(S, elem_size(dtype));
  ML_REQUIRE_ALIGNED(out, 8);
  cudaStream_t st = (cudaStream_t)stream;
  const int es = elem_size(dtype);
  i64 done = 0;
  const bool aligned = ((reinterpret_cast<uintptr_t>(T) | reinterpret_cast<uintptr_t>(S) | reinterpret_cast<uintptr_t>(out)) & 15u) == 0;
  if (aligned && dtype == ML_F32 && n >= 4 && n % 4 == 0 && tls().force_direct != 1)  // ring-staged streaming kernel (ml_stream.cu)
    return stream::launch_spice((const float*)T, (const float*)S, n, out, st);
  if (aligned && n >= 4) {
    const i64 n4 = n / 4;
    const unsigned grid = (unsigned)(cdiv(n4, kBlock) < 148 * 8 ? cdiv(n4, kBlock) : 148 * 8);
    if (dtype == ML_F32)
      k_spice_vec<float><<<grid, kBlock, 0, st>>>((const float*)T, (const float*)S, n4, out);
    else
      k_spice_vec<double><<<grid, kBlock, 0, st>>>((const double*)T, (const double*)S, n4, out);
    int rc = launched("k_spice_vec");
    if (rc) return rc;
    done = 4 * n4;
    if (done == n) return ML_OK;
  }
  const i64 rest = n - done;
  const unsigned grid = (unsigned)(cdiv(rest, kBlock) < 148 * 16 ? cdiv(rest, kBlock) : 148 * 16);
  const char* Tt = (const char*)T + done * es;
  const char* St = (const char*)S + done * es;
  if (dtype == ML_F32)
    k_spice<float><<<grid, kBlock, 0, st>>>((const float*)Tt, (const float*)St, rest, out + done);
  else
    k_spice<double><<<grid, kBlock, 0, st>>>((const double*)Tt, (const double*)St, rest, out + done);
  return launched("k_spice");
}

int ml_calc_dz(const double* z_i, const double* deptho, double top, double bottom, int has_bottom, int fraction,
               int64_t nz, int64_t ncol, double* out, void* stream) {
  ML_REQUIRE_PTR(z_i);
  ML_REQUIRE_PTR(deptho);
  ML_REQUIRE_PTR(out);
  if (nz <= 0 || ncol < 0 || nz > INT32_MAX) return fail(ML_ERR_SHAPE, "bad extents nz=%lld ncol=%lld", (long long)nz, (long long)ncol);
  if (int rcp = check_column_pressure(ncol)) return rcp;
  if (ncol == 0) return ML_OK;
  dim3 grid((unsigned)cdiv(ncol, kBlock), (unsigned)(nz < 65535 ? nz : 65535));
  k_calc_dz<<<grid, kBlock, 0, (cudaStream_t)stream>>>(z_i, deptho, top, bottom, has_bottom, fraction, (int)nz, ncol, out);
  return launched("k_calc_dz");
}

static int reference_state_impl(int eos, int dtype, const void* T0, const void* S0, const void* V0, int v_dtype,
                                const double* p_level, int64_t nz, int64_t ncol, double* rho_ref, double* sums,
                                void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_common(eos, dtype);
  if (rc) return rc;
  if (v_dtype != ML_F32 && v_dtype != ML_F64) return fail(ML_ERR_DTYPE, "unknown volcello dtype id %d", v_dtype);
  ML_REQUIRE_PTR(T0);
  ML_REQUIRE_PTR(S0);
  ML_REQUIRE_PTR(V0);
  ML_REQUIRE_PTR(p_level);
  ML_REQUIRE_PTR(rho_ref);
  ML_REQUIRE_PTR(sums);
  if (nz <= 0 || ncol <= 0 || nz > INT32_MAX) return fail(ML_ERR_SHAPE, "bad extents nz=%lld ncol=%lld", (long long)nz, (long long)ncol);
  if (int rcp = check_column_pressure(ncol)) return rcp;
  if (workspace == nullptr || workspace_bytes < ml_workspace_bytes(2, nz, ncol))
    return fail(ML_ERR_WORKSPACE, "workspace needs %zu bytes, got %zu", ml_workspace_bytes(2, nz, ncol), workspace_bytes);
  ML_REQUIRE_ALIGNED(workspace, 8);
  cudaStream_t st = (cudaStream_t)stream;
  double* partials = (double*)workspace;
  const int v_f32 = v_dtype == ML_F32;
  const uintptr_t bits = reinterpret_cast<uintptr_t>(T0) | reinterpret_cast<uintptr_t>(S0) |
                         reinterpret_cast<uintptr_t>(V0) | reinterpret_cast<uintptr_t>(rho_ref);
  if (dtype == ML_F32 && v_dtype == ML_F32 && direct_only() == false && stream::eligible(T0, S0, V0, rho_ref, ncol) &&
      (size_t)stream::refstate_blocks(nz, ncol) * 2 * sizeof(double) <= workspace_bytes) {
    // ring-staged streaming kernel (ml_stream.cu): persistent CTAs, block partials [2][blocks]
    if ((rc = stream::launch_refstate(eos, (const float*)T0, (const float*)S0, (const float*)V0, p_level, nz, ncol,
                                      rho_ref, partials, st)))
      return rc;
    k_reduce_rows<<<2, kBlock, 0, st>>>(partials, stream::refstate_blocks(nz, ncol), sums);
    return launched("k_reduce_rows");
  }
  if (v_dtype == dtype && ncol % 4 == 0 && (bits & 15u) == 0 && nz <= 65535 && tls().p_col == nullptr) {
    // ~12 resident blocks per SM over all levels; each thread walks its level in 2-quad trips
    i64 gx = cdiv(148 * 12, nz);
    const i64 need = cdiv(cdiv(ncol / 4, kBlock), 2);
    if (gx > need) gx = need;
    i64 cap = (i64)(workspace_bytes / sizeof(double) / 2 / nz);  // partials must fit the workspace
    if (cap > 512) cap = 512;
    if (gx > cap) gx = cap;
    if (gx >= 1) {
      dim3 grid((unsigned)gx, (unsigned)nz);
#define ML_LAUNCH_REFV(TIN, E) \
  k_reference_state_vec<TIN, E><<<grid, kBlock, 0, st>>>((const TIN*)T0, (const TIN*)S0, (const TIN*)V0, p_level, ncol, rho_ref, partials)
      if (dtype == ML_F32) {
        if (eos == ML_EOS_WRIGHT) ML_LAUNCH_REFV(float, 0); else ML_LAUNCH_REFV(float, 1);
      } else {
        if (eos == ML_EOS_WRIGHT) ML_LAUNCH_REFV(double, 0); else ML_LAUNCH_REFV(double, 1);
      }
#undef ML_LAUNCH_REFV
      if ((rc = launched("k_reference_state_vec"))) return rc;
      k_reduce_rows<<<2, kBlock, 0, st>>>(partials, gx * nz, sums);
      return launched("k_reduce_rows");
    }
  }
  const i64 nblk = cdiv(ncol, kBlock);
#define ML_LAUNCH_REF(TIN, E) \
  k_reference_state<TIN, E><<<(unsigned)nblk, kBlock, 0, st>>>((const TIN*)T0, (const TIN*)S0, V0, v_f32, p_level, tls().p_col, (int)nz, ncol, rho_ref, partials)
  if (dtype == ML_F32) {
    if (eos == ML_EOS_WRIGHT) ML_LAUNCH_REF(float, 0); else ML_LAUNCH_REF(float, 1);
  } else {
    if (eos == ML_EOS_WRIGHT) ML_LAUNCH_REF(double, 0); else ML_LAUNCH_REF(double, 1);
  }
#undef ML_LAUNCH_REF
  if ((rc = launched("k_reference_state"))) return rc;
  k_reduce_rows<<<2, kBlock, 0, st>>>(partials, nblk, sums);
  return launched("k_reduce_rows");
}

int ml_reference_state(int eos, int dtype, const void* T0, const void* S0, const void* V0, const double* p_level,
                       int64_t nz, int64_t ncol, double* rho_ref, double* sums, void* workspace, size_t workspace_bytes,
                       void* stream) {
  return reference_state_impl(eos, dtype, T0, S0, V0, dtype, p_level, nz, ncol, rho_ref, sums, workspace,
                              workspace_bytes, stream);
}

int ml_steric_local_selfref(int eos, int dtype, const void* T, const void* S, int t_bcast, int s_bcast,
                            const void* v_ref, int vref_dtype, const double* z_i, const double* deptho,
                            const double* p_level, double neg_inv_rhozero, int64_t nt, int64_t nz, int64_t ncol,
                            double* eta, double* rho_ref, double* sums, void* workspace, size_t workspace_bytes,
                            void* stream) {
  int rc = check_common(eos, dtype);
  if (rc) return rc;
  if ((rc = check_bcast(t_bcast, s_bcast))) return rc;
  if (vref_dtype != ML_F32 && vref_dtype != ML_F64) return fail(ML_ERR_DTYPE, "unknown vref dtype id %d", vref_dtype);
  ML_REQUIRE_PTR(T);
  ML_REQUIRE_PTR(S);
  ML_REQUIRE_PTR(v_ref);
  ML_REQUIRE_PTR(z_i);
  ML_REQUIRE_PTR(deptho);
  ML_REQUIRE_PTR(p_level);
  ML_REQUIRE_PTR(eta);
  ML_REQUIRE_PTR(sums);
  if (nt <= 0 || nz <= 0 || ncol <= 0 || nt > INT32_MAX || nz > INT32_MAX) return fail(ML_ERR_SHAPE, "bad extents nt=%lld nz=%lld ncol=%lld", (long long)nt, (long long)nz, (long long)ncol);
  if (int rcp = check_column_pressure(ncol)) return rcp;
  if (workspace == nullptr || workspace_bytes < ml_workspace_bytes(2, nz, ncol))
    return fail(ML_ERR_WORKSPACE, "workspace needs %zu bytes, got %zu", ml_workspace_bytes(2, nz, ncol), workspace_bytes);
  ML_REQUIRE_ALIGNED(workspace, 8);
  ML_REQUIRE_ALIGNED(T, elem_size(dtype));
  ML_REQUIRE_ALIGNED(S, elem_size(dtype));
  ML_REQUIRE_ALIGNED(v_ref, elem_size(vref_dtype));
  cudaStream_t st = (cudaStream_t)stream;
  const bool tma_ok = !direct_only() && tma::local_eligible(dtype, T, S, t_bcast, s_bcast, nullptr, v_ref,
                                                                 vref_dtype, nt, nz, ncol, eta, nullptr);
  // rho_ref is an output the caller may not want (8 bytes per reference point, 7 % of the traffic of a
  // 12-step call).  It can be left out when one fused chunk serves the whole call; longer series and the
  // direct family read it back for the later steps.
  if (rho_ref == nullptr && !(tma_ok && nt <= (dtype == ML_F32 ? 12 : 6)))
    return fail(ML_ERR_NULL, "rho_ref is NULL: it may only be omitted when one fused chunk serves the call "
                             "(aligned fields of at most 12 steps, 6 if stored as fp64)");
  if (tma_ok) {
    tls().last_path = ML_PATH_TMA;
    return tma::launch_selfref(eos, T, S, t_bcast, s_bcast, v_ref, vref_dtype, z_i, deptho, p_level, neg_inv_rhozero,
                               (int)nt, (int)nz, ncol, eta, rho_ref, sums, (double*)workspace, st);
  }
  // direct family: the reference-state pass, then the column integral against its rho_ref.
  // The reference T, S are the first step of whichever operand carries the time axis.
  rc = reference_state_impl(eos, dtype, T, S, v_ref, vref_dtype, p_level, nz, ncol, rho_ref, sums, workspace,
                            workspace_bytes, stream);
  if (rc) return rc;
  return ml_steric_local(eos, dtype, T, S, t_bcast, s_bcast, rho_ref, v_ref, vref_dtype, z_i, deptho, p_level,
                         neg_inv_rhozero, nt, nz, ncol, eta, nullptr, stream);
}

int ml_steric_local(int eos, int dtype, const void* T, const void* S, int t_bcast, int s_bcast, const double* rho_ref,
                    const void* v_ref, int vref_dtype, const double* z_i, const double* deptho, const double* p_level,
                    double neg_inv_rhozero, int64_t nt, int64_t nz, int64_t ncol, double* eta, double* delta_rho,
                    void* stream) {
  int rc = check_common(eos, dtype);
  if (rc) return rc;
  if ((rc = check_bcast(t_bcast, s_bcast))) return rc;
  if (vref_dtype != ML_F32 && vref_dtype != ML_F64) return fail(ML_ERR_DTYPE, "unknown vref dtype id %d", vref_dtype);
  ML_REQUIRE_PTR(T);
  ML_REQUIRE_PTR(S);
  ML_REQUIRE_PTR(rho_ref);
  ML_REQUIRE_PTR(v_ref);
  ML_REQUIRE_PTR(z_i);
  ML_REQUIRE_PTR(deptho);
  ML_REQUIRE_PTR(p_level);
  ML_REQUIRE_PTR(eta);
  if (nt < 0 || nz <= 0 || ncol < 0 || nt > INT32_MAX || nz > INT32_MAX) return fail(ML_ERR_SHAPE, "bad extents nt=%lld nz=%lld ncol=%lld", (long long)nt, (long long)nz, (long long)ncol);
  if (int rcp = check_column_pressure(ncol)) return rcp;
  ML_REQUIRE_ALIGNED(T, elem_size(dtype));
  ML_REQUIRE_ALIGNED(S, elem_size(dtype));
  ML_REQUIRE_ALIGNED(v_ref, elem_size(vref_dtype));
  if (nt == 0 || ncol == 0) return ML_OK;
  const i64 lvl = nz * ncol;
  const i64 ts = t_bcast ? 0 : lvl, ss = s_bcast ? 0 : lvl;
  cudaStream_t st = (cudaStream_t)stream;
  const int v_f32 = vref_dtype == ML_F32;

  if (direct_only() == false &&
      tma::local_eligible(dtype, T, S, t_bcast, s_bcast, rho_ref, v_ref, vref_dtype, nt, nz, ncol, eta, delta_rho)) {
    tls().last_path = ML_PATH_TMA;
    return tma::launch_local(eos, dtype, T, S, t_bcast, s_bcast, rho_ref, v_ref, vref_dtype, z_i, deptho, p_level,
                             neg_inv_rhozero, (int)nt, (int)nz, ncol, eta, delta_rho, st);
  }
  tls().last_path = ML_PATH_DIRECT;
  if (dtype == ML_F32) {
    if (eos == ML_EOS_WRIGHT) return launch_local_direct<float, 0>(T, S, ts, ss, rho_ref, v_ref, v_f32, z_i, deptho, p_level, neg_inv_rhozero, (int)nt, (int)nz, ncol, eta, delta_rho, st);
    return launch_local_direct<float, 1>(T, S, ts, ss, rho_ref, v_ref, v_f32, z_i, deptho, p_level, neg_inv_rhozero, (int)nt, (int)nz, ncol, eta, delta_rho, st);
  }
  if (eos == ML_EOS_WRIGHT) return launch_local_direct<double, 0>(T, S, ts, ss, rho_ref, v_ref, v_f32, z_i, deptho, p_level, neg_inv_rhozero, (int)nt, (int)nz, ncol, eta, delta_rho, st);
  return launch_local_direct<double, 1>(T, S, ts, ss, rho_ref, v_ref, v_f32, z_i, deptho, p_level, neg_inv_rhozero, (int)nt, (int)nz, ncol, eta, delta_rho, st);
}

int ml_steric_local_layers(int eos, int dtype, const void* T, const void* S, int t_bcast, int s_bcast,
                           const double* rho_ref, const void* v_ref, int vref_dtype, const double* z_i,
                           const double* deptho, const double* p_level, double neg_inv_rhozero, const double* edges,
                           int nlayers, int64_t nt, int64_t nz, int64_t ncol, double* eta, void* stream) {
  int rc = check_common(eos, dtype);
  if (rc) return rc;
  if ((rc = check_bcast(t_bcast, s_bcast))) return rc;
  if (vref_dtype != ML_F32 && vref_dtype != ML_F64) return fail(ML_ERR_DTYPE, "unknown vref dtype id %d", vref_dtype);
  ML_REQUIRE_PTR(T);
  ML_REQUIRE_PTR(S);
  ML_REQUIRE_PTR(rho_ref);
  ML_REQUIRE_PTR(v_ref);
  ML_REQUIRE_PTR(z_i);
  ML_REQUIRE_PTR(deptho);
  ML_REQUIRE_PTR(p_level);
  ML_REQUIRE_PTR(edges);
  ML_REQUIRE_PTR(eta);
  if ((rc = check_layers(edges, nlayers))) return rc;
  if (nt < 0 || nz <= 0 || ncol < 0 || nt > INT32_MAX || nz > INT32_MAX) return fail(ML_ERR_SHAPE, "bad extents nt=%lld nz=%lld ncol=%lld", (long long)nt, (long long)nz, (long long)ncol);
  if (int rcp = check_column_pressure(ncol)) return rcp;
  ML_REQUIRE_ALIGNED(T, elem_size(dtype));
  ML_REQUIRE_ALIGNED(S, elem_size(dtype));
  ML_REQUIRE_ALIGNED(v_ref, elem_size(vref_dtype));
  if (nt == 0 || ncol == 0) return ML_OK;
  const i64 lvl = nz * ncol;
  const i64 ts = t_bcast ? 0 : lvl, ss = s_bcast ? 0 : lvl;
  cudaStream_t st = (cudaStream_t)stream;
  const int v_f32 = vref_dtype == ML_F32;

  if (direct_only() == false &&
      tma::local_eligible(dtype, T, S, t_bcast, s_bcast, rho_ref, v_ref, vref_dtype, nt, nz, ncol, eta, nullptr)) {
    tls().last_path = ML_PATH_TMA;
    return tma::launch_local_layers(eos, T, S, t_bcast, s_bcast, rho_ref, v_ref, vref_dtype, z_i, deptho, p_level,
                                    neg_inv_rhozero, edges, nlayers, (int)nt, (int)nz, ncol, eta, st);
  }
  tls().last_path = ML_PATH_DIRECT;
  LayerEdges L;
  L.n = nlayers;
  for (int b = 0; b <= ML_MAX_LAYERS; ++b) L.e[b] = b <= nlayers ? edges[b] : 0.0;
  if (dtype == ML_F32) {
    if (eos == ML_EOS_WRIGHT) return launch_layers_direct<float, 0>(T, S, ts, ss, rho_ref, v_ref, v_f32, z_i, deptho, p_level, neg_inv_rhozero, (int)nt, (int)nz, ncol, eta, L, st);
    return launch_layers_direct<float, 1>(T, S, ts, ss, rho_ref, v_ref, v_f32, z_i, deptho, p_level, neg_inv_rhozero, (int)nt, (int)nz, ncol, eta, L, st);
  }
  if (eos == ML_EOS_WRIGHT) return launch_layers_direct<double, 0>(T, S, ts, ss, rho_ref, v_ref, v_f32, z_i, deptho, p_level, neg_inv_rhozero, (int)nt, (int)nz, ncol, eta, L, st);
  return launch_layers_direct<double, 1>(T, S, ts, ss, rho_ref, v_ref, v_f32, z_i, deptho, p_level, neg_inv_rhozero, (int)nt, (int)nz, ncol, eta, L, st);
}

int ml_steric_local_layers_variants(int eos, int dtype, const void* T, const void* S, const void* T_ref,
                                    const void* S_ref, const double* rho_ref, const void* v_ref, int vref_dtype,
                                    const double* z_i, const double* deptho, const double* p_level,
                                    double neg_inv_rhozero, const double* edges, int nlayers, int64_t nt, int64_t nz,
                                    int64_t ncol, double* eta_steric, double* eta_thermosteric,
                                    double* eta_halosteric, void* stream) {
  int rc = check_common(eos, dtype);
  if (rc) return rc;
  if (vref_dtype != ML_F32 && vref_dtype != ML_F64) return fail(ML_ERR_DTYPE, "unknown vref dtype id %d", vref_dtype);
  ML_REQUIRE_PTR(T);
  ML_REQUIRE_PTR(S);
  ML_REQUIRE_PTR(T_ref);
  ML_REQUIRE_PTR(S_ref);
  ML_REQUIRE_PTR(rho_ref);
  ML_REQUIRE_PTR(v_ref);
  ML_REQUIRE_PTR(z_i);
  ML_REQUIRE_PTR(deptho);
  ML_REQUIRE_PTR(p_level);
  ML_REQUIRE_PTR(edges);
  const int wanted = (eta_steric != nullptr) + (eta_thermosteric != nullptr) + (eta_halosteric != nullptr);
  if (wanted == 0) return fail(ML_ERR_NULL, "eta_steric, eta_thermosteric and eta_halosteric are all NULL");
  if ((rc = check_layers(edges, nlayers))) return rc;
  if (nt < 0 || nz <= 0 || ncol < 0 || nt > INT32_MAX || nz > INT32_MAX) return fail(ML_ERR_SHAPE, "bad extents nt=%lld nz=%lld ncol=%lld", (long long)nt, (long long)nz, (long long)ncol);
  if (int rcp = check_column_pressure(ncol)) return rcp;
  ML_REQUIRE_ALIGNED(T, elem_size(dtype));
  ML_REQUIRE_ALIGNED(S, elem_size(dtype));
  ML_REQUIRE_ALIGNED(T_ref, elem_size(dtype));
  ML_REQUIRE_ALIGNED(S_ref, elem_size(dtype));
  ML_REQUIRE_ALIGNED(v_ref, elem_size(vref_dtype));
  if (nt == 0 || ncol == 0) return ML_OK;
  // One pass over T and S for all the layered heights asked for (csrc/ml_tma3.cu, kLocalLayers3), on the fields the
  // one-pass kernel of ml_steric_local_variants takes and when more than one height is wanted.
  if (tls().force_direct == 0 && !direct_only() && wanted >= 2 &&
      tma::variants_eligible(dtype, T, S, T_ref, S_ref, vref_dtype, nt, nz, ncol)) {
    tls().last_path = ML_PATH_TMA;
    return tma::launch_local_layers_variants(eos, T, S, T_ref, S_ref, rho_ref, v_ref, z_i, deptho, p_level,
                                             neg_inv_rhozero, edges, nlayers, (int)nt, (int)nz, ncol, eta_steric,
                                             eta_thermosteric, eta_halosteric, (cudaStream_t)stream);
  }
  // one ml_steric_local_layers per wanted height; steric.py:115-121: thermosteric holds S at the reference slab,
  // halosteric holds T
  struct Variant {
    double* eta;
    const void *T, *S;
    int t_bcast, s_bcast;
  };
  const Variant todo[3] = {{eta_steric, T, S, 0, 0}, {eta_thermosteric, T, S_ref, 0, 1}, {eta_halosteric, T_ref, S, 1, 0}};
  for (const Variant& v : todo) {
    if (v.eta == nullptr) continue;
    if ((rc = ml_steric_local_layers(eos, dtype, v.T, v.S, v.t_bcast, v.s_bcast, rho_ref, v_ref, vref_dtype, z_i, deptho,
                                     p_level, neg_inv_rhozero, edges, nlayers, nt, nz, ncol, v.eta, stream)))
      return rc;
  }
  return ML_OK;
}

static int delta_rho_impl(int eos, int dtype, const void* T, const void* S, int t_bcast, int s_bcast,
                          const double* rho_ref, const void* v_ref, int vref_dtype, const double* p_level,
                          const double* weights, int64_t nt, int64_t nz, int64_t ncol, double* delta_rho, void* stream) {
  int rc = check_common(eos, dtype);
  if (rc) return rc;
  if ((rc = check_bcast(t_bcast, s_bcast))) return rc;
  if (vref_dtype != ML_F32 && vref_dtype != ML_F64) return fail(ML_ERR_DTYPE, "unknown vref dtype id %d", vref_dtype);
  ML_REQUIRE_PTR(T);
  ML_REQUIRE_PTR(S);
  ML_REQUIRE_PTR(rho_ref);
  ML_REQUIRE_PTR(v_ref);
  ML_REQUIRE_PTR(p_level);
  ML_REQUIRE_PTR(delta_rho);
  if (nt < 0 || nz <= 0 || ncol < 0 || nt > INT32_MAX || nz > INT32_MAX) return fail(ML_ERR_SHAPE, "bad extents nt=%lld nz=%lld ncol=%lld", (long long)nt, (long long)nz, (long long)ncol);
  if (int rcp = check_column_pressure(ncol)) return rcp;
  if (weights && nt % 12 != 0) return fail(ML_ERR_SHAPE, "annual averaging needs whole years of monthly data, got nt=%lld", (long long)nt);
  ML_REQUIRE_ALIGNED(T, elem_size(dtype));
  ML_REQUIRE_ALIGNED(S, elem_size(dtype));
  ML_REQUIRE_ALIGNED(v_ref, elem_size(vref_dtype));
  ML_REQUIRE_ALIGNED(delta_rho, 8);
  if (nt == 0 || ncol == 0) return ML_OK;
  const i64 lvl = nz * ncol;
  const i64 ts = t_bcast ? 0 : lvl, ss = s_bcast ? 0 : lvl;
  cudaStream_t st = (cudaStream_t)stream;
  const int v_f32 = vref_dtype == ML_F32;
  const uintptr_t bits = reinterpret_cast<uintptr_t>(T) | reinterpret_cast<uintptr_t>(S) |
                         reinterpret_cast<uintptr_t>(rho_ref) | reinterpret_cast<uintptr_t>(delta_rho);
  // fp32 fields, monthly output: the ring-staged streaming kernel (ml_stream.cu)
  if (weights == nullptr && dtype == ML_F32 && !direct_only() && stream::eligible(T, S, rho_ref, delta_rho, ncol) &&
      (reinterpret_cast<uintptr_t>(v_ref) & 15u) == 0 && nt <= INT32_MAX)
    return stream::launch_delta_rho(eos, (const float*)T, (const float*)S, ts, ss, rho_ref, v_ref, v_f32, p_level, (int)nt, nz,
                                    ncol, delta_rho, st);
  const bool vec = ncol % 4 == 0 && (bits & 15u) == 0 && tls().p_col == nullptr;
  const i64 gx = cdiv(vec ? ncol / 4 : ncol, kBlock);
  i64 gy = cdiv(148 * 16, gx);
  gy = gy < 1 ? 1 : (gy > nz ? nz : gy);
  dim3 grid((unsigned)gx, (unsigned)gy);
#define ML_LAUNCH_DRHO(TIN, E, V)                                                                                      \
  do {                                                                                                                 \
    if (weights)                                                                                                       \
      k_delta_rho<TIN, E, V, true><<<grid, kBlock, 0, st>>>((const TIN*)T, (const TIN*)S, ts, ss, rho_ref, v_ref, v_f32, \
                                                            p_level, tls().p_col, weights, (int)nt, (int)nz, ncol, delta_rho);     \
    else                                                                                                               \
      k_delta_rho<TIN, E, V, false><<<grid, kBlock, 0, st>>>((const TIN*)T, (const TIN*)S, ts, ss, rho_ref, v_ref,     \
                                                             v_f32, p_level, tls().p_col, nullptr, (int)nt, (int)nz, ncol, delta_rho); \
  } while (0)
  if (dtype == ML_F32) {
    if (eos == ML_EOS_WRIGHT) { if (vec) ML_LAUNCH_DRHO(float, 0, 4); else ML_LAUNCH_DRHO(float, 0, 1); }
    else { if (vec) ML_LAUNCH_DRHO(float, 1, 4); else ML_LAUNCH_DRHO(float, 1, 1); }
  } else {
    if (eos == ML_EOS_WRIGHT) { if (vec) ML_LAUNCH_DRHO(double, 0, 4); else ML_LAUNCH_DRHO(double, 0, 1); }
    else { if (vec) ML_LAUNCH_DRHO(double, 1, 4); else ML_LAUNCH_DRHO(double, 1, 1); }
  }
#undef ML_LAUNCH_DRHO
  return launched("k_delta_rho");
}

int ml_delta_rho(int eos, int dtype, const void* T, const void* S, int t_bcast, int s_bcast, const double* rho_ref,
                 const void* v_ref, int vref_dtype, const double* p_level, int64_t nt, int64_t nz, int64_t ncol,
                 double* delta_rho, void* stream) {
  return delta_rho_impl(eos, dtype, T, S, t_bcast, s_bcast, rho_ref, v_ref, vref_dtype, p_level, nullptr, nt, nz, ncol,
                        delta_rho, stream);
}

int ml_delta_rho_annual(int eos, int dtype, const void* T, const void* S, int t_bcast, int s_bcast,
                        const double* rho_ref, const void* v_ref, int vref_dtype, const double* p_level,
                        const double* weights, int64_t nt, int64_t nz, int64_t ncol, double* delta_rho_annual,
                        void* stream) {
  ML_REQUIRE_PTR(weights);
  return delta_rho_impl(eos, dtype, T, S, t_bcast, s_bcast, rho_ref, v_ref, vref_dtype, p_level, weights, nt, nz, ncol,
                        delta_rho_annual, stream);
}

int ml_steric_local_variants(int eos, int dtype, const void* T, const void* S, const void* T_ref, const void* S_ref,
                             const double* rho_ref, const void* v_ref, int vref_dtype, const double* z_i,
                             const double* deptho, const double* p_level, double neg_inv_rhozero, int64_t nt,
                             int64_t nz, int64_t ncol, double* eta_steric, double* eta_thermosteric,
                             double* eta_halosteric, double* rho_ref_out, double* sums, void* workspace,
                             size_t workspace_bytes, void* stream) {
  int rc = check_common(eos, dtype);
  if (rc) return rc;
  if (vref_dtype != ML_F32 && vref_dtype != ML_F64) return fail(ML_ERR_DTYPE, "unknown vref dtype id %d", vref_dtype);
  ML_REQUIRE_PTR(T);
  ML_REQUIRE_PTR(S);
  ML_REQUIRE_PTR(T_ref);
  ML_REQUIRE_PTR(S_ref);
  ML_REQUIRE_PTR(v_ref);
  ML_REQUIRE_PTR(z_i);
  ML_REQUIRE_PTR(deptho);
  ML_REQUIRE_PTR(p_level);
  if (rho_ref == nullptr) {  // the reference density is evaluated here (and handed back if rho_ref_out is given)
    ML_REQUIRE_PTR(sums);
    if (workspace == nullptr || workspace_bytes < ml_workspace_bytes(2, nz, ncol))
      return fail(ML_ERR_WORKSPACE, "workspace needs %zu bytes, got %zu", ml_workspace_bytes(2, nz, ncol), workspace_bytes);
    ML_REQUIRE_ALIGNED(workspace, 8);
  }
  if (nt <= 0 || nz <= 0 || ncol <= 0 || nt > INT32_MAX || nz > INT32_MAX) return fail(ML_ERR_SHAPE, "bad extents nt=%lld nz=%lld ncol=%lld", (long long)nt, (long long)nz, (long long)ncol);
  if (int rcp = check_column_pressure(ncol)) return rcp;
  ML_REQUIRE_ALIGNED(T, elem_size(dtype));
  ML_REQUIRE_ALIGNED(S, elem_size(dtype));
  ML_REQUIRE_ALIGNED(T_ref, elem_size(dtype));
  ML_REQUIRE_ALIGNED(S_ref, elem_size(dtype));
  ML_REQUIRE_ALIGNED(v_ref, elem_size(vref_dtype));
  // steric.py:115-121: thermosteric holds S at the reference slab, halosteric holds T.
  const bool self_reference = rho_ref == nullptr && T_ref == T && S_ref == S;  // the reference state is step 0
  // One pass over T and S for all the heights asked for (csrc/ml_tma3.cu): a point's three densities come from the
  // same two shared-memory words.  Taken when the fields suit the TMA family and more than one height is wanted.
  const int wanted = (eta_steric != nullptr) + (eta_thermosteric != nullptr) + (eta_halosteric != nullptr);
  const bool fused_ok = tls().force_direct == 0 && !direct_only() && wanted >= 2 &&
                        tma::variants_eligible(dtype, T, S, T_ref, S_ref, vref_dtype, nt, nz, ncol);
  if (fused_ok && (self_reference || rho_ref != nullptr)) {
    tls().last_path = ML_PATH_TMA;
    return tma::launch_variants(eos, T, S, T_ref, S_ref, rho_ref, v_ref, z_i, deptho, p_level, neg_inv_rhozero, (int)nt,
                                (int)nz, ncol, eta_steric, eta_thermosteric, eta_halosteric, rho_ref_out, sums,
                                static_cast<double*>(workspace), (cudaStream_t)stream);
  }
  if (rho_ref == nullptr) ML_REQUIRE_PTR(rho_ref_out);  // the launches below read the reference density from memory
  bool steric_done = false;
  if (rho_ref == nullptr) {
    if (self_reference && eta_steric) {  // reference state and steric height in one fused pass
      rc = ml_steric_local_selfref(eos, dtype, T, S, 0, 0, v_ref, vref_dtype, z_i, deptho, p_level, neg_inv_rhozero, nt,
                                   nz, ncol, eta_steric, rho_ref_out, sums, workspace, workspace_bytes, stream);
      steric_done = true;
    } else {
      rc = reference_state_impl(eos, dtype, T_ref, S_ref, v_ref, vref_dtype, p_level, nz, ncol, rho_ref_out, sums,
                                workspace, workspace_bytes, stream);
    }
    if (rc) return rc;
    rho_ref = rho_ref_out;
    if (fused_ok && !steric_done) {
      tls().last_path = ML_PATH_TMA;
      return tma::launch_variants(eos, T, S, T_ref, S_ref, rho_ref, v_ref, z_i, deptho, p_level, neg_inv_rhozero,
                                  (int)nt, (int)nz, ncol, eta_steric, eta_thermosteric, eta_halosteric, nullptr, nullptr,
                                  nullptr, (cudaStream_t)stream);
    }
  }
  // one single-variant launch per remaining height; with a self-reference the TMA family is told that step 0 is
  // the reference state itself, so that height is exactly zero there as in the reference (rho - rho_ref == 0)
  struct Variant {
    double* eta;
    const void *T, *S;
    int t_bcast, s_bcast;
  };
  const Variant todo[3] = {{steric_done ? nullptr : eta_steric, T, S, 0, 0},
                           {eta_thermosteric, T, S_ref, 0, 1},
                           {eta_halosteric, T_ref, S, 1, 0}};
  for (const Variant& v : todo) {
    if (v.eta == nullptr) continue;
    if (direct_only() == false && tma::local_eligible(dtype, v.T, v.S, v.t_bcast, v.s_bcast, rho_ref, v_ref, vref_dtype, nt,
                                                   nz, ncol, v.eta, nullptr)) {
      tls().last_path = ML_PATH_TMA;
      rc = tma::launch_local(eos, dtype, v.T, v.S, v.t_bcast, v.s_bcast, rho_ref, v_ref, vref_dtype, z_i, deptho,
                             p_level, neg_inv_rhozero, (int)nt, (int)nz, ncol, v.eta, nullptr, (cudaStream_t)stream,
                             self_reference ? 1 : 0);
    } else {
      rc = ml_steric_local(eos, dtype, v.T, v.S, v.t_bcast, v.s_bcast, rho_ref, v_ref, vref_dtype, z_i, deptho, p_level,
                           neg_inv_rhozero, nt, nz, ncol, v.eta, nullptr, stream);
    }
    if (rc) return rc;
  }
  return ML_OK;
}

int ml_steric_global(int eos, int dtype, const void* T, const void* S, int t_bcast, int s_bcast, const void* v_ref,
                     int vref_dtype, const double* p_level, int64_t nt, int64_t nz, int64_t ncol, double* masso,
                     void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_common(eos, dtype);
  if (rc) return rc;
  if ((rc = check_bcast(t_bcast, s_bcast))) return rc;
  if (vref_dtype != ML_F32 && vref_dtype != ML_F64) return fail(ML_ERR_DTYPE, "unknown vref dtype id %d", vref_dtype);
  ML_REQUIRE_PTR(T);
  ML_REQUIRE_PTR(S);
  ML_REQUIRE_PTR(v_ref);
  ML_REQUIRE_PTR(p_level);
  ML_REQUIRE_PTR(masso);
  if (nt < 0 || nz <= 0 || ncol <= 0 || nt > INT32_MAX || nz > INT32_MAX) return fail(ML_ERR_SHAPE, "bad extents nt=%lld nz=%lld ncol=%lld", (long long)nt, (long long)nz, (long long)ncol);
  if (int rcp = check_column_pressure(ncol)) return rcp;
  if (nt == 0) return ML_OK;
  if (workspace == nullptr || workspace_bytes < ml_workspace_bytes(nt, nz, ncol))
    return fail(ML_ERR_WORKSPACE, "workspace needs %zu bytes, got %zu", ml_workspace_bytes(nt, nz, ncol), workspace_bytes);
  ML_REQUIRE_ALIGNED(workspace, 8);
  ML_REQUIRE_ALIGNED(T, elem_size(dtype));
  ML_REQUIRE_ALIGNED(S, elem_size(dtype));
  ML_REQUIRE_ALIGNED(v_ref, elem_size(vref_dtype));
  const i64 lvl = nz * ncol;
  const i64 ts = t_bcast ? 0 : lvl, ss = s_bcast ? 0 : lvl;
  cudaStream_t st = (cudaStream_t)stream;
  const int v_f32 = vref_dtype == ML_F32;
  double* partials = (double*)workspace;

  if (direct_only() == false && tma::global_eligible(dtype, T, S, t_bcast, s_bcast, v_ref, vref_dtype, nt, nz, ncol)) {
    tls().last_path = ML_PATH_TMA;
    return tma::launch_global(eos, dtype, T, S, t_bcast, s_bcast, v_ref, vref_dtype, p_level, (int)nt, (int)nz, ncol,
                              masso, partials, st);
  }
  tls().last_path = ML_PATH_DIRECT;
  if (dtype == ML_F32) {
    if (eos == ML_EOS_WRIGHT) return launch_global_direct<float, 0>(T, S, ts, ss, v_ref, v_f32, p_level, (int)nt, (int)nz, ncol, masso, partials, st);
    return launch_global_direct<float, 1>(T, S, ts, ss, v_ref, v_f32, p_level, (int)nt, (int)nz, ncol, masso, partials, st);
  }
  if (eos == ML_EOS_WRIGHT) return launch_global_direct<double, 0>(T, S, ts, ss, v_ref, v_f32, p_level, (int)nt, (int)nz, ncol, masso, partials, st);
  return launch_global_direct<double, 1>(T, S, ts, ss, v_ref, v_f32, p_level, (int)nt, (int)nz, ncol, masso, partials, st);
}

int ml_steric_global_variants(int eos, int dtype, const void* T, const void* S, const void* T_ref, const void* S_ref,
                              const void* v_ref, int vref_dtype, const double* p_level, int64_t nt, int64_t nz,
                              int64_t ncol, double* masso_steric, double* masso_thermosteric,
                              double* masso_halosteric, double* sums, void* workspace, size_t workspace_bytes,
                              void* stream) {
  int rc = check_common(eos, dtype);
  if (rc) return rc;
  if (vref_dtype != ML_F32 && vref_dtype != ML_F64) return fail(ML_ERR_DTYPE, "unknown vref dtype id %d", vref_dtype);
  ML_REQUIRE_PTR(T);
  ML_REQUIRE_PTR(S);
  ML_REQUIRE_PTR(T_ref);
  ML_REQUIRE_PTR(S_ref);
  ML_REQUIRE_PTR(v_ref);
  ML_REQUIRE_PTR(p_level);
  const int wanted = (masso_steric != nullptr) + (masso_thermosteric != nullptr) + (masso_halosteric != nullptr);
  if (wanted == 0) return fail(ML_ERR_NULL, "no output: at least one of the three masses is required");
  // steric.py:105-107: without a supplied reference the reference state is step 0 of the fields (the same pointers)
  const bool self_reference = T_ref == T && S_ref == S;
  if (self_reference && sums == nullptr) return fail(ML_ERR_NULL, "sums is NULL: a self-reference call returns {volo, masso}");
  if (!self_reference && sums != nullptr) return fail(ML_ERR_MODE, "sums is only produced when T_ref, S_ref are T, S");
  if (nt <= 0 || nz <= 0 || ncol <= 0 || nt > INT32_MAX / 3 || nz > INT32_MAX)
    return fail(ML_ERR_SHAPE, "bad extents nt=%lld nz=%lld ncol=%lld", (long long)nt, (long long)nz, (long long)ncol);
  if (int rcp = check_column_pressure(ncol)) return rcp;
  if (workspace == nullptr || workspace_bytes < ml_workspace_bytes(3 * nt, nz, ncol))
    return fail(ML_ERR_WORKSPACE, "workspace needs %zu bytes, got %zu", ml_workspace_bytes(3 * nt, nz, ncol), workspace_bytes);
  ML_REQUIRE_ALIGNED(workspace, 8);
  ML_REQUIRE_ALIGNED(T, elem_size(dtype));
  ML_REQUIRE_ALIGNED(S, elem_size(dtype));
  ML_REQUIRE_ALIGNED(T_ref, elem_size(dtype));
  ML_REQUIRE_ALIGNED(S_ref, elem_size(dtype));
  ML_REQUIRE_ALIGNED(v_ref, elem_size(vref_dtype));
  cudaStream_t st = (cudaStream_t)stream;
  // One pass over T and S for all the masses asked for (csrc/ml_tma3.cu), bit-identical to the launches below.
  if (tls().force_direct == 0 && !direct_only() && wanted >= 2 &&
      tma::variants_eligible(dtype, T, S, T_ref, S_ref, vref_dtype, nt, nz, ncol) &&
      tma::global_variants_partials(nt, ncol) <= workspace_bytes) {
    tls().last_path = ML_PATH_TMA;
    return tma::launch_global_variants(eos, T, S, T_ref, S_ref, v_ref, p_level, (int)nt, (int)nz, ncol, masso_steric,
                                       masso_thermosteric, masso_halosteric, sums, static_cast<double*>(workspace), st);
  }
  if (self_reference) {
    // the scalars of the reference state (reference.py:71-80); the density field itself is not an output here
    double* rho = nullptr;
    cudaError_t e = cudaMallocAsync(reinterpret_cast<void**>(&rho), (size_t)nz * (size_t)ncol * sizeof(double), st);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMallocAsync(reference density)");
    rc = reference_state_impl(eos, dtype, T, S, v_ref, vref_dtype, p_level, nz, ncol, rho, sums, workspace,
                              workspace_bytes, stream);
    e = cudaFreeAsync(rho, st);
    if (rc) return rc;
    if (e != cudaSuccess) return cuda_fail(e, "cudaFreeAsync(reference density)");
  }
  // one single-height launch per wanted mass: thermosteric holds S at the reference slab, halosteric holds T
  struct Variant {
    double* masso;
    const void *T, *S;
    int t_bcast, s_bcast;
  };
  const Variant todo[3] = {{masso_steric, T, S, 0, 0}, {masso_thermosteric, T, S_ref, 0, 1}, {masso_halosteric, T_ref, S, 1, 0}};
  for (const Variant& v : todo) {
    if (v.masso == nullptr) continue;
    if ((rc = ml_steric_global(eos, dtype, v.T, v.S, v.t_bcast, v.s_bcast, v_ref, vref_dtype, p_level, nt, nz, ncol,
                               v.masso, workspace, workspace_bytes, stream)))
      return rc;
  }
  return ML_OK;
}

}  // extern "C"

int ml_calc_masso(int dtype, const void* rho, int w_dtype, const void* volcello, int64_t nrows, int64_t n, double* out,
                  void* workspace, size_t workspace_bytes, void* stream) {
  if (dtype != ML_F32 && dtype != ML_F64) return fail(ML_ERR_DTYPE, "unknown dtype id %d", dtype);
  if (volcello != nullptr && w_dtype != ML_F32 && w_dtype != ML_F64) return fail(ML_ERR_DTYPE, "unknown weight dtype id %d", w_dtype);
  ML_REQUIRE_PTR(rho);
  ML_REQUIRE_PTR(out);
  if (nrows < 0 || n < 0 || nrows > 65535) return fail(ML_ERR_SHAPE, "bad extents nrows=%lld n=%lld", (long long)nrows, (long long)n);
  if (nrows == 0) return ML_OK;
  ML_REQUIRE_ALIGNED(rho, elem_size(dtype));
  const i64 want = cdiv(n > 0 ? n : 1, (i64)kBlock * 8);
  const i64 nblk = want < 1 ? 1 : (want > 148 * 8 ? 148 * 8 : want);  // ~8 blocks per SM, each thread a strided serial sum
  if (workspace == nullptr || workspace_bytes < (size_t)(nrows * nblk) * sizeof(double))
    return fail(ML_ERR_WORKSPACE, "workspace needs %zu bytes, got %zu", (size_t)(nrows * nblk) * sizeof(double), workspace_bytes);
  ML_REQUIRE_ALIGNED(workspace, 8);
  cudaStream_t st = (cudaStream_t)stream;
  double* partials = (double*)workspace;
  dim3 grid((unsigned)nblk, (unsigned)nrows);
#define ML_WNS(TA, TW) k_weighted_nansum<TA, TW><<<grid, kBlock, 0, st>>>((const TA*)rho, (const TW*)volcello, n, partials)
  if (dtype == ML_F32) {
    if (volcello == nullptr || w_dtype == ML_F32) ML_WNS(float, float); else ML_WNS(float, double);
  } else {
    if (volcello == nullptr || w_dtype == ML_F64) ML_WNS(double, double); else ML_WNS(double, float);
  }
#undef ML_WNS
  int rc = launched("k_weighted_nansum");
  if (rc) return rc;
  k_reduce_rows<<<(unsigned)nrows, kBlock, 0, st>>>(partials, nblk, out);
  return launched("k_reduce_rows");
}
