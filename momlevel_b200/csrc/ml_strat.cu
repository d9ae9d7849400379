// ml_strat.cu -- stratification diagnostics that share the vertical sweep of the steric path
// (SURVEY.md section 8f, rank 4): buoyancy frequency, its Chelton adjustment, the stability
// (Turner) angle and the first-mode gravity-wave speed.
//
//   derived.calc_n2              src/momlevel/derived.py:391-411  (cell centres; the `interfaces`
//                                branch needs xgcm and stays out of scope)
//   derived.adjust_negative_n2   src/momlevel/derived.py:30-71
//   derived.calc_stability_angle src/momlevel/derived.py:714-766
//   derived.calc_wave_speed      src/momlevel/derived.py:798-828
//
// One thread owns one water column of one outer (time) slab and walks it top to bottom with a
// three-level window in registers (fed through a cp.async ring in shared memory, see k_strat), so
// T and S cross HBM once (8 B per point in, 8 B out) and the
// vertical derivative -- numpy.gradient(..., edge_order=2) on the uneven z grid, which is what
// DataArray.differentiate evaluates -- never materialises dT/dz, dS/dz, alpha or beta.  Threads
// are adjacent along x, so every load and store of a warp is one contiguous row segment.
#include "ml_common.cuh"
#include "ml_host.cuh"

namespace ml {
namespace {

constexpr int kBlock = 128;
constexpr int kMaxLevels = 512;  // gradient coefficients of every level live in shared memory (<= 48 KB with the ring)

// numpy.gradient's second-order coefficients for an uneven grid (numpy/lib/function_base.py,
// `gradient`: interior a,b,c from dx1 = x[i]-x[i-1], dx2 = x[i+1]-x[i]; one-sided three-point
// formulas at both ends for edge_order=2).  out[i] = a f[i-1] + b f[i] + c f[i+1], with the
// window shifted inwards at the ends.  Explicitly rounded like numpy evaluates them.
__device__ void gradient_coefficients(const double* __restrict__ z, int nz, double* __restrict__ coef /*[nz][3]*/) {
  for (int i = threadIdx.x; i < nz; i += blockDim.x) {
    double a, b, c;
    if (i == 0) {
      const double dx1 = __dsub_rn(z[1], z[0]), dx2 = __dsub_rn(z[2], z[1]);
      const double s = __dadd_rn(dx1, dx2);
      a = -__ddiv_rn(__dadd_rn(__dmul_rn(2.0, dx1), dx2), __dmul_rn(dx1, s));
      b = __ddiv_rn(s, __dmul_rn(dx1, dx2));
      c = -__ddiv_rn(dx1, __dmul_rn(dx2, s));
    } else if (i == nz - 1) {
      const double dx1 = __dsub_rn(z[nz - 2], z[nz - 3]), dx2 = __dsub_rn(z[nz - 1], z[nz - 2]);
      const double s = __dadd_rn(dx1, dx2);
      a = __ddiv_rn(dx2, __dmul_rn(dx1, s));
      b = -__ddiv_rn(__dadd_rn(dx2, dx1), __dmul_rn(dx1, dx2));
      c = __ddiv_rn(__dadd_rn(__dmul_rn(2.0, dx2), dx1), __dmul_rn(dx2, s));
    } else {
      const double dx1 = __dsub_rn(z[i], z[i - 1]), dx2 = __dsub_rn(z[i + 1], z[i]);
      const double s = __dadd_rn(dx1, dx2);
      a = -__ddiv_rn(dx2, __dmul_rn(dx1, s));
      b = __ddiv_rn(__dsub_rn(dx2, dx1), __dmul_rn(dx1, dx2));
      c = __ddiv_rn(dx1, __dmul_rn(dx2, s));
    }
    coef[3 * i + 0] = a;
    coef[3 * i + 1] = b;
    coef[3 * i + 2] = c;
  }
}

// alpha = -(drho/dT)/rho and beta = (drho/dS)/rho (wright.py:122-165) from ONE division:
// rho = pp/den and drho/dX = N_X/den^2 give alpha = -N_T/(den pp), beta = N_S/(den pp).
// Coefficients are DFMA operands straight from the constant bank (as literals each would be
// rebuilt from two 32-bit moves in front of its instruction, cf. ml_common.cuh).
struct WrightD {
  double b2x2, b3x3, c2x2, c3x3;  // coefficients of the T-derivatives of p0 and lambda (wright.py:75-78)
};
__constant__ WrightD kWrightD = {2.0 * wr::b2, 3.0 * wr::b3, 2.0 * wr::c2, 3.0 * wr::c3};

template <int EOS>
__device__ __forceinline__ void alpha_beta(double T, double S, double p, double& alpha, double& beta) {
  if (EOS == 0) {
    const WrightC K = kWrightC;  // warp-uniform copies: the compiler keeps them in uniform registers
    const WrightD D = kWrightD;
    const double al0 = fma(K.a2, S, fma(K.a1, T, K.a0));
    const double pp = fma(T, fma(K.b5, S, fma(T, fma(K.b3, T, K.b2), K.b1)), fma(K.b4, S, K.b0 + p));
    const double lam = fma(T, fma(K.c5, S, fma(T, fma(K.c3, T, K.c2), K.c1)), fma(K.c4, S, K.c0));
    const double den = fma(al0, pp, lam);
    const double dp0_t = fma(K.b5, S, fma(T, fma(D.b3x3, T, D.b2x2), K.b1));
    const double dlam_t = fma(K.c5, S, fma(T, fma(D.c3x3, T, D.c2x2), K.c1));
    const double n_t = fma(lam, dp0_t, -(pp * fma(pp, K.a1, dlam_t)));
    const double n_s = fma(lam, fma(K.b5, T, K.b4), -(pp * fma(pp, K.a2, fma(K.c5, T, K.c4))));
    const double r = div_checked(1.0, den * pp);
    alpha = -(n_t * r);
    beta = n_s * r;
  } else {
    const double r = 1.0 / linear_rho(T, S);  // linear.py:113-162
    alpha = -(lin::drho_dt * r);
    beta = lin::drho_ds * r;
  }
}

enum StratOut { kN2 = 0, kN2Adjusted = 1, kTurnerAngle = 2 };

// adjust_negative_n2 for one value (derived.py:56-69).  `fill` = this cell belongs to index 0 of
// the array's FIRST axis, which the reference fills with 1e-8 (time step 0 of a 4-D field, the
// surface level of a 3-D one); `carry` is the last positive value met further up the column.
// The kernels take the fill as `fill_slabs`, relative to the slabs of their own launch: < 0 fills
// the surface level of every slab, n >= 0 every level of the launch's slabs [0, n).
__device__ __forceinline__ double adjust_step(double n2, bool fill, double& carry) {
  const bool missing = isnan(n2);
  double adj = (missing || n2 <= 0.0) ? nan("") : n2;
  if (fill && isnan(adj)) adj = 1.0e-8;
  if (isnan(adj)) adj = carry;  // ffill along z
  else carry = adj;
  return missing ? nan("") : adj;
}

// Each thread streams its own column through a private slot of a shared-memory ring with
// cp.async: kRing - 3 levels of T and S are in flight per thread at no register cost (the
// three-level window itself lives in registers), and because a thread only ever reads what it
// copied itself, cp.async.wait_group is the only synchronisation.  With plain loads the sweep had
// two loads in flight per thread and ran latency-bound at a third of the HBM bandwidth.
constexpr int kRing = 16;

template <typename TIn>
__device__ __forceinline__ void cp_async(TIn* smem_dst, const TIn* gsrc) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  if (sizeof(TIn) == 4)
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(gsrc) : "memory");
  else
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

template <typename TIn, int EOS, int OUT>
__global__ void __launch_bounds__(kBlock) k_strat(const TIn* __restrict__ T, const TIn* __restrict__ S,
                                                  const double* __restrict__ z_l, const double* __restrict__ p_level,
                                                  double gravity, double patm, int fill_slabs, int nz, i64 ncol,
                                                  double* __restrict__ out) {
  extern __shared__ double s_coef[];  // [nz][3] gradient coefficients, [nz] pressure, then the two rings
  double* s_p = s_coef + 3 * nz;
  TIn* ringT = reinterpret_cast<TIn*>(s_p + nz) + threadIdx.x;  // [kRing][kBlock], this thread's slot
  TIn* ringS = ringT + kRing * kBlock;
  gradient_coefficients(z_l, nz, s_coef);
  for (int i = threadIdx.x; i < nz; i += blockDim.x)
    s_p[i] = p_level ? __ldg(p_level + i) : fma(__ldg(z_l + i), 1.0e4, patm);  // derived.py:396
  __syncthreads();
  const i64 c = (i64)blockIdx.x * kBlock + threadIdx.x;
  if (c >= ncol) return;
  const i64 slab = (i64)blockIdx.y * nz * ncol + c;
  const TIn* gT = T + slab;  // next level to fetch
  const TIn* gS = S + slab;
  double* oc = out + slab;
  int fetched = 0;
  auto fetch = [&]() {  // one commit group per level, empty past the bottom
    if (fetched < nz) {
      cp_async(ringT + (fetched % kRing) * kBlock, gT);
      cp_async(ringS + (fetched % kRing) * kBlock, gS);
      gT += ncol;
      gS += ncol;
    }
    ++fetched;
    cp_async_commit();
  };
  for (int l = 0; l < kRing - 1; ++l) fetch();
  const bool fill_slab = (int)blockIdx.y < fill_slabs;  // this slab belongs to adjusted[0]
  double carry = nan("");
  // one output cell: the EOS derivatives at (Tc, Sc, p_z) combined with the vertical gradients
  auto emit = [&](int z, double Tc, double Sc, double dtdz, double dsdz) {
    double alpha, beta;
    alpha_beta<EOS>(Tc, Sc, s_p[z], alpha, beta);
    double r;
    if (OUT == kTurnerAngle) {
      const double ratio = (beta * dsdz) / (alpha * dtdz);  // derived.py:753
      r = atan((1.0 + ratio) / (1.0 - ratio)) * 57.29577951308232;  // np.degrees: x * (180 / pi)
    } else {
      r = gravity * (alpha * dtdz - beta * dsdz);  // derived.py:401
      if (OUT == kN2Adjusted) r = adjust_step(r, fill_slab || (fill_slabs < 0 && z == 0), carry);
    }
    asm volatile("st.global.cs.f64 [%0], %1;" ::"l"(oc + (i64)z * ncol), "d"(r) : "memory");  // streamed, never re-read
  };
  // window (a, b, c) = levels (zc-1, zc, zc+1) in registers; nz >= 3 is checked by the host.
  // numpy.gradient's one-sided formulas at both ends use the same three levels as their neighbours,
  // so level 0 is emitted with level 1 and level nz-1 with level nz-2.
  cp_async_wait<kRing - 3>();  // groups 0 and 1 have landed
  double ta = 0.0, tb = (double)ringT[0], tc = (double)ringT[kBlock];
  double sa = 0.0, sb = (double)ringS[0], sc = (double)ringS[kBlock];
  for (int zc = 1; zc < nz - 1; ++zc) {
    fetch();                      // level zc + kRing - 2; its slot held level zc - 2, long consumed
    cp_async_wait<kRing - 3>();  // everything up to level zc + 1 has landed
    ta = tb; tb = tc; tc = (double)ringT[((zc + 1) % kRing) * kBlock];
    sa = sb; sb = sc; sc = (double)ringS[((zc + 1) % kRing) * kBlock];
    if (zc == 1) {  // forward three-point formula for the surface level
      const double a = s_coef[0], b = s_coef[1], cc = s_coef[2];
      emit(0, ta, sa, fma(cc, tc, fma(b, tb, a * ta)), fma(cc, sc, fma(b, sb, a * sa)));
    }
    {
      const double a = s_coef[3 * zc], b = s_coef[3 * zc + 1], cc = s_coef[3 * zc + 2];
      emit(zc, tb, sb, fma(cc, tc, fma(b, tb, a * ta)), fma(cc, sc, fma(b, sb, a * sa)));
    }
    if (zc == nz - 2) {  // backward three-point formula for the bottom level
      const double a = s_coef[3 * zc + 3], b = s_coef[3 * zc + 4], cc = s_coef[3 * zc + 5];
      emit(zc + 1, tc, sc, fma(cc, tc, fma(b, tb, a * ta)), fma(cc, sc, fma(b, sb, a * sa)));
    }
  }
}

// adjust_negative_n2 on an existing field (derived.py:30-71)
__global__ void __launch_bounds__(kBlock) k_adjust_n2(const double* __restrict__ n2, int fill_slabs, int nz, i64 ncol,
                                                      double* __restrict__ out) {
  const i64 c = (i64)blockIdx.x * kBlock + threadIdx.x;
  if (c >= ncol) return;
  const i64 slab = (i64)blockIdx.y * nz * ncol + c;
  const bool fill_slab = (int)blockIdx.y < fill_slabs;
  double carry = nan("");
  for (int z = 0; z < nz; ++z) {
    const double v = __ldg(n2 + slab + (i64)z * ncol);
    out[slab + (i64)z * ncol] = adjust_step(v, fill_slab || (fill_slabs < 0 && z == 0), carry);
  }
}

// calc_wave_speed (derived.py:821): sum_z sqrt(adjusted n2) dz / pi, skipna.  dz is [nz][ncol].
__global__ void __launch_bounds__(kBlock) k_wave_speed(const double* __restrict__ n2, const double* __restrict__ dz,
                                                       int fill_slabs, int nz, i64 ncol, double* __restrict__ out) {
  const i64 c = (i64)blockIdx.x * kBlock + threadIdx.x;
  if (c >= ncol) return;
  const i64 slab = (i64)blockIdx.y * nz * ncol + c;
  const bool fill_slab = (int)blockIdx.y < fill_slabs;
  double carry = nan(""), acc = 0.0;
  for (int z = 0; z < nz; ++z) {
    const double v = __ldg(n2 + slab + (i64)z * ncol);
    const double term = sqrt(adjust_step(v, fill_slab || (fill_slabs < 0 && z == 0), carry)) * __ldg(dz + (i64)z * ncol + c);
    if (!isnan(term)) acc += term;
  }
  out[(i64)blockIdx.y * ncol + c] = acc / 3.141592653589793;
}

// The outer slabs run on grid.y, which holds at most 65535 of them: a longer field (a level-last (y, x, z)
// field has y * x slabs, a daily record over 179 years 65535 time steps) is launched in chunks of
// kMaxSlabs, each with its pointers moved to its first slab.
constexpr i64 kMaxSlabs = 65535;

// fill_slabs of the kernels for the chunk [s0, s0 + n) of a call's slabs: fill_mode 0 = the surface level of
// every slab (-1); k >= 1 = every level of the call's slabs [0, k), i.e. the chunk's first k - s0 slabs, and
// none at all in a chunk past them
inline int chunk_fill(int fill_mode, i64 s0, i64 n) {
  if (fill_mode == 0) return -1;
  const i64 k = (i64)fill_mode - s0;
  return (int)(k <= 0 ? 0 : (k < n ? k : n));
}

inline int check_fill_mode(int fill_mode, int64_t nouter) {
  if (fill_mode < 0 || fill_mode > nouter)
    return fail(ML_ERR_MODE, "fill_mode must be 0 (surface level) or 1..nouter=%lld (leading slabs), got %d",
                (long long)nouter, fill_mode);
  return ML_OK;
}

template <int OUT>
int launch_strat(int eos, int dtype, const void* T, const void* S, const double* z_l, const double* p_level,
                 double gravity, double patm, int fill_mode, i64 nouter, int nz, i64 ncol, double* out,
                 cudaStream_t st) {
  const size_t smem = (size_t)4 * nz * sizeof(double) + (size_t)2 * kRing * kBlock * elem_size(dtype);
  for (i64 s0 = 0; s0 < nouter; s0 += kMaxSlabs) {
    const i64 n = nouter - s0 < kMaxSlabs ? nouter - s0 : kMaxSlabs;
    const i64 off = s0 * nz * ncol;
    const char* Tc = static_cast<const char*>(T) + off * elem_size(dtype);
    const char* Sc = static_cast<const char*>(S) + off * elem_size(dtype);
    const int fill = chunk_fill(fill_mode, s0, n);
    const dim3 grid((unsigned)((ncol + kBlock - 1) / kBlock), (unsigned)n);
#define ML_STRAT(TIN, E) \
  k_strat<TIN, E, OUT><<<grid, kBlock, smem, st>>>((const TIN*)Tc, (const TIN*)Sc, z_l, p_level, gravity, patm, fill, nz, ncol, out + off)
    if (dtype == ML_F32) {
      if (eos == ML_EOS_WRIGHT) ML_STRAT(float, 0); else ML_STRAT(float, 1);
    } else {
      if (eos == ML_EOS_WRIGHT) ML_STRAT(double, 0); else ML_STRAT(double, 1);
    }
#undef ML_STRAT
    const int rc = launched("k_strat");
    if (rc) return rc;
  }
  return ML_OK;
}

int check_strat(int eos, int dtype, const void* T, const void* S, const double* z_l, const double* out, int64_t nouter,
                int64_t nz, int64_t ncol) {
  if (eos != ML_EOS_WRIGHT && eos != ML_EOS_LINEAR) return fail(ML_ERR_EOS, "unknown equation of state id %d", eos);
  if (dtype != ML_F32 && dtype != ML_F64) return fail(ML_ERR_DTYPE, "unknown dtype id %d", dtype);
  ML_REQUIRE_PTR(T);
  ML_REQUIRE_PTR(S);
  ML_REQUIRE_PTR(z_l);
  ML_REQUIRE_PTR(out);
  // numpy.gradient(edge_order=2) needs three points; the coefficient table lives in shared memory
  if (nouter <= 0 || ncol <= 0 || nz < 3 || nz > kMaxLevels)
    return fail(ML_ERR_SHAPE, "bad extents nouter=%lld nz=%lld ncol=%lld (3 <= nz <= %d)",
                (long long)nouter, (long long)nz, (long long)ncol, kMaxLevels);
  ML_REQUIRE_ALIGNED(T, elem_size(dtype));
  ML_REQUIRE_ALIGNED(S, elem_size(dtype));
  return ML_OK;
}

}  // namespace
}  // namespace ml

using namespace ml;

extern "C" {

int ml_calc_n2(int eos, int dtype, const void* T, const void* S, const double* z_l, double gravity, double patm,
               int adjust_negative, int fill_mode, int64_t nouter, int64_t nz, int64_t ncol, double* out,
               void* stream) {
  int rc = check_strat(eos, dtype, T, S, z_l, out, nouter, nz, ncol);
  if (rc) return rc;
  if ((rc = check_fill_mode(fill_mode, nouter))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (adjust_negative)
    return launch_strat<kN2Adjusted>(eos, dtype, T, S, z_l, nullptr, gravity, patm, fill_mode, nouter, (int)nz, ncol, out, st);
  return launch_strat<kN2>(eos, dtype, T, S, z_l, nullptr, gravity, patm, fill_mode, nouter, (int)nz, ncol, out, st);
}

int ml_stability_angle(int eos, int dtype, const void* T, const void* S, const double* p_level, const double* z_l,
                       int64_t nouter, int64_t nz, int64_t ncol, double* out, void* stream) {
  int rc = check_strat(eos, dtype, T, S, z_l, out, nouter, nz, ncol);
  if (rc) return rc;
  ML_REQUIRE_PTR(p_level);
  return launch_strat<kTurnerAngle>(eos, dtype, T, S, z_l, p_level, 0.0, 0.0, 0, nouter, (int)nz, ncol, out,
                                    (cudaStream_t)stream);
}

int ml_adjust_negative_n2(const double* n2, int fill_mode, int64_t nouter, int64_t nz, int64_t ncol, double* out,
                          void* stream) {
  ML_REQUIRE_PTR(n2);
  ML_REQUIRE_PTR(out);
  if (nouter <= 0 || nz <= 0 || ncol <= 0 || nz > INT32_MAX)
    return fail(ML_ERR_SHAPE, "bad extents nouter=%lld nz=%lld ncol=%lld", (long long)nouter, (long long)nz, (long long)ncol);
  int rc = check_fill_mode(fill_mode, nouter);
  if (rc) return rc;
  for (i64 s0 = 0; s0 < nouter; s0 += kMaxSlabs) {
    const i64 n = nouter - s0 < kMaxSlabs ? nouter - s0 : kMaxSlabs;
    const i64 off = s0 * nz * ncol;
    const dim3 grid((unsigned)((ncol + kBlock - 1) / kBlock), (unsigned)n);
    k_adjust_n2<<<grid, kBlock, 0, (cudaStream_t)stream>>>(n2 + off, chunk_fill(fill_mode, s0, n), (int)nz, ncol, out + off);
    if ((rc = launched("k_adjust_n2"))) return rc;
  }
  return ML_OK;
}

int ml_wave_speed(const double* n2, const double* dz, int fill_mode, int64_t nouter, int64_t nz, int64_t ncol,
                  double* out, void* stream) {
  ML_REQUIRE_PTR(n2);
  ML_REQUIRE_PTR(dz);
  ML_REQUIRE_PTR(out);
  if (nouter <= 0 || nz <= 0 || ncol <= 0 || nz > INT32_MAX)
    return fail(ML_ERR_SHAPE, "bad extents nouter=%lld nz=%lld ncol=%lld", (long long)nouter, (long long)nz, (long long)ncol);
  int rc = check_fill_mode(fill_mode, nouter);
  if (rc) return rc;
  for (i64 s0 = 0; s0 < nouter; s0 += kMaxSlabs) {
    const i64 n = nouter - s0 < kMaxSlabs ? nouter - s0 : kMaxSlabs;
    const dim3 grid((unsigned)((ncol + kBlock - 1) / kBlock), (unsigned)n);
    k_wave_speed<<<grid, kBlock, 0, (cudaStream_t)stream>>>(n2 + s0 * nz * ncol, dz, chunk_fill(fill_mode, s0, n), (int)nz,
                                                            ncol, out + s0 * ncol);
    if ((rc = launched("k_wave_speed"))) return rc;
  }
  return ML_OK;
}

}  // extern "C"
