// ml_common.cuh -- device-side arithmetic shared by every kernel of libmomlevel_b200.
//
// Equations of state follow the reference's numpy expressions
// (src/momlevel/eos/wright.py:44-48, src/momlevel/eos/linear.py:55-58) evaluated in fp64
// registers with FMA contraction; inputs may be stored as fp32 and are widened on load.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace ml {

typedef long long i64;

// ----------------------------------------------------------------------------- constants
// Wright (1997) reduced-range coefficients, wright.py:6-20
namespace wr {
constexpr double a0 = 7.057924e-4, a1 = 3.480336e-7, a2 = -1.112733e-7;
constexpr double b0 = 5.790749e8, b1 = 3.516535e6, b2 = -4.002714e4, b3 = 2.084372e2,
                 b4 = 5.944068e5, b5 = -9.643486e3;
constexpr double c0 = 1.704853e5, c1 = 7.904722e2, c2 = -7.984422, c3 = 5.140652e-2,
                 c4 = -2.302158e2, c5 = -3.079464;
}  // namespace wr
// linear.py:17-23
namespace lin {
constexpr double rho_t0_s0 = 1000.0, drho_dt = -0.2, drho_ds = 0.8;
}

// --------------------------------------------------------------------------------- loads
// Streaming read-only loads; the fields are touched once per launch.
__device__ __forceinline__ double ldf(const float* p) { return (double)__ldg(p); }
__device__ __forceinline__ double ldf(const double* p) { return __ldg(p); }

// NaN test for a value PRODUCED by fp64 arithmetic (always a quiet NaN, so the quiet bit in
// the high word is set).  One integer compare instead of a DSETP on the fp64 pipe.
__device__ __forceinline__ bool is_nan_q(double x) {
  return (((unsigned)__double2hiint(x)) << 1) > 0xffe00000u;
}

// ------------------------------------------------------------------------------ division
// q = n / d for the Wright denominator (5.7e5 .. 7.3e5 over the oceanic range, never near
// zero).  MUFU.RCP64H seed (rel. error e ~ 2^-20) refined by one cubic step:
//   r = r0 (1 + e + e^2),  e = 1 - d r0   ->  rel. error e^3 < 2^-57.
// That is 3 DFMA + 1 DMUL instead of the ~10 fp64 slots of the IEEE division routine.
// NaN flows through.  Valid while 1/d is a normal number (2^-1022 <= |d| < 2^1022).
__device__ __forceinline__ double rcp_lean(double d) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(d));
  const double e = fma(-d, r, 1.0);
  const double t = fma(e, e, e);
  return fma(r, t, r);
}
__device__ __forceinline__ double div_lean(double n, double d) { return n * rcp_lean(d); }

// Same, but denominators whose reciprocal would leave the normal range take the IEEE path
// so inf / 0 behaviour matches numpy; used by the elementwise operator (ml_eos_eval), which
// may be handed arbitrary numbers.
__device__ __forceinline__ double div_checked(double n, double d) {
  const unsigned eh = (((unsigned)__double2hiint(d)) >> 20) & 0x7ffu;
  if (__builtin_expect(eh == 0u || (eh - 2045u) < 2u, 0)) return n / d;
  return div_lean(n, d);
}

// ---------------------------------------------------------------------------------- EOS
// The 15 Wright coefficients live in constant memory and are copied into (uniform)
// registers once per thread; literal doubles would be re-materialised as two 32-bit moves
// in front of every DFMA, which makes the point loop issue-bound instead of fp64-bound.
struct WrightC {
  double a0, a1, a2, b0, b1, b2, b3, b4, b5, c0, c1, c2, c3, c4, c5;
};
static __constant__ WrightC kWrightC = {wr::a0, wr::a1, wr::a2, wr::b0, wr::b1, wr::b2, wr::b3, wr::b4,
                                        wr::b5, wr::c0, wr::c1, wr::c2, wr::c3, wr::c4, wr::c5};

template <int EOS>
struct Eos;

// Wright: p enters only as (p + p0) and b0 is the constant term of p0, so b0p = b0 + p is
// formed once per level.  rho(T,S): 13 DFMA + the lean division (3 DFMA + 1 DMUL).
template <>
struct Eos<0> {
  WrightC K;
  double b0p;
  __device__ __forceinline__ Eos() : K(kWrightC), b0p(0.0) {}
  __device__ __forceinline__ void set_level(double p) { b0p = K.b0 + p; }
  __device__ __forceinline__ void terms(double T, double S, double b0p_, double& pp, double& den) const {
    const double al0 = fma(K.a2, S, fma(K.a1, T, K.a0));
    pp = fma(T, fma(K.b5, S, fma(T, fma(K.b3, T, K.b2), K.b1)), fma(K.b4, S, b0p_));
    const double lam = fma(T, fma(K.c5, S, fma(T, fma(K.c3, T, K.c2), K.c1)), fma(K.c4, S, K.c0));
    den = fma(al0, pp, lam);
  }
  __device__ __forceinline__ double rho(double T, double S) const {
    double pp, den;
    terms(T, S, b0p, pp, den);
    return div_lean(pp, den);
  }
  // density at another level's pressure without disturbing the current level
  __device__ __forceinline__ double rho_at(double T, double S, double p) const {
    double pp, den;
    terms(T, S, K.b0 + p, pp, den);
    return div_lean(pp, den);
  }
  __device__ __forceinline__ double rho_checked(double T, double S) const {
    double pp, den;
    terms(T, S, b0p, pp, den);
    return div_checked(pp, den);
  }
  // One operand pinned for a whole level (thermosteric holds S, halosteric holds T at the reference
  // slab, steric.py:115-121): p0 and lambda are cubic in T with S entering linearly, so the pinned
  // part of every coefficient is formed once and a point costs 6 (S pinned) or 4 (T pinned) fused
  // multiply-adds before the division instead of 13.  Same polynomial, different association: the
  // result differs from rho(T, S) by rounding (~1e-16 relative).
  struct Pinned {
    double a, b1, b0, c1, c0;
  };
  __device__ __forceinline__ Pinned pin_s(double S) const {  // at the current level
    return {fma(K.a2, S, K.a0), fma(K.b5, S, K.b1), fma(K.b4, S, b0p), fma(K.c5, S, K.c1), fma(K.c4, S, K.c0)};
  }
  __device__ __forceinline__ double rho_pinned_s(const Pinned& q, double T) const {
    const double pp = fma(T, fma(T, fma(K.b3, T, K.b2), q.b1), q.b0);
    const double lam = fma(T, fma(T, fma(K.c3, T, K.c2), q.c1), q.c0);
    return div_lean(pp, fma(fma(K.a1, T, q.a), pp, lam));
  }
  __device__ __forceinline__ Pinned pin_t(double T) const {
    return {fma(K.a1, T, K.a0), fma(K.b5, T, K.b4), fma(T, fma(T, fma(K.b3, T, K.b2), K.b1), b0p),
            fma(K.c5, T, K.c4), fma(T, fma(T, fma(K.c3, T, K.c2), K.c1), K.c0)};
  }
  __device__ __forceinline__ double rho_pinned_t(const Pinned& q, double S) const {
    const double pp = fma(S, q.b1, q.b0);
    return div_lean(pp, fma(fma(K.a2, S, q.a), pp, fma(S, q.c1, q.c0)));
  }
  // numerator and denominator on their own (same expressions as above), for callers that share one
  // reciprocal seed between several densities of a point
  __device__ __forceinline__ void terms_of(double T, double S, double& pp, double& den) const { terms(T, S, b0p, pp, den); }
  __device__ __forceinline__ void terms_pinned_s(const Pinned& q, double T, double& pp, double& den) const {
    pp = fma(T, fma(T, fma(K.b3, T, K.b2), q.b1), q.b0);
    den = fma(fma(K.a1, T, q.a), pp, fma(T, fma(T, fma(K.c3, T, K.c2), q.c1), q.c0));
  }
  __device__ __forceinline__ void terms_pinned_t(const Pinned& q, double S, double& pp, double& den) const {
    pp = fma(S, q.b1, q.b0);
    den = fma(fma(K.a2, S, q.a), pp, fma(S, q.c1, q.c0));
  }
};

// linear.py:55-58 -- pressure is ignored by design
__device__ __forceinline__ double linear_rho(double T, double S) {
  return lin::rho_t0_s0 + fma(lin::drho_ds, S, lin::drho_dt * T);
}
template <>
struct Eos<1> {
  __device__ __forceinline__ Eos() {}
  __device__ __forceinline__ void set_level(double) {}
  __device__ __forceinline__ double rho(double T, double S) const { return linear_rho(T, S); }
  __device__ __forceinline__ double rho_at(double T, double S, double) const { return linear_rho(T, S); }
  __device__ __forceinline__ double rho_checked(double T, double S) const { return linear_rho(T, S); }
  struct Pinned {
    double v;
  };
  __device__ __forceinline__ Pinned pin_s(double S) const { return {S}; }
  __device__ __forceinline__ double rho_pinned_s(const Pinned& q, double T) const { return linear_rho(T, q.v); }
  __device__ __forceinline__ Pinned pin_t(double T) const { return {T}; }
  __device__ __forceinline__ double rho_pinned_t(const Pinned& q, double S) const { return linear_rho(q.v, S); }
};

// Derivatives (wright.py:53-165); not on the steric path, plain IEEE division.
__device__ __forceinline__ void wright_terms(double T, double S, double& al0, double& p0, double& lam) {
  al0 = fma(wr::a2, S, fma(wr::a1, T, wr::a0));
  p0 = fma(T, fma(wr::b5, S, fma(T, fma(wr::b3, T, wr::b2), wr::b1)), fma(wr::b4, S, wr::b0));
  lam = fma(T, fma(wr::c5, S, fma(T, fma(wr::c3, T, wr::c2), wr::c1)), fma(wr::c4, S, wr::c0));
}
__device__ __forceinline__ double wright_drho_dtemp(double T, double S, double p) {
  double al0, p0, lam;
  wright_terms(T, S, al0, p0, lam);
  const double pp = p + p0;
  double i2 = 1.0 / fma(al0, pp, lam);
  i2 *= i2;
  const double dp0 = fma(wr::b5, S, fma(T, fma(3.0 * wr::b3, T, 2.0 * wr::b2), wr::b1));
  const double dlam = fma(wr::c5, S, fma(T, fma(3.0 * wr::c3, T, 2.0 * wr::c2), wr::c1));
  return i2 * (lam * dp0 - pp * fma(pp, wr::a1, dlam));
}
__device__ __forceinline__ double wright_drho_dsal(double T, double S, double p) {
  double al0, p0, lam;
  wright_terms(T, S, al0, p0, lam);
  const double pp = p + p0;
  double i2 = 1.0 / fma(al0, pp, lam);
  i2 *= i2;
  return i2 * (lam * fma(wr::b5, T, wr::b4) - pp * fma(pp, wr::a2, fma(wr::c5, T, wr::c4)));
}

// eos x func elementwise dispatch used by ml_eos_eval
template <int EOS, int FUNC>
__device__ __forceinline__ double eos_func(double T, double S, double p) {
  if (EOS == 0) {
    Eos<0> e;
    e.set_level(p);
    if (FUNC == 0) return e.rho_checked(T, S);
    if (FUNC == 1) return wright_drho_dtemp(T, S, p);
    if (FUNC == 2) return wright_drho_dsal(T, S, p);
    const double rho = e.rho_checked(T, S);
    if (FUNC == 3) return -1.0 * (wright_drho_dtemp(T, S, p) / rho);
    return wright_drho_dsal(T, S, p) / rho;
  } else {
    // linear.py:61-162: constant derivatives; alpha/beta keep numpy's NaN propagation
    // through density and np.full_like(T, ...)
    if (FUNC == 0) return linear_rho(T, S);
    if (FUNC == 1) return lin::drho_dt;
    if (FUNC == 2) return lin::drho_ds;
    const double rho = linear_rho(T, S);
    if (FUNC == 3) return -1.0 * (lin::drho_dt / rho);
    return lin::drho_ds / rho;
  }
}

// -------------------------------------------------------------------------------- spice
// Flament (2002), flament.py:7-40: pi = sum_ij b_ij T^i s^j, s = S - 35.
// Inner Horner in s for each power of T, outer Horner in T: 24 + 5 DFMA + 1 DADD.
// A result that is not finite is NaN, as in the reference's sum of power-table terms (flament.py:82-90): an infinite
// T or S, or a power that overflows, meets coefficients of both signs there (inf - inf), where the nested form alone
// would return +-inf.  Finite inputs in range never give an infinite result, so the test is on the result: one
// exponent-bit test on the integer pipe and a select, no branch and no extra fp64 work.
__device__ __forceinline__ double flament_spice(double T, double S) {
  const double s = S - 35.0;
  const double r0 = s * fma(s, fma(s, fma(s, -2.06e-4, -9.84e-4), -5.85e-3), 7.7442e-1);
  const double r1 = fma(s, fma(s, fma(s, fma(s, 1.36e-5, -8.5e-6), -2.742e-4), 2.034e-3), 5.1655e-2);
  const double r2 = fma(s, fma(s, fma(s, fma(s, 7.894e-6, 3.337e-5), -1.428e-5), -2.4681e-4), 6.64783e-3);
  const double r3 = fma(s, fma(s, fma(s, fma(s, -1.0853e-6, -3.0412e-6), 7.0036e-6), 7.326e-6), -5.4023e-5);
  const double r4 = fma(s, fma(s, fma(s, fma(s, 4.7133e-8, 1.0012e-7), -3.8209e-7), -3.029e-8), 3.949e-7);
  const double r5 = fma(s, fma(s, fma(s, fma(s, -6.676e-10, -1.1409e-9), 6.048e-9), -1.309e-9), -6.36e-10);
  const double r = fma(T, fma(T, fma(T, fma(T, fma(T, r5, r4), r3), r2), r1), r0);
  return (__double2hiint(r) & 0x7ff00000) == 0x7ff00000 ? __longlong_as_double(0x7ff8000000000000ll) : r;
}

// --------------------------------------------------------------------------- reductions
// Fixed-order block sum: lanes tree-reduce by shuffle, warp leaders through shared memory,
// warp 0 finishes.  The order depends only on the launch shape -> bitwise reproducible.
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;
}

template <int NWARPS>
__device__ __forceinline__ double block_sum(double v, double* smem /* NWARPS doubles */) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  v = warp_sum(v);
  __syncthreads();  // smem may still be read by a previous call
  if (lane == 0) smem[w] = v;
  __syncthreads();
  double r = 0.0;
  if (w == 0) {
    r = lane < NWARPS ? smem[lane] : 0.0;
    r = warp_sum(r);
  }
  return r;  // valid in thread 0
}

// dz of derived.py:308-318 for top = 0, bottom = None: the second clip min(max(zbot,0), .)
// is the identity because 0 <= ztop (asserted on the host, derived.py:284-292).
__device__ __forceinline__ double clipped_dz(double depth, double ztop, double zbot) {
  return fmin(fmax(depth - ztop, 0.0), zbot - ztop);
}

// --------------------------------------------------------------------- level profile (ml_steric_local_profile)
// Weight of one point in the area-weighted profile: coef * w * dz where the surface cell holds water (steric.py:166)
// and the column weight is a number; 0 elsewhere (a NaN weight counts as 0).  Both kernel families form it here.
__device__ __forceinline__ double profile_weight(bool surface_wet, double w, double dz, double coef) {
  return (surface_wet && !isnan(w)) ? __dmul_rn(__dmul_rn(w, dz), coef) : 0.0;
}
// One term of a profile sum, skipna: d = rho - rho_ref is rounded on its own (no contraction into an FMA), so a point
// at its reference state contributes exactly 0 and a NaN term (a hole, a missing reference volume) is skipped.
__device__ __forceinline__ double profile_add(double acc, double cw, double rho, double rref) {
  const double d = __dsub_rn(rho, rref);
  return is_nan_q(d) ? acc : fma(cw, d, acc);
}
// Region of a column for ml_steric_local_region_profile as a 4-bit field: its index if in [0, nregions), else 0xF
// (no region; nregions <= ML_MAX_REGIONS = 15).
__device__ __forceinline__ uint32_t region_nibble(const int8_t* region, i64 c, int nregions) {
  const int r = __ldg(region + c);
  return (r >= 0 && r < nregions) ? (uint32_t)r : 0xFu;
}

}  // namespace ml
