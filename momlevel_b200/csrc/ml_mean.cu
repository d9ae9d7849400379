// ml_mean.cu -- time mean of T, S and volcello over a baseline period (ml_mean_state_accumulate).
//
// A climatological reference state (setup_reference_state(period=...)) is the skipna weighted mean of each field
// over the period, x_mean = sum_t w_t x_t / sum_t w_t with both sums over the steps where x is not NaN (xarray's
// weighted(...).mean).  A thread owns consecutive cells and walks time fastest, so the six running sums -- a weighted
// sum and a weight sum per field -- stay in fp64 registers for the whole launch; they touch memory only between the
// launches of a period that arrives in blocks.
//
// Every step is added as acc = acc + w * x and wsum = wsum + w, rounded separately (no FMA contraction), in ascending
// t, and the mean is one IEEE division: the bits do not depend on how the period is cut into launches, on the kernel
// (vector or plain loads) or on the route, and equal a numpy loop over t doing the same three operations.
#include "ml_common.cuh"
#include "ml_host.cuh"

namespace ml {
namespace {

constexpr int kMeanBlock = 256;
// steps per launch: bounds one kernel's run time (1024 OM4p25 steps stream ~0.25 s at HBM rate); a longer call runs as
// several launches that carry the sums through the accumulator
constexpr int64_t kMeanStepsPerLaunch = 1024;
constexpr int kFirst = 1, kLast = 2;

__device__ __forceinline__ void mean_add(double& s, double& sw, double w, double x) {
  if (!isnan(x)) {  // skipna: a missing value adds to neither sum
    s = __dadd_rn(s, __dmul_rn(w, x));
    sw = __dadd_rn(sw, w);
  }
}

// four consecutive values, kept in their storage type until they are added
template <typename T>
struct Q4 {
  T v[4];
};
__device__ __forceinline__ void ldq(const float* p, Q4<float>& q) {
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(q.v[0]), "=f"(q.v[1]), "=f"(q.v[2]), "=f"(q.v[3]) : "l"(p));
}
__device__ __forceinline__ void ldq(const double* p, Q4<double>& q) {
  asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0, %1}, [%2];" : "=d"(q.v[0]), "=d"(q.v[1]) : "l"(p));
  asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0, %1}, [%2];" : "=d"(q.v[2]), "=d"(q.v[3]) : "l"(p + 2));
}
__device__ __forceinline__ void ldacc(const double* p, double v[4]) {  // the accumulator: read and written by this kernel
  const double2 a = *reinterpret_cast<const double2*>(p), b = *reinterpret_cast<const double2*>(p + 2);
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}
__device__ __forceinline__ void st4d(double* p, const double v[4]) {
  asm volatile("st.global.L1::no_allocate.v2.f64 [%0], {%1, %2};" ::"l"(p), "d"(v[0]), "d"(v[1]) : "memory");
  asm volatile("st.global.L1::no_allocate.v2.f64 [%0], {%1, %2};" ::"l"(p + 2), "d"(v[2]), "d"(v[3]) : "memory");
}

// Fast path: four consecutive cells per thread (n % 4 == 0, 16-byte aligned bases), U steps of T, S and V loaded before
// any of them is added so that 3 * U 16-byte loads per thread are in flight.  acc is [6][n]: sum and weight sum of T,
// of S, of V.  fp32 fields ask for three CTAs per SM: left unsaid, ptxas gives them 94 registers and two CTAs, and
// OM4p25 x 12 took 7.1 ms instead of 4.3 ms on a B200.  fp64 fields would spill under that bound; 0 leaves them unsaid.
template <typename TF, typename TV>
__global__ void __launch_bounds__(kMeanBlock, sizeof(TF) == 4 ? 3 : 0)
    k_mean_state_vec(const TF* __restrict__ T, const TF* __restrict__ S, const TV* __restrict__ V,
                     const double* __restrict__ w, i64 nt, i64 n, double* __restrict__ acc, int flags,
                     double* __restrict__ Tm, double* __restrict__ Sm, double* __restrict__ Vm) {
  constexpr int U = (sizeof(TF) == 4 && sizeof(TV) == 4) ? 4 : 2;
  const i64 c = 4 * ((i64)blockIdx.x * kMeanBlock + threadIdx.x);
  if (c >= n) return;
  double a[6][4];
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    if (flags & kFirst) {
      a[k][0] = a[k][1] = a[k][2] = a[k][3] = 0.0;
    } else {
      ldacc(acc + k * n + c, a[k]);
    }
  }
  i64 t = 0;
  for (; t + U <= nt; t += U) {
    Q4<TF> tq[U], sq[U];
    Q4<TV> vq[U];
    double wu[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const i64 o = (t + u) * n + c;
      ldq(T + o, tq[u]);
      ldq(S + o, sq[u]);
      ldq(V + o, vq[u]);
      wu[u] = w != nullptr ? __ldg(w + t + u) : 1.0;
    }
#pragma unroll
    for (int u = 0; u < U; ++u)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        mean_add(a[0][j], a[1][j], wu[u], (double)tq[u].v[j]);
        mean_add(a[2][j], a[3][j], wu[u], (double)sq[u].v[j]);
        mean_add(a[4][j], a[5][j], wu[u], (double)vq[u].v[j]);
      }
  }
  for (; t < nt; ++t) {
    Q4<TF> tq, sq;
    Q4<TV> vq;
    const i64 o = t * n + c;
    ldq(T + o, tq);
    ldq(S + o, sq);
    ldq(V + o, vq);
    const double wt = w != nullptr ? __ldg(w + t) : 1.0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      mean_add(a[0][j], a[1][j], wt, (double)tq.v[j]);
      mean_add(a[2][j], a[3][j], wt, (double)sq.v[j]);
      mean_add(a[4][j], a[5][j], wt, (double)vq.v[j]);
    }
  }
  if (flags & kLast) {
    double m[4];
    double* const out[3] = {Tm, Sm, Vm};
#pragma unroll
    for (int f = 0; f < 3; ++f) {
#pragma unroll
      for (int j = 0; j < 4; ++j) m[j] = __ddiv_rn(a[2 * f][j], a[2 * f + 1][j]);  // 0 / 0 = NaN: no value in the period
      st4d(out[f] + c, m);
    }
  } else {
#pragma unroll
    for (int k = 0; k < 6; ++k) st4d(acc + k * n + c, a[k]);
  }
}

// Plain loads: one cell per thread, any extent and alignment (ragged rows, offset bases, ml_set_force_direct(1)).
template <typename TF, typename TV>
__global__ void __launch_bounds__(kMeanBlock)
    k_mean_state(const TF* __restrict__ T, const TF* __restrict__ S, const TV* __restrict__ V,
                 const double* __restrict__ w, i64 nt, i64 n, double* __restrict__ acc, int flags,
                 double* __restrict__ Tm, double* __restrict__ Sm, double* __restrict__ Vm) {
  const i64 c = (i64)blockIdx.x * kMeanBlock + threadIdx.x;
  if (c >= n) return;
  double a[6];
#pragma unroll
  for (int k = 0; k < 6; ++k) a[k] = (flags & kFirst) ? 0.0 : acc[k * n + c];
  for (i64 t = 0; t < nt; ++t) {
    const i64 o = t * n + c;
    const double wt = w != nullptr ? __ldg(w + t) : 1.0;
    mean_add(a[0], a[1], wt, ldf(T + o));
    mean_add(a[2], a[3], wt, ldf(S + o));
    mean_add(a[4], a[5], wt, ldf(V + o));
  }
  if (flags & kLast) {
    Tm[c] = __ddiv_rn(a[0], a[1]);
    Sm[c] = __ddiv_rn(a[2], a[3]);
    Vm[c] = __ddiv_rn(a[4], a[5]);
  } else {
#pragma unroll
    for (int k = 0; k < 6; ++k) acc[k * n + c] = a[k];
  }
}

template <typename TF, typename TV>
int launch_mean(bool vec, const void* T, const void* S, const void* V, const double* w, i64 nt, i64 n, double* acc,
                int flags, double* Tm, double* Sm, double* Vm, cudaStream_t st) {
  if (vec) {
    const i64 nb = (n / 4 + kMeanBlock - 1) / kMeanBlock;
    k_mean_state_vec<TF, TV><<<(unsigned)nb, kMeanBlock, 0, st>>>((const TF*)T, (const TF*)S, (const TV*)V, w, nt, n,
                                                                  acc, flags, Tm, Sm, Vm);
    return launched("k_mean_state_vec");
  }
  const i64 nb = (n + kMeanBlock - 1) / kMeanBlock;
  k_mean_state<TF, TV><<<(unsigned)nb, kMeanBlock, 0, st>>>((const TF*)T, (const TF*)S, (const TV*)V, w, nt, n, acc,
                                                            flags, Tm, Sm, Vm);
  return launched("k_mean_state");
}

}  // namespace
}  // namespace ml

using namespace ml;

extern "C" {

size_t ml_mean_state_bytes(int64_t nz, int64_t ncol) {
  if (nz <= 0 || ncol <= 0 || nz > INT64_MAX / 48 / ncol) return 0;
  return (size_t)(6 * sizeof(double)) * (size_t)nz * (size_t)ncol;
}

int ml_mean_state_accumulate(int dtype, const void* T, const void* S, const void* V, int vdtype, const double* w,
                             int64_t nt, int64_t nz, int64_t ncol, void* acc, size_t acc_bytes, int flags,
                             double* T_mean, double* S_mean, double* V_mean, void* stream) {
  if (dtype != ML_F32 && dtype != ML_F64) return fail(ML_ERR_DTYPE, "unknown dtype id %d", dtype);
  if (vdtype != ML_F32 && vdtype != ML_F64) return fail(ML_ERR_DTYPE, "unknown volcello dtype id %d", vdtype);
  if (flags & ~(kFirst | kLast)) return fail(ML_ERR_MODE, "unknown flags %d (1 first, 2 last)", flags);
  ML_REQUIRE_PTR(T);
  ML_REQUIRE_PTR(S);
  ML_REQUIRE_PTR(V);
  if (nt <= 0 || nz <= 0 || ncol <= 0 || ml_mean_state_bytes(nz, ncol) == 0 || nt > INT64_MAX / (nz * ncol))
    return fail(ML_ERR_SHAPE, "bad extents nt=%lld nz=%lld ncol=%lld", (long long)nt, (long long)nz, (long long)ncol);
  if (flags & kLast) {
    ML_REQUIRE_PTR(T_mean);
    ML_REQUIRE_PTR(S_mean);
    ML_REQUIRE_PTR(V_mean);
    ML_REQUIRE_ALIGNED(T_mean, 8);
    ML_REQUIRE_ALIGNED(S_mean, 8);
    ML_REQUIRE_ALIGNED(V_mean, 8);
  }
  const int esz = elem_size(dtype), vsz = elem_size(vdtype);
  ML_REQUIRE_ALIGNED(T, esz);
  ML_REQUIRE_ALIGNED(S, esz);
  ML_REQUIRE_ALIGNED(V, vsz);
  if (w != nullptr) ML_REQUIRE_ALIGNED(w, 8);
  // the sums live in registers for a whole launch; they go through acc when the call does not start and end the period,
  // or when it is longer than one launch takes
  const bool need_acc = flags != (kFirst | kLast) || nt > kMeanStepsPerLaunch;
  if (need_acc) {
    if (acc == nullptr || acc_bytes < ml_mean_state_bytes(nz, ncol))
      return fail(ML_ERR_WORKSPACE, "accumulator needs %zu bytes, got %zu", ml_mean_state_bytes(nz, ncol),
                  acc == nullptr ? (size_t)0 : acc_bytes);
    ML_REQUIRE_ALIGNED(acc, 8);
  }
  const i64 n = nz * ncol;
  uintptr_t bits = reinterpret_cast<uintptr_t>(T) | reinterpret_cast<uintptr_t>(S) | reinterpret_cast<uintptr_t>(V);
  if (need_acc) bits |= reinterpret_cast<uintptr_t>(acc);
  if (flags & kLast)
    bits |= reinterpret_cast<uintptr_t>(T_mean) | reinterpret_cast<uintptr_t>(S_mean) | reinterpret_cast<uintptr_t>(V_mean);
  const bool vec = ncol % 4 == 0 && (bits & 15u) == 0 && tls().force_direct != 1;
  cudaStream_t st = (cudaStream_t)stream;
  double* a = need_acc ? (double*)acc : nullptr;
  for (i64 t0 = 0; t0 < nt; t0 += kMeanStepsPerLaunch) {
    const i64 k = nt - t0 < kMeanStepsPerLaunch ? nt - t0 : kMeanStepsPerLaunch;
    const int f = (t0 == 0 ? flags & kFirst : 0) | (t0 + k == nt ? flags & kLast : 0);
    const char* Tp = (const char*)T + t0 * n * esz;
    const char* Sp = (const char*)S + t0 * n * esz;
    const char* Vp = (const char*)V + t0 * n * vsz;
    const double* wp = w != nullptr ? w + t0 : nullptr;
    int rc;
    if (dtype == ML_F32)
      rc = vdtype == ML_F32 ? launch_mean<float, float>(vec, Tp, Sp, Vp, wp, k, n, a, f, T_mean, S_mean, V_mean, st)
                            : launch_mean<float, double>(vec, Tp, Sp, Vp, wp, k, n, a, f, T_mean, S_mean, V_mean, st);
    else
      rc = vdtype == ML_F32 ? launch_mean<double, float>(vec, Tp, Sp, Vp, wp, k, n, a, f, T_mean, S_mean, V_mean, st)
                            : launch_mean<double, double>(vec, Tp, Sp, Vp, wp, k, n, a, f, T_mean, S_mean, V_mean, st);
    if (rc) return rc;
  }
  return ML_OK;
}

}  // extern "C"
