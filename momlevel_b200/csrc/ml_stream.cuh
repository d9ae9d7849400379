// ml_stream.cuh -- interface of the ring-staged elementwise kernels (ml_stream.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace ml {
namespace stream {

// rows of ncol fp32 points start 16-byte aligned in every operand (pass NULL for an absent one)
bool eligible(const void* a, const void* b, const void* c, const void* out, long long ncol);

// spice.flament.spice over n points (n % 4 == 0)
int launch_spice(const float* T, const float* S, long long n, double* out, cudaStream_t st);

// eos.<name>.density over rows [nouter * nz][ncol]; p scalar / per level / absent (pmode as ml_eos_eval)
int launch_density(int eos, const float* T, const float* S, long long t_stride, long long s_stride, const double* p,
                   int pmode, long long nrows, int nz, long long ncol, double* out, cudaStream_t st);

// reference-state pass: rho_ref out, block partials [2][refstate_blocks()] for the fixed-order second stage
int refstate_blocks(long long nz, long long ncol);
int launch_refstate(int eos, const float* T0, const float* S0, const float* V0, const double* p_level, long long nz,
                    long long ncol, double* rho_ref, double* partials, cudaStream_t st);

// delta_rho[t][z][col] = rho(T, S, p_z) - rho_ref where the reference volume is present, NaN elsewhere (steric.py:151-153);
// t_stride / s_stride = 0 for an operand held at the reference slab
int launch_delta_rho(int eos, const float* T, const float* S, long long t_stride, long long s_stride, const double* rho_ref,
                     const void* v_ref, int v_f32, const double* p_level, int nt, long long nz, long long ncol, double* out,
                     cudaStream_t st);

// level profile (ml_steric_local_profile): per-warp partials of coef * m * w * dz * (rho_v - rho_ref) into part[v]
// ([nt * nz][profile_slots(ncol)], NULL for a variant not asked for), vm = the variants as bits (1 steric,
// 2 thermosteric, 4 halosteric); the fixed-order second stage is k_reduce_rows.  With a region index ([ncol],
// ml_steric_local_region_profile; NULL: none) part[v] is [nregions][nt * nz][profile_slots(ncol)].  ny > 0
// (ml_steric_local_zonal_profile): a level is ny grid rows of ncol = nx columns, T and S are [nt][nz][ny][nx] and
// part[v] is [nt * nz * ny][profile_slots(nx)], one partial row per grid row; ny = 0: a level is one row of ncol.
int profile_slots(long long ncol);
int launch_profile(int eos, int vm, const float* T, const float* S, const float* T_ref, const float* S_ref,
                   const double* rho_ref, const void* v_ref, int v_f32, const double* z_i, const double* deptho,
                   const double* weights, const double* p_level, double coef, int nt, long long nz, long long ncol,
                   double* const part[3], const int8_t* region, int nregions, int ny, cudaStream_t st);

}  // namespace stream
}  // namespace ml
