// ml_tma.cuh -- interface of the TMA-staged kernel family (ml_tma.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace ml {
namespace tma {

bool local_eligible(int dtype, const void* T, const void* S, int t_bcast, int s_bcast, const double* rho_ref,
                    const void* v_ref, int vref_dtype, int64_t nt, int64_t nz, int64_t ncol, const double* eta,
                    const double* delta_rho);
int launch_local(int eos, int dtype, const void* T, const void* S, int t_bcast, int s_bcast, const double* rho_ref,
                 const void* v_ref, int vref_dtype, const double* z_i, const double* deptho, const double* p_level,
                 double coef, int nt, int nz, int64_t ncol, double* eta, double* delta_rho, cudaStream_t st,
                 int first_is_reference = 0);  // step 0 of the fields is the reference state: its height is exactly 0

// kLocalLayers: launch_local split by depth layer, eta [nt][nlayers][ncol]; edges (host) as ml_steric_local_layers,
// eligibility is local_eligible without delta_rho
int launch_local_layers(int eos, const void* T, const void* S, int t_bcast, int s_bcast, const double* rho_ref,
                        const void* v_ref, int vref_dtype, const double* z_i, const double* deptho, const double* p_level,
                        double coef, const double* edges, int nlayers, int nt, int nz, int64_t ncol, double* eta,
                        cudaStream_t st);

// kSelfRef: reference state (rho_ref, volo, masso) and eta from one pass; reference = step 0
int launch_selfref(int eos, const void* T, const void* S, int t_bcast, int s_bcast, const void* v_ref, int vref_dtype,
                   const double* z_i, const double* deptho, const double* p_level, double coef, int nt, int nz,
                   int64_t ncol, double* eta, double* rho_ref, double* sums, double* partials, cudaStream_t st);

bool global_eligible(int dtype, const void* T, const void* S, int t_bcast, int s_bcast, const void* v_ref,
                     int vref_dtype, int64_t nt, int64_t nz, int64_t ncol);
int launch_global(int eos, int dtype, const void* T, const void* S, int t_bcast, int s_bcast, const void* v_ref,
                  int vref_dtype, const double* p_level, int nt, int nz, int64_t ncol, double* masso, double* partials,
                  cudaStream_t st);

// steric, thermosteric and halosteric height from one pass (ml_tma3.cu).  rho_ref != NULL: the reference is
// supplied (T_ref, S_ref, rho_ref); rho_ref == NULL: T_ref / S_ref are the step-0 slabs of T / S and the reference
// density, volo and masso are evaluated on the way (rho_ref_out optional).  Any eta may be NULL.
bool variants_eligible(int dtype, const void* T, const void* S, const void* T_ref, const void* S_ref, int vref_dtype,
                       int64_t nt, int64_t nz, int64_t ncol);
int launch_variants(int eos, const void* T, const void* S, const void* T_ref, const void* S_ref, const double* rho_ref,
                    const void* v_ref, const double* z_i, const double* deptho, const double* p_level, double coef, int nt,
                    int nz, int64_t ncol, double* eta_steric, double* eta_thermo, double* eta_halo, double* rho_ref_out,
                    double* sums, double* partials, cudaStream_t st);

// kLocalLayers3: launch_variants with a supplied reference (rho_ref read), split by depth layer; eta_* [nt][nlayers][ncol]
// each (NULL = not wanted), edges (host) as ml_steric_local_layers; eligibility is variants_eligible
int launch_local_layers_variants(int eos, const void* T, const void* S, const void* T_ref, const void* S_ref,
                                 const double* rho_ref, const void* v_ref, const double* z_i, const double* deptho,
                                 const double* p_level, double coef, const double* edges, int nlayers, int nt, int nz,
                                 int64_t ncol, double* eta_steric, double* eta_thermo, double* eta_halo, cudaStream_t st);

// the three global masses per step from one pass (ml_tma3.cu), each bit-identical to one launch_global with
// BC = 0 / 2 / 1; eligibility is variants_eligible.  sums != NULL: T_ref / S_ref are the step-0 slabs of T / S and
// {volo, masso} of the reference state are reduced on the way.  Any masso may be NULL.  `partials` holds
// global_variants_partials(nt, ncol) bytes.
size_t global_variants_partials(int64_t nt, int64_t ncol);
int launch_global_variants(int eos, const void* T, const void* S, const void* T_ref, const void* S_ref, const void* v_ref,
                           const double* p_level, int nt, int nz, int64_t ncol, double* masso_steric,
                           double* masso_thermo, double* masso_halo, double* sums, double* partials, cudaStream_t st);

// fixed-order second reduction stage (defined in ml_api.cu): out[r] = sum_b partials[r][b]
int reduce_rows(const double* partials, int64_t nblk, double* out, int nrows, cudaStream_t st);


}  // namespace tma
}  // namespace ml
