/* momlevel_b200.h -- C ABI of libmomlevel_b200.so (sm_100a CUDA kernels for momlevel's
 * steric sea-level path).
 *
 * The reference (jkrasting/momlevel) is pure Python and has no FFI of its own; its
 * operator boundary is "numpy arrays in, numpy array out" (`eos.<name>.density(T,S,p)`,
 * `spice.flament.spice(T,S)`) applied through `xr.apply_ufunc` (src/momlevel/derived.py:624-630).
 * Each entry point below names the reference code it replaces.  INTEGRATION.md shows the
 * ctypes stub a momlevel maintainer would add to call them.
 *
 * Conventions (all entry points)
 *   - return 0 on success, <0 = ml_status argument error, >0 = cudaError_t;
 *     `ml_last_error()` returns a thread-local message for the last non-zero return
 *   - DEVICE entry points take device pointers owned by the caller (any allocator: torch,
 *     cudaMalloc, DLPack imports), are asynchronous on `stream` (a cudaStream_t passed as
 *     void*, NULL = legacy default stream) and use the calling thread's current device
 *   - HOST entry points (`*_host`) take host pointers, do their own staging and
 *     synchronise before returning
 *   - field layout is MOM6 / C order [t][z][y][x], x fastest; (y,x) is passed flattened as
 *     `ncol = ny*nx` water columns; NaN marks a missing (land) value
 *   - `dtype` is the storage type of the 3-D/4-D input fields (ML_F32 or ML_F64); all
 *     arithmetic and all outputs are fp64
 *   - no exceptions cross the boundary; no global state besides __constant__ tables
 */
#ifndef MOMLEVEL_B200_H
#define MOMLEVEL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ML_ABI_VERSION 1

typedef enum ml_status {
  ML_OK = 0,
  ML_ERR_NULL = -1,      /* required pointer is NULL */
  ML_ERR_SHAPE = -2,     /* non-positive or inconsistent extent */
  ML_ERR_DTYPE = -3,     /* dtype is not ML_F32 / ML_F64 */
  ML_ERR_EOS = -4,       /* unknown equation of state / function id */
  ML_ERR_MODE = -5,      /* unknown pressure mode / flag combination */
  ML_ERR_WORKSPACE = -6, /* workspace too small or NULL */
  ML_ERR_ALIGN = -7,     /* pointer not aligned to its element size */
  ML_ERR_DEVICE = -8     /* no CUDA device / not an sm_100 device */
} ml_status;

typedef enum ml_dtype { ML_F32 = 0, ML_F64 = 1 } ml_dtype;

/* momlevel.eos.<name>: util.eos_func_from_str (src/momlevel/util.py:227-249) */
typedef enum ml_eos { ML_EOS_WRIGHT = 0, ML_EOS_LINEAR = 1 } ml_eos;

/* func_name argument of eos_func_from_str */
typedef enum ml_eos_func {
  ML_FUNC_DENSITY = 0,    /* wright.py:23-50,   linear.py:26-58   */
  ML_FUNC_DRHO_DTEMP = 1, /* wright.py:53-85,   linear.py:61-85   */
  ML_FUNC_DRHO_DSAL = 2,  /* wright.py:88-119,  linear.py:88-110  */
  ML_FUNC_ALPHA = 3,      /* wright.py:122-142, linear.py:113-136 */
  ML_FUNC_BETA = 4        /* wright.py:145-165, linear.py:139-162 */
} ml_eos_func;

/* how the pressure operand of ml_eos_eval broadcasts */
typedef enum ml_pmode {
  ML_P_SCALAR = 0,    /* one value (p[0]) for every point                   */
  ML_P_PER_LEVEL = 1, /* p[nz], what steric.py:96 builds from z_l           */
  ML_P_FULL = 2       /* p has the full [nouter][nz][ncol] shape            */
} ml_pmode;

/* which fused kernel family a launch used; see ml_last_path() */
typedef enum ml_path { ML_PATH_NONE = 0, ML_PATH_DIRECT = 1, ML_PATH_TMA = 2 } ml_path;

int ml_version(void);
const char* ml_last_error(void);
/* kernel family chosen by the most recent steric launch on this thread (ml_path) */
int ml_last_path(void);
/* number of kernels this library has launched from the calling thread (monotonic) */
int64_t ml_launch_count(void);
/* force ML_PATH_DIRECT (1) / allow ML_PATH_TMA (0) for this thread; 2 = TMA family without the one-pass
 * three-height kernels of the *_variants entry points (A/B); returns previous */
int ml_set_force_direct(int on);
/* Per-column pressure offset for this thread's next calls, until cleared with (NULL, 0): `patm` given as a 2-D
 * field instead of a scalar (src/momlevel/steric.py:96 and reference.py:54 broadcast `z_l * 1e4 + patm` by
 * dimension name).  p_col is a DEVICE array [ncol] of fp64; while it is set, ml_reference_state,
 * ml_steric_local(_selfref / _variants), ml_steric_global and ml_delta_rho(_annual) evaluate the EOS at
 * p_level[z] + p_col[col] and take the plain-load kernel family (ML_PATH_DIRECT); a call whose ncol differs
 * returns ML_ERR_SHAPE.  The *_host entry points do not read it. */
int ml_set_column_pressure(const double* p_col, int64_t ncol);
/* time steps per register chunk of the one-pass three-height kernel (4, 6, 8 or 12; 0 = default) for this
 * thread; a tuning knob for experiments and tests -- the results do not depend on it; returns previous */
int ml_set_variants_chunk(int tc);

/* ---------------------------------------------------------------------------------------
 * ml_eos_eval -- elementwise equation of state, fp64 out.
 * Replaces eos.wright.* / eos.linear.* as applied by derived.calc_rho
 * (src/momlevel/derived.py:597-639) and calc_alpha/calc_beta (:74-159).
 *   T, S      [nouter][nz][ncol] of `dtype`; if t_bcast / s_bcast is non-zero that operand
 *             is [nz][ncol] and is broadcast over nouter (thermosteric / halosteric,
 *             steric.py:115-121)
 *   p         fp64, shape per `pmode`
 *   out       [nouter][nz][ncol] fp64
 * ------------------------------------------------------------------------------------- */
int ml_eos_eval(int eos, int func, int dtype, const void* T, const void* S, int t_bcast,
                int s_bcast, const double* p, int pmode, int64_t nouter, int64_t nz,
                int64_t ncol, double* out, void* stream);

/* ---------------------------------------------------------------------------------------
 * ml_flament_spice -- Flament (2002) spiciness, elementwise, fp64 out.
 * Replaces spice.flament.spice (src/momlevel/spice/flament.py:43-95) as applied by
 * derived.calc_spice (src/momlevel/derived.py:669-711).  A point with an infinite or NaN
 * T or S, or whose powers overflow, is NaN, as in the reference (its power-table sum meets inf - inf).
 * ------------------------------------------------------------------------------------- */
int ml_flament_spice(int dtype, const void* T, const void* S, int64_t n, double* out,
                     void* stream);

/* ---------------------------------------------------------------------------------------
 * ml_calc_dz -- partial-bottom-cell thickness, out[nz][ncol] fp64.
 * Replaces derived.calc_dz (src/momlevel/derived.py:249-325); the sign asserts
 * (:284-292) stay on the host.  `has_bottom` = 0 means bottom=None.
 * ------------------------------------------------------------------------------------- */
int ml_calc_dz(const double* z_i, const double* deptho, double top, double bottom,
               int has_bottom, int fraction, int64_t nz, int64_t ncol, double* out,
               void* stream);

/* bytes of device scratch the reducing entry points need (block partials) */
size_t ml_workspace_bytes(int64_t nt, int64_t nz, int64_t ncol);

/* ---------------------------------------------------------------------------------------
 * ml_reference_state -- rho_ref = EOS(T0,S0,p) plus the two global sums, one pass.
 * Replaces reference.setup_reference_state (src/momlevel/reference.py:71-80) =
 * calc_rho + calc_volo (derived.py:787-789) + calc_masso (derived.py:435-438).
 *   T0,S0,V0  [nz][ncol] of `dtype` (the time_index slab)
 *   p_level   [nz] fp64
 *   rho_ref   [nz][ncol] fp64 out
 *   sums      device fp64[2] out: {volo = nansum(V0), masso = nansum(rho_ref*V0)}
 * ------------------------------------------------------------------------------------- */
int ml_reference_state(int eos, int dtype, const void* T0, const void* S0, const void* V0,
                       const double* p_level, int64_t nz, int64_t ncol, double* rho_ref,
                       double* sums, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * ml_steric_local -- fused EOS -> delta_rho -> clipped dz -> column integral.
 * Replaces the local branch of steric.steric (src/momlevel/steric.py:128,150-166) and the
 * inline use of derived.calc_dz (derived.py:295-318, top=0, bottom=None).
 *   T, S        [nt][nz][ncol] of `dtype` (or [nz][ncol] when *_bcast, see ml_eos_eval)
 *   rho_ref     [nz][ncol] fp64           reference["rho"]
 *   v_ref       [nz][ncol] of `vref_dtype` reference["volcello"]; NaN = dry cell
 *   z_i         [nz+1] fp64, deptho [ncol] fp64 (NaN = land -> 0, derived.py:295)
 *   p_level     [nz] fp64
 *   neg_inv_rhozero = -1.0/rhozero (steric.py:163)
 *   eta         [nt][ncol] fp64 out; NaN where v_ref[0][col] is NaN (steric.py:166)
 *   delta_rho   [nt][nz][ncol] fp64 out, or NULL to skip the 4-D field
 * ------------------------------------------------------------------------------------- */
int ml_steric_local(int eos, int dtype, const void* T, const void* S, int t_bcast, int s_bcast,
                    const double* rho_ref, const void* v_ref, int vref_dtype, const double* z_i,
                    const double* deptho, const double* p_level, double neg_inv_rhozero,
                    int64_t nt, int64_t nz, int64_t ncol, double* eta, double* delta_rho,
                    void* stream);

/* ---------------------------------------------------------------------------------------
 * ml_delta_rho -- the 4-D density anomaly on its own:
 *   delta_rho = where(v_ref notnull, rho(T,S,p) - rho_ref, NaN)   (src/momlevel/steric.py:151-158)
 * The reference always materialises this field; here the fused kernels integrate it without
 * storing it and this entry point produces it when a caller reads result["delta_rho"].
 *   delta_rho   [nt][nz][ncol] fp64 out; other arguments as ml_steric_local
 * ------------------------------------------------------------------------------------- */
int ml_delta_rho(int eos, int dtype, const void* T, const void* S, int t_bcast, int s_bcast,
                 const double* rho_ref, const void* v_ref, int vref_dtype, const double* p_level,
                 int64_t nt, int64_t nz, int64_t ncol, double* delta_rho, void* stream);

/* ---------------------------------------------------------------------------------------
 * ml_delta_rho_annual -- the density anomaly of ml_delta_rho averaged over each year of 12 monthly
 * steps with the weights of util.annual_average (src/momlevel/util.py:84-87, applied to the result
 * Dataset by steric.py:181-182): sum_m w_m d_m / sum_m w_m per cell, missing months skipped and the
 * weights renormalised (xarray's weighted(...).mean).  The monthly 4-D field is never stored.
 *   weights           device fp64[nt] (days in month); nt must be a multiple of 12
 *   delta_rho_annual  [nt/12][nz][ncol] fp64 out
 * ------------------------------------------------------------------------------------- */
int ml_delta_rho_annual(int eos, int dtype, const void* T, const void* S, int t_bcast, int s_bcast,
                        const double* rho_ref, const void* v_ref, int vref_dtype,
                        const double* p_level, const double* weights, int64_t nt, int64_t nz,
                        int64_t ncol, double* delta_rho_annual, void* stream);

/* ---------------------------------------------------------------------------------------
 * ml_steric_local_selfref -- ml_reference_state + ml_steric_local in one pass when the
 * reference state is the first time step of the dataset itself, which is what
 * steric.steric does when no `reference` is supplied (src/momlevel/steric.py:105-107 ->
 * reference.py:60-80 with time_index = 0).  rho_ref is evaluated from the step-0 rows that
 * the column integral reads anyway, stored for the caller and reduced into volo / masso,
 * so T and S cross HBM once for the whole call.
 *   T, S        as ml_steric_local; a broadcast operand IS the reference slab of that field
 *   v_ref       [nz][ncol] volcello at step 0
 *   rho_ref     [nz][ncol] fp64 out;  sums device fp64[2] out {volo, masso}
 *               rho_ref may be NULL when the caller does not need the field and one fused chunk serves the
 *               call (16-byte aligned fields with volcello stored alike, ncol >= 256, nt <= 12 for fp32
 *               storage or <= 6 for fp64): the store is
 *               7 % of the traffic of a 12-step call, and ml_reference_state produces the field on demand.
 *               Any other call with rho_ref == NULL returns ML_ERR_NULL.
 * ------------------------------------------------------------------------------------- */
int ml_steric_local_selfref(int eos, int dtype, const void* T, const void* S, int t_bcast,
                            int s_bcast, const void* v_ref, int vref_dtype, const double* z_i,
                            const double* deptho, const double* p_level, double neg_inv_rhozero,
                            int64_t nt, int64_t nz, int64_t ncol, double* eta, double* rho_ref,
                            double* sums, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * ml_steric_local_variants -- steric, thermosteric and halosteric height in one call.
 * steric.py:115-121 selects per call which operand of the EOS is held at its reference value;
 * BASELINE config 2 asks for all three:
 *   rho(T,S) - rho_ref,  rho(T,S_ref) - rho_ref,  rho(T_ref,S) - rho_ref        (steric.py:128,151-153)
 * Fields that suit the TMA family (fp32, 16-byte aligned, ncol % 4 == 0, ncol >= 256) take ONE pass for
 * all the heights asked for (csrc/ml_tma3.cu: T and S cross HBM once, a point's three densities come from
 * the same two shared-memory words; bit-identical to the single-height kernels); anything else, or a call
 * that asks for one height only, runs one single-height launch per height.  ml_set_force_direct(2) keeps
 * the TMA family but turns the one-pass kernel off (A/B).
 *   T, S          [nt][nz][ncol] of `dtype`
 *   T_ref, S_ref  [nz][ncol] of `dtype`: reference["thetao"], reference["so"]; when they are step 0
 *                 of T, S themselves (the same pointers) the heights of step 0 are exactly zero
 *   rho_ref       [nz][ncol] fp64 in, or NULL: evaluate it from T_ref, S_ref (reference.py:71-80),
 *                 store it in rho_ref_out [nz][ncol] and put {volo, masso} into sums (workspace as
 *                 for ml_reference_state).  rho_ref_out may be NULL when the one-pass kernel serves a
 *                 self-reference call (it needs only the sums); any other call with both NULL returns
 *                 ML_ERR_NULL
 *   eta_*         [nt][ncol] fp64 out each; a NULL pointer skips that variant's store
 * ------------------------------------------------------------------------------------- */
int ml_steric_local_variants(int eos, int dtype, const void* T, const void* S, const void* T_ref,
                             const void* S_ref, const double* rho_ref, const void* v_ref,
                             int vref_dtype, const double* z_i, const double* deptho,
                             const double* p_level, double neg_inv_rhozero, int64_t nt, int64_t nz,
                             int64_t ncol, double* eta_steric, double* eta_thermosteric,
                             double* eta_halosteric, double* rho_ref_out, double* sums,
                             void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * ml_steric_local_layers -- the local height of ml_steric_local split by depth layer, from one pass:
 *   eta[t][b][col] = coef * sum_z calc_dz(top=edges[b], bottom=edges[b+1]) * (rho - rho_ref),
 * masked where v_ref at the surface is missing (NaN in every layer); a layer wholly below a wet column's
 * sea floor is 0.0.  calc_dz is derived.calc_dz (derived.py:295-318), so at a partial bottom cell that
 * straddles an inner edge the layers add up to more than the full column, as in the reference.
 *   edges       HOST pointer to nlayers + 1 strictly increasing values >= 0; the last may be +inf
 *               (to the sea floor).  1 <= nlayers <= ML_MAX_LAYERS; anything else returns ML_ERR_SHAPE
 *   eta         [nt][nlayers][ncol] fp64 out
 * Other arguments as ml_steric_local (no delta_rho output); reads the thread's column pressure like it.
 * nlayers == 1 with edges {0, +inf} is bit-identical to ml_steric_local.
 * ------------------------------------------------------------------------------------- */
#define ML_MAX_LAYERS 8
int ml_steric_local_layers(int eos, int dtype, const void* T, const void* S, int t_bcast, int s_bcast,
                           const double* rho_ref, const void* v_ref, int vref_dtype, const double* z_i,
                           const double* deptho, const double* p_level, double neg_inv_rhozero,
                           const double* edges, int nlayers, int64_t nt, int64_t nz, int64_t ncol,
                           double* eta, void* stream);

/* ---------------------------------------------------------------------------------------
 * ml_steric_local_layers_variants -- the steric, thermosteric and halosteric heights of
 * ml_steric_local_variants split by depth layer as ml_steric_local_layers, in one call: how much of a
 * layer's change is warming and how much is freshening.
 * Fields that suit the one-pass kernel of ml_steric_local_variants (fp32, 16-byte aligned, ncol % 4 == 0,
 * ncol >= 256) take ONE pass over T and S for all the heights asked for (csrc/ml_tma3.cu), each bit-identical
 * to its ml_steric_local_layers launch; anything else, a column pressure (ml_set_column_pressure) or a call
 * that asks for one height only runs one ml_steric_local_layers per height.  ml_set_force_direct(2) turns
 * the one-pass kernel off (A/B).
 *   T, S          [nt][nz][ncol] of `dtype`
 *   T_ref, S_ref  [nz][ncol] of `dtype`: reference["thetao"], reference["so"]
 *   rho_ref       [nz][ncol] fp64: reference["rho"] (ml_reference_state or a supplied reference); required
 *   edges         HOST pointer, nlayers as ml_steric_local_layers (ML_ERR_SHAPE otherwise)
 *   eta_*         [nt][nlayers][ncol] fp64 out each; a NULL pointer skips that variant; at least one is
 *                 required (ML_ERR_NULL)
 * Other arguments as ml_steric_local_layers; reads the thread's column pressure like it.
 * ------------------------------------------------------------------------------------- */
int ml_steric_local_layers_variants(int eos, int dtype, const void* T, const void* S, const void* T_ref,
                                    const void* S_ref, const double* rho_ref, const void* v_ref,
                                    int vref_dtype, const double* z_i, const double* deptho,
                                    const double* p_level, double neg_inv_rhozero, const double* edges,
                                    int nlayers, int64_t nt, int64_t nz, int64_t ncol, double* eta_steric,
                                    double* eta_thermosteric, double* eta_halosteric, void* stream);

/* ---------------------------------------------------------------------------------------
 * ml_steric_local_profile -- the area-weighted steric, thermosteric and halosteric height change by
 * model level, from one pass over T and S:
 *   prof_v[t][z] = neg_inv_rhozero * nansum_col( m * w * dz * delta_rho_v[t][z][col] )
 * with delta_rho_v the anomaly of ml_delta_rho for variant v (steric.py:115-121, :151-153), dz the
 * thickness of derived.calc_dz (derived.py:295-318, top=0, bottom=None), m = v_ref[0][col] present (the
 * surface mask of steric.py:166) and w = weights[col] (a NaN weight counts as 0).  A NaN term (a hole at
 * a wet cell, a missing reference volume) is skipped.  Summed over z this is nansum_col(w * eta) of
 * ml_steric_local's height eta: dividing by nansum(w) is left to the caller.
 * fp32 fields with 16-byte aligned rows (ncol % 4 == 0) stream through a shared-memory ring
 * (csrc/ml_stream.cu); fp64 storage, ragged rows, a column pressure (ml_set_column_pressure) or
 * ml_set_force_direct(1) take the plain-load kernel, which gives the same bits.  All the heights asked
 * for come from one pass; each is bit-identical to a call that asks for it alone, and
 * ml_set_force_direct(2) runs one launch per height (A/B).  Sums run in a fixed order: reproducible.
 *   T, S          [nt][nz][ncol] of `dtype`
 *   T_ref, S_ref  [nz][ncol] of `dtype`: reference["thetao"], reference["so"]
 *   rho_ref       [nz][ncol] fp64: reference["rho"]
 *   weights       [ncol] fp64 (device), e.g. areacello or areacello * basin mask
 *   prof_*        [nt][nz] fp64 out each (device); a NULL pointer skips that variant; at least one is
 *                 required (ML_ERR_NULL)
 *   workspace     ml_profile_workspace_bytes(number of prof_* given, nt, nz, ncol) bytes
 * Other arguments as ml_steric_local.  Every argument error returns before any launch.
 * ------------------------------------------------------------------------------------- */
size_t ml_profile_workspace_bytes(int nvariants, int64_t nt, int64_t nz, int64_t ncol);
int ml_steric_local_profile(int eos, int dtype, const void* T, const void* S, const void* T_ref,
                            const void* S_ref, const double* rho_ref, const void* v_ref,
                            int vref_dtype, const double* z_i, const double* deptho,
                            const double* weights, const double* p_level, double neg_inv_rhozero,
                            int64_t nt, int64_t nz, int64_t ncol, double* prof_steric,
                            double* prof_thermosteric, double* prof_halosteric, void* workspace,
                            size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * ml_steric_local_region_profile -- ml_steric_local_profile for every region of a region map at once
 * (basins side by side), from one pass over T and S:
 *   prof_v[r][t][z] = neg_inv_rhozero * nansum_{col: region[col] == r}( m * w * dz * delta_rho_v[t][z][col] )
 * Region r is exactly what ml_steric_local_profile gives with weights where(region == r, w, 0), and a map that
 * puts every column in region 0 gives exactly its one-region result.  Every density is evaluated once per step
 * whatever the number of regions; a warp of 32 x 8 columns spread over many regions sums once per region it
 * touches.  Routes and switches are those of ml_steric_local_profile (the ring for eligible fp32 fields, the
 * plain-load kernel with the same bits otherwise, ml_set_force_direct(2) one launch per variant).
 *   region        [ncol] int8 (device): the region index of each column, in [0, nregions); any other value
 *                 (e.g. -1) puts the column in no region.  NULL returns ML_ERR_NULL.
 *   nregions      1 <= nregions <= ML_MAX_REGIONS; anything else returns ML_ERR_SHAPE
 *   prof_*        [nregions][nt][nz] fp64 out each (device): numerators only, the caller divides by each
 *                 region's nansum(w); a NULL pointer skips that variant; at least one is required (ML_ERR_NULL)
 *   workspace     at least one step: ml_region_profile_workspace_bytes(number of prof_* given, nregions, 1, nz,
 *                 ncol) bytes (ML_ERR_WORKSPACE otherwise).  The time axis runs in chunks of as many steps as
 *                 the workspace holds; the bits of a step do not depend on the chunks.
 * Other arguments as ml_steric_local_profile.  Every argument error returns before any launch.
 * ------------------------------------------------------------------------------------- */
#define ML_MAX_REGIONS 15
size_t ml_region_profile_workspace_bytes(int nvariants, int nregions, int64_t nt, int64_t nz, int64_t ncol);
int ml_steric_local_region_profile(int eos, int dtype, const void* T, const void* S, const void* T_ref,
                                   const void* S_ref, const double* rho_ref, const void* v_ref, int vref_dtype,
                                   const double* z_i, const double* deptho, const double* weights,
                                   const int8_t* region, int nregions, const double* p_level,
                                   double neg_inv_rhozero, int64_t nt, int64_t nz, int64_t ncol,
                                   double* prof_steric, double* prof_thermosteric, double* prof_halosteric,
                                   void* workspace, size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * ml_steric_local_zonal_profile -- ml_steric_local_profile for every grid row at once (a latitude-depth
 * section), from one pass over T and S:
 *   prof_v[t][z][j] = neg_inv_rhozero * nansum_i( m * w * dz * delta_rho_v[t][z][j][i] )
 * Row j is bit for bit what ml_steric_local_profile gives on the fields, reference slabs, deptho, weights and
 * column pressure of row j alone (sliced to [..., j:j+1, :], contiguous, ncol = nx): a (level, row) is split into
 * the same 2048-column sub-tiles, summed in the same order into the same per-warp partials.  Routes and switches
 * are those of ml_steric_local_profile (the ring for fp32 fields with nx % 4 == 0 and 16-byte aligned bases, the
 * plain-load kernel with the same bits otherwise, ml_set_force_direct(2) one launch per variant).
 *   T, S          [nt][nz][ny][nx] of `dtype`; T_ref, S_ref, rho_ref, v_ref [nz][ny][nx]
 *   deptho, weights [ny][nx] fp64 (device); a column pressure (ml_set_column_pressure) has ny * nx values
 *   prof_*        [nt][nz][ny] fp64 out each (device): numerators only, the caller divides row j by the row's
 *                 nansum(w); a NULL pointer skips that variant; at least one is required (ML_ERR_NULL)
 *   workspace     at least one step: ml_zonal_profile_workspace_bytes(number of prof_* given, 1, nz, ny, nx)
 *                 bytes (ML_ERR_WORKSPACE otherwise).  The time axis runs in chunks of as many steps as the
 *                 workspace holds; the bits of a step do not depend on the chunks.
 * Other arguments as ml_steric_local_profile.  Every argument error returns before any launch.
 * ------------------------------------------------------------------------------------- */
size_t ml_zonal_profile_workspace_bytes(int nvariants, int64_t nt, int64_t nz, int64_t ny, int64_t nx);
int ml_steric_local_zonal_profile(int eos, int dtype, const void* T, const void* S, const void* T_ref,
                                  const void* S_ref, const double* rho_ref, const void* v_ref, int vref_dtype,
                                  const double* z_i, const double* deptho, const double* weights,
                                  const double* p_level, double neg_inv_rhozero, int64_t nt, int64_t nz,
                                  int64_t ny, int64_t nx, double* prof_steric, double* prof_thermosteric,
                                  double* prof_halosteric, void* workspace, size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * ml_steric_global -- fused EOS -> sum_{z,col} rho * v_ref per time step.
 * Replaces calc_masso(rho, reference["volcello"]) in the global branch
 * (src/momlevel/steric.py:135, derived.py:435-438); the ln() formula (steric.py:136-142)
 * is host arithmetic on nt doubles.
 *   masso       device fp64[nt] out
 * ------------------------------------------------------------------------------------- */
int ml_steric_global(int eos, int dtype, const void* T, const void* S, int t_bcast, int s_bcast,
                     const void* v_ref, int vref_dtype, const double* p_level, int64_t nt,
                     int64_t nz, int64_t ncol, double* masso, void* workspace,
                     size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * ml_steric_global_variants -- the masses of the global steric, thermosteric and halosteric
 * series in one call.  Replaces calc_masso(rho, reference["volcello"]) of the global branch
 * (src/momlevel/steric.py:134-135, derived.py:435-438) for the three variants of steric.py:115-121:
 *   sum rho(T,S) V,   sum rho(T,S_ref) V,   sum rho(T_ref,S) V        per step, V = reference volcello
 * Fields that suit the TMA family (fp32, 16-byte aligned, ncol % 4 == 0, ncol >= 256) take ONE pass for
 * all the masses asked for (csrc/ml_tma3.cu), each bit-identical to one ml_steric_global launch; anything
 * else, a column pressure (ml_set_column_pressure) or a call that asks for one mass only runs one
 * ml_steric_global per mass.  ml_set_force_direct(2) turns the one-pass kernel off.
 *   T, S          [nt][nz][ncol] of `dtype`
 *   T_ref, S_ref  [nz][ncol] of `dtype`: reference["thetao"], reference["so"]; when they are T, S themselves
 *                 (the same pointers: the reference is step 0, steric.py:105-107) `sums` gets {volo, masso}
 *                 of the reference state (reference.py:74-80), and must be NULL otherwise
 *   v_ref         [nz][ncol] reference volcello of `vref_dtype`
 *   masso_*       device fp64[nt] out each; a NULL pointer skips that variant; at least one is required
 *   sums          device fp64[2] out (self-reference calls only)
 *   workspace     ml_workspace_bytes(3 * nt, nz, ncol) bytes
 * ------------------------------------------------------------------------------------- */
int ml_steric_global_variants(int eos, int dtype, const void* T, const void* S, const void* T_ref,
                              const void* S_ref, const void* v_ref, int vref_dtype,
                              const double* p_level, int64_t nt, int64_t nz, int64_t ncol,
                              double* masso_steric, double* masso_thermosteric,
                              double* masso_halosteric, double* sums, void* workspace,
                              size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * ml_calc_masso -- skipna sums of a field that already exists: out[r] = sum_i rho[r][i] * volcello[i].
 * Replaces derived.calc_masso (src/momlevel/derived.py:414-444: `(rho * volcello).sum(...)` per time step, without
 * the rho * volcello temporary) and, with volcello == NULL, derived.calc_volo (derived.py:769-795:
 * `volcello.sum()`, the field passed as `rho` with nrows = 1).  Two fixed-order stages: bitwise reproducible.
 *   rho        device [nrows][n] of `dtype`;  volcello device [n] of `w_dtype` or NULL
 *   out        device fp64[nrows];  workspace: nrows * 1184 doubles are always enough
 *   nrows      any count up to INT32_MAX: more than 65535 rows (a time axis of 3-hourly output over 23 years)
 *              are launched in chunks of 65535; a row's result does not depend on nrows or on its chunk.
 * ------------------------------------------------------------------------------------- */
int ml_calc_masso(int dtype, const void* rho, int w_dtype, const void* volcello, int64_t nrows, int64_t n,
                  double* out, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * ml_steric_local_host -- the same computation as reference_state + steric_local for
 * variant="steric" on HOST buffers: time steps are staged to the device through two
 * pinned/registered windows so the copy of step k+1 overlaps the kernels of step k.
 * This is the end-to-end call bench.py times as `e2e`.
 *   T, S        host [nt][nz][ncol] of `dtype`;  v0 host [nz][ncol] of `dtype`
 *               (volcello at time_index 0); reference state = time step 0 (reference.py:60-68)
 *   eta         host [nt][ncol] fp64 out
 *   rho_ref_out host [nz][ncol] fp64 out or NULL; sums_out host fp64[2] {volo, masso}
 *   steps_per_window  time steps per staging window (>=1)
 * ------------------------------------------------------------------------------------- */
int ml_steric_local_host(int eos, int dtype, const void* T, const void* S, const void* v0,
                         const double* z_i, const double* deptho, const double* p_level,
                         double neg_inv_rhozero, int64_t nt, int64_t nz, int64_t ncol,
                         int steps_per_window, double* eta, double* rho_ref_out,
                         double* sums_out);

/* ---------------------------------------------------------------------------------------
 * ml_steric_global_host -- the masses of ml_steric_global for fields in HOST memory (a daily global
 * series does not fit in HBM: BASELINE config 4 is 1.4 TB), streamed through the same two windows.
 *   T, S    host [nt][nz][ncol] of `dtype`;  v_ref host [nz][ncol] of `dtype` (reference["volcello"])
 *   masso   host fp64[nt] out; the ln() formula of steric.py:136-142 stays with the caller
 * ------------------------------------------------------------------------------------- */
int ml_steric_global_host(int eos, int dtype, const void* T, const void* S, const void* v_ref,
                          const double* p_level, int64_t nt, int64_t nz, int64_t ncol,
                          int steps_per_window, double* masso);

/* ---------------------------------------------------------------------------------------
 * ml_steric_local_variants_host -- ml_steric_local_host that also returns the thermosteric and
 * halosteric heights: the fields cross PCIe once (the transfer is what bounds the host path) and each
 * window is integrated three times on the device.  eta_thermosteric / eta_halosteric are host
 * [nt][ncol] fp64 outputs and may be NULL; the other arguments are those of ml_steric_local_host.
 * ------------------------------------------------------------------------------------- */
int ml_steric_local_variants_host(int eos, int dtype, const void* T, const void* S, const void* v0,
                                  const double* z_i, const double* deptho, const double* p_level,
                                  double neg_inv_rhozero, int64_t nt, int64_t nz, int64_t ncol,
                                  int steps_per_window, double* eta_steric, double* eta_thermosteric,
                                  double* eta_halosteric, double* rho_ref_out, double* sums_out);

/* ---------------------------------------------------------------------------------------
 * ml_host_stream_* -- the host path for fields that arrive block by block.
 * The reference works on dask-backed Datasets (src/momlevel/derived.py:624-630 `dask="allowed"`;
 * examples/example.ipynb cell 4 opens the model output with chunks={"time": 1, ...}): the fields never exist as
 * one array.  begin() takes everything that does not depend on time, push() one block of consecutive time
 * steps -- staged, packed and copied like a window of ml_steric_local_host while the previous block computes --
 * and finish() waits for the tail.  ml_steric_local_host, ml_steric_local_variants_host and
 * ml_steric_global_host are begin + one push per window + finish.
 *
 *   domain        ML_DOMAIN_LOCAL: heights eta[nt_block][ncol] per push (steric.py:150-166);
 *                 ML_DOMAIN_GLOBAL: masses masso[nt_block] per push (steric.py:135)
 *   variants      bit 0 steric, bit 1 thermosteric, bit 2 halosteric (steric.py:115-121); at least one
 *   v_ref         host [nz][ncol] of vref_dtype: reference["volcello"]; must stay valid until the first push returns
 *   T_ref, S_ref, rho_ref   host reference slabs / density of a SUPPLIED reference (steric.py:98-103), or all NULL:
 *                 the reference state is step 0 of the first block (steric.py:105-107, reference.py:60-80).
 *                 rho_ref is needed by the local domain, T_ref / S_ref by the thermo- / halosteric variants
 *   z_i, deptho   host, local domain only;  p_level host [nz]
 *   max_block_steps   upper bound of nt_block (sizes the two device windows)
 *   want_reference    bit 0: finish() will be asked for rho_ref_out (every row then crosses as it is);
 *                     bit 1: global domain with a self-reference: evaluate volo / masso from step 0 (sums_out)
 * push(): T_block, S_block host [nt_block][nz][ncol] of `dtype` (pinned memory keeps the copies asynchronous;
 *   pageable memory is staged by the library's own threads); out_* host [nt_block][ncol] (local) or [nt_block]
 *   (global) for the variants asked for.  The block's memory may be reused once the NEXT push (or finish) has
 *   returned; the outputs are complete when finish() returns.
 * finish(): rho_ref_out host [nz][ncol] or NULL; sums_out host fp64[2] {volo, masso} or NULL; frees the stream.
 * abort(): drains the device and frees the stream (after an error, or to give up).
 * A stream belongs to the thread that began it; a thread has one open stream at a time.
 * ------------------------------------------------------------------------------------- */
#define ML_DOMAIN_LOCAL 0
#define ML_DOMAIN_GLOBAL 1
int ml_host_stream_begin(int domain, int eos, int dtype, int variants, const void* v_ref, int vref_dtype,
                         const void* T_ref, const void* S_ref, const double* rho_ref, const double* z_i,
                         const double* deptho, const double* p_level, double neg_inv_rhozero, int64_t nz,
                         int64_t ncol, int64_t max_block_steps, int want_reference, void** stream_out);
int ml_host_stream_push(void* stream, const void* T_block, const void* S_block, int64_t nt_block,
                        double* out_steric, double* out_thermosteric, double* out_halosteric);
int ml_host_stream_finish(void* stream, double* rho_ref_out, double* sums_out);
int ml_host_stream_abort(void* stream);

/* Frees the device staging buffers, streams and events that the *_host entry points keep per
 * host thread between calls. */
int ml_host_release(void);

/* ---------------------------------------------------------------------------------------
 * Wet-cell packing of the host path.  The reference never uses T or S where the reference
 * volcello is missing: delta_rho is NaN there (src/momlevel/steric.py:151-153), the column sum
 * skips it (:163) and so do volo / masso (derived.py:435-438, 787-789).  ml_steric_local_host,
 * ml_steric_local_variants_host and ml_steric_global_host therefore move a level row either as it is (DMA straight from the
 * caller's buffer) or as its present cells only (compressed by host threads into pinned staging,
 * expanded on the device with NaN in the absent cells), whichever side -- PCIe or the host cores --
 * has time left; the heights are bit-identical either way.  fp32 fields only; a call that asks for
 * rho_ref_out moves every row as it is (rho_ref is defined on absent cells too).  Fields in PAGEABLE memory
 * (plain malloc / numpy; a DMA from it is a slow synchronous bounce through the driver) send every row through the
 * packers and the pinned staging, full rows included, and volcello and the heights cross through pinned
 * buffers of the library's own, unless mode is 0.
 *   ml_host_set_packing(mode, threads)  mode 0 = never pack, 1 = balance dynamically (default),
 *                                       2 = pack every row that has absent cells, 3 = as 1 but the packed
 *                                       rows wait for the copy engine in a six-row ring of pinned memory
 *                                       written with ordinary stores (meant to stay in the last-level cache,
 *                                       so that the packed bytes never touch DRAM), 4 = as 3 but a row goes
 *                                       as it is only while no packed row is waiting for the copy stream
 *                                       (modes 3 and 4 measured slower than 1: profiles/r02_experiments.md).
 *                                       threads <= 0 leaves the number of packing threads to the library: it starts
 *                                       from half the calling thread's CPU affinity count divided by the ranks on the
 *                                       host (LOCAL_WORLD_SIZE) and, in mode 1, times every window on the copy stream
 *                                       and settles on the fastest of {that, none, twice, half} for this machine and
 *                                       load -- packing has to beat plain copies by 6 % to be chosen, and the ranks of
 *                                       a host (LOCAL_WORLD_SIZE > 1 under torchrun) choose from the element-wise
 *                                       maximum of their tables, i.e. together and for the slowest of them -- (kept
 *                                       per host thread between calls, tried afresh every 256 windows);
 *                                       a call that starts while "none" is in front moves every row as it is and does
 *                                       not build the presence index either.
 *                                       Applies to the calling host thread.
 *   ml_host_last_packed_fraction()      share of the level rows of the last host call that crossed packed
 *   ml_host_last_h2d_bytes()            bytes the last host call of this thread copied host -> device
 *   ml_host_last_timings(ms4)           host wall time of the last ml_steric_local*_host call, milliseconds:
 *                                       presence index (made on the device behind the upload of volcello and read
 *                                       back: k_presence_words / k_presence_before), windows, drain (kernels of the
 *                                       last window + read-back), whole call
 * The two loops underneath are exported for testing (csrc/ml_pack.cpp, no CUDA inside):
 *   ml_pack_index_rows  v [nrows][ncol] fp32 -> words / before [nrows][ceil(ncol/32)]: bit i of a word
 *                       = column 32 g + i is not NaN; before = present cells of the row in front of the
 *                       group; row_count [nrows]; returns the total
 *   ml_pack_rows        present cells of groups [g0, g1) of one T row and one S row, written to
 *                       t_out / s_out (the row's packed base) at offset before[g0]
 *   ml_pack_rows_cached the same with ordinary instead of non-temporal stores (mode 3)
 *   ml_pack_simd        512 when the AVX-512 bodies are in use, 0 for the scalar ones
 * ------------------------------------------------------------------------------------- */
int ml_host_set_packing(int mode, int threads);
double ml_host_last_packed_fraction(void);
/* packing threads of the calling thread's last window (what the tuner of ml_host_set_packing(1, 0) has settled on) */
int ml_host_last_pack_threads(void);
uint64_t ml_host_last_h2d_bytes(void);
int ml_host_last_timings(double* ms4);
/* Test entry of the table the ranks of a host share for that decision (POSIX shared memory named after the job's
 * MASTER_ADDR / MASTER_PORT / TORCHELASTIC_RUN_ID and the user id): attaches to a made-up job `port` as `rank` of
 * `ranks`, publishes ms4 (ms per step of {default, none, twice, half}; negative = unknown), waits up to wait_ms for the
 * others, writes the element-wise maximum over the ranks to combined4 (unknown anywhere = unknown) and returns the
 * number of ranks it saw.  No CUDA inside. */
int ml_host_tuner_share_selftest(const char* port, int rank, int ranks, int64_t nz, int64_t ncol, const double* ms4,
                                 double* combined4, int wait_ms);
uint64_t ml_pack_index_rows(const float* v, int64_t nrows, int64_t ncol, uint32_t* words,
                            uint32_t* before, uint64_t* row_count);
void ml_pack_rows(const float* t_row, const float* s_row, const uint32_t* words, const uint32_t* before,
                  int64_t g0, int64_t g1, int64_t ncol, float* t_out, float* s_out);
void ml_pack_rows_cached(const float* t_row, const float* s_row, const uint32_t* words, const uint32_t* before,
                         int64_t g0, int64_t g1, int64_t ncol, float* t_out, float* s_out);
int ml_pack_simd(void);

/* =======================================================================================
 * Stratification diagnostics that share the vertical sweep of the steric path (csrc/ml_strat.cu).
 * T, S are [nouter][nz][ncol] of `dtype`, z_l is [nz] fp64 (3 <= nz <= 512: the vertical
 * derivative is numpy.gradient(f, z_l, edge_order=2), what DataArray.differentiate evaluates).
 * `fill_mode` selects which cells adjust_negative_n2's `adjusted[0] = adjusted[0].fillna(1e-8)`
 * (src/momlevel/derived.py:63) touches: index 0 of the array's FIRST axis, i.e.
 *   0 = the surface level of every slab   (a 3-D field [z][y][x], passed with nouter = 1)
 *   k = every level of outer slabs [0, k), 1 <= k <= nouter: the outer slabs whose first index
 *       is 0, i.e. the product of the extents between the first axis and the level axis --
 *       1 for [t][z][y][x] (its first time step), nt for [member][t][z][y][x] (every time
 *       step of member 0), nx for a level-last [y][x][z] (the row y = 0, with ncol = 1).
 *   Any other value returns ML_ERR_MODE.
 * nouter has no upper limit: above 65535 slabs (the grid.y limit of one launch) the entry points
 * launch their kernel once per 65535 slabs, and the fill follows the slab index of the whole call.
 * ===================================================================================== */

/* ml_calc_n2 -- squared buoyancy frequency at cell centres, g * (alpha dT/dz - beta dS/dz) with
 * locally referenced pressure p = z_l * 1e4 + patm.
 * Replaces derived.calc_n2 without `interfaces` (src/momlevel/derived.py:391-411), including
 * adjust_negative=True (:409 -> :30-71).  out is [nouter][nz][ncol] fp64. */
int ml_calc_n2(int eos, int dtype, const void* T, const void* S, const double* z_l, double gravity,
               double patm, int adjust_negative, int fill_mode, int64_t nouter, int64_t nz,
               int64_t ncol, double* out, void* stream);

/* ml_adjust_negative_n2 -- Chelton et al. (1998) adjustment of an existing N2 field:
 * non-positive values are replaced by the last positive value above them in the column.
 * Replaces derived.adjust_negative_n2 (src/momlevel/derived.py:30-71). */
int ml_adjust_negative_n2(const double* n2, int fill_mode, int64_t nouter, int64_t nz, int64_t ncol,
                          double* out, void* stream);

/* ml_stability_angle -- Turner angle degrees(arctan((1 + R) / (1 - R))), R = beta dS/dz / (alpha dT/dz).
 * Replaces derived.calc_stability_angle (src/momlevel/derived.py:714-766); p_level is the
 * caller's pressure per level, [nz] fp64. */
int ml_stability_angle(int eos, int dtype, const void* T, const void* S, const double* p_level,
                       const double* z_l, int64_t nouter, int64_t nz, int64_t ncol, double* out,
                       void* stream);

/* ml_wave_speed -- first-baroclinic-mode gravity wave speed, sum_z sqrt(adjusted N2) dz / pi (skipna).
 * Replaces the arithmetic of derived.calc_wave_speed (src/momlevel/derived.py:821); the mask of
 * :822 is array bookkeeping done by the host.  n2 [nouter][nz][ncol], dz [nz][ncol],
 * out [nouter][ncol], all fp64. */
int ml_wave_speed(const double* n2, const double* dz, int fill_mode, int64_t nouter, int64_t nz,
                  int64_t ncol, double* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MOMLEVEL_B200_H */
