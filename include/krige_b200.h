/*
 * krige_b200.h — C ABI of libkrige_b200.so, the B200-native kriging execute() backend.
 *
 * This is the drop-in boundary for PyKrige's `execute(..., backend='cuda')`.
 * It replaces, one level higher (coordinates in, not dense a/bd matrices), the
 * reference's own native plug-in entry points:
 *
 *   _c_exec_loop(a_all, bd_all, mask, n, pars)                       src/pykrige/lib/cok.pyx:14-96
 *   _c_exec_loop_moving_window(a_all, bd_all, mask, bd_idx, n_max, pars)
 *                                                                    src/pykrige/lib/cok.pyx:98-193
 * and the Python bodies they mirror:
 *   OrdinaryKriging._get_kriging_matrix / _exec_vector               src/pykrige/ok.py:626-683
 *   OrdinaryKriging._exec_loop_moving_window                         src/pykrige/ok.py:722-758
 *   UniversalKriging._get_kriging_matrix / _exec_vector              src/pykrige/uk.py:861-1009
 *   OrdinaryKriging3D / UniversalKriging3D equivalents               src/pykrige/ok3d.py:603-657, uk3d.py:688-811
 *   core._adjust_for_anisotropy                                      src/pykrige/core.py:120-193
 *   variogram_models.*                                               src/pykrige/variogram_models.py:25-81
 *
 * Conventions
 *   - plain C types only; all array arguments are caller-owned.
 *   - "host" pointers are ordinary host memory (pinned or pageable);
 *     "dev" pointers are CUDA device memory on the handle's device.
 *   - every function returns KB200_OK (0) or a negative KB200_E* code;
 *     kb200_last_error() gives a human-readable message for the handle.
 *   - a handle is bound to one CUDA device and one stream and is not thread-safe.
 *   - there is NO CPU fallback: without a CUDA device every entry point
 *     that computes returns KB200_ECUDA.
 */
#ifndef KRIGE_B200_H
#define KRIGE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- status codes ------------------------------------------------------- */
#define KB200_OK            0
#define KB200_EBADARG      -1   /* -> ValueError                                        */
#define KB200_EUNSUPPORTED -2   /* -> NotImplementedError (cok.pyx / variogram_models.pyx:20-21 convention) */
#define KB200_ESINGULAR    -3   /* -> numpy.linalg.LinAlgError (global) / ValueError('Singular matrix') (kNN, cok.pyx:176-179) */
#define KB200_ECUDA        -4   /* -> RuntimeError (no device / CUDA runtime failure)   */
#define KB200_ENOMEM       -5   /* -> MemoryError                                       */
#define KB200_ESTATE       -6   /* -> RuntimeError (call order)                         */

/* ---- variogram model ids (keyed on the reference's function __name__,
 *      src/pykrige/lib/variogram_models.pyx:5-21; hole-effect added) ------- */
#define KB200_VG_LINEAR       0  /* params [slope, nugget]            variogram_models.py:25 */
#define KB200_VG_POWER        1  /* params [scale, exponent, nugget]  variogram_models.py:32 */
#define KB200_VG_GAUSSIAN     2  /* params [psill, range, nugget]     variogram_models.py:40 */
#define KB200_VG_EXPONENTIAL  3  /* params [psill, range, nugget]     variogram_models.py:48 */
#define KB200_VG_SPHERICAL    4  /* params [psill, range, nugget]     variogram_models.py:56 */
#define KB200_VG_HOLE_EFFECT  5  /* params [psill, range, nugget]     variogram_models.py:73 */
#define KB200_VG_TABLE        6  /* 'custom' / GSTools callables (ok.py:224-253): tabulated by the host, see kb200_set_variogram_table; no params */

/* ---- arithmetic of the big contraction ---------------------------------- */
#define KB200_F64 0   /* fp64 contraction: with a positive definite covariance form and 512 <= n <= 65535 on the INT8
                         tensor cores with 8 exact slices (55 bits, as accurate as the fp64 product), else on the fp64
                         DMMA tensor cores (small n, pseudo_inv, the indefinite general path) */
#define KB200_F32 1   /* factorisation stays fp64; contraction in 3xTF32 on tcgen05 (fp32-class accuracy) */
#define KB200_F64X 2  /* fp64-class contraction on the INT8 tensor cores: error-free slicing into 6 signed slices (41 bits),
                         exact int32 accumulation (tcgen05 kind::i8), exact int64 recombination; agrees with KB200_F64
                         to ~1e-10 */
#define KB200_F64X5 3 /* the same with 5 slices (34 bits, 15 instead of 21 MMAs per k-step) */
#define KB200_F64X4 4 /* the same with 4 slices (27 bits, 10 MMAs per k-step): between float32 and float64 */

/* ---- coordinates (ok.py:292-318) -------------------------------------------- */
#define KB200_EUCLIDEAN  0
#define KB200_GEOGRAPHIC 1   /* (x, y) = (lon, lat) degrees; great-circle distances, core.py:36-97; OK 2-D only */

#define KB200_MAX_DRIFT 15   /* drift columns (regional-linear + host supplied), excluding the unbiasedness column */

typedef struct kb200_ctx* kb200_handle;

/* Create a handle on CUDA device `device` (-1 = current device). */
int  kb200_create(kb200_handle* out, int device);
void kb200_destroy(kb200_handle h);
const char* kb200_last_error(kb200_handle h);
/* Library/ABI version (major*1000+minor). */
int  kb200_version(void);

/*
 * Describe the kriging system (the data side) and factor it on the device.
 * Replaces _get_kriging_matrix + scipy.linalg.inv of the reference
 * (ok.py:626-648,663; uk.py:861-920,935).
 *
 *  dim            2 or 3
 *  dtype          KB200_F64 (DMMA) / KB200_F32 (tcgen05 3xTF32) / KB200_F64X, KB200_F64X5, KB200_F64X4 (tcgen05 INT8 slices)
 *  n              number of data points
 *  x,y,z          host, length n, ORIGINAL (un-adjusted) coordinates; z may be NULL when dim==2
 *  values         host, length n (self.Z / self.VALUES)
 *  center[dim]    anisotropy centre (XCENTER, YCENTER[, ZCENTER])                 ok.py:278-279
 *  aniso[dim*dim] row-major matrix Mt = stretch @ rot of core._adjust_for_anisotropy  core.py:148-189
 *                 (adjusted = Mt @ (p - center) + center); identity when isotropic
 *  model          KB200_VG_*,  vparams: the reference's *stored* parameter list (psill form);
 *                 KB200_VG_TABLE: no parameters (vparams may be NULL, n_vparams = 0), the table set by
 *                 kb200_set_variogram_table is used
 *  exact_values   ok.py:671-672 semantics;  eps: |d| <= eps counts as an exact hit (ok.py:177)
 *  n_rl           0, or dim: regional-linear drift columns built on device from the adjusted coordinates
 *                 (uk.py:877-883, uk3d.py:708-717)
 *  n_hd           number of host-supplied drift columns (point_log, external_Z, specified, functional;
 *                 uk.py:884-910) ; drift_data is host, column-major n x n_hd (column c at drift_data + c*n)
 *  Work is asynchronous on the handle's stream; errors of the factorisation
 *  (non positive-definite / singular) are reported here (the call synchronises once).
 */
int kb200_set_problem(kb200_handle h, int dim, int dtype, int64_t n,
                      const double* x, const double* y, const double* z,
                      const double* values,
                      const double* center, const double* aniso,
                      int model, const double* vparams, int n_vparams,
                      int exact_values, double eps,
                      int n_rl, int n_hd, const double* drift_data);

/*
 * Krige explicit points (style='points', and 'masked' after compaction).
 *   px,py,pz   host, length m, ORIGINAL coordinates (anisotropy is applied on device, ok.py:880-885)
 *   drift_pts  host, column-major m x (n_hd - n_dev) values of the host-supplied drift terms at the points (or NULL);
 *              the first n_dev drift terms are evaluated on the device when kb200_set_device_drift described them
 *   z_out, ss_out  host, length m  (zvalues, sigmasq of ok.py:680-681)
 */
int kb200_execute_points(kb200_handle h, int64_t m,
                         const double* px, const double* py, const double* pz,
                         const double* drift_pts,
                         double* z_out, double* ss_out);

/*
 * Krige a rectangular grid (style='grid'): points are generated on the device
 * in the reference's order — 2-D: meshgrid(x, y) flattened, x fastest (ok.py:864-866);
 * 3-D: meshgrid(z, y, x, indexing='ij') flattened, x fastest (ok3d.py:863-866).
 *   gx,gy,gz   host axis vectors of length nx, ny, nz (gz NULL and nz=1 for 2-D)
 *   first,count  the slice [first, first+count) of the flattened grid to compute (multi-GPU sharding);
 *                z_out/ss_out are host arrays of length `count`.
 */
int kb200_execute_grid(kb200_handle h,
                       int64_t nx, int64_t ny, int64_t nz,
                       const double* gx, const double* gy, const double* gz,
                       const double* drift_pts,
                       int64_t first, int64_t count,
                       double* z_out, double* ss_out);

/* Same as the two calls above but with DEVICE pointers for the point coordinates /
 * axis vectors and for the outputs; nothing is copied to or from the host. */
int kb200_execute_points_dev(kb200_handle h, int64_t m,
                             const double* d_px, const double* d_py, const double* d_pz,
                             const double* d_drift_pts,
                             double* d_z_out, double* d_ss_out);
int kb200_execute_grid_dev(kb200_handle h,
                           int64_t nx, int64_t ny, int64_t nz,
                           const double* d_gx, const double* d_gy, const double* d_gz,
                           const double* d_drift_pts,
                           int64_t first, int64_t count,
                           double* d_z_out, double* d_ss_out);

/*
 * Moving-window kriging (n_closest_points=k): exact k nearest data points per
 * prediction point (cKDTree.query(k, eps=0.0), ok.py:957-960), local (k+1)x(k+1)
 * system assembled on the fly and solved per point (ok.py:722-758, cok.pyx:98-193).
 * Ordinary kriging only (the reference has no moving window for UK, uk.py:1090-1098).
 * Point sources as above: explicit points (grid = 0) or a grid slice (grid = 1).
 */
int kb200_execute_knn_points(kb200_handle h, int k, int64_t m,
                             const double* px, const double* py, const double* pz,
                             double* z_out, double* ss_out);
int kb200_execute_knn_grid(kb200_handle h, int k,
                           int64_t nx, int64_t ny, int64_t nz,
                           const double* gx, const double* gy, const double* gz,
                           int64_t first, int64_t count,
                           double* z_out, double* ss_out);
int kb200_execute_knn_grid_dev(kb200_handle h, int k,
                               int64_t nx, int64_t ny, int64_t nz,
                               const double* d_gx, const double* d_gy, const double* d_gz,
                               int64_t first, int64_t count,
                               double* d_z_out, double* d_ss_out);
/* Set the data for the moving window only (no global factorisation, SURVEY F4). */
int kb200_set_problem_knn(kb200_handle h, int dim, int64_t n,
                          const double* x, const double* y, const double* z,
                          const double* values,
                          const double* center, const double* aniso,
                          int model, const double* vparams, int n_vparams,
                          int exact_values, double eps);

/*
 * Multi-GPU: the factor blob (packed inverse Cholesky factor + dual vectors +
 * constants + adjusted data coordinates) lives in ONE contiguous device
 * allocation so that rank 0 can factor and a single NCCL broadcast ships it.
 *   kb200_blob_bytes    size of the blob for the current problem description
 *   kb200_blob_ptr      device pointer of the blob owned by the handle
 *   kb200_describe_problem  same arguments as kb200_set_problem but performs NO
 *                       device work: it only records the description and allocates the blob,
 *                       so that a non-root rank can receive the broadcast into kb200_blob_ptr()
 *   kb200_blob_commit   mark the (received) blob as valid: the handle is ready to execute
 */
int64_t kb200_blob_bytes(kb200_handle h);
void*   kb200_blob_ptr(kb200_handle h);
int kb200_describe_problem(kb200_handle h, int dim, int dtype, int64_t n,
                           const double* x, const double* y, const double* z,
                           const double* values,
                           const double* center, const double* aniso,
                           int model, const double* vparams, int n_vparams,
                           int exact_values, double eps,
                           int n_rl, int n_hd, const double* drift_data);
int kb200_blob_commit(kb200_handle h);

/*
 * Drift terms evaluated at the prediction points ON THE DEVICE (universal kriging, 2-D): the point-logarithmic
 * terms -strength * log(distance to the well), log(0) -> -100 (uk.py:884-896, 955-966) and the external-Z term
 * sampled from a raster with the reference's bilinear rule incl. its on-node / on-line cases (uk.py:512-628,
 * 967-971). They are the FIRST n_wells + (raster ? 1 : 0) of the n_hd drift columns of every following
 * kb200_set_problem / kb200_describe_problem on this handle (the reference's column order, uk.py:884-900); their
 * values at the DATA points still arrive in drift_data, their values at the prediction points are no longer part
 * of drift_pts. n_wells = 0 and ext_nx = ext_ny = 0 switch the feature off.
 *   wells      host, [n_wells][3]: well x, y in the ADJUSTED frame (uk.py:458-467) and strength
 *   ext_x/y    host raster axes (length ext_nx / ext_ny), ext_z host raster [ext_ny][ext_nx]; sampled at the
 *              ORIGINAL prediction coordinates; the caller checks that the raster covers the prediction domain
 *              (uk.py:545-551 raises ValueError). Arrays are copied.
 */
int kb200_set_device_drift(kb200_handle h, int n_wells, const double* wells,
                           int64_t ext_nx, int64_t ext_ny, const double* ext_x, const double* ext_y,
                           const double* ext_z);

/*
 * Single-process multi-GPU (SURVEY.md 8b/8e): a group of handles on n_gpus devices of this box (devices = NULL:
 * 0 .. n_gpus-1) behind ONE call from ONE host thread — what execute(..., backend='cuda', n_gpus=G) binds.
 * kb200_group_set_problem: device 0 assembles and factors, the factor blob is copied to the peers over NVLink
 * (cudaMemcpyPeerAsync), no other transfer. kb200_group_execute_*: the work list is cut into n_gpus contiguous
 * blocks of the reference's flattened point order (ok.py:864-866); every device kriges its block and writes it
 * into the caller's z_out / ss_out at its offset, so the result equals the single-GPU result bit for bit.
 * Arguments as in the single-handle calls. Configuration that precedes a problem description
 * (kb200_set_coordinates, kb200_set_pseudo_inverse, kb200_set_variogram_table, kb200_set_device_drift) is applied
 * per member through kb200_group_member(). Errors: the code of the first failing member;
 * kb200_group_last_error names the device.
 */
typedef struct kb200_group_ctx* kb200_group;
int  kb200_group_create(kb200_group* out, int n_gpus, const int* devices);
void kb200_group_destroy(kb200_group g);
const char* kb200_group_last_error(kb200_group g);
int  kb200_group_size(kb200_group g);
kb200_handle kb200_group_member(kb200_group g, int i);       /* borrowed; destroyed with the group */
int kb200_group_set_problem(kb200_group g, int dim, int dtype, int64_t n,
                            const double* x, const double* y, const double* z,
                            const double* values,
                            const double* center, const double* aniso,
                            int model, const double* vparams, int n_vparams,
                            int exact_values, double eps,
                            int n_rl, int n_hd, const double* drift_data);
int kb200_group_set_problem_knn(kb200_group g, int dim, int64_t n,
                                const double* x, const double* y, const double* z,
                                const double* values,
                                const double* center, const double* aniso,
                                int model, const double* vparams, int n_vparams,
                                int exact_values, double eps);
int kb200_group_execute_points(kb200_group g, int64_t m,
                               const double* px, const double* py, const double* pz,
                               const double* drift_pts,
                               double* z_out, double* ss_out);
int kb200_group_execute_grid(kb200_group g,
                             int64_t nx, int64_t ny, int64_t nz,
                             const double* gx, const double* gy, const double* gz,
                             const double* drift_pts,
                             int64_t first, int64_t count,
                             double* z_out, double* ss_out);
int kb200_group_execute_knn_points(kb200_group g, int k, int64_t m,
                                   const double* px, const double* py, const double* pz,
                                   double* z_out, double* ss_out);
int kb200_group_execute_knn_grid(kb200_group g, int k,
                                 int64_t nx, int64_t ny, int64_t nz,
                                 const double* gx, const double* gy, const double* gz,
                                 int64_t first, int64_t count,
                                 double* z_out, double* ss_out);

/* Select the coordinate type of the NEXT kb200_set_problem / kb200_set_problem_knn / kb200_describe_problem
 * call (default KB200_EUCLIDEAN). Geographic mode requires dim == 2 and no drift terms; anisotropy is ignored,
 * as in the reference (ok.py:296-306). */
int kb200_set_coordinates(kb200_handle h, int coordinates_type);

/* Use an existing CUDA stream (cudaStream_t passed as void*) for all work of the handle. */
int kb200_set_stream(kb200_handle h, void* cuda_stream);

/*
 * Device-side timings (CUDA events on the handle's stream) of the last calls, in ms:
 *  [0] assemble  [1] cholesky  [2] triangular inverse  [3] pack + dual vectors
 *  [4] solve kernel (sum over chunks)  [5] finalize (sum)  [6] h2d  [7] d2h
 *  [8] knn search  [9] knn local solve
 *  [10] solve-kernel launches  [11] total kernel launches since the last kb200_reset_counters
 *  [12] slices of the INT8 contraction kernel of the current problem (0 = fp64 DMMA or 3xTF32 kernel)
 * Returns the number of entries written (<= n).
 */
int  kb200_last_timings(kb200_handle h, double* ms, int n);
void kb200_reset_counters(kb200_handle h);

/* 'custom' variogram callables and GSTools covariance models (variogram_function f(params, d), ok.py:224-253;
 * the reference's own native backend refuses them, lib/variogram_models.pyx:20-21). A Python callable cannot
 * run on the device, so the host samples it once: gamma_nodes[i] = f(params, d_i) at the n_nodes (>= 16)
 * square-root-spaced distances d_i = dmax * (i / (n_nodes - 1))^2, i = 0 .. n_nodes-1 (dense near 0, where
 * variograms bend). The device evaluates model KB200_VG_TABLE by cubic Hermite interpolation in sqrt(d)
 * (DESIGN.md 5c: <= 3e-12 relative for smooth models at 2^20 nodes). Every distance that the following
 * problem evaluates must be <= dmax (data-data and data-prediction); the host wrapper sizes dmax from the
 * bounding boxes. All nodes must be finite (KB200_EBADARG otherwise). The table is copied; it stays
 * attached to the handle until replaced. Call before kb200_set_problem / kb200_describe_problem /
 * kb200_set_problem_knn with model = KB200_VG_TABLE (vparams may be NULL, n_vparams = 0).
 */
int kb200_set_variogram_table(kb200_handle h, int64_t n_nodes, double dmax, const double* gamma_nodes);

/* pseudo_inv=True (ok.py:156-165,660-661; uk.py:932-933; ok3d.py / uk3d.py likewise): the NEXT
 * kb200_set_problem / kb200_describe_problem on this handle inverts the bordered kriging matrix with a
 * pseudo-inverse (singular values below max(M,N)*eps*s_max dropped, as scipy.linalg.pinv / pinvh), so that
 * redundant data points are averaged instead of raising KB200_ESINGULAR. float64 only
 * (KB200_EUNSUPPORTED otherwise); the moving window ignores the flag, as the reference does
 * (ok.py:753 always calls scipy.linalg.solve). Resets the handle's problem state.
 */
int kb200_set_pseudo_inverse(kb200_handle h, int enable);

/* ---- constructor-side helpers (SURVEY.md 8f next-2) ----------------------------------------------
 *
 * kb200_experimental_variogram replaces the pdist binning of core._initialize_variogram_model
 * (core.py:432-505): over all n(n-1)/2 data pairs, d = pair distance (euclidean on the ALREADY
 * ADJUSTED coordinates x, y[, z], dim = 2 | 3; great-circle degrees of (lon, lat) = (x, y) when the
 * handle is in KB200_GEOGRAPHIC mode, dim = 2), g = 0.5 (v_i - v_j)^2, binned into `nlags` equal-width
 * lags from dmin to dmax (last edge dmax + 0.001, core.py:471-476). Host arrays in and out:
 *   counts[nlags], lag_sum[nlags] (sum of d), semi_sum[nlags] (sum of g), dminmax[2] = (dmin, dmax);
 * the caller forms the means and drops empty lags (core.py:493-505). Stateless with respect to the
 * factored problem of the handle. Returns KB200_EBADARG for n < 2, nlags < 1 or nlags > 4096.
 */
int kb200_experimental_variogram(kb200_handle h, int dim, int64_t n,
                                 const double* x, const double* y, const double* z, const double* values,
                                 int nlags, double* counts, double* lag_sum, double* semi_sum, double* dminmax);

/* kb200_statistics replaces core._find_statistics (core.py:759-836): for every data point i >= 1 the
 * ordinary-kriging estimate from points [0, i) and its variance, read off the Cholesky factor that
 * kb200_set_problem computed on THIS handle (any dtype; not after kb200_blob_commit alone, not for the
 * indefinite fallback -> KB200_EUNSUPPORTED, not for a kNN-only problem -> KB200_ESTATE).
 * delta[i] = Z_i - zhat_i, sigma[i] = sqrt(sigmasq_i); entries 0 and points that coincide with an
 * earlier point (distance <= 1e-10, core.py:729-731) are returned as 0 — the caller drops
 * sigma <= eps entries exactly as core.py:829-831. Host arrays of length n.
 */
int kb200_statistics(kb200_handle h, double* delta, double* sigma);

/* Debug/verification taps (used by tests only): copy device intermediates to host.
 *  what = 1: Cholesky factor L of the shifted covariance matrix (n_pad x n_pad, row-major, lower triangle valid)
 *  what = 2: W = inv(L) (same layout)
 *  what = 3: dual block: Uz (n x (K+2), column-major), then Sinv ((K+1)^2), then phi (K+1), then c0
 * `cap` is the capacity of `out` in doubles; returns the number of doubles written or a negative code. */
int64_t kb200_debug_fetch(kb200_handle h, int what, double* out, int64_t cap);

#ifdef __cplusplus
}
#endif
#endif /* KRIGE_B200_H */
