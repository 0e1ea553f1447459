/*
 * grates_b200 -- C ABI of the B200 (sm_100a) spherical-harmonic hot path of akvas/grates.
 *
 * The reference (pure Python/numpy) has no FFI; the boundary it offers is its Python method
 * signatures.  Each entry point below replaces the numpy/BLAS body of one of those methods
 * (citations are relative to /root/reference/grates/).  The Python host side
 * (the grates_b200 Python package) builds the small epoch-independent tables with the reference's exact
 * numpy expressions and calls these functions through ctypes; see INTEGRATION.md for the
 * binding a maintainer of the reference would add.
 *
 * Conventions
 *  - All floating-point data are IEEE double, C-contiguous.
 *  - "packed" coefficient arrays are the reference's anm[L][L] layout (gravityfield.py:149-159):
 *    C_nm = anm[n][m] (m <= n), S_nm = anm[m-1][n] (m >= 1), L = nmax + 1.
 *  - Grid values are [nlat][nlon], rows north -> south, columns west -> east (grid.py:1149-1150).
 *  - Covariance matrices and ravelled vectors are in the degree-wise order of
 *    utilities.py:310-360 (index of C_nm = n^2 + max(2m-1, 0), of S_nm = n^2 + 2m), offset nmin^2.
 *  - Pointers named d_* are device pointers on the plan's device, h_* are host pointers.
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Device entry
 *    points are asynchronous with respect to the host; *_host entry points return after the
 *    result is in the host buffer.
 *  - The library never frees caller memory and returns no owning pointer except gb_plan*.
 *  - Return value: GB_OK or an error code; gb_last_error() gives the thread-local message.
 *  - There is no CPU fallback anywhere: without a CUDA device every compute call fails.
 *  - Re-entrancy: a gb_plan owns ONE workspace (packed coefficients, spectral intermediate, analysis and covariance
 *    scratch).  Calls on one plan may use different streams -- the library orders a call behind the previous call's
 *    work on whatever stream that ran (an event wait, free when the stream is the same) -- but two host threads must
 *    not be inside calls on the same plan at the same time (the Python layer holds a per-plan lock).  Different plans
 *    are independent.
 *  - Stream order: the kernels of a synthesis call are chained with programmatic dependent launch and signal
 *    `launch_dependents` early.  Work the caller enqueues behind a call with an ordinary launch (or a copy) starts
 *    after the call's last kernel has completed, as usual; only a kernel the CALLER launches with
 *    cudaLaunchAttributeProgrammaticStreamSerialization directly behind a call must execute griddepcontrol.wait
 *    (cudaGridDependencySynchronize) before it touches the call's output.  The first kernel of every call waits
 *    for all prior work of the stream before it reads the caller's input.
 */
#ifndef GRATES_B200_H
#define GRATES_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GB_OK 0
#define GB_ERR_ARGUMENT 1
#define GB_ERR_CUDA 2
#define GB_ERR_UNSUPPORTED 3
#define GB_ERR_MEMORY 4

typedef struct gb_plan gb_plan;

/* Library version (major*10000 + minor*100 + patch); bumped with every change of this header.  The Python binding
 * refuses a library whose version differs from the one it was written for (grates_b200/_lib.py). */
#define GB_VERSION 203
int gb_version(void);

/* Thread-local description of the last error returned on this thread. */
const char* gb_last_error(void);

/* Number of visible CUDA devices (fails with GB_ERR_CUDA if the driver is unusable). */
int gb_device_count(int* count);

/* Temporaries of a call (covariance tiles, filter batches; up to a few GB) are stream-ordered allocations from a memory
 * pool the library owns per device; the pool keeps them between calls.  gb_trim synchronises the device and returns
 * the pool's unused memory to the driver.  The device's default pool is never touched. */
int gb_trim(int device);

/*
 * Plan = the epoch-independent tables of one (grid geometry, nmax, kernel, GM, R) combination,
 * resident on one device.  Replaces the per-call table construction of
 * PotentialCoefficients.to_grid (gravityfield.py:353-365) and
 * RegularGrid.covariance_propagation (grid.py:819-831).
 *
 *   cos_theta, sin_theta [nlat]   cos / sin of the geocentric colatitude of each parallel
 *                                 (utilities.py:438-459 then np.cos / np.sin, utilities.py:38-39)
 *   kn [nlat][nmax+1]             inverse kernel factor x upward continuation x GM/R
 *                                 (gravityfield.py:356 == grid.py:657 == grid.py:823)
 *   cos_mlon, sin_mlon [nmax+1][nlon]   cos(m*lon_j), sin(m*lon_j) (utilities.py:271-273)
 *
 * The fully normalised Legendre functions themselves are NOT passed in: the kernels run the
 * recursion of utilities.py:37-54 on the fly, per latitude tile, with unfused IEEE multiplies
 * and subtracts so that every P_nm is bit-identical to the reference's table.
 */
int gb_plan_create(gb_plan** plan, int nmax, int nlat, int nlon,
                   const double* cos_theta, const double* sin_theta, const double* kn,
                   const double* cos_mlon, const double* sin_mlon, int device);
int gb_plan_destroy(gb_plan* plan);

/* Geometry queries (for the host wrapper). */
int gb_plan_info(const gb_plan* plan, int* nmax, int* nlat, int* nlon, int* device);

/*
 * 1 if the plan's meridians are symmetric about 0 and invariant under a half turn (all grids the
 * reference constructs itself: GeographicGrid, GaussGrid with a meridian count divisible by 8).
 * gb_synthesis then evaluates only the first quadrant of meridians and obtains the other three by
 * sign changes (one quarter of the multiply-adds of the direct longitude contraction); set the
 * environment variable GB_NO_SYMMETRY=1 to force the direct contraction.
 * Returns 2 if in addition the first-quadrant meridians mirror about pi/4 (meridian count divisible by 16, e.g. the
 * 0.5 and 0.25 degree GeographicGrid): gb_synthesis then evaluates the first OCTANT only -- the orders 0, 2 (mod 4) change
 * the sign of their cosine / sine rows under mu -> pi/2 - mu, the odd orders swap them -- for three quarters of the
 * four-fold kernel's multiply-adds.  Both gates are measured on the plan's own tables.  GB_S2_QUADRANT=1 at call time
 * keeps the four-fold kernel.
 */
int gb_plan_is_symmetric(const gb_plan* plan);

/*
 * 1 if the plan's parallels are mirror images about the equator closely enough for the folded Legendre stage
 * (GeographicGrid / GaussGrid down to about 0.5 degree spacing): gb_synthesis then runs the recursion for the northern
 * parallels only and obtains the southern ones from P_nm(pi - theta) = (-1)^(n-m) P_nm(theta) -- half the recursion steps
 * and multiply-adds of the Legendre stage.  The gate is measured at plan creation: the zonal functions of both
 * hemispheres, computed with the reference's own (not exactly mirrored) cos(theta) tables, must agree to 2e-13 of their
 * largest value in every degree.  Parallels next to the poles that fail (the reference's arccos is ill-conditioned
 * there; e.g. one parallel of a 0.25 degree grid) keep the unfolded stage in tiles of 32 per hemisphere: the return
 * value is 0 (not folded) or 1 + the number of such polar tiles (at most two).  GB_NO_FOLD=1 forces the unfolded stage.
 */
int gb_plan_is_folded(const gb_plan* plan);

/*
 * Spherical-harmonic synthesis of n_epochs coefficient sets onto the plan's grid.
 * Replaces the body of PotentialCoefficients.to_grid, gravityfield.py:358-368, for a batch:
 *   out[e][i][j] = sum_n kn[i][n] sum_m P_nm(theta_i) (C_nm^e cos m lon_j + S_nm^e sin m lon_j)
 *   d_anm [n_epochs][L][L] packed, d_out [n_epochs][nlat][nlon].
 * d_out must be 16-byte aligned (the kernels store pairs of doubles); GB_ERR_ARGUMENT otherwise, before any launch.
 */
int gb_synthesis(gb_plan* plan, const double* d_anm, int n_epochs, double* d_out, void* stream);

/*
 * Same through host buffers: copies the coefficients to the device, runs the kernels in
 * epoch chunks and copies each finished chunk back while the next one computes.
 * Pinned host buffers (gb_host_alloc) give the full PCIe rate; pageable ones work too.
 */
int gb_synthesis_host(gb_plan* plan, const double* h_anm, int n_epochs, double* h_out);

/*
 * Bit-exact check hook: the on-the-fly Legendre recursion written out as a table, scaled by
 * kn, in the reference's packed layout.  d_out [nlat][L][L]; with scaled == 0 the kn factor is
 * left out and the result equals utilities.legendre_functions (utilities.py:13-59) bit for bit.
 */
int gb_legendre_table(gb_plan* plan, double* d_out, int scaled, void* stream);

/*
 * Spherical-harmonic analysis (area-weighted least squares, order by order), batched.
 * Replaces RegularGrid.to_potential_coefficients, grid.py:776-785.  The per-order operators
 * solve(A'WA, A'W) of grid.py:690-696 are separable on a regular grid with rank-one area
 * weights (SURVEY 3.3); the host builds the small Legendre-side factor once per plan:
 *
 *   lon_ops [2L][nlon]     row 2m   : u_j cos(m lon_j) / sum_j u_j cos^2(m lon_j)
 *                          row 2m+1 : u_j sin(m lon_j) / sum_j u_j sin^2(m lon_j)   (row 1 = 0)
 *   lat_ops                concatenation over m = 0..nmax of op_m [cnt_m][nlat] row-major,
 *                          cnt_m = nmax + 1 - max(m, nmin); op_m = solve(P'WP, P'W)
 *   lat_op_offsets [L+1]   element offsets of op_m inside lat_ops
 */
int gb_plan_set_analysis(gb_plan* plan, int nmin, const double* lon_ops, const double* lat_ops,
                         const int64_t* lat_op_offsets);
/* The same with the latitude-side operators built ON THE DEVICE from the latitude factor w_lat [nlat] (host) of the
 * separable area weights: P by the bit-exact recursion, per order the normal matrix, its Cholesky factor and two
 * triangular solves (gb_dgemm / gb_dpotrf_upper / gb_dtrsm_upper).  Fails with GB_ERR_ARGUMENT if a normal matrix is
 * not positive definite (the grid does not resolve the degree). */
int gb_plan_set_analysis_weights(gb_plan* plan, int nmin, const double* lon_ops, const double* w_lat);
/*   d_grid [n_epochs][nlat][nlon] -> d_anm [n_epochs][L][L] packed (degrees < nmin zero). */
int gb_analysis(gb_plan* plan, const double* d_grid, int n_epochs, double* d_anm, void* stream);
int gb_analysis_host(gb_plan* plan, const double* h_grid, int n_epochs, double* h_anm);

/*
 * Explicit operators in degree-wise order (dense, for small grids / window matrices):
 *   gb_synthesis_matrix  d_out [nlat*nlon][K'] , K' = (nmax+1)^2 - nmin^2   (Grid.synthesis_matrix, grid.py:412-443)
 *   gb_analysis_matrix   d_out [K'][nlat*nlon] for the nmin of gb_plan_set_analysis (RegularGrid.analysis_matrix,
 *                        grid.py:698-730)
 */
int gb_synthesis_matrix(gb_plan* plan, int nmin, double* d_out, void* stream);
int gb_analysis_matrix(gb_plan* plan, double* d_out, void* stream);

/*
 * Covariance propagation to per-point variances, diag(F Sigma F'), for the parallels
 * [row0, row0 + nrows) of the plan's grid.  Replaces grid.py:833-835 (the reference then takes
 * the square root, grid.py:837-839; pass GB_COV_SQRT for that).
 *   d_sigma [K'][K'] row-major, K' = (nmax+1)^2 - nmin^2, degree-wise order
 *   d_out   [nrows][nlon]  ([2 nrows][nlon] with GB_COV_MIRRORED)
 *   flags   GB_COV_SQRT: return standard deviations.  GB_COV_SYMMETRIC: the caller states that
 *           Sigma is symmetric (a covariance matrix is); only its order-block pairs k <= k' are
 *           contracted, which halves the work.  Without the flag the full matrix is used.
 */
#define GB_COV_SQRT 1
#define GB_COV_SYMMETRIC 2
/* GB_COV_MIRRORED: the block is the `nrows` NORTHERN parallels [row0, row0 + nrows) (2 (row0 + nrows) <= nlat) together
 * with their mirror images about the equator; d_out is [2 nrows][nlon]: the northern rows, then the parallels
 * [nlat - row0 - nrows, nlat - row0) in increasing order.  On grids that are symmetric about the equator the Legendre
 * factors of a parallel and its mirror image differ by the sign (-1)^(n-m) only, so the first contraction runs once for
 * both (half its flops); this is how row blocks should be cut for several GPUs.  A full-grid call folds by itself. */
#define GB_COV_MIRRORED 4
int gb_covariance_propagation(gb_plan* plan, const double* d_sigma, int nmin, int row0, int nrows,
                              double* d_out, int flags, void* stream);
/*
 * Propagation of a FILTERED covariance, diag(A F Sigma F' A'), without forming F Sigma F' (the reference
 * multiplies the dense matrices, F = SpatialFilter.matrix(nmin, nmax), filter.py:72-92, :120-127, :193-222):
 * a degree-wise or order-wise F keeps the product structure of A, so the filter is applied to the small
 * Legendre factor instead (K^2-sized products disappear).
 *   d_blocks / block_offsets / nf   order-wise blocks as for gb_orderwise_filter, or NULL
 *   d_wn [nmax+1]                   degree weights of an isotropic filter, or NULL
 * Both may be given (F = diag(w) * F_blocks: the blocks act first).
 */
int gb_covariance_propagation_filtered(gb_plan* plan, const double* d_sigma, int nmin, int row0, int nrows,
                                       double* d_out, int flags, const double* d_blocks,
                                       const int64_t* block_offsets, int nf, const double* d_wn, void* stream);

/*
 * Isotropic (degree-wise) filters: Gaussian and Butterworth, filter.py:31-130, scale every
 * coefficient of degree n by a weight w_n.
 *   gb_scale_by_degree      d_anm_out[e][r][c] = d_anm_in[e][r][c] * d_wn[max(r, c)]   (may alias)
 *   gb_synthesis_weighted   gb_synthesis of the scaled coefficients without materialising them: the
 *                           weights are multiplied in while the coefficients are packed order-wise
 *   d_wn [nmax+1] device array (the reference leaves degrees 0, 1 unscaled for the Gaussian: w = 1)
 *   d_out of gb_synthesis_weighted: 16-byte aligned, as for gb_synthesis
 */
int gb_scale_by_degree(const double* d_anm_in, const double* d_wn, int n_epochs, int nmax,
                       double* d_anm_out, int device, void* stream);
int gb_synthesis_weighted(gb_plan* plan, const double* d_anm, const double* d_wn, int n_epochs,
                          double* d_out, void* stream);

/*
 * Order-wise block filter (gb_orderwise_filter) followed by gb_synthesis of the filtered batch, without materialising
 * it: the filter writes its result in the layout the Legendre stage of the synthesis reads.  Replaces
 * OrderWiseFilter.filter (filter.py:180-189) + PotentialCoefficients.to_grid (gravityfield.py:331-368) per epoch;
 * bit-identical to the two calls in sequence.  nf >= the plan's nmax.  d_out: 16-byte aligned, as for gb_synthesis.
 */
int gb_synthesis_orderwise_filtered(gb_plan* plan, const double* d_blocks, const int64_t* block_offsets, int nf,
                                    const double* d_anm, int n_epochs, double* d_out, void* stream);

/*
 * Dense filter matrices (GeneralMatrix / VDK, filter.py:430-572), batched over epochs: x_e = ravel(anm_e, nmin,
 * nmax_filter), y_e = W x_e, unravel up to min(nmax_in, nmax_filter), degrees below nmin copied through.
 *   gb_dense_filter_tile_elements   doubles needed for the operand tiles of a k x k matrix
 *   gb_dense_filter_prepare         d_matrix [k][k] row-major (degree-wise order) -> d_tiles, once per filter
 *   gb_dense_filter                 d_anm_in [n_epochs][nmax_in+1]^2 -> d_anm_out [n_epochs][min(nmax_in, nmax_filter)+1]^2
 */
int64_t gb_dense_filter_tile_elements(int64_t k);
int gb_dense_filter_prepare(const double* d_matrix, int64_t k, double* d_tiles, int device, void* stream);
int gb_dense_filter(const double* d_tiles, int nmin, int nmax_filter, const double* d_anm_in, int n_epochs,
                    int nmax_in, double* d_anm_out, int device, void* stream);

/*
 * Order-wise block filter, batched over epochs.  Replaces OrderWiseFilter.filter,
 * filter.py:180-189: order 0 block on C_n0, blocks 2m-1 / 2m on C_nm / S_nm, each block
 * truncated to its top-left (nmax+1-m)^2 corner; degrees 0 and 1 pass through unchanged.
 *   d_blocks        all blocks concatenated; block b is [(nf+1-m_b)][(nf+1-m_b)] row-major
 *   block_offsets   [2*nf+2] element offsets of each block inside d_blocks (host array)
 *   nf              maximum degree of the filter; nmax <= nf required
 *   d_anm_in/out    [n_epochs][L][L] packed (may not alias)
 */
int gb_orderwise_filter(const double* d_blocks, const int64_t* block_offsets, int nf,
                        const double* d_anm_in, int n_epochs, int nmax, double* d_anm_out,
                        int device, void* stream);

/*
 * Arbitrary point sets (the reference's IrregularGrid path).  Tables are per point:
 *   cos_theta, sin_theta [npts], kn [npts][nmax+1], cos_mlon, sin_mlon [npts][nmax+1]
 *   (cos(m*lon_p), sin(m*lon_p), utilities.py:303-304).
 * gb_points_synthesis replaces gravityfield.py:376-388: d_anm [n_epochs][L][L] -> d_out [n_epochs][npts].
 * gb_points_covariance replaces grid.py:1103-1116: direct blocked diag(F Sigma F') with Sigma
 *   [K'][K'] (degree-wise order, offset nmin^2) -> d_out [npts] variances; flags as for gb_covariance_propagation
 *   (GB_COV_SQRT: std-devs; GB_COV_SYMMETRIC: only the lower triangle of Sigma is contracted, half the flops).
 * gb_points_adjoint replaces the sum over nodal points of RadialBasisFunctions.to_potential_coefficients,
 *   gravityfield.py:707-724 (the transposed design matrix): d_values [n_epochs][npts] -> d_anm [n_epochs][L][L],
 *   anm[n, m] = sum_p kn[p][n] Y_nm(p) v[p]; the shape factors K[n, m] are applied by the caller.
 */
typedef struct gb_points gb_points;
int gb_points_create(gb_points** points, int nmax, int npts, const double* cos_theta, const double* sin_theta,
                     const double* kn, const double* cos_mlon, const double* sin_mlon, int device);
int gb_points_destroy(gb_points* points);
int gb_points_synthesis(gb_points* points, const double* d_anm, int n_epochs, double* d_out, void* stream);
int gb_points_covariance(gb_points* points, const double* d_sigma, int nmin, double* d_out, int flags,
                         void* stream);
int gb_points_adjoint(gb_points* points, const double* d_values, int n_epochs, double* d_anm, void* stream);
/* Dense synthesis operator of the point set: d_out [npts][K'], K' = (nmax+1)^2 - nmin^2, degree-wise order
 * (Grid.synthesis_matrix, grid.py:412-443, with IrregularGrid.synthesis_matrix_per_order, grid.py:957-991). */
int gb_points_synthesis_matrix(gb_points* points, int nmin, double* d_out, void* stream);

/*
 * Consumers of gridded epoch batches that keep the grids on the device.
 *   gb_temporal_rms       d_out[p] = sqrt(sum_e v[e][p]^2 / n_epochs); replaces the accumulation loop of
 *                         gridded_rms, gravityfield.py:1165-1170 (same summation order, bit-identical)
 *   gb_weighted_moments   d_out[e][0] = sum_p w[p] (v[e][p] - c[e]),  d_out[e][1] = sum_p w[p] (v[e][p] - c[e])^2
 *                         with w = area element * mask and c = d_shift (NULL: 0): the sums behind
 *                         Grid.mean / rms / std, grid.py:174-260, for a whole batch
 *   d_values [n_epochs][n_points], d_weights [n_points], d_shift [n_epochs] or NULL
 */
int gb_temporal_rms(const double* d_values, int n_epochs, int64_t n_points, double* d_out, int device,
                    void* stream);
int gb_weighted_moments(const double* d_values, const double* d_weights, const double* d_shift,
                        int n_epochs, int64_t n_points, double* d_out, int device, void* stream);

/*
 * Variances of linear functionals of the coefficients (basin means): var_b = a_b' Sigma a_b.
 *   gb_ravel_coefficients   packed d_anm [n_sets][L][L] -> degree-wise vectors d_vec [n_sets][K'],
 *                           K' = (nmax+1)^2 - nmin^2 (reference utilities.py:310-360)
 *   gb_quadratic_forms      d_out[b] = d_vec[b]' * d_sigma * d_vec[b]  for n_vec vectors of length k;
 *                           d_sigma [k][k] row-major is read once per eight vectors
 * The functional of an area-weighted basin mean is a_b = A' w_b (A: synthesis operator of
 * grid.py:412-443); A' runs through gb_analysis with adjoint operators (grates_b200/plan.py: set_adjoint).
 */
int gb_ravel_coefficients(const double* d_anm, int n_sets, int nmax, int nmin, double* d_vec, int device,
                          void* stream);
int gb_quadratic_forms(const double* d_sigma, int64_t k, const double* d_vec, int n_vec, double* d_out,
                       int device, void* stream);

/*
 * Gravitational acceleration (gradient of the potential, no centrifugal term) as three scalar syntheses.  The general
 * form of the zonal gradient of PotentialCoefficients.gravitational_acceleration (gravityfield.py:423-481, restated for
 * GRS80 normal gravity in kernel.py): each Cartesian component of grad V of a degree-nmax field is a synthesis at degree
 * nmax + 1 of linearly transformed coefficients, with degree factors GM/R^2 (R/r)^(n'+1) (Cunningham's relation).
 *   gb_gradient_coefficients   d_anm [n_sets][L][L] packed -> d_out [n_sets][3][L+1][L+1] packed, components (x, y, z)
 *                              Earth-fixed; with q = (2n+1)/(2n+3), (C_nm, S_nm) contributes
 *                                Z[n+1][m]   -sqrt((n-m+1)(n+m+1) q) (C, S)
 *                                X[n+1][m+1] -fp (C, S),  Y[n+1][m+1] (+fp S, -fp C)
 *                                X[n+1][m-1] +fm (C, S),  Y[n+1][m-1] (+fm S, -fm C)   (m >= 1)
 *                              fp = sqrt((n+m+1)(n+m+2) q)/2 (x sqrt 2 at m = 0), fm = sqrt((n-m+1)(n-m+2) q)/2
 *                              (x sqrt 2 at m = 1); sines of order 0 dropped; degree 0 of d_out is zero.  Deterministic
 *                              (a gather, no atomics).
 *   gb_rotate_to_local         d_xyz [n_sets][3][n_points] (gx, gy, gz) -> (east, north, up) in place, with
 *                              d_frame [4][n_points] = (cos theta, sin theta, cos lon, sin lon) of each point:
 *                                east  = -sin lon gx + cos lon gy
 *                                north = -cos theta cos lon gx - cos theta sin lon gy + sin theta gz
 *                                up    =  sin theta cos lon gx + sin theta sin lon gy + cos theta gz
 *                              theta is the GEOCENTRIC colatitude: the frame is geocentric spherical, not the ellipsoidal
 *                              normal.  Grid values are the [nlat][nlon] points flattened row by row.
 */
int gb_gradient_coefficients(const double* d_anm, int n_sets, int nmax, double* d_out, int device, void* stream);
int gb_rotate_to_local(double* d_xyz, const double* d_frame, int n_sets, int64_t n_points, int device, void* stream);

/* Pinned host memory for the *_host entry points. */
int gb_host_alloc(void** ptr, uint64_t bytes);
int gb_host_free(void* ptr);

/*
 * FP64 pipe probes used by bench.py for the roofline denominator (MEASURED_PEAKS.json holds
 * no FP64 figure): sustained DMMA (tensor) and DFMA (vector) rate in TFLOP/s on `device`.
 */
int gb_probe_fp64_peak(int device, double* dmma_tflops, double* dfma_tflops);

/*
 * Per-kernel device timing of gb_synthesis calls (for the roofline figures of bench.py):
 * with capacity > 0 every following gb_synthesis on this plan records CUDA events on the
 * caller's stream around its three kernels (pack, Legendre stage 1, Fourier stage 2), for up to
 * `capacity` calls; capacity = 0 switches it off.  gb_plan_stage_times synchronises those events,
 * writes ms[call][3] for the recorded calls (at most max_calls), returns their number in
 * n_calls and clears the record.
 */
int gb_plan_set_profiling(gb_plan* plan, int capacity);
int gb_plan_stage_times(gb_plan* plan, double* ms, int max_calls, int* n_calls);

/* Number of kernel launches issued by this library on the calling thread since the last reset. */
int64_t gb_launch_count(int reset);

/*
 * Covariance producers (SURVEY 8 f4).  BlockMatrix.cholesky / sparse_inverse / inverse of the reference
 * (lstsq.py:698-717, 823-846, 848-882; used by NormalEquations.compute_covariance, lstsq.py:1026-1042) are loops over
 * matrix blocks around four library calls: scipy.linalg.cholesky(lower=False), scipy.linalg.solve_triangular,
 * scipy.linalg.inv and numpy's `@`.  The three entry points below replace them on device-resident blocks
 * (row-major FP64, arbitrary leading dimension); the Python mirror (grates_b200/lstsq.py) keeps the block loops.
 *
 *   gb_dgemm         C[m][n] = alpha * op(A) * op(B) + beta * C; trans_a: A is stored [k][m], trans_b: B is stored
 *                    [n][k]; upper_only: tiles strictly below the diagonal are skipped (symmetric updates)
 *   gb_dpotrf_upper  A = W' W in place, W upper triangular, strict lower triangle zeroed; *d_info (device int) = 0 or
 *                    the 1-based index of the first non-positive pivot (scipy raises LinAlgError there)
 *   gb_dtrsm_upper   solves W X = B (trans = 0) or W' X = B (trans = 1) in place of B[n][m], W upper triangular
 */
int gb_dgemm(int trans_a, int trans_b, int64_t m, int64_t n, int64_t k, double alpha, const double* d_a, int64_t lda,
             const double* d_b, int64_t ldb, double beta, double* d_c, int64_t ldc, int upper_only, int device, void* stream);
int gb_dpotrf_upper(double* d_a, int64_t n, int64_t lda, int* d_info, int device, void* stream);
int gb_dtrsm_upper(int trans, const double* d_w, int64_t n, int64_t ldw, double* d_b, int64_t m, int64_t ldb, int device,
                   void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GRATES_B200_H */
