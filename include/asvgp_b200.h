/* libasvgp_sm100a — C ABI of the B200-native ASVGP hot path.
 *
 * This is the drop-in boundary (SURVEY.md §8(b), DESIGN.md §2).  Each entry point replaces the arithmetic that the
 * reference delegates to SciPy sparsetools / banded_matrices / CHOLMOD / dense TF linalg at the cited lines
 * (paths relative to the reference repository root).  The reference-side binding a maintainer would add is a
 * ctypes stub: see INTEGRATION.md.
 *
 * Conventions
 *  - plain C: pointers and sizes only, no torch/CUDA types in signatures; `stream` is a cudaStream_t passed as void*
 *    (NULL = the legacy default stream).
 *  - every data pointer is a DEVICE pointer to caller-owned, contiguous memory unless it is named `h_*`.
 *  - all floating point is IEEE fp64; indices are int64 (reference basis.py:58,72-73).
 *  - symmetric banded matrices travel as LOWER bands, row-major (k+1) x M with band[d*M + j] = A[j+d, j] and the last
 *    d entries of row d zero — exactly the layout of banded_matrices / reference utils.py:24-30.
 *  - return value: 0 = ok, <0 = error (asvgp_last_error() gives the message).  No entry point synchronises the host
 *    with the device; numerical failure (non-positive pivot) is reported through the `info` slot of the output
 *    buffer (0 = ok, j+1 = first failing pivot), LAPACK style.
 *  - nothing here falls back to the CPU: without a CUDA device every compute entry point returns an error.
 */
#ifndef ASVGP_B200_H
#define ASVGP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ASVGP_ABI_VERSION 1

#if defined(__GNUC__)
#define ASVGP_API __attribute__((visibility("default")))
#else
#define ASVGP_API
#endif

/* Matern kernel kinds (reference inducing_features.py:16,22,32). */
#define ASVGP_MATERN12 0
#define ASVGP_MATERN32 1
#define ASVGP_MATERN52 2

ASVGP_API int asvgp_abi_version(void);
/* Message of the last failing call on this thread (empty string if none). */
ASVGP_API const char* asvgp_last_error(void);
/* Number of CUDA kernels this library has launched in this process so far (all streams, all entry points). */
ASVGP_API int64_t asvgp_launch_count(void);
/* Test aid: fills every SM's shared memory with a NaN bit pattern (kernels inherit the previous kernel's shared memory; the GPU
 * test suite calls this before every test so that a read of a never-written slot fails deterministically). */
ASVGP_API int asvgp_debug_poison_smem(void* stream);

/* ---- a2/a6: basis evaluation = the non-zeros of Kuf -------------------------------------------------------------
 * Replaces SplineBasis.evaluate_basis (basis.py:51-80) / SplineFeatures1D.make_Kuf (inducing_features.py:47-48).
 * For point i: idx[i] = max(searchsorted_left(mesh, x[i]) - 1, 0) and vals[r*n + i] = d^dx/dx^dx of basis row
 * idx[i]+r at x[i], r = 0..order (the reference's b_{order+1-r}).  `coef` = (order+1)^2 exact piece coefficients in
 * t (ascending powers), required for dx > 0, ignored (may be NULL) for dx = 0. */
ASVGP_API int asvgp_basis_eval_1d(const double* x, int64_t n, const double* mesh, int n_knots, int order, int dx,
                        const double* coef, int64_t* idx, double* vals, void* stream);

/* ---- a7: O(N) accumulation of the banded Gram, the projection and sum(y^2) ------------------------------------------
 * Replaces GPR_1d.__init__'s `Kuf @ y`, `Kuf @ Kuf.T`, utils.sparse_to_band and sum(y^2) (gpr.py:39-44,
 * utils.py:24-30) without materialising Kuf.  Adds into (does NOT zero) the packed accumulator
 *   acc = [ G_band (order+1)*M | b M | sum(y^2) | count ]            ((order+2)*M + 2 doubles)
 * so that shards / chunks can be accumulated by repeated calls and all-reduced as one buffer.  M = n_knots+order-1. */
ASVGP_API int asvgp_accum_1d(const double* x, const double* y, int64_t n, const double* mesh, int n_knots, int order,
                   double* acc, void* stream);

/* Same sums for points in NO PARTICULAR ORDER (SURVEY 8(d) C3-ii: "random order, any binning pass included").
 * asvgp_accum_1d is exact for any order but spends one fp64 RED per band entry per point once consecutive points stop
 * sharing knot intervals; this variant first partitions the points into <= 256 buckets of consecutive intervals
 * (histogram, scan, shared-memory staged scatter), then sorts each 4096-point unit by interval in shared memory and
 * accumulates every run in registers.  `work`: asvgp_accum_1d_binned_work_bytes(n) bytes of device scratch
 * (16 B per point + 8 KB).  asvgp_order_probe_1d writes to out[0] (device) the fraction of 4096 sampled neighbour
 * pairs that lie more than one knot interval apart (~0 time-series order, ~1 shuffled) so a caller can choose. */
ASVGP_API int64_t asvgp_accum_1d_binned_work_bytes(int64_t n);
ASVGP_API int asvgp_accum_1d_binned(const double* x, const double* y, int64_t n, const double* mesh, int n_knots,
                                    int order, double* acc, void* work, int64_t work_bytes, void* stream);
ASVGP_API int asvgp_order_probe_1d(const double* x, int64_t n, const double* mesh, int n_knots, double* out, void* stream);

/* ---- element types of the training points ------------------------------------------------------------------------------
 * The *_typed twins below read x / X and y as float64 or float32, each independently (x_type, y_type: ASVGP_F64 or
 * ASVGP_F32).  A float32 value converts to float64 exactly, so the kernels convert every loaded value in registers and the
 * results equal those for the same points converted to float64 first, up to summation order; the accumulators stay
 * float64.  float32 halves the bytes the O(N) pass reads and needs no widened copy of the data.  The untyped functions are
 * these with ASVGP_F64 for both arrays.  An unknown type code returns an error before any CUDA call.  Alignment rules are
 * those of the untyped functions; binned scratch records stay float64 (the *_work_bytes queries do not depend on the
 * types). */
#define ASVGP_F64 0
#define ASVGP_F32 1
ASVGP_API int asvgp_accum_1d_typed(const void* x, int x_type, const void* y, int y_type, int64_t n, const double* mesh,
                                   int n_knots, int order, double* acc, void* stream);
ASVGP_API int asvgp_accum_1d_binned_typed(const void* x, int x_type, const void* y, int y_type, int64_t n, const double* mesh,
                                          int n_knots, int order, double* acc, void* work, int64_t work_bytes, void* stream);
ASVGP_API int asvgp_order_probe_1d_typed(const void* x, int x_type, int64_t n, const double* mesh, int n_knots, double* out,
                                         void* stream);

/* ---- a10: 1-D posterior mean / variance over test points ----------------------------------------------------------------
 * Replaces GPR_1d.predict_f (gpr.py:91-136): mean[i] = sum_r w_r alpha[idx+r],
 * var[i] = variance + sum_{r,s} w_r w_s S[idx+r, idx+s] with S = band(P^-1) - band(Kuu^-1) (lower band, (order+1) x M). */
ASVGP_API int asvgp_predict_1d(const double* xnew, int64_t n, const double* mesh, int n_knots, int order, const double* alpha,
                     const double* S_band, double variance, double* mean, double* var, void* stream);

/* ---- a5: Kuu assembly ----------------------------------------------------------------------------------------------------
 * Replaces SplineFeatures1D.make_Kuu (inducing_features.py:12-44): Kuu = sum_t coef[t] * tables[t] over the static
 * bands A, B, C, D, BC, BC_grad, BC_ggrad of the basis (basis.py:31-45,82-114), each (order+1) x M, stacked
 * contiguously in `tables`.  `h_coef` / `h_dcoef` are HOST arrays of the Matern coefficients and of their
 * derivatives w.r.t. the lengthscale; dKuu (may be NULL) receives sum_t dcoef[t] * tables[t]. */
ASVGP_API int asvgp_kuu_assemble(const double* tables, int n_terms, const double* h_coef, const double* h_dcoef, int M,
                                 int order, double* Kuu, double* dKuu, void* stream);

/* Scratch bytes needed by asvgp_elbo_grad_1d / asvgp_posterior_1d (chunks = 0: library default). */
ASVGP_API int64_t asvgp_workspace_bytes_1d(int M, int order, int chunks);

/* ---- a8 + a9: collapsed ELBO and its hyper-parameter gradients ------------------------------------------------------------
 * Replaces GPR_1d.elbo (gpr.py:49-89: cholesky_band x2, inverse_from_cholesky_band, product_band_band,
 * solve_triang_mat) and the TF reverse-mode gradient the optimiser asks for (example.py:31-32).
 * `acc` is the packed accumulator of asvgp_accum_1d (after any all-reduce).  `chunks`: number of partitions of the
 * banded sweeps (0 = default).  out[16] (device):
 *   [0] ELBO  [1] dELBO/dvariance  [2] dELBO/dlengthscale  [3] dELBO/dsigma2
 *   [4] log|Kuu|  [5] log|P|  [6] b^T P^-1 b  [7] trace(Kuu^-1 G)  [8] info (0 ok, j+1 first non-positive pivot)
 *   [9..14] diagnostics (SM cycles of the chain phases)  [15] d trace(Kuu^-1 G) / d lengthscale. */
ASVGP_API int asvgp_elbo_grad_1d(const double* Kuu, const double* dKuu, const double* acc, int M, int order,
                                 double variance, double sigma2, int chunks, double* out, void* work,
                                 int64_t work_bytes, void* stream);

/* The same bound in two calls, split where its data dependencies are.  The Kuu chain (log|Kuu|, band(Kuu^-1), both with
 * their lengthscale tangents: gpr.py:56-70's cholesky_band(Kuu) / inverse_from_cholesky_band) depends on the
 * hyper-parameters only, so a caller can launch it on a side stream WHILE asvgp_accum_1d streams the data, and finish with
 * the P chains once the accumulator (and its all-reduce) is complete:
 *   asvgp_kuu_chain_1d(Kuu, dKuu, ..., kuu_state, work_a, side_stream);
 *   asvgp_accum_1d(..., acc, stream);  [all-reduce];
 *   asvgp_elbo_grad_1d_prepared(kuu_state, Kuu, dKuu, acc, ..., out, work_b, kuu_ready_event, stream);
 * `gate_event` (cudaEvent_t or NULL) is recorded on the side stream right before the chain kernel, after its parallel pre-pass:
 * a caller about to launch a machine-filling kernel on `stream` lets `stream` wait for it, so that the chain's few CTAs are
 * dispatched first instead of queueing behind the streaming kernel's thousands.
 * `kuu_ready_event`: a cudaEvent_t recorded on the side stream after asvgp_kuu_chain_1d (NULL if `stream` is already ordered
 * after it).  join_late = 0: `stream` waits for it up front and the trace(Kuu^-1 G) partial sums ride in the P chains'
 * pre-pass launch (the Kuu chain was launched long ago, e.g. before the accumulate).  join_late = 1: `stream` waits only where
 * the Kuu state is first read — after the P chains — so that without an accumulate in between (an optimiser iteration) the
 * Kuu chain and the P chains still run side by side.
 * `kuu_state`: asvgp_kuu_state_doubles(M, order) doubles on the device; the two calls need separate workspaces of
 * asvgp_workspace_bytes_1d bytes each when they may overlap.  asvgp_elbo_grad_1d is exactly these two calls on one stream. */
ASVGP_API int64_t asvgp_kuu_state_doubles(int M, int order);
ASVGP_API int asvgp_kuu_chain_1d(const double* Kuu, const double* dKuu, int M, int order, int chunks, double* kuu_state,
                                 void* work, int64_t work_bytes, void* gate_event, void* stream);
ASVGP_API int asvgp_elbo_grad_1d_prepared(const double* kuu_state, const double* Kuu, const double* dKuu, const double* acc,
                                          int M, int order, double variance, double sigma2, int chunks, double* out,
                                          void* work, int64_t work_bytes, void* kuu_ready_event, int join_late, void* stream);

/* ---- batched hyper-parameter evaluation -----------------------------------------------------------------------------------
 * B settings (v_b, l_b, sigma2_b) of the bound over the same data, in one stream of launches (a multi-start optimiser, a
 * lengthscale scan).  The data term does not depend on the hyper-parameters, so all slots share the accumulators.
 *
 * asvgp_kuu_assemble_batched: asvgp_kuu_assemble for B coefficient sets.  h_coef / h_dcoef are HOST arrays [B][n_terms]
 * (h_dcoef may be NULL: zeros); Kuu and dKuu (may be NULL) are [B][order+1][M].  Slot b's band equals asvgp_kuu_assemble with
 * row b of the coefficients bit for bit.
 *
 * asvgp_elbo_grad_1d_batched: `acc` holds D packed accumulators of asvgp_accum_1d, one per output column, contiguous
 * ([D][(order+2) M + 2]); Kuu / dKuu are [B][order+1][M]; h_variance / h_sigma2 are HOST arrays [B].  out[B][D][16] (device)
 * has the 16 slots of asvgp_elbo_grad_1d.  For the same `chunks`, out[b][d][0..8] and [15] equal asvgp_elbo_grad_1d on
 * (Kuu[b], dKuu[b], accumulator d, v_b, sigma2_b) bit for bit, whatever B, the other slots and the position of b in the batch;
 * [9..14] are that evaluation's own clock diagnostics.  A slot whose factorisation fails reports its pivot in its own info
 * slot and leaves the others untouched.  B outside 1..ASVGP_MAX_BATCH, D outside 1..ASVGP_MAX_BATCH_COLUMNS, a
 * non-positive v_b or sigma2_b and a workspace smaller than asvgp_workspace_bytes_1d_batched(M, order, chunks, B, D) bytes
 * are rejected before any CUDA call (the query returns -1 for arguments out of range). */
#define ASVGP_MAX_BATCH 64
#define ASVGP_MAX_BATCH_COLUMNS 64
ASVGP_API int asvgp_kuu_assemble_batched(const double* tables, int n_terms, int B, const double* h_coef, const double* h_dcoef,
                                         int M, int order, double* Kuu, double* dKuu, void* stream);
ASVGP_API int64_t asvgp_workspace_bytes_1d_batched(int M, int order, int chunks, int B, int D);
ASVGP_API int asvgp_elbo_grad_1d_batched(const double* Kuu, const double* dKuu, const double* acc, int M, int order, int B, int D,
                                         const double* h_variance, const double* h_sigma2, int chunks, double* out, void* work,
                                         int64_t work_bytes, void* stream);

/* ---- many independent series on one basis -----------------------------------------------------------------------------------
 * S series of 1-D data share the basis (mesh, order) but nothing else.  They travel concatenated: x[n], y[n] hold all points,
 * series s being points offsets[s] .. offsets[s+1] - 1, with offsets[S+1] int64, offsets[0] = 0, non-decreasing and
 * offsets[S] = n (the library does not check this contract; the Python layer does, on the host).  Empty series are allowed.
 *
 * asvgp_accum_1d_segmented_typed: asvgp_accum_1d_typed for every series at once.  acc holds S packed accumulators
 * ([S][(order+2) M + 2], layout of asvgp_accum_1d); series s's points are added into row s (nothing is zeroed), its count slot
 * receives offsets[s+1] - offsets[s].  Any order within a series is exact; sorted order is fast, as for asvgp_accum_1d.  x / y
 * element types as for asvgp_accum_1d_typed.  `offsets` is a DEVICE array.  S < 1 and unknown type codes are rejected before
 * any CUDA call.
 *
 * asvgp_elbo_grad_1d_batched_rows: asvgp_elbo_grad_1d_batched where slot b reads accumulator row h_row[b] of acc[R][D][L]
 * (column d of slot b at acc + (h_row[b] D + d) L, L = (order+2) M + 2).  h_row is a HOST array [B] of rows in 0..R-1 (repeats
 * allowed).  out[b][d][0..8] and [15] equal asvgp_elbo_grad_1d on (Kuu[b], dKuu[b], row h_row[b] column d, v_b, sigma2_b) bit for
 * bit, whatever B, the rows and the other slots.  asvgp_elbo_grad_1d_batched is this call with R = 1 and every row 0.  A row out
 * of range, a NULL h_row and the range checks of asvgp_elbo_grad_1d_batched are rejected before any CUDA call.
 *
 * asvgp_posterior_1d_batched: asvgp_posterior_1d for B slots (Kuu[B][order+1][M], sigma2_b from the HOST array h_sigma2[B],
 * accumulator row h_row[b] of acc[R][L]); alpha[B][M], S_band[B][order+1][M], info[B][2].  Slot b equals asvgp_posterior_1d on
 * its operands bit for bit; a failing slot reports its pivot in its own info and leaves the others untouched.  B lies in
 * 1..ASVGP_MAX_BATCH; the workspace needs asvgp_workspace_bytes_posterior_1d_batched(M, order, chunks, B) bytes (-1 for
 * arguments out of range).  asvgp_posterior_1d is the one-slot case.
 *
 * asvgp_predict_1d_segmented: asvgp_predict_1d per series: test points offsets_new[s] .. offsets_new[s+1] - 1 (DEVICE int64
 * [S+1], same contract as above) use alpha[s] of [S][M], S_band[s] of [S][order+1][M] and variance[s] of the DEVICE array
 * variance[S].  The per-point arithmetic is asvgp_predict_1d's. */
ASVGP_API int asvgp_accum_1d_segmented_typed(const void* x, int x_type, const void* y, int y_type, int64_t n, const int64_t* offsets,
                                             int S, const double* mesh, int n_knots, int order, double* acc, void* stream);
ASVGP_API int asvgp_elbo_grad_1d_batched_rows(const double* Kuu, const double* dKuu, const double* acc, int R, const int64_t* h_row,
                                              int M, int order, int B, int D, const double* h_variance, const double* h_sigma2,
                                              int chunks, double* out, void* work, int64_t work_bytes, void* stream);
ASVGP_API int64_t asvgp_workspace_bytes_posterior_1d_batched(int M, int order, int chunks, int B);
ASVGP_API int asvgp_posterior_1d_batched(const double* Kuu, const double* acc, int R, const int64_t* h_row, int M, int order, int B,
                                         const double* h_sigma2, int chunks, double* alpha, double* S_band, double* info, void* work,
                                         int64_t work_bytes, void* stream);
ASVGP_API int asvgp_predict_1d_segmented(const double* xnew, int64_t n, const int64_t* offsets_new, int S, const double* mesh,
                                         int n_knots, int order, const double* alpha, const double* S_band, const double* variance,
                                         double* mean, double* var, void* stream);

/* ---- a10 (factorisation half): posterior weights -------------------------------------------------------------------------
 * Replaces the CHOLMOD factorisations and solves of GPR_1d.predict_f (gpr.py:96-108):
 * alpha = P^-1 Kuf_y / sigma2 and S = band(P^-1) - band(Kuu^-1), P = Kuu + G / sigma2.  info[2] (device): failing
 * pivot of the Kuu / P factorisation or 0. */
ASVGP_API int asvgp_posterior_1d(const double* Kuu, const double* acc, int M, int order, double sigma2, int chunks,
                                 double* alpha, double* S_band, double* info, void* work, int64_t work_bytes,
                                 void* stream);

/* ---- band(A^-1) and log|A| with one tangent ------------------------------------------------------------------------------
 * Replaces banded.cholesky_band + banded.inverse_from_cholesky_band (gpr.py:56-59) and their TF gradients for ONE banded
 * SPD matrix A (lower band (order+1) x M) with tangent dA: sig_val = band(A^-1), sig_tan = band(-A^-1 dA A^-1),
 * scal[4] = { log|A|, d log|A|, info, 0 }.  Used per dimension by the Kronecker model (gpr.py:287-289,307). */
ASVGP_API int asvgp_band_inverse_1d(const double* A, const double* dA, int M, int order, int chunks, double* sig_val,
                                    double* sig_tan, double* scal, void* work, int64_t work_bytes, void* stream);

/* ==== 2-D (Kronecker) model =================================================================================================
 * Basis index (i1, i2) -> i1*m2 + i2 (kronecker.py:7-30), M = m1*m2.  Block-banded matrices travel in STENCIL layout:
 * S[e*M + j], e = d1*(2*order+1) + (d2+order), holding A[(j1+d1, j2+d2), (j1, j2)] for d1 in [0,order],
 * d2 in [-order,order], stored for d1 > 0 or (d1 == 0 and d2 >= 0); everything else is zero. */

/* Doubles of the per-cell moment table used by asvgp_accum_2d ((2o+1)^2 + (o+1)^2 per cell, plus one trailing slot the
 * library uses to select between its gridded-input and general kernels without a host round trip). */
ASVGP_API int64_t asvgp_accum_2d_moment_doubles(int n_knots1, int n_knots2, int order);

/* ---- a11 + a12: O(N) accumulation for the Kronecker model -----------------------------------------------------------------
 * Replaces GPR_kron.__init__'s per-dimension make_Kuf, kron.make_kvs_sparse (row-wise Khatri-Rao, kronecker.py:7-33),
 * `Kuf @ y` and `Kuf @ Kuf.T` (gpr.py:268-274).  X is row-major [n, 2].  Adds (does not zero) per-cell moments into
 * `cellmom` and { sum y^2, count } into scal[2]; both can be all-reduced across ranks before expansion. */
ASVGP_API int asvgp_accum_2d(const double* X, const double* y, int64_t n, const double* mesh1, int n_knots1,
                             const double* mesh2, int n_knots2, int order, double* cellmom, double* scal,
                             void* stream);

/* Same sums when the CALLER KNOWS the points are a flattened raster (np.meshgrid(x1, x2, indexing="ij"), x1 slow, rows of
 * `row_len` points whose x2 repeat from row to row — the eNATL60-shaped inputs): skips asvgp_accum_2d's on-device
 * classification probe and its unselected candidate kernels and launches the coalesced column sweep alone.  Every lane
 * still bit-compares each point with what the statement implies and falls back per row / per point, so a wrong statement
 * costs time, never correctness. */
ASVGP_API int asvgp_accum_2d_raster(const double* X, const double* y, int64_t n, int64_t row_len, const double* mesh1,
                                    int n_knots1, const double* mesh2, int n_knots2, int order, double* cellmom,
                                    double* scal, void* stream);

/* Same sums for points in NO PARTICULAR ORDER (SURVEY 8(d) C4 "shuffled-order variant").  asvgp_accum_2d is exact for
 * any order but pays (2o+1)^2 + (o+1)^2 fp64 REDs per point once consecutive points stop sharing a cell; this variant
 * partitions the points into <= 256 buckets of dimension-1 knot intervals, sorts each 4096-point unit by cell in
 * shared memory and accumulates every run in registers.  `work`: asvgp_accum_2d_binned_work_bytes(n) bytes of device
 * scratch (24 B per point + 8 KB).  asvgp_order_probe_2d writes to out[0] (device) the fraction of 4096 sampled
 * neighbour pairs that lie more than one cell apart (~0 raster / run order, ~1 shuffled). */
ASVGP_API int64_t asvgp_accum_2d_binned_work_bytes(int64_t n);
ASVGP_API int asvgp_accum_2d_binned(const double* X, const double* y, int64_t n, const double* mesh1, int n_knots1,
                                    const double* mesh2, int n_knots2, int order, double* cellmom, double* scal,
                                    void* work, int64_t work_bytes, void* stream);
ASVGP_API int asvgp_order_probe_2d(const double* X, int64_t n, const double* mesh1, int n_knots1, const double* mesh2,
                                   int n_knots2, double* out, void* stream);

/* Typed twins of the four entry points above (element types as for asvgp_accum_1d_typed; X [n, 2] has one type). */
ASVGP_API int asvgp_accum_2d_typed(const void* X, int x_type, const void* y, int y_type, int64_t n, const double* mesh1,
                                   int n_knots1, const double* mesh2, int n_knots2, int order, double* cellmom, double* scal,
                                   void* stream);
ASVGP_API int asvgp_accum_2d_raster_typed(const void* X, int x_type, const void* y, int y_type, int64_t n, int64_t row_len,
                                          const double* mesh1, int n_knots1, const double* mesh2, int n_knots2, int order,
                                          double* cellmom, double* scal, void* stream);
ASVGP_API int asvgp_accum_2d_binned_typed(const void* X, int x_type, const void* y, int y_type, int64_t n, const double* mesh1,
                                          int n_knots1, const double* mesh2, int n_knots2, int order, double* cellmom,
                                          double* scal, void* work, int64_t work_bytes, void* stream);
ASVGP_API int asvgp_order_probe_2d_typed(const void* X, int x_type, int64_t n, const double* mesh1, int n_knots1,
                                         const double* mesh2, int n_knots2, double* out, void* stream);

/* Expands the moment table into the Gram stencil Gs[(o+1)(2o+1) x M] and the projection b[M] (both must be zeroed by
 * the caller).  Cprod[(o+1)(o+1)(2o+1)], Dy[(o+1)(o+1)]: exact Bernstein-type expansion tables (host-computed). */
ASVGP_API int asvgp_expand_moments_2d(const double* cellmom, const double* Cprod, const double* Dy, int n_knots1,
                                      int n_knots2, int order, double* Gs, double* b, void* stream);

/* ---- a13 + a14: factorisation of P = K1 (x) K2 + G / sigma2 and its selected inverse ---------------------------------------------
 * Replaces utils.bands_to_kron_cholesky (utils.py:45-51), tf.linalg.cholesky(P), its log-det and
 * triangular_solve(L_P, Kuf_y) (gpr.py:287-295), and what the reference's dense cholesky_solve / TF reverse mode extract
 * from P^-1 (gpr.py:293-307, 319-326).
 *
 * asvgp_kron_*: nested-dissection multifrontal method (csrc/ndfront_2d.cu).  The m1 x m2 grid of basis functions is bisected
 * recursively by order-wide strips; every tree level is one batch of independent dense fronts (persistent tile-DAG kernels,
 * fp64 tensor cores); the dependency chain is 1751 columns at 200 x 200, order 3, instead of 40 000.  Kuf_y rides along as
 * an extra row of every front, so ||L^-1 Kuf_y||^2 and P^-1 Kuf_y need no separate solves.
 * Buffer sizes (doubles) come from the four queries below.
 *   band:   receives the factor (opaque);  rhs_io[m1 m2]: Kuf_y (input of asvgp_kron_factor; asvgp_kron_selinv overwrites it
 *           with P^-1 Kuf_y);  scal[3] = { log|P|, ||L^-1 Kuf_y||^2, info } with info = 0 ok, j+1 = basis function whose pivot
 *           was not positive, -1 internal time-out.
 *   asvgp_kron_selinv: sigma_stencil = entries of P^-1 in stencil layout, x_io = P^-1 Kuf_y.  `band` is CONSUMED; sig_band:
 *           asvgp_kron_sig_doubles of scratch; work: asvgp_kron_work_doubles.  An internal time-out poisons the outputs with NaN.
 * asvgp_kron_plan_info: diagnostics of the elimination tree, out[8] = { fronts, levels, tiles per pool, separator block
 *   columns, dependency chain in columns, in 64-column blocks, largest front, flops }; idx_out (may be NULL, capacity in ints):
 *   per front { level, ns, nb, ns separator ids, nb boundary ids (m1*m2 = the right-hand-side row) }; returns the ints needed. */
ASVGP_API int64_t asvgp_kron_band_doubles(int m1, int m2, int order);
ASVGP_API int64_t asvgp_kron_sig_doubles(int m1, int m2, int order);
ASVGP_API int64_t asvgp_kron_work_doubles(int m1, int m2, int order);
ASVGP_API int64_t asvgp_kron_rhs_doubles(int m1, int m2, int order);
ASVGP_API int64_t asvgp_kron_plan_info(int m1, int m2, int order, double* out, int32_t* idx_out, int64_t idx_capacity);
ASVGP_API int asvgp_kron_factor(const double* K1, const double* K2, const double* Gs, int m1, int m2, int order,
                                double sigma2, double* band, double* rhs_io, double* scal, void* stream);
ASVGP_API int asvgp_kron_selinv(double* band, int m1, int m2, int order, double* sig_band, double* x_io,
                                double* sigma_stencil, double* work, void* stream);

/* ---- several right-hand sides (multi-output targets y[N, D]) -----------------------------------------------------------------
 * P does not depend on y: one factorisation and one selected inverse serve D = n_rhs columns b_d = Kuf y_d, which ride along
 * as D extra boundary unknowns of every front (the root's boundary is exactly these D, one 64-wide tile).
 *   rhs_io[n_rhs x M]: column d at d*M (input of the factor; the selected inverse overwrites it with x_d = P^-1 b_d, same layout);
 *   scal[2 + n_rhs] = { log|P|, info, ||L^-1 b_1||^2, ..., ||L^-1 b_D||^2 } (info as for asvgp_kron_factor);
 *   sigma_stencil: entries of P^-1 in stencil layout, as for asvgp_kron_selinv.
 * asvgp_kron_doubles_multi: h_sizes[4] (HOST) = { band, sig, work, rhs } doubles of the buffers for this n_rhs.
 * asvgp_kron_plan_info_multi: asvgp_kron_plan_info for this n_rhs (rhs nodes m1*m2 ... m1*m2 + n_rhs - 1, the last n_rhs
 *   boundary ids of every front); -1 (with asvgp_last_error set) for invalid arguments.
 * The dense twins take rhs[n_rhs x n] and return x_out[n_rhs x n] and scal in the same layouts.
 * n_rhs lies in [1, ASVGP_MAX_RHS]: every front's boundary grows by n_rhs - 1 rows, and 32 keeps that growth within half a
 * 64-wide tile block (and the root's boundary within one tile); anything else is rejected before any CUDA call.  With
 * n_rhs = 1 every _multi function runs the plan and the arithmetic of its single-rhs counterpart, bit for bit. */
#define ASVGP_MAX_RHS 32
ASVGP_API int asvgp_kron_doubles_multi(int m1, int m2, int order, int n_rhs, int64_t* h_sizes);
ASVGP_API int64_t asvgp_kron_plan_info_multi(int m1, int m2, int order, int n_rhs, double* out, int32_t* idx_out,
                                             int64_t idx_capacity);
ASVGP_API int asvgp_kron_factor_multi(const double* K1, const double* K2, const double* Gs, int m1, int m2, int order, int n_rhs,
                                      double sigma2, double* band, double* rhs_io, double* scal, void* stream);
ASVGP_API int asvgp_kron_selinv_multi(double* band, int m1, int m2, int order, int n_rhs, double* sig_band, double* x_io,
                                      double* sigma_stencil, double* work, void* stream);

/* asvgp_kronband_*: the same two operations on the scalar band of P in the natural order (bandwidth order*(m2+1), gpr.py:262)
 * as one tile DAG over the band (csrc/tiledag_2d.cu) — a single chain over all m1 m2 columns, 10x slower at 200 x 200; kept
 * as an independent second implementation (the tests compare the two).  Same arguments, except that rhs_io has
 * asvgp_kronband_rhs_doubles entries (zero padded) and holds L^-1 Kuf_y between the two calls.
 * asvgp_kronband_colstat_offset: offset (doubles) inside `band` of the per-block-column diagnostics record, 20 doubles per
 * block column: [0] 2 sum log L_cc, [1] ||y_C||^2, [2..7] %globaltimer stamps of the factorisation's critical path,
 * [8..11] SM-cycle split of the diagonal tile's POTRF, [12..18] stamps of the selected inverse (tools/kron_chain_times.py). */
ASVGP_API int64_t asvgp_kronband_band_doubles(int m1, int m2, int order);
ASVGP_API int64_t asvgp_kronband_sig_doubles(int m1, int m2, int order);
ASVGP_API int64_t asvgp_kronband_work_doubles(int m1, int m2, int order);
ASVGP_API int64_t asvgp_kronband_rhs_doubles(int m1, int m2, int order);
ASVGP_API int64_t asvgp_kronband_colstat_offset(int m1, int m2, int order);
ASVGP_API int asvgp_kronband_factor(const double* K1, const double* K2, const double* Gs, int m1, int m2, int order,
                                    double sigma2, double* band, double* rhs_io, double* scal, void* stream);
ASVGP_API int asvgp_kronband_selinv(double* band, int m1, int m2, int order, double* sig_band, double* x_io,
                                    double* sigma_stencil, double* work, void* stream);

/* Scalar contractions for the ELBO gradient and the Kronecker trace term; out[11] (device):
 *   [0..3]  sum P^-1 .* Op,  [4..7]  x^T Op x   for Op = G, dK1(x)K2, K1(x)dK2, K1(x)K2
 *   [8..10] sum G .* (T1 (x) T2) for (T1,T2) = (S1,S2), (dS1,S2), (S1,dS2), S_i = band(K_i^-1). */
ASVGP_API int asvgp_kron_terms(const double* SigP, const double* Gs, const double* x, const double* K1,
                               const double* dK1, const double* K2, const double* dK2, const double* S1,
                               const double* dS1, const double* S2, const double* dS2, int m1, int m2, int order,
                               double* out, void* stream);

/* ---- a15: 2-D posterior mean / variance ----------------------------------------------------------------------------------------
 * Replaces GPR_kron.predict_f / predict_f_sparse (gpr.py:310-359): mean = w^T alpha, var = prior_var + w^T P^-1 w -
 * (a^T K1^-1 a)(b^T K2^-1 b), w = a (x) b.  SigP in stencil layout, S1/S2 lower bands of K1^-1/K2^-1.  The posterior is
 * first converted to per-cell polynomial form in `work` (asvgp_predict_2d_work_doubles doubles), then streamed over
 * the test points (32 B of traffic per point). */
ASVGP_API int64_t asvgp_predict_2d_work_doubles(int n_knots1, int n_knots2, int order);
/* The two halves of asvgp_predict_2d for callers that predict in several batches (the reference predicts in chunks of
 * 10 000 points, eNATL60.py:96-102): _prepare converts the posterior to per-cell polynomial form in `work` ONCE per set of
 * hyper-parameters, _apply streams one batch of test points through it.  row_len > 0 states that the batch is a flattened
 * raster with rows of row_len points (as asvgp_accum_2d_raster); 0 = classify on the device. */
ASVGP_API int asvgp_predict_2d_prepare(int n_knots1, int n_knots2, int order, const double* alpha, const double* SigP,
                                       const double* S1, const double* S2, double* work, void* stream);
ASVGP_API int asvgp_predict_2d_apply(const double* Xnew, int64_t n, int64_t row_len, const double* mesh1, int n_knots1,
                                     const double* mesh2, int n_knots2, int order, double prior_var, double* mean,
                                     double* var, double* work, void* stream);
ASVGP_API int asvgp_predict_2d(const double* Xnew, int64_t n, const double* mesh1, int n_knots1, const double* mesh2,
                               int n_knots2, int order, const double* alpha, const double* SigP, const double* S1,
                               const double* S2, double prior_var, double* mean, double* var, double* work,
                               void* stream);

/* ---- the one collective of the data-parallel path (SURVEY 8(e)) ---------------------------------------------------------------------------
 * One-shot all-reduce of a packed accumulator over NVLink peer memory: every rank's partial sums live in a symmetric buffer
 * (mapped into every peer); one kernel per rank does the cross-rank barrier (signal pads, system-scope release / acquire),
 * reads all peers' buffers and adds them in rank order (bit-identical result on every rank).  buffer_ptrs / pad_ptrs: device
 * arrays of `world` 64-bit addresses of every rank's buffer / signal pad.  `epoch` increases by one per call, identically on all
 * ranks; callers double-buffer the symmetric buffers (asvgp_b200/dist.py).  status[1] (device int): 1 if a peer never arrived
 * (the output is then NaN; waits are bounded).  Replaces torch.distributed.all_reduce (NCCL) for this buffer. */
ASVGP_API int asvgp_allreduce_oneshot(const void* buffer_ptrs, const void* pad_ptrs, int rank, int world, int64_t offset_doubles,
                                      int64_t n, unsigned epoch, int pad_offset, double* out, int* status, void* stream);

/* ---- dense SPD matrices on the front kernels ----------------------------------------------------------------------------------------
 * Replaces tf.linalg.cholesky / triangular_solve / cholesky_solve of a DENSE matrix (GPR_additive, gpr.py:192-195, 221-231):
 * one front of the nested-dissection machinery above.  A: n x n row-major (lower triangle read), n <= 32768.
 * asvgp_dense_factor: scal[3] = { log|A|, rhs^T A^-1 rhs, info }.  asvgp_dense_selinv (consumes band): x_out = A^-1 rhs,
 * inv_out[n x n] = A^-1 (full, symmetric). */
ASVGP_API int64_t asvgp_dense_band_doubles(int n);
ASVGP_API int64_t asvgp_dense_sig_doubles(int n);
ASVGP_API int64_t asvgp_dense_work_doubles(int n);
ASVGP_API int asvgp_dense_factor(const double* A, int n, const double* rhs, double* band, double* scal, void* stream);
ASVGP_API int asvgp_dense_selinv(double* band, int n, double* sig_band, double* x_out, double* inv_out, double* work,
                                 void* stream);
/* n_rhs right-hand sides (layouts as for asvgp_kron_factor_multi): rhs[n_rhs x n], scal[2 + n_rhs] = { log|A|, info,
 * rhs_d^T A^-1 rhs_d ... }, x_out[n_rhs x n]; h_sizes[4] (HOST) = { band, sig, work, rhs } doubles. */
ASVGP_API int asvgp_dense_doubles_multi(int n, int n_rhs, int64_t* h_sizes);
ASVGP_API int asvgp_dense_factor_multi(const double* A, int n, int n_rhs, const double* rhs, double* band, double* scal,
                                       void* stream);
ASVGP_API int asvgp_dense_selinv_multi(double* band, int n, int n_rhs, double* sig_band, double* x_out, double* inv_out,
                                       double* work, void* stream);

/* ---- GPR_additive (gpr.py:139-236): sum of 1-D models, Kuf = stacked per-dimension features ------------------------------------------
 * asvgp_accum_cross: C[m_a x m_b] += Kuf_a Kuf_b^T for two dimensions of the same points (xa[i * stride], xb[i * stride]) — the
 *   dense off-diagonal blocks of `Kuf @ Kuf.T` (gpr.py:174-175); the banded diagonal blocks are asvgp_accum_1d's.
 * asvgp_additive_put_band / _put_cross: write (add != 0: add) scale * (a lower band as a symmetric block) at `offset` on the
 *   diagonal of the dense M x M matrix `out`; write a cross block and its transpose.  asvgp_additive_scale: P = G / sigma2.
 *   Together: KufKfu (gpr.py:175) and `Kuu.to_dense() + KufKfu / sigma2` (gpr.py:192).
 * asvgp_additive_terms: out4 = { sum S_dd .* K_d, sum S_dd .* dK_d, x_d^T K_d x_d, x_d^T dK_d x_d } for the diagonal block of
 *   dimension d of S = P^-1 (dense) and x = P^-1 Kuf_y;  asvgp_dense_terms: out2 = { sum S .* G, x^T G x }.  These are what the
 *   derivatives of the bound need (TF reverse mode in the reference).
 * asvgp_predict_additive: GPR_additive.predict_f (gpr.py:212-236).  Xnew[n, D] row-major, D <= 8; meshes = all knot arrays
 *   concatenated; meta[4 d ..] = { knot offset, number of knots, first basis function, m_d } (device ints); S_all = the lower
 *   bands of K_d^-1 concatenated in dimension order. */
ASVGP_API int asvgp_accum_cross(const double* xa, const double* xb, int64_t stride, int64_t n, const double* mesh_a,
                                int n_knots_a, const double* mesh_b, int n_knots_b, int order, double* C, void* stream);
ASVGP_API int asvgp_additive_put_band(const double* band, int m, int order, int offset, int M, double scale, int add,
                                      double* out, void* stream);
ASVGP_API int asvgp_additive_put_cross(const double* C, int m_a, int m_b, int offset_a, int offset_b, int M, double* out,
                                       void* stream);
ASVGP_API int asvgp_additive_scale(const double* G, int M, double sigma2, double* P, void* stream);
ASVGP_API int asvgp_additive_terms(const double* Pinv, const double* x, int M, int offset, int m, int order, const double* Kd,
                                   const double* dKd, double* out4, void* stream);
ASVGP_API int asvgp_dense_terms(const double* Pinv, const double* G, const double* x, int M, double* out2, void* stream);
ASVGP_API int asvgp_predict_additive(const double* Xnew, int64_t n, int D, const double* meshes, const int* meta, int M,
                                     int order, const double* alpha, const double* Pinv, const double* S_all,
                                     double prior_var, double* mean, double* var, void* stream);

/* ---- name-for-name counterparts of the reference's Kronecker helpers (not used by the models) -------------------------------
 * asvgp_khatri_rao_csc replaces kronecker.make_kvs_two_sparse (kronecker.py:7-27; make_kvs_sparse folds it over a list,
 * :29-33): row-wise Khatri-Rao product of two sparse feature matrices in CSC form with int64 indices, column n of the
 * result holding A[ia, n] * B[ib, n] at row ia * m_b + ib.  out_indptr[n_cols + 1] is the caller's prefix sum of
 * nnzA(n) * nnzB(n); out_indices / out_data have out_indptr[n_cols] entries.
 * asvgp_kron_dense / asvgp_cholesky_dense replace the dense Kronecker products and the per-dimension tf.linalg.cholesky
 * of utils.bands_to_kron_cholesky (utils.py:45-51): row-major dense in, row-major dense out ((m_a m_b)^2 doubles);
 * info[1] (device) = 0 or the 1-based first non-positive pivot. */
ASVGP_API int asvgp_khatri_rao_csc(const int64_t* indptr_a, const int64_t* indices_a, const double* data_a,
                                   const int64_t* indptr_b, const int64_t* indices_b, const double* data_b,
                                   int64_t n_cols, int64_t m_b, const int64_t* out_indptr, int64_t* out_indices,
                                   double* out_data, void* stream);
ASVGP_API int asvgp_kron_dense(const double* A, int m_a, const double* B, int m_b, double* out, void* stream);
ASVGP_API int asvgp_cholesky_dense(const double* A, int m, double* L, double* info, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ASVGP_B200_H */
