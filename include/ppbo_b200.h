/* ppbo_b200 -- C ABI of the B200 (sm_100a) implementation of the PPBO hot path.
 *
 * Drop-in boundary: the reference (AaltoPML/PPBO) is pure Python; its hot path calls numpy / scipy /
 * LAPACK from src/gp_model.py, src/kernels.py, src/misc.py, src/acquisition.py and
 * src/random_fourier_sampler.py.  A maintainer binds this library with ctypes (INTEGRATION.md) and the
 * entry points below replace those call sites one for one; each comment names the reference lines it
 * replaces.  All matrices are row-major (numpy C order) float64.  Unless a parameter name ends in `_h`,
 * every pointer is a DEVICE pointer (torch tensor .data_ptr()); `stream` is a cudaStream_t passed as
 * void*.  Return value: 0 = OK, > 0 = LAPACK-style info (e.g. index of the first non-positive pivot),
 * < 0 = error (-1 bad argument, -2 CUDA failure); ppbo_last_error() gives the message.
 * There is no CPU fallback anywhere in this library.
 */
#ifndef PPBO_B200_H
#define PPBO_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define PPBO_KERNEL_SE 0       /* src/kernels.py:19-25 (ARD generalisation: one length-scale per dim) */
#define PPBO_KERNEL_RQ 1       /* src/kernels.py:27-34 (alpha = 2)                                     */
#define PPBO_KERNEL_CAMPHOR 2  /* src/kernels.py:36-53                                                 */
#define PPBO_KERNEL_SQDIST 3   /* internal: squared Euclidean distance (ppbo_sqdist)                   */
#define PPBO_KERNEL_MATERN32 4 /* sf^2 (1 + sqrt3 r) exp(-sqrt3 r), r = |(x - y) / l| (ARD as for SE)   */
#define PPBO_KERNEL_MATERN52 5 /* sf^2 (1 + sqrt5 r + 5 r^2 / 3) exp(-sqrt5 r)                          */

int ppbo_version(void);
const char* ppbo_last_error(void);
/* device properties the host layer reports (SM count etc.); dev = CUDA ordinal */
int ppbo_device_sm_count(int dev);
/* number of CUDA kernels this library has launched so far in this process (bench.py: gpu_launches) */
long long ppbo_launch_count(void);
/* Switches for reference paths and launch shapes; 0 is the default of every key.  Any other key returns -1.
 *   4  column-tile groups of the INT8 contraction (> 0: that many)
 *   8  1: panel and look-ahead GEMMs of the Cholesky through the general GEMM kernel
 *   9  1: trailing update of the Cholesky through the general GEMM kernel (0 or 1 only)
 *   11 1: difference-form covariance and posterior-mean kernels instead of the tensor-pipe ones
 *   14 SMs the INT8 contraction leaves free (> 0: that many; -1: one CTA per work item)
 *   15 grid of the symmetric mat-vec tile kernel (> 0: that many CTAs) */
int ppbo_set_tuning(int key, int value);
/* host-thread role for concurrent fits (no reference counterpart: the reference is single-threaded, ppbo_numerical_main.py:192);
 * background threads get lowest-priority internal streams */
int ppbo_set_thread_background(int on);

/* ---- K1: covariance matrices -------------------------------------------------------------------- */
/* out[n1 x n2] = k(X1_i, X2_j).  Replaces kernels.SE_kernel / RQ_kernel / camphor_copper_kernel and
 * GPModel.create_Gramian_nonsquare (src/gp_model.py:153-155).  lengthscales_h: D host doubles. */
int ppbo_kernel_matrix(int kind, const double* X1, int n1, const double* X2, int n2, int D,
                       const double* lengthscales_h, double sigma_f, double* out, long long ld, void* stream);
/* out[n1 x n2] = |X1_i - X2_j|^2.  Replaces kernels.dist (src/kernels.py:3-11). */
int ppbo_sqdist(const double* X1, int n1, const double* X2, int n2, int D, double* out, long long ld, void* stream);
/* out[n x n] = (1-s) K(X,X) + s * (tr K / n) I, tr K / n == sigma_f^2 for these stationary kernels.
 * Replaces GPModel.create_Gramian = kernel + misc.regularize_covariance (src/gp_model.py:147-151,
 * src/misc.py:71-88: the SVD round trip is the identity, the shrinkage is fused). */
int ppbo_gram_regularized(int kind, const double* X, int n, int D, const double* lengthscales_h,
                          double sigma_f, double shrinkage, double* out, long long ld, void* stream);
/* K <- (1-s) K + s (tr K / n) I in place for an arbitrary square matrix (misc.regularize_covariance on a caller-supplied
 * matrix, src/misc.py:71-88).  scratch1: one device double. */
int ppbo_shrink_inplace(double* K, long long ld, int n, double shrinkage, double* scratch1, void* stream);
/* Rows / columns [n_old, n_new) of the regularised covariance of X[0 : n_new] written in place into out (leading dimension
 * ld >= n_new); the leading n_old x n_old block is not touched.  One (m+1)-row block is appended per PPBO iteration
 * (FeedbackProcessing.update_X, src/feedback_processing.py:133-154) while the reference rebuilds Sigma from scratch
 * (GPModel.update_Sigma, src/gp_model.py:157); the shrinkage term is N-independent for these stationary kernels, so the old
 * matrix is the leading block of the new one.  Bit-identical to ppbo_gram_regularized on X[0 : n_new]. */
int ppbo_gram_append(int kind, const double* X, int n_old, int n_new, int D, const double* lengthscales_h, double sigma_f,
                     double shrinkage, double* out, long long ld, void* stream);
/* analytic dK/dlog(l_d) and dK/dlog(sigma_f) for the SE kernel (north_star piece 1; the reference has
 * no gradient -- checked against finite differences of SE_kernel).  dK: [(D+1)][n1 x n2] */
int ppbo_kernel_se_grad(const double* X1, int n1, const double* X2, int n2, int D,
                        const double* lengthscales_h, double sigma_f, double* dK, long long ld,
                        long long stride, void* stream);

/* ---- K2: preference-likelihood terms and the Laplace fit ---------------------------------------- */
/* Comparison-set layout: set q = rows q(m+1) .. q(m+1)+m of f, winner first
 * (src/feedback_processing.py:121-123).  Outputs (any may be NULL):
 *   lik_sum[1]  = sum_q sum_j Phi(Delta_qj / sqrt 2)             (GPModel.sum_Phi order 0, src/gp_model.py:176-193)
 *   beta[N]     = likelihood gradient                            (GPModel.T_grad, src/gp_model.py:234-238)
 *   arrow[Q*m]  = a_qj = -Delta phi~(Delta) / (2 m sigma^2)      (GPModel.create_Lambda, src/gp_model.py:249-274) */
int ppbo_lik_terms(const double* f, int Q, int m, double sigma, double* lik_sum, double* beta,
                   double* arrow, void* stream);
/* set_sums[Q]: the per-comparison-set values sum_j Phi(Delta_qj / sqrt 2) (GPModel.sum_Phi_vec order 0, src/gp_model.py:206-218) */
int ppbo_lik_set_sums(const double* f, int Q, int m, double sigma, double* set_sums, void* stream);
/* dense Lambda[N x N] from the arrow coefficients (public attr GPModel.Lambda_MAP) */
int ppbo_lambda_dense(const double* arrow, int Q, int m, double* out, long long ld, void* stream);
/* G[Qm x Qm] = B^T Sigma B, the prior covariance of the latent differences f_j - f_winner.  Qm <= 65535 (one grid row per row of G;
 * the same limit holds for ppbo_diffspace_gram_append, ppbo_laplace_fit and ppbo_laplace_refactor) */
int ppbo_diffspace_gram(const double* Sigma, long long lds, int Q, int m, double* G, long long ldg, void* stream);

/* the same for appended comparison sets: entries of G with a row or a column in [Q_old m, Q_new m), in place (bit-identical to
 * ppbo_diffspace_gram on the grown Sigma) */
int ppbo_diffspace_gram_append(const double* Sigma, long long lds, int Q_old, int Q_new, int m, double* G, long long ldg,
                               void* stream);

/* doubles in a "factor object" of capacity n: n*n matrix (leading dimension n) followed by the inverted 128x128 diagonal blocks */
long long ppbo_factor_doubles(int n);
/* workspace (bytes) needed by ppbo_laplace_fit */
long long ppbo_laplace_workspace_bytes(int Q, int m);
/* MAP of T(f) = -1/2 f' Sigma^-1 f - (1/m) sum Phi(Delta/sqrt2)  (GPModel.update_fMAP, src/gp_model.py:354-389,
 * replaces scipy trust-exact): damped Newton in difference space, every Newton step one Cholesky of
 * I + a^1/2 (B' Sigma B) a^1/2 (size Qm), followed by factor-reusing chord steps.  f_init may be NULL (start at 0).
 * G [>= Qm x Qm, leading dimension ldg] and Lfac (factor object of capacity cap >= Qm) may be larger than the problem so that a
 * model can grow in place.  flags:
 *   PPBO_FIT_G_READY        G already holds B' Sigma B (ppbo_diffspace_gram / _append); otherwise it is formed here
 *   PPBO_FIT_FACTOR_WARM    Lfac holds chol(I + s G s) of the leading warm_rows x warm_rows system for s = sa_fac (the previous
 *                           iteration's factor; warm_rows = Qm when nothing was appended).  The fit starts with chord steps
 *                           from (f_init, alpha_init = Sigma^-1 f_init) and factorises only if they contract too slowly; up to
 *                           64 appended rows are carried as a BORDER of the old factor (Schur complement of the new rows with
 *                           their current coefficients in every step), so the steady-state iteration is O(M^2 m)
 *                           (the reference's warm start pads the previous fMAP, src/gp_model.py:375-377)
 *   PPBO_FIT_FACTOR_AT_MODE finish with the factor of I + a+^1/2 G a+^1/2 AT the mode (what ppbo_predict with covariance and
 *                           ppbo_neg_corr_build need); without it Lfac keeps the last factor used and ppbo_laplace_refactor
 *                           builds the mode factor on demand (the posterior mean needs alpha only)
 * binv_cache (may be NULL; ppbo_blockinv_bytes(cap) bytes) with binv_state_h[2] (host, in/out; {0, 0} initially): persistent home
 *          of the factor's 1024-block inverses -- a factor that only grows at its end keeps its leading blocks between fits.
 * alpha_init (may be NULL): Sigma^-1 f_init when the caller knows it (a warm start from the previous (f, alpha) with zeros
 *          appended to alpha and Sigma_new,old alpha_old appended to f is consistent by construction).
 * Outputs: f_map[N], alpha[N] = Sigma^-1 f_map, arrow[Qm] (signed coefficients at the mode), sa_fac[Qm] (may be NULL) = the
 *          clamped square roots the factor left in Lfac was built with (a bordered fit writes the grown factor back),
 *          stats_h[12] host doubles: iterations, last step inf-norm, last relative step, T(f_map), line-search halvings,
 *          info, Cholesky factorisations, chord steps, factor state (2 at the mode / 1 last Newton or warm factor / 0 none),
 *          converged (1/0), relative size of the first warm step, border rows */
#define PPBO_FIT_G_READY 1
#define PPBO_FIT_FACTOR_WARM 2
#define PPBO_FIT_FACTOR_AT_MODE 4
int ppbo_laplace_fit(const double* Sigma, long long lds, int Q, int m, double sigma, const double* f_init,
                     const double* alpha_init, int max_iter, double tol, int flags, double* G, long long ldg, double* Lfac,
                     int cap, double* sa_fac, int warm_rows, double* binv_cache, int* binv_state_h, double* f_map, double* alpha,
                     double* arrow, void* workspace, long long workspace_bytes, double* stats_h, void* stream);
/* factor of I + a+^1/2 G a+^1/2 for the coefficients `arrow` (a fit that skipped PPBO_FIT_FACTOR_AT_MODE); sa_fac[M] receives
 * sqrt(max(arrow, 0)).  Returns 0 or the index of the first non-positive pivot. */
int ppbo_laplace_refactor(const double* G, long long ldg, int M, const double* arrow, double* Lfac, int cap, double* sa_fac,
                          void* stream);
/* Grow chol(I + s G s) from M_old to M_new rows after comparison sets were appended (G grown by ppbo_diffspace_gram_append).
 * The coefficients of the new rows, sa_fac[M_old : M_new), are taken as given (f_new_sets == NULL) or computed here from the
 * warm-start values f_new_sets[(M_new - M_old) / m * (m + 1)] of the appended sets (winner first), s = sqrt(max(a(f), 0)).
 * Only the block rows from the last 128-row boundary on are recomputed -- O(M^2 m) work instead of the O(M^3 / 3) of a new
 * factorisation.  The reference refactors its N x N Hessian from scratch inside every trust-exact iteration
 * (src/gp_model.py:382-384).  Returns 0 or the first non-positive pivot. */
int ppbo_factor_extend(const double* G, long long ldg, int M_old, int M_new, double* sa_fac, const double* f_new_sets, int m,
                       double sigma, double* Lfac, int cap, void* stream);

/* out[N x N] = I + Sigma W (reference_sign = 0) or I - Sigma W = I + Sigma Lambda_MAP (reference_sign = 1: the matrix
 * GPModel.evidence factors, src/gp_model.py:301-302), W = B diag(arrow) B' with the SIGNED coefficients.  N = Q (m+1) <= 65535. */
int ppbo_evidence_matrix(const double* Sigma, long long lds, int Q, int m, const double* arrow, int reference_sign, double* out,
                         long long ldo, void* stream);

/* ---- dense FP64 linear algebra (replaces the LAPACK/BLAS calls under numpy/scipy) ---------------- */
/* C[M x N] = alpha * A[M x K] . B[N x K]^T + beta * C   (row-major, K contiguous in A and B) */
int ppbo_gemm_nt(const double* A, long long lda, const double* B, long long ldb, double* C, long long ldc,
                 int M, int N, int K, double alpha, double beta, void* stream);
/* lower tiles of C = alpha A B^T + beta C for a square C[N x N], in the tile configuration of ppbo_gemm_nt (same bits below the
 * diagonal); tiles above the diagonal are not written */
int ppbo_gemm_nt_lower(const double* A, long long lda, const double* B, long long ldb, double* C, long long ldc, int N, int K,
                       double alpha, double beta, void* stream);
/* tuning entry: ppbo_gemm_nt with an explicit tile configuration index (scripts/ubench_ops.py) */
int ppbo_gemm_nt_cfg(int cfg, const double* A, long long lda, const double* B, long long ldb, double* C, long long ldc,
                     int M, int N, int K, double alpha, double beta, void* stream);
long long ppbo_potrf_workspace_bytes(int n);
/* in-place lower Cholesky of the lower triangle of A[n x n]; the upper triangle is never read, and it is untouched outside the
 * 128 x 128 diagonal blocks (inside them the trailing updates write whole tiles: scratch there).  info_h: host int,
 * 0 or 1-based index of the first non-positive pivot.  Replaces dpotrf under scipy.linalg.solve(assume_a='pos')
 * (src/misc.py:96-100) and under scipy's trust-exact. */
int ppbo_potrf_lower(double* A, long long lda, int n, void* workspace, long long workspace_bytes, int* info_h,
                     void* stream);
/* X[nrhs x n] (row-major, one right-hand side per ROW) <- X . L^-T (trans=0)  or  X . L^-1 (trans=1) */
int ppbo_trsm_right_lower(const double* L, long long ldl, int n, double* X, long long ldx, int nrhs, int trans,
                          void* workspace, long long workspace_bytes, void* stream);
/* x <- (L L^T)^-1 x for one right-hand side; x must have room for n + 128 doubles (scratch tail).  Replaces cho_solve
 * under scipy's trust-exact (src/gp_model.py:382-384). */
int ppbo_potrs_vec(const double* L, long long ldl, int n, double* x, void* workspace, long long workspace_bytes, void* stream);
/* The same solve for a factor that serves MANY right-hand sides (chord steps of the Newton iterations): the diagonal blocks of
 * L are inverted once at 1024 x 1024 granularity (from the 128 x 128 inverses ppbo_potrf_lower left in its workspace), after
 * which each solve is n/1024 steps of two bandwidth-bound matrix-vector kernels instead of a 40-link dependency chain.
 * Replaces the cho_solve calls inside scipy's trust-exact (src/gp_model.py:382, src/random_fourier_sampler.py:128). */
long long ppbo_blockinv_bytes(int n);
int ppbo_blockinv_build(const double* L, long long ldl, int n, const void* potrf_workspace, void* blockinv,
                        long long blockinv_bytes, void* stream);
int ppbo_potrs_vec_blockinv(const double* L, long long ldl, int n, void* blockinv, long long blockinv_bytes, double* x,
                            void* stream);
/* out = (L L^T)^-1 (dense, symmetric) from the factor and workspace of ppbo_potrf_lower; work: n*n doubles.
 * Replaces misc.pd_inverse (src/misc.py:96-100; LAPACK dposv with an identity right-hand side) where a caller reads an
 * explicit inverse (GPModel.Sigma_inv, posterior_covariance). */
int ppbo_potri_lower(const double* L, long long ldl, int n, void* workspace, long long workspace_bytes, double* work,
                     double* out, long long ldo, void* stream);
/* In-place LU with partial pivoting (largest magnitude, first index on ties -- LAPACK dgetrf's rule) of A[n x n];
 * result_h[3] = { sign(det U), log|det A|, sign of the row permutation }.  Replaces scipy.linalg.lu + numpy.linalg.slogdet in
 * GPModel.evidence (src/gp_model.py:303-308).  Returns 1 when a pivot is exactly zero. */
long long ppbo_lu_workspace_bytes(int n);
int ppbo_lu_logdet(double* A, long long lda, int n, void* workspace, long long workspace_bytes, double* result_h, void* stream);
/* y = A x for row-major A[M x N] */
int ppbo_gemv(const double* A, long long lda, int M, int N, const double* x, double* y, void* stream);
/* y = A x for a symmetric A[n x n], reading only its lower triangle; the bits do not depend on the launch grid */
int ppbo_symv_lower(const double* A, long long lda, int n, const double* x, double* y, void* stream);

/* ---- K4: prediction and exact-GP acquisition ----------------------------------------------------- */
long long ppbo_predict_workspace_bytes(int N, int Q, int m, int P, int batch);
/* workspace of a mean-only call (Sigma_p == NULL): the mat-vec mode of the SE / RQ / Matern / camphor kernels (camphor as an SE
 * kernel on lifted coordinates) never materialises the cross-covariance */
long long ppbo_predict_mean_workspace_bytes(int kind, int N, int P, int batch);
/* Posterior mean and covariance on `batch` grids of P points each (Xp: [batch*P x D]).
 * mu = k*' alpha ; Sigma_p = reg(K**) - k*' (Sigma^-1 - Sigma^-1 Post Sigma^-1) k*  evaluated as
 * reg(K**) - Y'Y (+ low-rank term for negative arrow coefficients), Y = Lfac^-1 a+^1/2 B' k*.
 * Replaces GPModel.mu_Sigma_pred (src/gp_model.py:441-452).  mu: [batch*P], Sigma_p: [batch][P x P] (may be NULL).
 * P * batch is not bounded by a launch dimension (the per-point kernels loop over grid rows). */
/* Negative arrow coefficients at the mode (data that contradict the fit) make W = B a B' indefinite; the factor
 * object only carries a+ = max(a,0).  These three calls build the exact low-rank correction
 * (Woodbury on the r negative columns) that ppbo_predict adds: count (host sync; indices to idx_h), size, build. */
int ppbo_neg_count(const double* arrow, int M, int* idx_h, int idx_capacity, void* stream);
long long ppbo_neg_corr_doubles(int M, int r);
int ppbo_neg_corr_build(const double* G, long long ldg, int M, const double* arrow, const double* Lfac, int cap,
                        const int* idx_h, int r, double* neg_corr, void* stream);
/* Lfac: factor object of capacity cap holding the factor AT the mode (only read when Sigma_p != NULL) */
int ppbo_predict(int kind, const double* X, int N, int D, const double* lengthscales_h, double sigma_f,
                 double shrinkage, int Q, int m, const double* alpha, const double* arrow, const double* Lfac, int cap,
                 const double* neg_corr, int n_neg, const double* Xp, int P, int batch, double* mu,
                 double* Sigma_p, void* workspace, long long workspace_bytes, void* stream);
/* mu_h[0] = k(x, X) alpha for ONE point given and returned in HOST memory (x_h[D], mu_h[1]); one launch, no allocation, the
 * call returns when the value is on the host.  Replaces GPModel.mu_pred (src/gp_model.py:454-458) inside the sequential
 * differential evolution of GPModel.mu_star (src/gp_model.py:415-437: ~10^4 dependent evaluations per model update). */
int ppbo_mu_pred_point(int kind, const double* X, int N, int D, const double* lengthscales_h, double sigma_f, const double* alpha,
                       const double* x_h, double* mu_h, void* stream);
/* The sequential differential evolution of GPModel.mu_star (src/gp_model.py:415-437: scipy.optimize.differential_evolution(
 * mu_pred_neq, bounds, updating='immediate', maxiter=2000)) with the loop on the host in C++ instead of in scipy's Python: strategy
 * 'best1bin', latin-hypercube start, population popsize x D, dither in [mutation_lo, mutation_hi), stop when
 * std(energies) <= atol + tol |mean(energies)|.  It replays scipy 1.18 on numpy's legacy global stream draw for draw: mt_key[624] /
 * mt_pos are the MT19937 state of numpy.random.get_state() on entry and the state to hand to set_state() on return, and the
 * trial vectors, accepted members, stopping generation and result are bit for bit those of the scipy call on the same objective.
 * The L-BFGS-B polish scipy runs afterwards is left to the caller.  All pointers are HOST pointers.
 * x_h[D] / fun_h[1]: best member in problem units and its value; stats_h[6] (may be NULL): generations, evaluations (as scipy
 * counts them), converged, population size, discarded evaluations, calls of f / f_batch.  An objective that returns NaN stops the
 * search with an error.
 * window > 1: under 'immediate' updating a trial reads the best member, two sampled members and its own, so the next `window`
 * trials are built from the population as it is and evaluated in one call (f_batch: B rows of x_h -> f_h[B], return 0; one launch
 * on the device); the results are walked in order, and the window is cut at the first trial made stale by an earlier acceptance
 * (a new best member, or a replaced row among its two sampled ones), the stream put back to where it was before that trial was
 * built.  Same draws, same comparisons, same result bits; about one launch per ten retained evaluations at window 16 .. 32.
 * window = 1 (or f_batch NULL): one call of f per trial.
 *   ppbo_de_minimize : any objective given as a callback (the CPU tests compare it with scipy through this entry)
 *   ppbo_mu_star_de  : objective -mu(x) = -k(x, X) alpha on the device (X, alpha: DEVICE), ppbo_mu_pred_point(s) per trial / window */
typedef double (*ppbo_objective_fn)(const double* x_h, int D, void* ctx);
typedef int (*ppbo_objective_batch_fn)(const double* x_h, int B, int D, double* f_h, void* ctx);
int ppbo_de_minimize(ppbo_objective_fn f, ppbo_objective_batch_fn f_batch, int window, void* ctx, int D, const double* lower_h,
                     const double* upper_h, int popsize, int maxiter, double tol, double atol, double mutation_lo,
                     double mutation_hi, double recombination, unsigned int* mt_key, int* mt_pos, double* x_h, double* fun_h,
                     int* stats_h);
int ppbo_mu_star_de(int kind, const double* X, int N, int D, const double* lengthscales_h, double sigma_f, const double* alpha,
                    const double* lower_h, const double* upper_h, int popsize, int maxiter, double tol, double atol,
                    double mutation_lo, double mutation_hi, double recombination, int window, unsigned int* mt_key, int* mt_pos,
                    double* x_h, double* fun_h, int* stats_h, void* stream);
/* B <= 64 points per launch, arguments and results in HOST memory (x_h[B][D], mu_h[B]); point b is evaluated by one CTA with the
 * arithmetic of ppbo_mu_pred_point (same bits).  GPModel.mu_pred (src/gp_model.py:454-458) for the windows above. */
int ppbo_mu_pred_points(int kind, const double* X, int N, int D, const double* lengthscales_h, double sigma_f, const double* alpha,
                        const double* x_h, int B, double* mu_h, void* stream);
/* Multi-start ascent of the posterior mean mu(x) = sum_i alpha_i k(x, X_i) over [0,1]^D (X [N][D], alpha [N], X0 [R][D]: DEVICE),
 * one CTA per start: the projected gradient ascent of ppbo_rff_maximize with the value and the analytic gradient of mu fused in
 * one pass over the design.  Stops when the projected gradient is below gtol * sigma_f^2 * sum_i |alpha_i| (relative to the bound
 * on |mu|) or after max_iter steps; periodic_mask as for ppbo_rff_maximize (camphor: 0b111011).  Per start (DEVICE): the end point
 * xout[R][D], mu there fout[R], the gradient there gout[R][D] and the steps taken iters[R]; xbest[D], fbest[1] = the best start
 * (the lowest index on ties).  max_iter = 0: mu and its gradient at the starts (projected onto the box / wrapped).
 * D <= 32; every kernel kind but PPBO_KERNEL_SQDIST. */
int ppbo_mu_maximize(int kind, const double* X, int N, int D, const double* lengthscales_h, double sigma_f, const double* alpha,
                     const double* X0, int R, int max_iter, double gtol, int periodic_mask, double* xout, double* fout, double* gout,
                     int* iters, double* xbest, double* fbest, void* stream);
/* fmax[b][s] = max_p ( mu[b][p] + sum_k Z[b][s][k] Fac[b][p][k] ), arg[b][s] = first arg-max.
 * Replaces the S calls of np.random.multivariate_normal + np.max in acquisition.EI / varmax
 * (src/acquisition.py:78-80, 175-177); Fac is the (P x P) sampling factor (row p = coefficients of point p). */
int ppbo_mvn_rowmax(const double* Z, long long ldz, long long strideZ, const double* Fac, long long ldf,
                    long long strideF, const double* mu, long long strideMu, int S, int P, int K, int batch,
                    double* fmax, int* arg, void* stream);
/* per batch entry: out[b][0] = sum_s max(fmax-mustar,0), out[b][1] = sum_s fmax, out[b][2] = sum_s fmax^2
 * (EI: src/acquisition.py:80-81; varmax: :178).  Deterministic fixed-order reduction. */
int ppbo_acq_reduce(const double* fmax, int S, int batch, double mustar, double* out, void* stream);
/* same with mu* read from device memory (no host round trip between the mu* search and the reduction) */
int ppbo_acq_reduce_dev(const double* fmax, int S, int batch, const double* mustar_dev, double* out, void* stream);
/* Greedy batch selection by joint expected improvement (q-EI) over the SAME draws behind fmax[batch][S]: the maxima of grid b and
 * grid b' in sample s are values of one sampled function, so q-EI(A) = E_s[max(max_{b in A} fmax[b][s] - mu*, 0)].  Step k of q
 * (no addition to the reference, which proposes one query; no host synchronisation between the steps):
 *   ppbo_acq_batch_gain : gain[b] = sum_s max(max(cur[s], fmax[b][s]) - mu*, 0) for every candidate (mu* in device memory; cur is
 *                         not read at k = 0), in the order of ppbo_acq_reduce_dev (step 0: its column 0, bit for bit);
 *                         gain[batch] = S.  gain: batch + 1 doubles, which several ranks sum (one all-reduce) before the pick.
 *   ppbo_acq_batch_pick : w = arg-max of gain[0..batch) over the candidates not in idx[0..k), lowest index on ties; idx[k] = w,
 *                         val[k] = gain[w] / gain[batch] (the joint EI of the first k+1 picks), cur[s] = max(cur[s], fmax[w][s])
 *                         (k = 0: cur = fmax[w]).  S = 0 (a rank without samples) picks without touching cur or fmax.
 * Both: argument error unless 0 <= k < q <= batch <= PPBO_ACQ_BATCH_MAX; ppbo_acq_batch_gain also needs S >= 1 and mu*. */
#define PPBO_ACQ_BATCH_MAX 65535
int ppbo_acq_batch_gain(const double* fmax, int S, int batch, const double* mustar_dev, const double* cur, int k, int q,
                        double* gain, void* stream);
int ppbo_acq_batch_pick(const double* gain, int batch, const double* fmax, int S, int k, int q, int* idx, double* val, double* cur,
                        void* stream);
/* out[0] = max_i x[i] (accumulate != 0: also over the previous out[0]).  Batched candidate form of the max the reference's
 * GPModel.mu_star looks for (src/gp_model.py:415-437): mu* over a set of candidate points. */
int ppbo_vec_max(const double* x, long long n, int accumulate, double* out, void* stream);

/* ---- K3: random Fourier features ------------------------------------------------------------------ */
/* sqrt(2 sigma_f^2 / F) cos(W X^T + b).  feature_major = 1: Phi[F x n] (the reference's layout, used for the
 * training points); 0: PhiT[n x F] (point-major, the K-contiguous operand of the sampling GEMM, used for grids).
 * Replaces Hsampler.phiVec / phi (src/random_fourier_sampler.py:45-50). */
int ppbo_rff_features(const double* W, const double* b, int F, int D, const double* X, int n, double sigma_f,
                      double* Phi, long long ld, int feature_major, void* stream);
/* J[F x D] = -sqrt(2 sigma_f^2/F) sin(W x + b) * W   (Hsampler.Dphi, src/random_fourier_sampler.py:51-53) */
int ppbo_rff_jacobian(const double* W, const double* b, int F, int D, const double* x, double sigma_f,
                      double* J, void* stream);
/* out[0] = phi(x)' omega and out[1..D] = its gradient in x, one launch (the objective / jac pair of Hsampler.return_xstar,
 * src/random_fourier_sampler.py:166-167). */
int ppbo_rff_value_grad(const double* W, const double* b, int F, int D, const double* omega, const double* x, double sigma_f,
                        double* out, void* stream);
/* Maximisers of S sampled functions g_s(x) = phi(x)' Omega[s] over [0,1]^D, R restarts each from X0[S][R][D]: one CTA per
 * (sample, restart) runs projected gradient ascent (Barzilai-Borwein steps, Armijo backtracking) until the projected gradient is
 * below gtol or max_iter; xbest[S][D], fbest[S] = the best restart per sample.  work: S R (D + 1) doubles.  Batched form of
 * Hsampler.return_xstar / sample_xstar (src/random_fourier_sampler.py:143-178,215-220: sequential scipy L-BFGS-B restarts).
 * periodic_mask: bit d set = coordinate d has period 1 (the camphor kernel's basis: 0b111011); such a coordinate is reduced modulo
 * 1 after every step instead of being projected, and its whole gradient counts in the stationarity test.  0: the box [0,1]^D. */
int ppbo_rff_maximize(const double* W, const double* b, int F, int D, double sigma_f, const double* Omega, long long ldo, int S,
                      const double* X0, int R, int max_iter, double gtol, int periodic_mask, double* xbest, double* fbest,
                      double* work, void* stream);
/* weight-space objective pieces (Hsampler.S / S_grad / S_hessian, src/random_fourier_sampler.py:106-122):
 * f = Phi_X' omega (Phi_X feature-major [F x N]); S = -1/2|omega|^2 - lik_sum/m (host double); grad[F];
 * hess_diag[F] (the reference Hessian is diagonal).  Any output may be NULL. */
long long ppbo_rff_workspace_bytes(int F, int Q, int m);
int ppbo_rff_objective(const double* Phi_X, long long ld, int F, int Q, int m, double sigma, const double* omega,
                       double* S_out_h, double* grad, double* hess_diag, void* workspace, long long workspace_bytes,
                       void* stream);
/* omega_MAP (Hsampler.update_omega_MAP, src/random_fourier_sampler.py:124-132, replaces scipy trust-exact): Newton in
 * weight space with the exact clamped Hessian I + Psi' a+ Psi (F x F Cholesky) and backtracking; hess_diag[F] is the
 * reference's diagonal Hessian at the optimum (its Laplace covariance is 1 / -hess_diag, :134-137).
 * factor_cache (may be NULL; ppbo_rff_factor_cache_doubles(F) doubles): persistent home of the Hessian factor; with
 * warm_factor = 1 it holds the previous fit's factor and the iteration starts with chord steps from omega0 (a design that grew by
 * one comparison set changes the F x F Hessian by a rank-m term); warm_factor = 2: its 1024-block inverses are in the cache too.
 * Chord steps are Anderson-mixed (depth 5).
 * stats_h[5]: iterations, last relative step, S(omega_MAP), factorisations + chord steps / 1000, 1 if the cache's block inverses are
 * valid for the cache's factor on return. */
long long ppbo_rff_factor_cache_doubles(int F);
int ppbo_rff_fit(const double* Phi_X, long long ld, int F, int Q, int m, double sigma, const double* omega0,
                 int max_iter, double tol, double* factor_cache, int warm_factor, double* omega_map, double* hess_diag,
                 void* workspace, long long workspace_bytes, double* stats_h, void* stream);
/* Full Laplace covariance of the weight-space posterior (opt-in; the reference's covariance is diagonal,
 * src/random_fourier_sampler.py:134-137, and so is the default path above).  L[F x ldl] (followed by the inverted 128-blocks the
 * solves read: ppbo_rff_hessian_factor_doubles(F, ldl) doubles in all) receives the Cholesky factor of the EXACT Hessian
 * -grad^2 S(omega) = I + Psi' diag(a) Psi with the signed likelihood coefficients a at omega -- the precision of the Laplace
 * approximation, whose diagonal is -hess_diag.  A caller buffer: the fit's factor_cache (clamped chord matrix) is not touched.
 * info_h (host, may be NULL = no synchronisation): 0 or the first non-positive pivot, also the return value; no fall-back. */
long long ppbo_rff_hessian_factor_workspace_bytes(int F, int Q, int m);
long long ppbo_rff_hessian_factor_doubles(int F, long long ldl);
int ppbo_rff_hessian_factor(const double* Phi_X, long long ld, int F, int Q, int m, double sigma, const double* omega, double* L,
                            long long ldl, void* workspace, long long workspace_bytes, int* info_h, void* stream);
/* out[i] = standard normal number (offset + i) of Philox4x32-10 stream `stream_id` under `seed` (Box-Muller on 53-bit uniforms).
 * Counter-based: the value of a given index does not depend on launch shape or on which GPU draws it.  Replaces the host
 * np.random draws of the reference where the caller does not inject its own (oracle: oracle/ppbo_oracle.py philox_normals). */
int ppbo_normal_fill(unsigned long long seed, unsigned int stream_id, long long offset, double* out, long long n, void* stream);
/* Omega[s][f] = omega_map[f] + z[s][f] / sqrt(-hess_diag[f]): S posterior weight draws from the diagonal Laplace covariance
 * (Hsampler.update_covariancematrix + sample_omega, src/random_fourier_sampler.py:134-137,207-213).  Z[S x F] are injected
 * standard normals (parity tests); Z == NULL draws z[s][f] as normal number (sample0 + s) * F + f of the Philox stream, so
 * shards of the sample range over several GPUs reproduce the single-GPU draw exactly. */
int ppbo_rff_sample_omega(const double* omega_map, const double* hess_diag, const double* Z, long long ldz,
                          unsigned long long seed, unsigned int stream_id, long long sample0, int S, int F, double* Omega,
                          long long ldo, void* stream);
/* Omega = 1 omega_map' + Z L^-1: S draws from N(omega_map, H^-1) for the factor L of ppbo_rff_hessian_factor (the full-covariance
 * Hsampler.sample_omega, src/random_fourier_sampler.py:207-213, numpy's multivariate_normal with the dense covariance).  Z as in
 * ppbo_rff_sample_omega (injected, or Philox numbers (sample0 + s) F + f).  S <= 65535 per call.
 * workspace: ppbo_rff_sample_omega_full_workspace_bytes(S, F) bytes. */
long long ppbo_rff_sample_omega_full_workspace_bytes(int S, int F);
int ppbo_rff_sample_omega_full(const double* omega_map, const double* L, long long ldl, const double* Z, long long ldz,
                               unsigned long long seed, unsigned int stream_id, long long sample0, int S, int F, double* Omega,
                               long long ldo, void* workspace, long long workspace_bytes, void* stream);
/* Fs = Omega[S x F] . PhiT_grid[P x F]^T per batch entry (grid), fused per-sample max / first arg-max over P
 * (batched form of the objective in Hsampler.return_xstar, src/random_fourier_sampler.py:166,170).
 * Fs_full (optional, tests only): dense [batch][S x P]. */
int ppbo_rff_eval_argmax(const double* Omega, long long ldo, int S, int F, const double* PhiT_grid, long long ldp,
                         long long stridePhi, int P, int batch, double* fmax, int* arg, double* Fs_full,
                         void* stream);

/* ---- K3 on the tcgen05 INT8 tensor pipe (csrc/ozaki.cu) -----------------------------------------------------------------
 * The same contraction as ppbo_rff_eval_argmax (Hsampler.return_xstar's objective, src/random_fourier_sampler.py:166,170,
 * batched over samples and grid points), evaluated to FP64 accuracy by error-free splitting: every operand row is scaled by a
 * power of two and cut into `slices` balanced base-256 digit planes (INT8); slices (slices+1)/2 exact INT8 x INT8 -> INT32
 * tensor-core GEMMs are recombined in INT64/FP64.  Deterministic and bit-reproducible (oracle: ppbo_oracle.ozaki_matmul).
 * Truncation error <= (slices+1) K 2^(-8 slices - 2) |row|_max |col|_max (slices = 6: 1e-11 .. 1e-12 relative in practice). */
/* tile height of the digit-plane layout: operand 0 = samples (A, 128 rows), 1 = grid points (B, 64 rows) */
int ppbo_ozaki_tile_rows(int operand);
/* bytes of the digit planes / doubles of the row scales for `batch` matrices of rows x K */
long long ppbo_ozaki_plane_bytes(int rows, int K, int tile_rows, int batch, int slices);
long long ppbo_ozaki_scale_doubles(int rows, int tile_rows, int batch);
/* X[batch][rows x K] (row stride ldx, batch stride strideX) -> scale[batch][rows_pad] (powers of two) and the INT8 digit planes
 * in the tiled shared-memory image of the tensor-core operand (layout: csrc/ozaki.cu, tile_offset) */
int ppbo_ozaki_slice(const double* X, long long ldx, long long strideX, int rows, int K, int tile_rows, int batch, int slices,
                     double* scale, signed char* planes, void* stream);
/* The S posterior weight draws of ppbo_rff_sample_omega (Philox path) written directly as the A-operand digit planes and row
 * scales (sized by ppbo_ozaki_plane_bytes / ppbo_ozaki_scale_doubles for S rows, K = F, tile_rows(0), batch 1): the draws are
 * generated in shared memory and never reach HBM.  Bit-identical to ppbo_rff_sample_omega followed by ppbo_ozaki_slice.
 * (Hsampler.sample_omega, src/random_fourier_sampler.py:207-213, batched over S samples.) */
int ppbo_ozaki_sample_slice(const double* omega_map, const double* hess_diag, unsigned long long seed, unsigned int stream_id,
                            long long sample0, int S, int F, int slices, double* scale, signed char* planes, void* stream);
/* The standard normals z[s][f] = Philox number (sample0 + s) F + f themselves as A-operand digit planes (no mean, no scale): the
 * draws of the full-covariance contraction max_p (mu_p + z_s . Phi~_p), which do not depend on the fit.  Bit-identical to
 * ppbo_normal_fill followed by ppbo_ozaki_slice. */
int ppbo_ozaki_normal_slice(unsigned long long seed, unsigned int stream_id, long long sample0, int S, int F, int slices,
                            double* scale, signed char* planes, void* stream);
/* fmax[batch][S], arg[batch][S] = per-sample max / first arg-max over the P grid points of A . B_b^T from digit planes
 * (A sliced with tile_rows(0), batch 1; B with tile_rows(1), `batch` grids).  Fs_full (optional, tests): dense [batch][S x P].
 * workspace: ppbo_ozaki_rowmax_workspace_bytes(S, P, batch) bytes (partial maxima of the column-tile groups).
 * err_flag (optional, device int): set to the id of a starved pipeline wait before the kernel traps (never on a healthy run). */
long long ppbo_ozaki_rowmax_workspace_bytes(int S, int P, int batch);
int ppbo_ozaki_rowmax(const signed char* Aplanes, const double* ascale, int S, const signed char* Bplanes, const double* bscale,
                      int P, int batch, int K, int slices, double* fmax, int* arg, double* Fs_full, void* workspace,
                      long long workspace_bytes, int* err_flag, void* stream);
/* The same with a column offset: fmax[b][s] = max_p (bias[b][p] + (A . B_b^T)[s][p]), each element formed as ONE fma of the exact
 * scaled product and the offset (so equal to ozaki_matmul + bias, bit for bit); first arg-max on ties as above.  The posterior
 * mean mu_p = phi(x_p)' omega_MAP of the full-covariance draws f_s(x_p) = mu_p + z_s . (L^-1 phi(x_p)).  bias: [batch][P]. */
int ppbo_ozaki_rowmax_bias(const signed char* Aplanes, const double* ascale, int S, const signed char* Bplanes, const double* bscale,
                           const double* bias, int P, int batch, int K, int slices, double* fmax, int* arg, double* Fs_full,
                           void* workspace, long long workspace_bytes, int* err_flag, void* stream);
/* diagnostic: SM clocks for `iters` back-to-back 128 x N x 32 INT8 MMAs on `blocks` SMs, rotating over `nacc` accumulators
 * (mode 0: A, B from shared memory; 1: A from TMEM; 2: B plane re-used); clocks_out[blocks] device int64.
 * Used by scripts/ozaki_probe.py --ubench. */
int ppbo_ozaki_mma_rate(int N, int mode, int nacc, int iters, int blocks, long long* clocks_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PPBO_B200_H */
