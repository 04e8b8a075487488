/* gegp.h -- C ABI of the B200-native gradient-enhanced Gaussian-process hot path (libgegp.so).
 *
 * Drop-in boundary for marchildon/gpgradpy v1.3.2.  The reference has no FFI; the operator interface it
 * exposes is the set of bound Python methods listed below, and each entry point here is what a ctypes
 * binding behind that method calls (see INTEGRATION.md for the binding stubs):
 *
 *   gegp_build_cov      <- Kernel.calc_all_K_w_chofac   gpgradpy/src/kernel/Kernel.py:140-307
 *                          KernelSqExpGradMod.sq_exp_calc_KernGrad  kernel/KernelSqExp.py:322-410
 *                          CommonFun.calc_Rtensor       base/CommonFun.py:58-84
 *   gegp_potrf          <- scipy cho_factor call sites  kernel/Kernel.py:251,291
 *   gegp_trsm_rows      <- scipy cho_solve (forward half) eval/GpEvalModel.py:154, eval/GpMeanFun.py:102
 *   gegp_potri          <- cho_solve(chofac, eye(N))    optz/CalcLkd.py:174,234
 *   gegp_dgemm          <- the BLAS dgemm behind `@`     kernel/Kernel.py:227,237,252
 *   gegp_lml_eval       <- CalcLkd.calc_lkd_all         optz/CalcLkd.py:270-346  (noise-free :30-95,149-181;
 *                          noisy :185-251), GpHparaGrad.calc_KernGrad_hp / calc_Kcov_grad_hp
 *                          optz/GpHparaGrad.py:13-155, GpMeanFunPoly.calc_model_max_lkd_poly
 *                          eval/GpMeanFun.py:69-122; with B > 1 the candidate loops
 *                          optz/GpHparaX0.py:39-45 and optz/OptzLkd.py:249-270
 *   gegp_predict_setup  <- GpEvalModel.setup_eval_model eval/GpEvalModel.py:17-57
 *   gegp_predict        <- GpEvalModel.eval_model       eval/GpEvalModel.py:59-198 (mu, sigma)
 *   gegp_cross_cov      <- calc_KernGrad(X, X*) use at  eval/GpEvalModel.py:133-139
 *
 * Conventions
 *   - every pointer is a DEVICE pointer to fp64 unless stated; matrices are row-major with an explicit
 *     leading dimension (must be even; bases 16-byte aligned);
 *   - N = n + n_g*d; row/column order is dimension-major: value of point a -> a, d/dx_i at gradient slot g ->
 *     n + i*n_g + g (base/CommonFun.py:170, kernel/Kernel.py:353);
 *   - grad_slot[n] (int32, device) maps a point to its gradient slot or -1; NULL means all points carry gradients;
 *   - every function that evaluates the kernel takes (int kernel, double kernel_hp) right after theta: the kernel
 *     family GEGP_KERNEL_* and its extra hyper-parameter (alpha of the rational-quadratic kernel; ignored otherwise);
 *   - every call is asynchronous on `stream` (a cudaStream_t), never allocates, never throws;
 *   - re-entrant: no call keeps mutable state between or across calls except caches that are keyed and locked
 *     (tensor maps) and pooled per call (the look-ahead streams of the factorisation); concurrent calls from several
 *     host threads and on several devices are supported.  gegp_set_option and gegp_profile_* are process-wide tuning /
 *     instrumentation hooks and must not race with running calls;
 *   - return value: 0 ok; < 0 bad argument (a small negative code naming the argument: its position in the ABI-3
 *     argument list, i.e. not counting (kernel, kernel_hp); -50: bad kernel family / kernel hyper-parameter) or
 *     -1000-cudaError for a launch failure.
 *     Numerical failure (matrix not positive definite) is reported LAPACK-style in a device int / the
 *     GEGP_OUT_INFO slot: 0 ok, k > 0 leading minor of order k is not positive definite.
 */
#ifndef GEGP_H_
#define GEGP_H_
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GEGP_ABI_VERSION 4

/* covariance assembly modes (kernel/Kernel.py:220-237 vs :268-277) */
#define GEGP_MODE_BASE 0       /* varK * (K + diag(noise) + eta*I)                                  */
#define GEGP_MODE_PRECON 1     /* varK * (P^-1 (K + diag(noise)) P^-1 + eta*I), P = diag sqrt(diag)    */
#define GEGP_MODE_PRECON_COV 2 /* varK * (K + diag(noise) + eta*diag(K + noise))  (= P * PRECON * P)   */

/* kernel families (kernel/Kernel.py:27-107 binds one of three kernel files); kernel_hp is the extra hyper-parameter
 * of the family (alpha of the rational-quadratic kernel, kernel/KernelRatQuad.py:849-850; ignored by the others) */
#define GEGP_KERNEL_SQEXP 0     /* 'SqExp'  kernel/KernelSqExp.py     exp(-s),  s = sum_i theta_i r_i^2            */
#define GEGP_KERNEL_MATERN52 1  /* 'Ma5f2'  kernel/KernelMatern5f2.py (1 + sqrt5 nu + 5/3 nu^2) exp(-sqrt5 nu)    */
#define GEGP_KERNEL_RATQUAD 2   /* 'RatQu'  kernel/KernelRatQuad.py   (1 + s / alpha)^-alpha                      */

/* layout of the per-candidate result vector of gegp_lml_eval (doubles) */
#define GEGP_OUT_LML 0     /* log marginal likelihood (no N/2 ln 2pi term, optz/CalcLkd.py:168,226)      */
#define GEGP_OUT_SIGMA2 1  /* noise-free: closed-form varK = res^T K^-1 res / N (floor 1e-32); noisy: varK */
#define GEGP_OUT_BETA 2    /* GLS constant mean                                                         */
#define GEGP_OUT_LOGDET 3  /* ln det of the (un-preconditioned) factored matrix                          */
#define GEGP_OUT_INFO 4    /* 0 or the order of the first non-positive leading minor                     */
#define GEGP_OUT_QUAD 5    /* res^T K^-1 res                                                            */
#define GEGP_OUT_DVARK 6   /* noisy only: dLML/dvarK                                                    */
#define GEGP_OUT_DVARF 7   /* noisy only: dLML/dvar_fval                                                */
#define GEGP_OUT_DVARG 8   /* noisy only: dLML/dvar_fgrad                                               */
#define GEGP_OUT_DKERN 9   /* dLML/dkernel_hp (rational-quadratic alpha; 0 for the other kernels)        */
#define GEGP_OUT_GRAD 10   /* dLML/dtheta[0..d-1] (w.r.t. theta, not log10 theta)                        */
#define GEGP_OUT_LEN(d) (GEGP_OUT_GRAD + (d))

/* operations for gegp_workspace_bytes */
#define GEGP_OP_LML 0       /* gegp_lml_eval without gradient : arg = B */
#define GEGP_OP_LML_GRAD 1  /* gegp_lml_eval with gradient    : arg = B */
#define GEGP_OP_PREDICT 2   /* gegp_predict                   : arg = nx chunk */

int gegp_abi_version(void);

/* Tuning knobs (process-wide).  Returns the previous value (>= 0) or a negative argument error.
 * GEGP_OPT_TMA_MIN_TILES: the 128 x 128-tile TMA GEMM kernel is used for products with at least this many output
 * tiles per problem (default 400, measured); smaller products run on the 64 x 64-tile cp.async kernel.  The
 * choice depends on the shape of one problem only, never on the batch count (bit-identical results across
 * batch sizes and ranks). */
#define GEGP_OPT_TMA_MIN_TILES 1
#define GEGP_OPT_LOOKAHEAD 2       /* 0: single-stream factorisation; 1 (default): look-ahead on priority streams */
#define GEGP_OPT_SMALL_TILE_MAX 3  /* products with at most this many 64 x 64 tiles in total use 32 x 32 tiles (36) */
#define GEGP_OPT_CHAIN_CLUSTER 4   /* CTAs per cluster of the factorisation's chain step: 0 automatic (default), 1, 2, 4 */
/* Pieces of K^-1 = U U^T that only need the left part of the factor are issued while the factorisation is still running
 * (LML + gradient evaluations): 0 off, 1 the aa block only, 2 also the first columns of the root's pair product,
 * 3 (default) level 2 up to N = 8192 and off above (a function of the shape of one problem only).  The levels differ in
 * the summation order of K^-1 (agreement to rounding). */
#define GEGP_OPT_INV_EARLY 5
int gegp_set_option(int key, int value);

size_t gegp_workspace_bytes(int op, int n, int n_g, int d, int arg);

/* leading dimension this library uses for an N-column work matrix (multiple of 16 doubles) */
int64_t gegp_ld(int N);

/* K1: fused covariance builder.  theta[d]; noise[N] (already divided by varK where the reference divides,
 * kernel/Kernel.py:218) or NULL; p_out[2N] receives p and 1/p (required for GEGP_MODE_PRECON, else may be NULL);
 * uplo 0: full matrix, 1: lower triangle only (strict upper part is left untouched). */
int gegp_build_cov(int n, int n_g, int d, const double* X, const int32_t* grad_slot, const double* theta, int kernel, double kernel_hp,
                   const double* noise, int mode, double eta, double varK, double* K_out, int64_t ldk,
                   double* p_out, int uplo, void* stream);

/* Cross covariance, transposed: Kx[x, c] = cov(test point x, training datum c) * (pinv ? pinv[c] : 1);
 * Kx is [nx, ld]. */
int gegp_cross_cov(int n, int n_g, int d, const double* X, const int32_t* grad_slot, const double* Xs, int nx,
                   const double* theta, int kernel, double kernel_hp, const double* pinv, double* Kx, int64_t ld, void* stream);

/* K2: blocked Cholesky on the fp64 tensor cores.  A is (N + n_extra) x lda, lower triangle of the leading
 * N x N block holds the SPD matrix; on exit it holds L (lower) and the n_extra appended rows R are
 * overwritten with R * L^-T (forward-solved right-hand sides).  info_dev: device int, must be 0 on entry.
 * dinv[gegp_dinv_doubles(N)] receives the inverse-transposed 128 x 128 diagonal blocks of L (block b, row-major
 * with ld 128, at dinv + b*128*128).  They are part of the factor: later solves against L multiply with their
 * 32 x 32 diagonal sub-blocks on the tensor cores (each product followed by one refinement step, so the result is
 * as accurate as a substitution) and the explicit inverse starts from them (scipy cho_factor returns
 * (c, lower); here the factor is (A, dinv)). */
int64_t gegp_dinv_doubles(int N);
int gegp_potrf(int N, int n_extra, double* A, int64_t lda, double* dinv, int* info_dev, void* stream);

/* B (r x ldb, r rows of length N) <- B * L^-T against an existing factor (L, dinv). */
int gegp_trsm_rows(int N, const double* L, int64_t ldl, const double* dinv, double* B, int64_t ldb, int r,
                   void* stream);

/* Explicit inverse from the factor (scipy cho_solve(chofac, eye(N)), optz/CalcLkd.py:174):
 * U (N x ldu) receives L^-T in its upper triangle, Kinv (N x ldk) the full symmetric (L L^T)^-1. */
int gegp_potri(int N, const double* L, int64_t ldl, const double* dinv, double* U, int64_t ldu, double* Kinv,
               int64_t ldk, void* stream);

/* The DMMA GEMM engine every O(N^3) step runs on: C = alpha * A * op(B) + beta * C, row-major;
 * transb = 0: B is K x N; transb = 1: B is N x K (C = A B^T).  lda, ldb even, A and B 16-byte aligned. */
int gegp_dgemm(int transb, int M, int N, int K, double alpha, const double* A, int64_t lda, const double* B,
               int64_t ldb, double beta, double* C, int64_t ldc, void* stream);

/* K3/K5: LML (+ hyper-parameter gradient) for B candidate theta rows, fused build -> factor -> reduce.
 * theta_batch[B, d]; y[N] data vector (values then Fortran-flattened gradients); noise[N] or NULL
 * (NOT divided by varK; used only when noisy != 0); noisy = 0: varK := 1 inside K and sigma^2 in closed form
 * (kernel/Kernel.py:128-138, optz/CalcLkd.py:149-181); noisy = 1: varK_batch[B] given, LML of
 * optz/CalcLkd.py:185-251.  mode is GEGP_MODE_BASE or GEGP_MODE_PRECON.  pnlt_grad is the varK-penalty
 * derivative term of optz/CalcLkd.py:175 (0 when lkd_varK_pnlt_use is False).
 * kernel: GEGP_KERNEL_*; kernel_hp_batch[B] (device): the kernel's extra hyper-parameter per candidate (alpha of the
 * rational-quadratic kernel; may be NULL for the kernels without one); dLML/dalpha comes back in GEGP_OUT_DKERN.
 * out[B, GEGP_OUT_LEN(d)].  alpha_out[B, N] (K^-1 (y - H beta), un-preconditioned) or NULL. */
int gegp_lml_eval(int B, const double* theta_batch, const double* varK_batch, int kernel,
                  const double* kernel_hp_batch, int n, int n_g, int d,
                  const double* X, const int32_t* grad_slot, const double* y, const double* noise, int mode,
                  double eta, int noisy, double pnlt_grad, int want_grad, double* out, double* alpha_out,
                  void* work, size_t work_bytes, void* stream);

/* K4 setup: build (varK := 1, kernel/Kernel.py:196-197) + factor + forward-solve of P^-1 (y - H beta).
 * A is (N + 1) x lda; dinv[gegp_dinv_doubles(N)]; p_out[2N]; on exit row N of A holds
 * w = L^-1 P^-1 (y - H beta).  alpha_out[N] (optional) receives K^-1 (y - H beta) (eval/GpEvalModel.py:57). */
int gegp_predict_setup(int n, int n_g, int d, const double* X, const int32_t* grad_slot, const double* theta, int kernel, double kernel_hp,
                       const double* noise, int mode, double eta, const double* y, double beta, double* A,
                       int64_t lda, double* dinv, double* p_out, double* alpha_out, int* info_dev, void* stream);

/* K4: posterior mean and standard deviation at nx test points (eval/GpEvalModel.py:154-168):
 * mu = beta + k*^T K^-1 (y - H beta), sig = sqrt(varK) sqrt(max(0, 1 - k*^T K^-1 k*)); sig2_out (optional)
 * receives the unclipped 1 - k*^T K^-1 k*, n_negative_dev counts entries < 0 (the reference asserts on them). */
int gegp_predict(int n, int n_g, int d, const double* X, const int32_t* grad_slot, const double* theta, int kernel, double kernel_hp,
                 const double* A, int64_t lda, const double* dinv, const double* p, int mode, double beta, double varK,
                 const double* Xs, int nx, double* mu, double* sig, double* sig2_out, int* n_negative_dev,
                 void* work, size_t work_bytes, void* stream);

/* K4 with x-derivatives (eval_model(calc_grad=True), eval/GpEvalModel.py:170-173, 319-354): additionally
 * dmudx[nx, d] = d mu / d x and dsigdx[nx, d] = d sig / d x.  The derivative columns of K(X, X*) are generated on the
 * fly and forward-solved beside k* (d + 1 rows per test point): work >= (d + 1) * gegp_ld(N) * 8 bytes per point. */
int gegp_predict_grad(int n, int n_g, int d, const double* X, const int32_t* grad_slot, const double* theta, int kernel, double kernel_hp,
                      const double* A, int64_t lda, const double* dinv, const double* p, int mode, double beta,
                      double varK, const double* Xs, int nx, double* mu, double* sig, double* sig2_out, double* dmudx,
                      double* dsigdx, int* n_negative_dev, void* work, size_t work_bytes, void* stream);

/* Surrogate Hessians at ONE test point xs[d] (eval_model(calc_grad=True, calc_hess=True), eval/GpEvalModel.py:175-180,
 * 356-382; the reference also takes one point per call).  alpha[N] = K^-1 (y - H beta) from gegp_predict_setup.
 * Besides mu, sig, dmudx[d], dsigdx[d] it returns hess3[3, d, d]:
 *   hess3[0] = d2mu/dx2,  hess3[1] = (d2 kstar / dx2) . (K^-1 kstar)  (term1),
 *   hess3[2] = (d kstar / dx) K^-1 (d kstar / dx)^T  (term2), kstar = K(X, xs);
 * the caller forms d2sig2/dx2 = -2 varK (term1 + term2) and d2sig/dx2 = (d2sig2/dx2 - 2 dsig dsig^T) / (2 sig).
 * Each d x d slab is exactly symmetric.  work >= (d + 2) * gegp_ld(N) * 8 bytes. */
int gegp_predict_hess(int n, int n_g, int d, const double* X, const int32_t* grad_slot, const double* theta, int kernel, double kernel_hp,
                      const double* A, int64_t lda, const double* dinv, const double* p, const double* alpha, int mode,
                      double beta, double varK, const double* xs, double* mu, double* sig, double* sig2_out,
                      double* dmudx, double* dsigdx, double* hess3, int* n_negative_dev, void* work, size_t work_bytes,
                      void* stream);

/* Surrogate Hessians at nx test points Xs[nx, d] in one chunked pass (a second-order optimiser of an acquisition function
 * run from many starts at once).  Arguments as gegp_predict_hess with xs replaced by (Xs, nx); outputs mu[nx], sig[nx],
 * sig2_out[nx] (optional), dmudx[nx, d], dsigdx[nx, d] and hess3[nx, 3, d, d], each point's slab with the meaning of the
 * one-point call (d2mu/dx2, term1, term2); n_negative_dev counts the negative sig2 entries.  Per chunk of points: one
 * cross-covariance launch, one forward solve of the (d + 1) rows of every point, one back substitution of all the points'
 * K^-1 k* at once and one contraction launch.  mu, sig, sig2, dmudx and dsigdx are those of gegp_predict_grad for the same
 * chunk; hess3 agrees with the one-point call to rounding (the one-point call solves for K^-1 k* with its own back
 * substitution; the contraction is the same) and every d x d slab is exactly symmetric.  d <= 421, where the
 * contraction's shared-memory tiles fit (else -3); gegp_predict_setup itself accepts d up to about 353.
 * work >= gegp_dinv_doubles(N) * 8 bytes, plus ((d + 1) * gegp_ld(N) + 128) * 8 bytes per point of a chunk; the chunk is as many points as fit (at least one, else -25).  nx = 0 writes nothing. */
int gegp_predict_hess_batch(int n, int n_g, int d, const double* X, const int32_t* grad_slot, const double* theta, int kernel,
                            double kernel_hp, const double* A, int64_t lda, const double* dinv, const double* p,
                            const double* alpha, int mode, double beta, double varK, const double* Xs, int nx, double* mu,
                            double* sig, double* sig2_out, double* dmudx, double* dsigdx, double* hess3, int* n_negative_dev,
                            void* work, size_t work_bytes, void* stream);

/* Where gegp_lml_eval keeps its per-candidate arrays inside `work` (candidate 0; candidate c adds
 * c * per_candidate_doubles), so that a caller can go on working with the factor and the explicit inverse of the
 * evaluation it has just run (condition number, below).  out[8] = { header_bytes, ld, per_candidate_doubles,
 * offset of A (factor L, lower), of p (p then p^-1, ld apart), of dinv, of U (= L^-T, upper), of Kinv (full inverse) },
 * offsets in doubles after the header; U and Kinv are -1 unless want_grad. */
int gegp_lml_layout(int n, int n_g, int d, int want_grad, int B, int64_t* out8);

/* Condition number kappa_2 of the regularised matrix and its hyper-parameter gradient (kernel/Kernel.py:240,280:
 * np.linalg.cond(., 2); optz/GpHparaCon.py:161-235: full np.linalg.eig, then
 * dkappa/dhp = (v_max^T dK v_max - kappa v_min^T dK v_min) / lambda_min).  Here the two extreme eigenpairs come from
 * a Lanczos iteration with full re-orthogonalisation whose kernels are below (the k x k tridiagonal eigenproblem
 * and the restart loop are host logic): lambda_max from products with K (gegp_symv on the matrix gegp_build_cov
 * wrote), lambda_min from products with the explicit inverse gegp_lml_eval / gegp_potri left on the device.
 *   gegp_symv:         y = M x, M row-major N x ld (ld even, M 16-byte aligned).
 *   gegp_lanczos_step: V[(k+1), ldv] rows 0..j orthonormal, w = M v_j on entry; on exit alpha[j] = v_j.w,
 *                      beta[j] = |w_orth| (device scalars) and V row j+1 = w_orth / beta[j].   j < 255.
 *   gegp_lincomb:      out = normalised sum_i coef[i] V_i (Ritz vector), coef[k] on the device, k <= 256.
 *   gegp_quad_grad:    q_hp = v^T (dKcov/dhp) v for hp = theta_1..theta_d (out[GEGP_OUT_GRAD + m]) and, when
 *                      noisy, varK / var_fval / var_fgrad (GEGP_OUT_DVARK/DVARF/DVARG), dKcov/dtheta generated on
 *                      the fly (optz/GpHparaGrad.py:13-56, :58-98).  GEGP_MODE_BASE only (the reference has no
 *                      condition-number gradient in precon mode).  work >= gegp_quad_grad_work_bytes(n, d). */
int gegp_symv(int N, const double* M, int64_t ld, const double* x, double* y, void* stream);
/* out[row] = sum_c |M[row, c]|: Gershgorin row sums of the built matrix for the variable nugget
 * eta = max_row / (cond_max_target - 1) of wellcond_mtd = 'rescale_eta_vary' (kernel/Kernel.py:229-234, 269-274). */
int gegp_row_abs_sum(int N, const double* M, int64_t ld, double* out, void* stream);
/* out[row] = sum_c M[row, c]^2 (Frobenius norms for cond_norm = 'fro', optz/GpHparaCon.py:237-261). */
int gegp_row_sq_sum(int N, const double* M, int64_t ld, double* out, void* stream);
/* sum(W .* dKcov/dhp) for a symmetric device matrix W (N x ldw) and every hyper-parameter, dKcov/dhp generated on the
 * fly; layout of `out` as gegp_quad_grad.  The Frobenius condition-number gradient contracts
 * W = frac K - K^-3 / frac this way (optz/GpHparaCon.py:252-259).  work >= gegp_quad_grad_work_bytes + 8 (N + 1). */
int gegp_weighted_grad(int n, int n_g, int d, const double* X, const int32_t* grad_slot, const double* theta, int kernel, double kernel_hp,
                       const double* W, int64_t ldw, int mode, double eta, int noisy, const double* varK_dev,
                       double* out, void* work, size_t work_bytes, void* stream);
int gegp_lanczos_step(int N, int j, double* V, int64_t ldv, double* w, double* alpha, double* beta, void* stream);
int gegp_lincomb(int N, int k, const double* V, int64_t ldv, const double* coef, double* out, void* stream);
size_t gegp_quad_grad_work_bytes(int n, int n_g, int d);
int gegp_quad_grad(int n, int n_g, int d, const double* X, const int32_t* grad_slot, const double* theta, int kernel, double kernel_hp,
                   const double* v, int mode, double eta, int noisy, const double* varK_dev, double* out,
                   void* work, size_t work_bytes, void* stream);

/* Batched forms of the condition-number building blocks for B candidates of one problem geometry (the B matrices that
 * B likelihood evaluations leave in the gegp_lml_eval workspace, gegp_lml_layout): candidate z's arrays sit
 * z * stride doubles after candidate 0's.  `active` (int32[B] on the device, or NULL for 0 .. B-1) names the candidate
 * of each of the B launch rows, so candidates that have converged drop out without copying.  A candidate's results do
 * not depend on B, on the other candidates or on `active`: each is bit-identical to the single-candidate call.
 *   gegp_symv_batch:          y_z = M_z x_z (M 16-byte aligned, ld and strideM even, x 16-byte aligned, strideX even);
 *                             B <= 65535.
 *   gegp_lanczos_step_batch:  gegp_lanczos_step on every candidate at the same step j; alpha_z, beta_z are strideAB apart.
 *   gegp_lincomb_batch:       gegp_lincomb per candidate; ks (int32[.] on the device, indexed by candidate, or NULL)
 *                             gives candidate z its own basis size ks[z] (clamped to 1 .. k), k <= 256.
 *   gegp_quad_grad_batch:     gegp_quad_grad for B vectors V + z * ldv, each with its own theta row (theta_batch[B, d]),
 *                             varK (varK_batch[B], when noisy) and kernel hyper-parameter (kernel_hp_batch[B], required
 *                             for the rational-quadratic kernel); out[B, GEGP_OUT_LEN(d)] (zeroed by the caller).
 *                             work >= gegp_quad_grad_batch_work_bytes(B, n, n_g, d).
 *   gegp_build_cov_batch:     gegp_build_cov for B theta rows into K_out + z * strideK.  varK_batch[B] or NULL (1); with
 *                             both noise and varK_batch the noise is divided by varK_z (kernel/Kernel.py:218).  p_out
 *                             (p then 1/p, strideP >= 2N apart) is required for GEGP_MODE_PRECON, else may be NULL. */
int gegp_symv_batch(int B, int N, const double* M, int64_t ld, int64_t strideM, const double* x, int64_t strideX,
                    double* y, int64_t strideY, const int32_t* active, void* stream);
int gegp_lanczos_step_batch(int B, int N, int j, double* V, int64_t ldv, int64_t strideV, double* w, int64_t strideW,
                            double* alpha, double* beta, int64_t strideAB, const int32_t* active, void* stream);
int gegp_lincomb_batch(int B, int N, int k, const int32_t* ks, const double* V, int64_t ldv, int64_t strideV,
                       const double* coef, int64_t strideCoef, double* out, int64_t strideOut, const int32_t* active,
                       void* stream);
size_t gegp_quad_grad_batch_work_bytes(int B, int n, int n_g, int d);
int gegp_quad_grad_batch(int B, const double* theta_batch, const double* varK_batch, int kernel,
                         const double* kernel_hp_batch, int n, int n_g, int d, const double* X, const int32_t* grad_slot,
                         const double* V, int64_t ldv, int mode, double eta, int noisy, double* out, void* work,
                         size_t work_bytes, void* stream);
int gegp_build_cov_batch(int B, const double* theta_batch, const double* varK_batch, int kernel,
                         const double* kernel_hp_batch, int n, int n_g, int d, const double* X, const int32_t* grad_slot,
                         const double* noise, int mode, double eta, double* K_out, int64_t ldk, int64_t strideK,
                         double* p_out, int64_t strideP, int uplo, void* stream);

/* Direct (non-adjoint) likelihood form, lkd_use_adj_mtd = False (optz/CalcLkd.py:64-85, 104-116, 135-147, 349-367;
 * eval/GpMeanFun.py:110-120; noisy data: optz/CalcLkd.py:206-207, 238-241, 253-265).  The reference forms, for every
 * hyper-parameter hp_k with D_k = dKcov/dhp_k:  a^T D_k a,  h^T D_k a  and  tr(K^-1 D_k)  (a = K^-1 (y - H beta),
 * h = K^-1 H) and from them hp_beta_grad, hp_varK_grad, ln_det_Kmat_grad and ln_lkd_grad.  This call produces those sums
 * from what a preceding gegp_lml_eval(B = 1, want_grad = 1) on the same `work` left behind (factor rows, L^-T, the
 * explicit inverse), generating D_k on the fly:
 *   out[0 .. 3][GEGP_OUT_LEN(d)]: rows laid out as GEGP_OUT_* (GRAD + m, DKERN, and when noisy DVARK / DVARF / DVARG):
 *       row 0: a^T D a     row 1: (a + h)^T D (a + h)     row 2: (a - h)^T D (a - h)     row 3: tr(K^-1 D)
 *       (h^T D a = (row 1 - row 2) / 4)
 *   out[4 * GEGP_OUT_LEN(d) + 0] = H^T K^-1 H,   out[4 * GEGP_OUT_LEN(d) + 1] = H^T a.
 * theta, kernel, mode, eta, noisy, varK_dev must be those of that evaluation; scratch: 4 * gegp_ld(N) doubles. */
int gegp_lml_direct_terms(int n, int n_g, int d, const double* X, const int32_t* grad_slot, const double* theta,
                          int kernel, double kernel_hp, int mode, double eta, int noisy, const double* varK_dev,
                          void* work, size_t work_bytes, double* scratch, double* out, void* stream);

/* Instrumentation for bench.py (not on the product path): count kernel launches, and (time_gemm != 0)
 * bracket every DMMA GEMM launch with CUDA events on its stream.  gegp_profile_end synchronises the device. */
void gegp_profile_begin(int time_gemm);
int gegp_profile_end(long* launches, long* gemm_launches, double* gemm_ms, double* gemm_flops);

/* Roofline denominator, measured on the device the caller is about to time: issue peak of the fp64 tensor-core
 * instruction (mma.sync.m8n8k4.f64, SASS DMMA.8x8x4) with 16 warps per SM, best of `reps` runs, in TFLOP/s.
 * Synchronous (it times itself with CUDA events).  scratch: device buffer of >= 512 * (number of SMs) doubles.
 * No reference counterpart: the reference has no device path; bench.py reports every O(N^3) kernel against this. */
int gegp_dmma_peak(double* scratch, size_t scratch_doubles, int reps, double* tflops_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GEGP_H_ */
