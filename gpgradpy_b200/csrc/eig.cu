// Extreme eigenpairs of a dense symmetric matrix on the device: the kernels of a Lanczos iteration with full
// re-orthogonalisation (the loop, the k x k tridiagonal eigenproblem and the restart logic stay on the host side of
// the C ABI, gpgradpy_b200/backend.py).  Used for the 2-norm condition number kappa = lambda_max / lambda_min of the
// regularised covariance matrix and its hyper-parameter gradient, which the reference obtains from a full
// np.linalg.cond + np.linalg.eig (optz/GpHparaCon.py:161-235, kernel/Kernel.py:240,280).  lambda_max comes from
// iterating with K (symv on the rebuilt matrix), lambda_min from iterating with the explicit inverse K^-1 the
// likelihood gradient has already produced (largest eigenvalue of K^-1 = 1 / lambda_min).
#include "linalg.h"

namespace gegp {

namespace {

// Batched launches put one candidate matrix per gridDim.y row (symv) or per CTA (Lanczos step, Ritz combination);
// `active` (int32, optional) maps that index to a candidate, so converged candidates drop out without copying.
__device__ __forceinline__ int cand_of(const int* __restrict__ active, int i) { return active ? active[i] : i; }

// y = M x, M row-major N x ld (every row read once, coalesced; x stays in L1/L2): HBM-read bound, 8 N^2 bytes.
constexpr int SYMV_ROWS = 8;   // rows (warps) per CTA
__global__ void __launch_bounds__(SYMV_ROWS * 32)
symv_kernel(int N, const double* __restrict__ M_all, int64_t ld, int64_t strideM, const double* __restrict__ x_all,
            int64_t strideX, double* __restrict__ y_all, int64_t strideY, const int* __restrict__ active) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int row = blockIdx.x * SYMV_ROWS + w;
  if (row >= N) return;
  const int z = cand_of(active, blockIdx.y);
  const double* x = x_all + z * strideX;
  const double* mr = M_all + z * strideM + (int64_t)row * ld;
  double s0 = 0.0, s1 = 0.0;
  const int N2 = N & ~1;
  for (int c = 2 * lane; c < N2; c += 64) {   // ld is even and M 16-byte aligned: double2 loads
    const double2 m = *reinterpret_cast<const double2*>(mr + c);
    const double2 v = *reinterpret_cast<const double2*>(x + c);
    s0 += m.x * v.x;
    s1 += m.y * v.y;
  }
  if ((N & 1) && lane == 0) s0 += mr[N - 1] * x[N - 1];
  const double s = warp_sum(s0 + s1);
  if (lane == 0) y_all[z * strideY + row] = s;
}

// out[row] = sum_c |M[row, c]| : the Gershgorin row sums behind the variable nugget
// eta = max_row sum|K| / (cond_max_target - 1)  (kernel/Kernel.py:229-234, 269-274).
template <bool SQ>
__global__ void __launch_bounds__(SYMV_ROWS * 32)
row_abs_sum_kernel(int N, const double* __restrict__ M, int64_t ld, double* __restrict__ out) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int row = blockIdx.x * SYMV_ROWS + w;
  if (row >= N) return;
  const double* mr = M + (int64_t)row * ld;
  double s0 = 0.0, s1 = 0.0;
  const int N2 = N & ~1;
  for (int c = 2 * lane; c < N2; c += 64) {
    const double2 m = *reinterpret_cast<const double2*>(mr + c);
    s0 += SQ ? m.x * m.x : fabs(m.x);
    s1 += SQ ? m.y * m.y : fabs(m.y);
  }
  if ((N & 1) && lane == 0) s0 += SQ ? mr[N - 1] * mr[N - 1] : fabs(mr[N - 1]);
  const double s = warp_sum(s0 + s1);
  if (lane == 0) out[row] = s;
}

// One Lanczos step in ONE CTA per candidate (fixed reduction order: deterministic, and the same in any batch).  On entry V rows 0..j hold the orthonormal
// basis and w = M v_j.  alpha_j = v_j . w ;  w -= alpha_j v_j + beta_{j-1} v_{j-1} ;  two classical Gram-Schmidt
// sweeps against v_0..v_j ;  beta_j = |w| ;  v_{j+1} = w / beta_j.
constexpr int LZ_T = 1024;
__device__ __forceinline__ void gs_sweep(int N, int nv, const double* __restrict__ V, int64_t ldv, double* w,
                                         double* coef, int tid) {
  const int lane = tid & 31, warp = tid >> 5;
  for (int i = warp; i < nv; i += LZ_T / 32) {   // warp `warp` owns the dots with rows warp, warp + 32, ...
    const double* vi = V + (int64_t)i * ldv;
    double s = 0.0;
    for (int e = lane; e < N; e += 32) s += vi[e] * w[e];
    s = warp_sum(s);
    if (lane == 0) coef[i] = s;
  }
  __syncthreads();
  for (int e = tid; e < N; e += LZ_T) {
    double acc = w[e];
    for (int i = 0; i < nv; i++) acc -= coef[i] * V[(int64_t)i * ldv + e];
    w[e] = acc;
  }
  __syncthreads();
}

__global__ void __launch_bounds__(LZ_T)
lanczos_step_kernel(int N, int j, double* __restrict__ V_all, int64_t ldv, int64_t strideV, double* __restrict__ w_all,
                    int64_t strideW, double* __restrict__ alpha_all, double* __restrict__ beta_all, int64_t strideAB,
                    const int* __restrict__ active) {
  __shared__ double coef[256];
  __shared__ double sh[32];
  const int tid = threadIdx.x;
  const int z = cand_of(active, blockIdx.x);
  double* V = V_all + z * strideV;
  double* w = w_all + z * strideW;
  double* alpha = alpha_all + z * strideAB;
  double* beta = beta_all + z * strideAB;
  const double* vj = V + (int64_t)j * ldv;
  double s = 0.0;
  for (int e = tid; e < N; e += LZ_T) s += vj[e] * w[e];
  const double a = block_sum(s, sh);
  const double bprev = (j > 0) ? beta[j - 1] : 0.0;
  const double* vp = (j > 0) ? V + (int64_t)(j - 1) * ldv : vj;
  for (int e = tid; e < N; e += LZ_T) w[e] -= a * vj[e] + bprev * vp[e];
  __syncthreads();
  gs_sweep(N, j + 1, V, ldv, w, coef, tid);
  gs_sweep(N, j + 1, V, ldv, w, coef, tid);
  s = 0.0;
  for (int e = tid; e < N; e += LZ_T) s += w[e] * w[e];
  const double nrm = sqrt(block_sum(s, sh));
  if (tid == 0) { alpha[j] = a; beta[j] = nrm; }
  const double inv = nrm > 0.0 ? 1.0 / nrm : 0.0;
  double* vn = V + (int64_t)(j + 1) * ldv;
  for (int e = tid; e < N; e += LZ_T) vn[e] = w[e] * inv;
}

// out = normalised sum_i coef[i] V_i  (Ritz vector; also used to normalise a start vector with k = 1, coef = 1).
// ks (optional): each candidate's own basis size, at most k (Lanczos breakdown can leave a candidate a shorter basis).
__global__ void __launch_bounds__(LZ_T)
lincomb_kernel(int N, int k, const int* __restrict__ ks, const double* __restrict__ V_all, int64_t ldv, int64_t strideV,
               const double* __restrict__ coef_all, int64_t strideCoef, double* __restrict__ out_all, int64_t strideOut,
               const int* __restrict__ active) {
  __shared__ double sh[32];
  __shared__ double c[256];
  const int tid = threadIdx.x;
  const int z = cand_of(active, blockIdx.x);
  const int kz = ks ? max(1, min(ks[z], k)) : k;
  const double* V = V_all + z * strideV;
  const double* coef = coef_all + z * strideCoef;
  double* out = out_all + z * strideOut;
  if (tid < kz) c[tid] = coef[tid];
  __syncthreads();
  double s = 0.0;
  for (int e = tid; e < N; e += LZ_T) {
    double acc = 0.0;
    for (int i = 0; i < kz; i++) acc += c[i] * V[(int64_t)i * ldv + e];
    out[e] = acc;
    s += acc * acc;
  }
  const double nrm = sqrt(block_sum(s, sh));
  const double inv = nrm > 0.0 ? 1.0 / nrm : 0.0;
  for (int e = tid; e < N; e += LZ_T) out[e] *= inv;
}

}  // namespace

int symv_full(const Ctx& ctx, int N, const double* M, int64_t ld, int64_t strideM, const double* x, int64_t strideX,
              double* y, int64_t strideY, const int* active) {
  if (N <= 0 || ctx.batch <= 0) return 0;
  symv_kernel<<<dim3((N + SYMV_ROWS - 1) / SYMV_ROWS, ctx.batch), SYMV_ROWS * 32, 0, ctx.stream>>>(
      N, M, ld, strideM, x, strideX, y, strideY, active);
  GEGP_CHECK_LAUNCH();
  return 0;
}

int row_abs_sum(const Ctx& ctx, int N, const double* M, int64_t ld, double* out, bool squares) {
  if (N <= 0) return 0;
  if (squares) row_abs_sum_kernel<true><<<(N + SYMV_ROWS - 1) / SYMV_ROWS, SYMV_ROWS * 32, 0, ctx.stream>>>(N, M, ld, out);
  else row_abs_sum_kernel<false><<<(N + SYMV_ROWS - 1) / SYMV_ROWS, SYMV_ROWS * 32, 0, ctx.stream>>>(N, M, ld, out);
  GEGP_CHECK_LAUNCH();
  return 0;
}

int lanczos_step(const Ctx& ctx, int N, int j, double* V, int64_t ldv, int64_t strideV, double* w, int64_t strideW,
                 double* alpha, double* beta, int64_t strideAB, const int* active) {
  if (j < 0 || j >= 255) return -2;
  if (ctx.batch <= 0) return 0;
  lanczos_step_kernel<<<ctx.batch, LZ_T, 0, ctx.stream>>>(N, j, V, ldv, strideV, w, strideW, alpha, beta, strideAB, active);
  GEGP_CHECK_LAUNCH();
  return 0;
}

int lincomb_rows(const Ctx& ctx, int N, int k, const int* ks, const double* V, int64_t ldv, int64_t strideV,
                 const double* coef, int64_t strideCoef, double* out, int64_t strideOut, const int* active) {
  if (k < 1 || k > 256) return -2;
  if (ctx.batch <= 0) return 0;
  lincomb_kernel<<<ctx.batch, LZ_T, 0, ctx.stream>>>(N, k, ks, V, ldv, strideV, coef, strideCoef, out, strideOut, active);
  GEGP_CHECK_LAUNCH();
  return 0;
}

}  // namespace gegp
