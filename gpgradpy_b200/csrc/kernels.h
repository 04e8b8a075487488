// Internal kernel launchers of the gradient-enhanced GP path (covariance build, LML reductions, predict).
#pragma once
#include "common.cuh"
#include "../../include/gegp.h"

namespace gegp {

// Problem geometry: n points in d dimensions, n_g of them carry gradients.
// Matrix/data order (dimension-major): value of point a -> a ; d/dx_i at gradient slot g -> n + i*ng + g.
struct Geom {
  int n, ng, d, N;
  const double* X;   // [n, d] row-major, device
  const int* slot;   // [n] gradient slot of each point or -1 ; nullptr when every point has a gradient
  // kernel family (GEGP_KERNEL_*) and its extra hyper-parameter (alpha of the rational-quadratic kernel): one scalar, or
  // one value per problem of a batch (device array, index blockIdx.z)
  int ktype;
  double khp;
  const double* khp_batch;
  __host__ __device__ double kernel_hp(int z) const { return khp_batch ? khp_batch[z] : khp; }
};

// ------------------------------------------------------------------------------------------------
// Radial profiles.  All three kernel families of the reference are functions phi(s) of the scaled squared distance
// s = sum_i theta_i r_i^2, r = x - x'.  With u_i = theta_i r_i every block of the gradient-enhanced matrix and of its
// hyper-parameter / x derivatives follows from phi and its s-derivatives f1, f2, f3 (first to third):
//   K_00 = phi            K_i0 = 2 u_i f1          K_0j = -2 u_j f1          K_ij = -2 theta_i delta_ij f1 - 4 u_i u_j f2
//   d/dtheta_m: r_m^2 times the same blocks one derivative up, plus the explicit theta_m dependence of u and theta
//   SqExp      (kernel/KernelSqExp.py:18-46, 322-410):      phi = exp(-s)
//   Matern-5/2 (kernel/KernelMatern5f2.py:17-52, 354-451):  phi = (1 + sqrt5 nu + 5/3 nu^2) exp(-sqrt5 nu), nu = sqrt(s)
//   RatQuad    (kernel/KernelRatQuad.py:18-51, 439-553):     phi = (1 + s / alpha)^-alpha
// ------------------------------------------------------------------------------------------------
struct RadialProfile { double f0, f1, f2, f3; };

__device__ __forceinline__ RadialProfile radial_profile(int ktype, double alpha, double s) {
  RadialProfile p;
  if (ktype == GEGP_KERNEL_SQEXP) {
    const double k = exp(-s);
    p.f0 = k; p.f1 = -k; p.f2 = k; p.f3 = -k;
  } else if (ktype == GEGP_KERNEL_MATERN52) {
    const double sqrt5 = 2.23606797749978969641;
    const double nu = sqrt(s), e = exp(-sqrt5 * nu);
    p.f0 = (1.0 + sqrt5 * nu + (5.0 / 3.0) * s) * e;
    p.f1 = -(5.0 / 6.0) * (1.0 + sqrt5 * nu) * e;
    p.f2 = (25.0 / 12.0) * e;
    // 1 / nu is singular at r = 0, where it only ever multiplies r_i r_j r_m^2 = 0: clamp like the reference
    // (kernel/KernelMatern5f2.py:574: inv_nu_mat = 1 / max(nu_mat, 1e-16))
    p.f3 = -(25.0 * sqrt5 / 24.0) * e / fmax(nu, 1e-16);
  } else {
    const double B = 1.0 + s / alpha, Binv = 1.0 / B;
    p.f0 = pow(B, -alpha);
    p.f1 = -p.f0 * Binv;
    p.f2 = ((alpha + 1.0) / alpha) * p.f0 * Binv * Binv;
    p.f3 = -((alpha + 1.0) * (alpha + 2.0) / (alpha * alpha)) * p.f0 * Binv * Binv * Binv;
  }
  return p;
}

// d/dalpha of (phi, f1, f2) for the rational-quadratic kernel (kernel/KernelRatQuad.py:133-163, 752-843); zero for
// the kernels without an extra hyper-parameter.
__device__ __forceinline__ RadialProfile radial_profile_dalpha(int ktype, double alpha, double s, const RadialProfile& p) {
  RadialProfile g;
  g.f0 = g.f1 = g.f2 = g.f3 = 0.0;
  if (ktype == GEGP_KERNEL_RATQUAD) {
    const double t = s / alpha, lnB = log1p(t), q = t / (1.0 + t);
    g.f0 = p.f0 * (q - lnB);
    g.f1 = p.f1 * ((alpha + 1.0) / alpha * q - lnB);
    g.f2 = p.f2 * ((alpha + 2.0) / alpha * q - lnB - 1.0 / (alpha * (alpha + 1.0)));
  }
  return g;
}

// diag(K) of a gradient row of dimension i is kernel_diag_coef * theta_i (minus twice the slope of phi at 0, times
// theta_i): 2 for the Gaussian and the rational-quadratic kernel, 5/3 for Matern-5/2 (gamma_i^2 of each kernel
// file's theta2gamma: kernel/KernelSqExp.py:581, kernel/KernelMatern5f2.py:655, kernel/KernelRatQuad.py:853)
__host__ __device__ __forceinline__ double kernel_diag_coef(int ktype) {
  return ktype == GEGP_KERNEL_MATERN52 ? 5.0 / 3.0 : 2.0;
}

// Observation noise as the kernels see it: noise[z*stride + row], optionally divided by varK (per problem).
struct NoiseSpec {
  const double* noise;     // nullptr: noise-free
  int64_t stride;          // 0: one vector shared by every problem of the batch
  const double* varK_all;  // per-problem varK (device) or nullptr -> use the scalar
  double varK;             // scalar varK when varK_all == nullptr
  int divide;              // 1: use noise / varK (kernel/Kernel.py:218)
};

int launch_prep_p(const Ctx& ctx, const Geom& gm, const double* theta, int64_t strideTheta, NoiseSpec ns, int mode,
                  double* p, double* pinv, int64_t strideP);
int launch_build_cov(const Ctx& ctx, const Geom& gm, const double* theta, int64_t strideTheta, NoiseSpec ns,
                     const double* pinv, int64_t strideP, int mode, double eta, double* out, int64_t ld,
                     int64_t strideOut, int lower_only);
int launch_append_res(const Ctx& ctx, int N, int n, const double* y, double beta, const double* pinv, double* row);
int launch_scale_vec(const Ctx& ctx, int N, const double* a, int64_t strideA, const double* pinv, int64_t strideP,
                     double* out, int64_t strideOut);
int launch_cross_cov(const Ctx& ctx, const Geom& gm, const double* theta, const double* pinv, const double* Xs, int nx,
                     double* out, int64_t ld);
int launch_cross_cov_dx(const Ctx& ctx, const Geom& gm, const double* theta, const double* pinv, const double* Xs, int nx,
                        double* out, int64_t ld);
// mu, sig, sig2 of nx points from their (d + 1) solved rows each (ld ldz), and dmu, dsig [nx, d] when d > 0
int launch_predict_grad_rows(const Ctx& ctx, int N, int d, const double* Z, int64_t ldz, int nx, const double* w,
                             double beta, double varK, double* mu, double* sig, double* sig2, double* dmu, double* dsig,
                             int* n_negative);
// Training points per shared-memory tile of the Hessian contraction at dimension d; 0 where its tiles cannot fit.
int hess_batch_tile_height(int d);
// nx test points at once: bt[x * ldb + c] holds L^-T z0 of point x (b = pinv .* bt), Z the (d + 1) solved rows per point
// (ld ldz); out[nx, 3, d, d].  -908 where hess_batch_tile_height(d) = 0.
int launch_predict_hess_batch(const Ctx& ctx, const Geom& gm, const double* theta, const double* Xs, int nx, const double* a,
                              const double* bt, int64_t ldb, const double* pinv, const double* Z, int64_t ldz, double* out);
int launch_append_rhs(const Ctx& ctx, int N, int n, const double* y, const double* pinv, int64_t strideP, double* rows,
                      int64_t ld, int64_t strideRows);

// out layout per problem (GEGP_OUT_* in gegp.h)
int launch_lml_finalize(const Ctx& ctx, int N, const double* A, int64_t lda, int64_t strideA, const double* pinv,
                        int64_t strideP, int noisy, const double* varK, double* w, int64_t strideW, double* out,
                        int64_t strideOut, const int* info, int zero_grad_d);
int launch_lml_grad(const Ctx& ctx, const Geom& gm, const double* theta, int64_t strideTheta, const double* Kinv,
                    int64_t ldk, int64_t strideK, const double* alpha_t, int64_t strideAlpha, const double* pinv,
                    int64_t strideP, int mode, double eta, int noisy, const double* varK, double pnlt_grad, double* partial,
                    int64_t stridePartial, double* out, int64_t strideOut, int quad = 0);

size_t lml_grad_partial_doubles(int n, int d);

}  // namespace gegp
