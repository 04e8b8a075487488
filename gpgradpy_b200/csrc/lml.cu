// K3: log marginal likelihood and its hyper-parameter gradient from the Cholesky factor, with dK/dtheta
// generated on the fly (never materialised), and the K4 posterior row reductions.
//
// Reference: calc_lkd_w_Kern_mtd_adjoint (optz/CalcLkd.py:149-181), calc_lkd_all_w_noise (:185-251),
// calc_model_max_lkd_poly (eval/GpMeanFun.py:98-108), sq_exp_calc_KernGrad_grad_th
// (kernel/KernelSqExp.py:471-568), calc_KernGrad_hp / calc_Kcov_grad_hp (optz/GpHparaGrad.py:13-155),
// eval_model (eval/GpEvalModel.py:154-168).
#include "kernels.h"

namespace gegp {

// ------------------------------------------------------------------------------------------------
// finalize: rows N and N+1 of the factored trapezoid hold z_y = L^-1 P^-1 y and z_h = L^-1 P^-1 H.
//   beta = (z_h.z_y)/(z_h.z_h) ; w = z_y - beta z_h ; quad = w.w = res^T K^-1 res
//   logdet = 2 sum log(L_ii * p_i)
//   noise-free: sigma2 = max(1e-32, quad/N), LML = -(N ln sigma2 + logdet)/2
//   noisy     : LML = -(logdet + quad)/2
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024)
lml_finalize_kernel(int N, const double* __restrict__ A_all, int64_t lda, int64_t strideA,
                    const double* __restrict__ pinv_all, int64_t strideP, int noisy, const double* __restrict__ varK,
                    double* __restrict__ w_all, int64_t strideW, double* __restrict__ out_all, int64_t strideOut,
                    const int* __restrict__ info, int zero_grad_d) {
  __shared__ double sh[32];
  const int z = blockIdx.x;
  const double* A = A_all + z * strideA;
  const double* pinv = pinv_all + z * strideP;
  const double* zy = A + (int64_t)N * lda;
  const double* zh = zy + lda;
  double hh = 0, hy = 0, ld = 0;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    const double h = zh[i];
    hh += h * h;
    hy += h * zy[i];
    ld += log(A[(int64_t)i * lda + i]) - log(pinv[i]);
  }
  hh = block_sum(hh, sh);
  hy = block_sum(hy, sh);
  ld = block_sum(ld, sh);
  const double beta = hy / hh;
  double quad = 0;
  double* w = w_all + z * strideW;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    const double wi = zy[i] - beta * zh[i];
    w[i] = wi;
    quad += wi * wi;
  }
  quad = block_sum(quad, sh);
  if (threadIdx.x == 0) {
    double* out = out_all + z * strideOut;
    const double logdet = 2.0 * ld;
    double s2, lml;
    if (noisy) {
      s2 = varK[z];
      lml = -(logdet + quad) / 2.0;
    } else {
      s2 = fmax(1e-32, quad / N);
      lml = -(N * log(s2) + logdet) / 2.0;
    }
    out[GEGP_OUT_LML] = lml;
    out[GEGP_OUT_SIGMA2] = s2;
    out[GEGP_OUT_BETA] = beta;
    out[GEGP_OUT_LOGDET] = logdet;
    out[GEGP_OUT_INFO] = (double)info[z];
    out[GEGP_OUT_QUAD] = quad;
    out[GEGP_OUT_DVARK] = 0.0;
    out[GEGP_OUT_DVARF] = 0.0;
    out[GEGP_OUT_DVARG] = 0.0;
    out[GEGP_OUT_DKERN] = 0.0;
    for (int m = 0; m < zero_grad_d; m++) out[GEGP_OUT_GRAD + m] = 0.0;   // gradient not requested: defined zeros
  }
}

int launch_lml_finalize(const Ctx& ctx, int N, const double* A, int64_t lda, int64_t strideA, const double* pinv,
                        int64_t strideP, int noisy, const double* varK, double* w, int64_t strideW, double* out,
                        int64_t strideOut, const int* info, int zero_grad_d) {
  lml_finalize_kernel<<<ctx.batch, 1024, 0, ctx.stream>>>(N, A, lda, strideA, pinv, strideP, noisy, varK, w, strideW, out,
                                                          strideOut, info, zero_grad_d);
  GEGP_CHECK_LAUNCH();
  return 0;
}

// alpha_t <- alpha_t .* pinv  (un-preconditioned alpha = K^-1 res) into a separate output
__global__ void scale_vec_kernel(int N, const double* __restrict__ a, int64_t strideA, const double* __restrict__ pinv,
                                 int64_t strideP, double* __restrict__ out, int64_t strideOut) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < N) out[blockIdx.z * strideOut + i] = a[blockIdx.z * strideA + i] * pinv[blockIdx.z * strideP + i];
}

int launch_scale_vec(const Ctx& ctx, int N, const double* a, int64_t strideA, const double* pinv, int64_t strideP,
                     double* out, int64_t strideOut) {
  scale_vec_kernel<<<dim3((N + 255) / 256, 1, ctx.batch), 256, 0, ctx.stream>>>(N, a, strideA, pinv, strideP, out,
                                                                             strideOut);
  GEGP_CHECK_LAUNCH();
  return 0;
}

// ------------------------------------------------------------------------------------------------
// gradient contraction:  g_m = sum_{rows,cols} (dK/dtheta_m) .* W ,  W = P^-1 (c1 a a^T - Kinv/2) P^-1
// (a = preconditioned alpha, Kinv = inverse of the factored matrix).  One CTA per (point a, 128 points b);
// each thread owns one pair and walks the (d+1) x (d+1) block of W that belongs to it, reading Kinv
// coalesced along b.  Using the symmetry of W and K, only rows i of the pair block are needed:
//   A0 = W00,  A1 = 4 sum_i u_i W_i0 - 2 sum_i th_i W_ii,  A2 = -4 sum_i u_i (W u)_i      (u_i = th_i r_i)
//   sum(K .* W)        = sum_pairs  f0 A0 + f1 A1 + f2 A2        (f0..f3: radial profile and its s-derivatives, kernels.h)
//   g_m                = sum_pairs  r_m^2 (f1 A0 + f2 A1 + f3 A2) + f1 (4 r_m W_m0 - 2 W_mm) - 8 f2 r_m (W u)_m
//   g_alpha (RatQuad)  = sum_pairs  (df0 A0 + df1 A1 + df2 A2) / dalpha
// For the Gaussian kernel (f1 = f3 = -k, f0 = f2 = k) this is  g_m = sum_pairs k (t_m - r_m^2 S)  with
//   S = W00 - 4 sum u_i W_i0 + 2 sum th_i W_ii - 4 sum u_i (W u)_i,  t_m = -4 r_m W_m0 + 2 W_mm - 8 r_m (W u)_m.
// Per-CTA partial sums are written to `partial` and reduced in a fixed order by the finalize kernel.
// ------------------------------------------------------------------------------------------------
constexpr int GB = 128;
constexpr int LML_GRAD_MAX_GRID_Y = 65535;

// quad 0: LML gradient weights; 1: W = alpha alpha^T (Kinv not read); 2: W = the matrix passed as Kinv.
// WIDE (d >= 8): four independent Kinv loads in flight per thread; otherwise the plain loop -- measured: the wide form
// is 1.5x faster at d = 10 and 20, the narrow one at d = 5.  72 registers / 7 CTAs per SM for the Gaussian kernel,
// 80 / 6 (narrow) and 96 / 5 (wide) for the other families (ptxas -v: no spills).
// GAUSS: the Gaussian kernel as a compile-time constant (f0 = f2 = k, f1 = f3 = -k fold into one register and the
// alpha row disappears: no spills under the occupancy bound); false = kernel family read from gm.ktype.
template <int quad, bool WIDE, bool GAUSS>
__global__ void __launch_bounds__(GB, GAUSS ? 7 : (WIDE ? 5 : 6))
lml_grad_kernel(Geom gm, const double* __restrict__ theta_all, int64_t strideTheta, const double* __restrict__ Kinv_all,
                int64_t ldk, int64_t strideK, const double* __restrict__ alpha_all, int64_t strideAlpha,
                const double* __restrict__ pinv_all, int64_t strideP, const double* __restrict__ out_all,
                int64_t strideOut, int noisy, double pnlt_grad, double* __restrict__ partial_all,
                int64_t stridePartial, int a0) {
  extern __shared__ double sm[];
  const int d = gm.d, n = gm.n, ng = gm.ng, N = gm.N;
  double* vs = sm;              // [d][GB]  v_j = pinv[col_j] * u_j
  double* gs = vs + d * GB;     // [d+1][GB] per-thread t_m, then g_m ; row d = k*S
  double* xa = gs + (d + 1) * GB;  // [d]
  double* th = xa + d;             // [d]

  const int tid = threadIdx.x, z = blockIdx.z;
  const int a = a0 + blockIdx.y, b = blockIdx.x * GB + tid;
  const double* theta = theta_all + z * strideTheta;
  const double* Kinv = Kinv_all + z * strideK;
  const double* alpha = alpha_all + z * strideAlpha;
  const double* pinv = pinv_all + z * strideP;
  const double* outz = out_all + z * strideOut;
  const int np = 2 * d + 3;
  double* part = partial_all + z * stridePartial + ((int64_t)a * gridDim.x + blockIdx.x) * np;

  for (int e = tid; e < d; e += GB) { xa[e] = gm.X[(int64_t)a * d + e]; th[e] = theta[e]; }
  __syncthreads();

  // quad: W = alpha alpha^T only (quadratic forms v^T dK/dhp v for the condition-number gradient); Kinv is not read
  // quad == 2: W = the symmetric matrix passed in place of Kinv (general weighted sum  sum(W .* dK/dhp))
  const double c1 = quad == 2 ? 0.0 : quad ? 1.0 : (noisy ? 0.5 : (pnlt_grad / N + 1.0 / (2.0 * outz[GEGP_OUT_SIGMA2])));
  const double c2 = quad == 2 ? -1.0 : quad ? 0.0 : 0.5;
  const int sa = gm.slot ? gm.slot[a] : a;
  const bool valid = (b < n);
  const int sb = valid ? (gm.slot ? gm.slot[b] : b) : -1;
  const bool same = valid && (a == b);

  double A0 = 0.0, A1 = 0.0, A2 = 0.0, Ab = 0.0;
  double dv = 0.0;
  RadialProfile ph;
  ph.f0 = ph.f1 = ph.f2 = ph.f3 = 0.0;
  const int ktype = GAUSS ? GEGP_KERNEL_SQEXP : gm.ktype;
  const double kalpha = GAUSS ? 0.0 : gm.kernel_hp(z);
  double ssum = 0.0;
  if (valid) {
    double e = 0.0;
    for (int j = 0; j < d; j++) {
      const double r = xa[j] - gm.X[(int64_t)b * d + j];
      const double u = th[j] * r;
      e += u * r;
      double v = 0.0;
      if (sb >= 0) {
        const int col = n + j * ng + sb;
        v = pinv[col] * u;
        Ab += v * alpha[col];
      }
      vs[j * GB + tid] = v;
    }
    ssum = e;
    ph = radial_profile(ktype, kalpha, e);
    const double pa0 = pinv[a], pb0 = pinv[b];
    const double W00 = pa0 * pb0 * (c1 * alpha[a] * alpha[b] - (quad == 1 ? 0.0 : c2 * Kinv[(int64_t)a * ldk + b]));
    A0 = W00;
    if (same) dv = W00;
  } else {
    for (int j = 0; j < d; j++) vs[j * GB + tid] = 0.0;
  }
  // diagonal sums are produced by the single thread with b == a
  if (same) {
    part[d + 1] = dv;
    if (sa < 0) for (int i = 0; i < d; i++) part[d + 2 + i] = 0.0;
  }

  for (int i = 0; i < d; i++) {
    double t = 0.0;
    if (valid && sa >= 0) {
      const int row = n + i * ng + sa;
      const double pr = pinv[row], ar = alpha[row];
      const double* krow = Kinv + (int64_t)row * ldk;
      const double rb = gm.X[(int64_t)b * d + i];
      const double ri = xa[i] - rb, ui = th[i] * ri;
      const double Wi0 = pr * pinv[b] * (c1 * ar * alpha[b] - (quad == 1 ? 0.0 : c2 * krow[b]));
      double rowdot = 0.0, Wii = 0.0;
      if (sb >= 0) {
        double dot = 0.0, kii = 0.0;
        if (quad != 1) {
          const double* kp = krow + n + sb;
          if (WIDE) {
            // four independent loads in flight per thread (the kernel is HBM-read bound: 8 N^2 bytes of Kinv; eight
            // cost more in occupancy than they gain: measured 82 us with four, 112 us with eight at N = 5500)
            double d0 = 0.0, d1 = 0.0, d2 = 0.0, d3 = 0.0;
            int j = 0;
            for (; j + 3 < d; j += 4) {
              const double k0 = kp[(int64_t)j * ng], k1 = kp[(int64_t)(j + 1) * ng], k2 = kp[(int64_t)(j + 2) * ng],
                           k3 = kp[(int64_t)(j + 3) * ng];
              d0 += vs[j * GB + tid] * k0;
              d1 += vs[(j + 1) * GB + tid] * k1;
              d2 += vs[(j + 2) * GB + tid] * k2;
              d3 += vs[(j + 3) * GB + tid] * k3;
            }
            for (; j < d; j++) d0 += vs[j * GB + tid] * kp[(int64_t)j * ng];
            dot = (d0 + d1) + (d2 + d3);
            kii = kp[(int64_t)i * ng];
          } else {   // few dimensions: the plain loop (one pass, no extra load for the diagonal entry) is faster
            for (int j = 0; j < d; j++) {
              const double kv = krow[n + j * ng + sb];
              dot += vs[j * GB + tid] * kv;
              if (j == i) kii = kv;
            }
          }
        }
        rowdot = pr * (c1 * ar * Ab - c2 * dot);
        const int coli = n + i * ng + sb;
        Wii = pr * pinv[coli] * (c1 * ar * alpha[coli] - c2 * kii);
      }
      if constexpr (GAUSS) {   // A0 holds S = A0 - A1 + A2, the common factor k is applied once at the end
        A0 += -4.0 * ui * Wi0 + 2.0 * th[i] * Wii - 4.0 * ui * rowdot;
        t = -4.0 * ri * Wi0 + 2.0 * Wii - 8.0 * ri * rowdot;
      } else {
        A1 += 4.0 * ui * Wi0 - 2.0 * th[i] * Wii;
        A2 -= 4.0 * ui * rowdot;
        t = ph.f1 * (4.0 * ri * Wi0 - 2.0 * Wii) - 8.0 * ph.f2 * (ri * rowdot);
      }
      if (same) part[d + 2 + i] = Wii;
    }
    gs[i * GB + tid] = t;
  }
  // g_m = t_m + r_m^2 (f1 A0 + f2 A1 + f3 A2)
  // (Gaussian kernel: g_m = k (t_m - r_m^2 S), sum(K .* W) = k S, with S accumulated in A0)
  const double Sth = GAUSS ? -A0 : ph.f1 * A0 + ph.f2 * A1 + ph.f3 * A2;
  const double wk = GAUSS ? ph.f0 : 1.0;
  for (int m = 0; m < d; m++) {
    double g = 0.0;
    if (valid) {
      const double r = xa[m] - gm.X[(int64_t)b * d + m];
      g = wk * (gs[m * GB + tid] + (r * r) * Sth);
    }
    gs[m * GB + tid] = g;
  }
  gs[d * GB + tid] = valid ? (GAUSS ? wk * A0 : ph.f0 * A0 + ph.f1 * A1 + ph.f2 * A2) : 0.0;
  // the kernel hyper-parameter (one block-wide sum more; only the rational-quadratic kernel has one)
  if (ktype == GEGP_KERNEL_RATQUAD) {
    double ga = 0.0;
    if (valid) {
      const RadialProfile da = radial_profile_dalpha(ktype, kalpha, ssum, ph);
      ga = da.f0 * A0 + da.f1 * A1 + da.f2 * A2;
    }
    ga = warp_sum(ga);
    __shared__ double ga_sh[GB / 32];
    if ((tid & 31) == 0) ga_sh[tid >> 5] = ga;
    __syncthreads();
    if (tid == 0) {
      double t = 0.0;
      for (int q = 0; q < GB / 32; q++) t += ga_sh[q];
      part[2 * d + 2] = t;
    }
  } else if (tid == 0) {
    part[2 * d + 2] = 0.0;
  }
  __syncthreads();
  // reduce d+1 rows of GB values: warp w handles rows w, w+4, ...
  const int lane = tid & 31, w = tid >> 5;
  for (int m = w; m <= d; m += GB / 32) {
    double s = 0.0;
#pragma unroll
    for (int q = 0; q < GB / 32; q++) s += gs[m * GB + lane + 32 * q];
    s = warp_sum(s);
    if (lane == 0) part[m] = s;
  }
  // CTAs that do not contain the diagonal pair contribute zeros to the diagonal sums
  const bool has_diag = (a / GB == (int)blockIdx.x);
  if (!has_diag && tid < d + 1) part[d + 1 + tid] = 0.0;
}

// Sum the per-CTA partials in a fixed order and assemble the gradient entries of `out`.
//   noise-free: dLML/dtheta_m = G_m + [precon] c eta DG_m          (c = kernel_diag_coef: 2, Matern-5/2: 5/3)
//   noisy     : dLML/dtheta_m = varK (G_m + [precon] c eta DG_m)
//               dLML/dvarK    = SK + eta (DV + sum_m c th_m DG_m) [precon]  |  SK + eta (DV + sum DG_m) [base]
//               dLML/dalpha   = [varK] G_alpha                      (rational-quadratic kernel only)
//               dLML/dvar_f   = (1 + eta) DV [precon] | DV [base] ; dLML/dvar_g likewise with sum_m DG_m
// stage 1: one CTA per (column c of the partial table, problem z): fixed-order sum over the CTAs' partials
__global__ void __launch_bounds__(256)
lml_grad_colsum_kernel(int np, int64_t nparts, double* __restrict__ partial_all, int64_t stridePartial) {
  __shared__ double sh[32];
  const int c = blockIdx.x, z = blockIdx.y;
  double* part = partial_all + z * stridePartial;
  double s = 0.0;
  for (int64_t p = threadIdx.x; p < nparts; p += blockDim.x) s += part[p * np + c];
  s = block_sum(s, sh);
  if (threadIdx.x == 0) part[nparts * np + c] = s;     // the column sums sit right behind the partial table
}

// stage 2: assemble the gradient entries of `out` from the 2d+2 column sums
__global__ void __launch_bounds__(64)
lml_grad_finalize_kernel(int d, int64_t nparts, const double* __restrict__ partial_all, int64_t stridePartial,
                         const double* __restrict__ theta_all, int64_t strideTheta, int mode, double eta, int noisy,
                         const double* __restrict__ varK, double* __restrict__ out_all, int64_t strideOut, int B,
                         int ktype) {
  const int z = blockIdx.x * blockDim.x + threadIdx.x;
  if (z >= B) return;
  const int np = 2 * d + 3;
  const double cd = kernel_diag_coef(ktype);   // d diag(K) / d theta_m on gradient block m (optz/GpHparaGrad.py:40-50)
  const double* tot = partial_all + z * stridePartial + nparts * np;
  const double* th = theta_all + z * strideTheta;
  double* out = out_all + z * strideOut;
  const bool precon = (mode == GEGP_MODE_PRECON);
  const double vk = noisy ? varK[z] : 1.0;
  const double SK = tot[d], DV = tot[d + 1];
  double sdg = 0.0, sdg_th = 0.0;
  for (int m = 0; m < d; m++) {
    const double DG = tot[d + 2 + m];
    sdg += DG;
    sdg_th += cd * th[m] * DG;
    out[GEGP_OUT_GRAD + m] = vk * (tot[m] + (precon ? cd * eta * DG : 0.0));
  }
  // diag(K) does not depend on the kernel hyper-parameter: no nugget term (optz/GpHparaGrad.py:52-55, 111-123)
  out[GEGP_OUT_DKERN] = vk * tot[2 * d + 2];
  if (noisy) {
    out[GEGP_OUT_DVARK] = SK + eta * (precon ? (DV + sdg_th) : (DV + sdg));
    out[GEGP_OUT_DVARF] = (precon ? 1.0 + eta : 1.0) * DV;
    out[GEGP_OUT_DVARG] = (precon ? 1.0 + eta : 1.0) * sdg;
  }
}

size_t lml_grad_partial_doubles(int n, int d) {   // per-CTA partials followed by the 2d+3 column sums
  return (size_t)n * ((n + GB - 1) / GB) * (2 * d + 3) + (size_t)(2 * d + 3);
}

int launch_lml_grad(const Ctx& ctx, const Geom& gm, const double* theta, int64_t strideTheta, const double* Kinv,
                    int64_t ldk, int64_t strideK, const double* alpha_t, int64_t strideAlpha, const double* pinv,
                    int64_t strideP, int mode, double eta, int noisy, const double* varK, double pnlt_grad,
                    double* partial, int64_t stridePartial, double* out, int64_t strideOut, int quad) {
  const int d = gm.d;
  const size_t smem = (size_t)(d * GB + (d + 1) * GB + 2 * d) * sizeof(double);
  if (quad < 0 || quad > 2) return -906;
  if (smem > (size_t)GEGP_MAX_DYN_SMEM) return -907;
  const bool wide = d >= 8;
  const bool gauss = gm.ktype == GEGP_KERNEL_SQEXP;
  if (smem > 48 * 1024) {   // (only reached with d > 20: the wide kernels); once per device, largest size
    if (gauss) {
      if (quad == 0) GEGP_SET_SMEM((lml_grad_kernel<0, true, true>), GEGP_MAX_DYN_SMEM);
      else if (quad == 1) GEGP_SET_SMEM((lml_grad_kernel<1, true, true>), GEGP_MAX_DYN_SMEM);
      else GEGP_SET_SMEM((lml_grad_kernel<2, true, true>), GEGP_MAX_DYN_SMEM);
    } else {
      if (quad == 0) GEGP_SET_SMEM((lml_grad_kernel<0, true, false>), GEGP_MAX_DYN_SMEM);
      else if (quad == 1) GEGP_SET_SMEM((lml_grad_kernel<1, true, false>), GEGP_MAX_DYN_SMEM);
      else GEGP_SET_SMEM((lml_grad_kernel<2, true, false>), GEGP_MAX_DYN_SMEM);
    }
  }
  // point a is a0 + blockIdx.y: the launch is issued in slices of at most 65535 points a (the gridDim.y limit), each
  // CTA computing and storing exactly what it would in one launch
  const int nbt = (gm.n + GB - 1) / GB;
  timeline_begin(ctx.stream, "lmlgrad", gm.N, d, quad);
  for (int a0 = 0; a0 < gm.n; a0 += LML_GRAD_MAX_GRID_Y) {
    const dim3 grid(nbt, (gm.n - a0 < LML_GRAD_MAX_GRID_Y) ? gm.n - a0 : LML_GRAD_MAX_GRID_Y, ctx.batch);
#define GEGP_LAUNCH_LML_GRAD(Q, W, G)                                                                                    \
    lml_grad_kernel<Q, W, G><<<grid, GB, smem, ctx.stream>>>(gm, theta, strideTheta, Kinv, ldk, strideK, alpha_t,        \
                                                             strideAlpha, pinv, strideP, out, strideOut, noisy, pnlt_grad, \
                                                             partial, stridePartial, a0)
#define GEGP_LAUNCH_LML_GRAD_W(Q, G) do { if (wide) GEGP_LAUNCH_LML_GRAD(Q, true, G); else GEGP_LAUNCH_LML_GRAD(Q, false, G); } while (0)
    if (gauss) {
      if (quad == 0) GEGP_LAUNCH_LML_GRAD_W(0, true);
      else if (quad == 1) GEGP_LAUNCH_LML_GRAD_W(1, true);
      else GEGP_LAUNCH_LML_GRAD_W(2, true);
    } else {
      if (quad == 0) GEGP_LAUNCH_LML_GRAD_W(0, false);
      else if (quad == 1) GEGP_LAUNCH_LML_GRAD_W(1, false);
      else GEGP_LAUNCH_LML_GRAD_W(2, false);
    }
#undef GEGP_LAUNCH_LML_GRAD_W
#undef GEGP_LAUNCH_LML_GRAD
    GEGP_CHECK_LAUNCH();
  }
  timeline_end(ctx.stream);
  const int64_t nparts = (int64_t)nbt * gm.n;
  const int np = 2 * d + 3;
  lml_grad_colsum_kernel<<<dim3(np, ctx.batch), 256, 0, ctx.stream>>>(np, nparts, partial, stridePartial);
  GEGP_CHECK_LAUNCH();
  lml_grad_finalize_kernel<<<(ctx.batch + 63) / 64, 64, 0, ctx.stream>>>(d, nparts, partial, stridePartial, theta,
                                                                        strideTheta, mode, eta, noisy, varK, out,
                                                                        strideOut, ctx.batch, gm.ktype);
  GEGP_CHECK_LAUNCH();
  return 0;
}

// Posterior with x-derivatives: per test point the d + 1 solved rows z0 = L^-1 P^-1 k*, z_j = L^-1 P^-1 dk*/dx_j give
//   mu = beta + z0.w ; sig2 = 1 - |z0|^2 ; dmu/dx_j = z_j.w ; dsig/dx_j = -varK (z_j.z0) / sig   (0 where sig = 0)
// (eval/GpEvalModel.py:319-354: calc_dmudx, calc_dsigdx).  With d = 0 (one row per point, dmu and dsig unused) it is
// the plain posterior of gegp_predict.
__global__ void __launch_bounds__(256)
predict_grad_rows_kernel(int N, int d, const double* __restrict__ Z, int64_t ldz, const double* __restrict__ w,
                         double beta, double varK, double* __restrict__ mu, double* __restrict__ sig,
                         double* __restrict__ sig2, double* __restrict__ dmu, double* __restrict__ dsig,
                         int* __restrict__ n_negative) {
  __shared__ double sh[32];
  __shared__ double sig_sh;
  const int x = blockIdx.x;
  const double* z0 = Z + (int64_t)x * (d + 1) * ldz;
  double d1 = 0, d2 = 0;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    const double v = z0[i];
    d1 += v * w[i];
    d2 += v * v;
  }
  d1 = block_sum(d1, sh);
  d2 = block_sum(d2, sh);
  if (threadIdx.x == 0) {
    const double s2 = 1.0 - d2;
    mu[x] = beta + d1;
    if (sig2) sig2[x] = s2;
    if (s2 < 0 && n_negative) atomicAdd(n_negative, 1);
    sig_sh = sqrt(fmax(s2, 0.0)) * sqrt(varK);
    sig[x] = sig_sh;
  }
  __syncthreads();
  const double sg = sig_sh;
  for (int j = 0; j < d; j++) {
    const double* zj = z0 + (int64_t)(1 + j) * ldz;
    double a = 0, b = 0;
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
      const double v = zj[i];
      a += v * w[i];
      b += v * z0[i];
    }
    a = block_sum(a, sh);
    b = block_sum(b, sh);
    if (threadIdx.x == 0) {
      dmu[(int64_t)x * d + j] = a;
      dsig[(int64_t)x * d + j] = (sg != 0.0) ? -(varK * b) / sg : 0.0;
    }
  }
}

int launch_predict_grad_rows(const Ctx& ctx, int N, int d, const double* Z, int64_t ldz, int nx, const double* w,
                             double beta, double varK, double* mu, double* sig, double* sig2, double* dmu, double* dsig,
                             int* n_negative) {
  if (nx <= 0) return 0;
  predict_grad_rows_kernel<<<nx, 256, 0, ctx.stream>>>(N, d, Z, ldz, w, beta, varK, mu, sig, sig2, dmu, dsig, n_negative);
  GEGP_CHECK_LAUNCH();
  return 0;
}

// Surrogate Hessians (eval/GpEvalModel.py:175-180, 356-382; the second x-derivatives of the cross covariance are
// kernel/KernelSqExp.py:66-88 for value entries and :432-468 for gradient entries, kernel/KernelMatern5f2.py:54-96,
// 272-331 and kernel/KernelRatQuad.py:54-97, 556-633 for the other two families).  Per test point, with r = x_p - x* and
// the radial profile f1, f2, f3 (kernels.h), the second derivatives of k* are
//   value entry p        : 4 th_i th_k r_i r_k f2 + 2 th_i delta_ik f1
//   gradient entry (j, p): (4 th_i th_j (delta_ik r_j + delta_jk r_i) + 4 delta_ij th_i th_k r_k) f2
//                           + 8 th_i th_j th_k r_i r_j r_k f3.
// Summing the gradient entries over j gives, per training point p with value coefficient c_p, gradient coefficients
// G_p[j] (zero where slot[p] < 0) and s_p = sum_j th_j r_j G_p[j]:
//   H[i,k] = th_i th_k M[i,k] + delta_ik th_i W,   W = sum_p (2 f1 c_p + 4 f2 s_p),
//   M[i,k] = sum_p (r_i q_k + r_k q_i),           q_j = 2 (f2 c_p + 2 f3 s_p) r_j + 4 f2 G_p[j],
// so each radial profile is computed once per (test point, training point) pair: O(n d^2) per point instead of O(n d^3).
// Applied with c, G from a = K^-1 (y - H beta) (-> d2mu/dx2) and from b = P^-1 L^-T z0 = K^-1 k* (-> term1).
// term2[i,k] = z_i . z_k reads the point's d solved derivative rows once, in column tiles through shared memory.
// CTA (x, y) is point x, page y of its d(d+1)/2 upper-triangle pairs (2048 pairs a page).  Thread t owns the pairs
// y 2048 + t, + 256, ... (d(d+1)/2 >= 256) or, for small d, pair t % P of the point / column subset t / P; the subsets
// are summed in a fixed order.  Every entry is computed once for i <= k and mirrored, so each Hessian is exactly
// symmetric.  Every page recomputes the training-point tiles and W, which only its diagonal pairs use.
constexpr int HB_T = 256;     // threads per CTA
constexpr int HB_TP = 64;     // training points per tile where it fits (every d <= 145)
constexpr int HB_CT = 64;     // columns per term2 tile
constexpr int HB_MAXI = 8;    // upper-triangle pairs per thread and page
constexpr int HB_PAGE = HB_T * HB_MAXI;

static size_t hess_batch_smem_bytes(int d, int tp) {   // dynamic shared memory of a CTA, tile height tp
  const size_t tile = (size_t)tp * (3 * (size_t)d + 1), gram = (size_t)d * (HB_CT + 1);
  return (2 * (size_t)d + 3 * HB_T + (tile > gram ? tile : gram)) * sizeof(double);
}

int hess_batch_tile_height(int d) {
  for (int tp = HB_TP; tp >= 1; tp /= 2)   // 32 doubles of static shared memory: block_sum's scratch
    if (hess_batch_smem_bytes(d, tp) + 32 * sizeof(double) <= (size_t)GEGP_MAX_DYN_SMEM) return tp;
  return 0;
}

__global__ void __launch_bounds__(HB_T)
predict_hess_batch_kernel(Geom gm, const double* __restrict__ theta, const double* __restrict__ Xs,
                          const double* __restrict__ a, const double* __restrict__ bt, int64_t ldb,
                          const double* __restrict__ pinv, const double* __restrict__ Z, int64_t ldz, int tp,
                          double* __restrict__ out) {
  extern __shared__ double sm[];
  __shared__ double sh[32];
  const int d = gm.d, n = gm.n, ng = gm.ng, N = gm.N;
  const int x = blockIdx.x, t = threadIdx.x;
  bt += (int64_t)x * ldb;          // this point's solved row b~ = L^-T z0 (b = pinv .* b~)
  double* xs = sm;                 // [d]
  double* th = xs + d;             // [d]
  double* red = th + d;            // [3][HB_T] subset partial sums
  double* tile = red + 3 * HB_T;   // [tp][3d + 1] (r | q_a | q_b) or [d][HB_CT + 1] (derivative rows)
  const int P = d * (d + 1) / 2;
  const int G = P >= HB_T ? 1 : HB_T / P;    // subsets of the point / column range
  const int g = G > 1 ? t / P : 0;
  const bool active = G == 1 || t < G * P;
  const int e0 = G > 1 ? t % P : blockIdx.y * HB_PAGE + t;
  const int nit = G > 1 ? 1 : HB_MAXI;
  for (int j = t; j < d; j += HB_T) { xs[j] = Xs[(int64_t)x * d + j]; th[j] = theta[j]; }
  int ii[HB_MAXI], kk[HB_MAXI];
#pragma unroll
  for (int m = 0; m < HB_MAXI; m++) {
    int e = e0 + m * HB_T, i = 0;
    if (m >= nit || e >= P) { ii[m] = kk[m] = -1; continue; }
    while (e >= d - i) { e -= d - i; i++; }
    ii[m] = i;
    kk[m] = i + e;
  }
  double acc0[HB_MAXI], acc1[HB_MAXI], acc2[HB_MAXI];
#pragma unroll
  for (int m = 0; m < HB_MAXI; m++) acc0[m] = acc1[m] = acc2[m] = 0.0;

  // ---- term2: Gram matrix of the d derivative rows z_1 .. z_d
  const double* z0 = Z + (int64_t)x * (d + 1) * ldz;
  constexpr int GLD = HB_CT + 1;
  for (int c0 = 0; c0 < N; c0 += HB_CT) {
    __syncthreads();
    for (int e = t; e < d * HB_CT; e += HB_T) {
      const int j = e / HB_CT, c = e % HB_CT;
      tile[j * GLD + c] = (c0 + c < N) ? z0[(int64_t)(1 + j) * ldz + c0 + c] : 0.0;
    }
    __syncthreads();
    if (active) {
#pragma unroll
      for (int m = 0; m < HB_MAXI; m++) {
        if (ii[m] < 0) continue;
        const double* zi = tile + ii[m] * GLD;
        const double* zk = tile + kk[m] * GLD;
        double s = acc2[m];
        for (int c = g; c < HB_CT; c += G) s += zi[c] * zk[c];
        acc2[m] = s;
      }
    }
  }

  // ---- d2mu/dx2 and term1: the closed-form contraction over the training points
  const int TLD = 3 * d + 1;
  double wa = 0.0, wb = 0.0;
  for (int p0 = 0; p0 < n; p0 += tp) {
    __syncthreads();
    if (t < tp) {
      double* rr = tile + t * TLD;
      double* qa = rr + d;
      double* qb = qa + d;
      const int p = p0 + t;
      if (p < n) {
        const int sp = gm.slot ? gm.slot[p] : p;
        const double* xp = gm.X + (int64_t)p * d;
        double s = 0.0, sa = 0.0, sb = 0.0;
        for (int j = 0; j < d; j++) {
          const double r = xp[j] - xs[j], u = th[j] * r;
          s += u * r;
          double ga = 0.0, gb = 0.0;
          if (sp >= 0) {
            const int col = n + j * ng + sp;
            ga = a[col];
            gb = bt[col] * pinv[col];
          }
          sa += u * ga;
          sb += u * gb;
          rr[j] = r;
          qa[j] = ga;
          qb[j] = gb;
        }
        const RadialProfile ph = radial_profile(gm.ktype, gm.khp, s);
        const double ca = a[p], cb = bt[p] * pinv[p];
        const double ua = 2.0 * (ph.f2 * ca + 2.0 * ph.f3 * sa), ub = 2.0 * (ph.f2 * cb + 2.0 * ph.f3 * sb);
        const double v = 4.0 * ph.f2;
        for (int j = 0; j < d; j++) {
          qa[j] = ua * rr[j] + v * qa[j];
          qb[j] = ub * rr[j] + v * qb[j];
        }
        wa += 2.0 * ph.f1 * ca + 4.0 * ph.f2 * sa;
        wb += 2.0 * ph.f1 * cb + 4.0 * ph.f2 * sb;
      } else {
        for (int j = 0; j < 3 * d; j++) rr[j] = 0.0;
      }
    }
    __syncthreads();
    if (active) {
#pragma unroll
      for (int m = 0; m < HB_MAXI; m++) {
        if (ii[m] < 0) continue;
        const int i = ii[m], k = kk[m];
        double s0 = acc0[m], s1 = acc1[m];
        for (int q = g; q < tp; q += G) {
          const double* rr = tile + q * TLD;
          const double ri = rr[i], rk = rr[k];
          s0 += ri * rr[d + k] + rk * rr[d + i];
          s1 += ri * rr[2 * d + k] + rk * rr[2 * d + i];
        }
        acc0[m] = s0;
        acc1[m] = s1;
      }
    }
  }
  wa = block_sum(wa, sh);
  wb = block_sum(wb, sh);

  // ---- sum the subsets in a fixed order, scale, mirror
  if (G > 1) {
    __syncthreads();
    if (active) {
      red[t] = acc0[0];
      red[HB_T + t] = acc1[0];
      red[2 * HB_T + t] = acc2[0];
    }
    __syncthreads();
    if (t < P) {
      double s0 = 0.0, s1 = 0.0, s2 = 0.0;
      for (int q = 0; q < G; q++) {
        s0 += red[q * P + t];
        s1 += red[HB_T + q * P + t];
        s2 += red[2 * HB_T + q * P + t];
      }
      acc0[0] = s0;
      acc1[0] = s1;
      acc2[0] = s2;
    }
  }
  if (G == 1 || t < P) {
    double* o = out + (int64_t)x * 3 * d * d;
#pragma unroll
    for (int m = 0; m < HB_MAXI; m++) {
      if (ii[m] < 0) continue;
      const int i = ii[m], k = kk[m];
      const double tt = th[i] * th[k];
      const double h0 = tt * acc0[m] + (i == k ? th[i] * wa : 0.0);
      const double h1 = tt * acc1[m] + (i == k ? th[i] * wb : 0.0);
      const double h2 = acc2[m];
      o[i * d + k] = h0;
      o[d * d + i * d + k] = h1;
      o[2 * d * d + i * d + k] = h2;
      if (i != k) {
        o[k * d + i] = h0;
        o[d * d + k * d + i] = h1;
        o[2 * d * d + k * d + i] = h2;
      }
    }
  }
}

int launch_predict_hess_batch(const Ctx& ctx, const Geom& gm, const double* theta, const double* Xs, int nx, const double* a,
                              const double* bt, int64_t ldb, const double* pinv, const double* Z, int64_t ldz, double* out) {
  if (nx <= 0) return 0;
  const int tp = hess_batch_tile_height(gm.d);
  if (tp == 0) return -908;
  const size_t smem = hess_batch_smem_bytes(gm.d, tp);
  if (smem > 48 * 1024) GEGP_SET_SMEM(predict_hess_batch_kernel, GEGP_MAX_DYN_SMEM);
  const int pages = (gm.d * (gm.d + 1) / 2 + HB_PAGE - 1) / HB_PAGE;
  predict_hess_batch_kernel<<<dim3(nx, pages), HB_T, smem, ctx.stream>>>(gm, theta, Xs, a, bt, ldb, pinv, Z, ldz, tp, out);
  GEGP_CHECK_LAUNCH();
  return 0;
}

}  // namespace gegp
