// K1: fused covariance builder for the gradient-enhanced GP (Gaussian kernel: specialised fast path; Matern-5/2 and
// rational-quadratic kernels: the generic tile kernel with the radial profiles of kernels.h).
//
// Writes the N x N matrix (N = n + n_g*d, dimension-major order) in ONE pass: value block, dK/dx
// blocks, d2K/dxdx' blocks, observation noise, diagonal preconditioner P^-1 . P^-1 and nugget.
// Replaces sq_exp_calc_KernGrad (kernel/KernelSqExp.py:322-410), calc_Rtensor (base/CommonFun.py:58-84)
// and the dense diag-matrix products of calc_all_K_w_chofac (kernel/Kernel.py:213-237, 268-277).
//
// Each CTA owns a tile of point pairs (TA x TB); the squared distance and exp are evaluated once per
// pair, then all (d+1)^2 block entries of the pair are emitted.  Threads run along b, so every store
// instruction of a warp writes one contiguous 256-byte row segment.  HBM-write bound: 8*N^2 bytes.
#include "kernels.h"

namespace gegp {

constexpr int TA = 16;   // a-points per CTA
constexpr int TB = 64;   // b-points per CTA (2 warps wide)
constexpr int BUILD_THREADS = 256;

// p[row] = sqrt(diag(K) + noise[row]), pinv = 1/p.  diag(K) = 1 (value rows), c theta_i (gradient rows; c = 2, or 5/3
// for Matern-5/2: kernel_diag_coef).
__device__ __forceinline__ double noise_at(const NoiseSpec& ns, int z, int row) {
  const double v = ns.noise[z * ns.stride + row];
  if (!ns.divide) return v;
  return v / (ns.varK_all ? ns.varK_all[z] : ns.varK);
}

__global__ void prep_p_kernel(Geom gm, const double* __restrict__ theta, int64_t strideTheta, NoiseSpec ns, int mode,
                              double* __restrict__ p, double* __restrict__ pinv, int64_t strideP) {
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= gm.N) return;
  const int z = blockIdx.z;
  double pv = 1.0, pi = 1.0;
  if (mode == GEGP_MODE_PRECON) {
    const double* th = theta + z * strideTheta;
    double dg = 1.0;
    if (row >= gm.n) dg = kernel_diag_coef(gm.ktype) * th[(row - gm.n) / gm.ng];
    if (ns.noise) dg += noise_at(ns, z, row);
    pv = sqrt(dg);
    pi = 1.0 / pv;
  }
  if (p) p[z * strideP + row] = pv;
  pinv[z * strideP + row] = pi;
}

// mode: GEGP_MODE_BASE   out = varK * (K + diag(noise) + eta I)
//       GEGP_MODE_PRECON out = varK * (P^-1 (K + diag(noise)) P^-1 + eta I)
//       GEGP_MODE_PRECON_COV out = varK * (K + diag(noise) + eta * diag(K + noise))   (= P Ktilde P)
__global__ void __launch_bounds__(BUILD_THREADS)
build_cov_kernel(Geom gm, const double* __restrict__ theta_all, int64_t strideTheta, NoiseSpec ns,
                 const double* __restrict__ pinv_all, int64_t strideP, int mode, double eta,
                 double* __restrict__ out_all, int64_t ld, int64_t strideOut, int lower_only) {
  extern __shared__ double sm[];
  const int d = gm.d, n = gm.n, ng = gm.ng;
  double* xa = sm;                 // [TA][d]
  double* xb = xa + TA * d;        // [d][TB]  (transposed: conflict-free along b)
  double* th = xb + d * TB;        // [d]
  double* sg = th + d;             // [d] gradient-row scale 1/sqrt(2 theta_i) (precon, noise-free) or 1
  int* slot_a = reinterpret_cast<int*>(sg + d);  // [TA]
  int* slot_b = slot_a + TA;                     // [TB]

  const int tid = threadIdx.x;
  const int a0 = blockIdx.y * TA, b0 = blockIdx.x * TB;
  const int z = blockIdx.z;
  const double* theta = theta_all + z * strideTheta;
  const double* pinv = pinv_all ? pinv_all + z * strideP : nullptr;
  double* out = out_all + z * strideOut;
  const bool noise = (ns.noise != nullptr);
  const double varK = ns.varK_all ? ns.varK_all[z] : ns.varK;

  for (int e = tid; e < TA * d; e += BUILD_THREADS) {
    const int a = e / d, i = e % d;
    xa[e] = (a0 + a < n) ? gm.X[(int64_t)(a0 + a) * d + i] : 0.0;
  }
  for (int e = tid; e < TB * d; e += BUILD_THREADS) {
    const int b = e / d, i = e % d;
    xb[i * TB + b] = (b0 + b < n) ? gm.X[(int64_t)(b0 + b) * d + i] : 0.0;
  }
  const bool precon = (mode == GEGP_MODE_PRECON);
  const int ktype = gm.ktype;
  const double kalpha = gm.kernel_hp(z), cdiag = kernel_diag_coef(ktype);
  for (int e = tid; e < d; e += BUILD_THREADS) {
    th[e] = theta[e];
    sg[e] = precon ? 1.0 / sqrt(cdiag * theta[e]) : 1.0;
  }
  for (int e = tid; e < TA; e += BUILD_THREADS) slot_a[e] = (a0 + e < n) ? (gm.slot ? gm.slot[a0 + e] : a0 + e) : -1;
  for (int e = tid; e < TB; e += BUILD_THREADS) slot_b[e] = (b0 + e < n) ? (gm.slot ? gm.slot[b0 + e] : b0 + e) : -1;
  __syncthreads();

  const int tb = tid & (TB - 1);        // b within tile
  const int ta0 = tid / TB;             // 0..3 ; thread owns a = ta0 + 4*q, q = 0..3
  const int b = b0 + tb;
  if (b >= n) return;
  const int sb = slot_b[tb];
  const bool use_pvec = precon && noise;  // per-row scales only differ from sg[] with noise

#pragma unroll 1
  for (int q = 0; q < TA / 4; q++) {
    const int al = ta0 + 4 * q, a = a0 + al;
    if (a >= n) continue;
    const int sa = slot_a[al];
    const double* xav = xa + al * d;
    double e = 0.0;
    for (int i = 0; i < d; i++) {
      const double r = xav[i] - xb[i * TB + tb];
      e += th[i] * (r * r);
    }
    const RadialProfile ph = radial_profile(ktype, kalpha, e);
    const double k = ph.f0, k1 = ph.f1, k2 = ph.f2;
    const bool same = (a == b);
    // ---- value-value entry
    {
      const double sr = use_pvec ? pinv[a] : 1.0, sc = use_pvec ? pinv[b] : 1.0;
      double v = k;
      if (same && noise) v += noise_at(ns, z, a);
      double dadd = 0.0;
      if (same) dadd = (mode == GEGP_MODE_PRECON_COV) ? eta * v : eta;
      v = (v * sr) * sc + dadd;
      if (!lower_only || a >= b) out[(int64_t)a * ld + b] = varK * v;
    }
    // ---- value row, gradient columns: K_0j = -2 th_j r_j f1  (SqExp: +2 th_j r_j k; upper part: skipped when lower_only)
    if (sb >= 0 && !lower_only) {
      const double sr = use_pvec ? pinv[a] : 1.0;
      for (int j = 0; j < d; j++) {
        const int col = n + j * ng + sb;
        const double r = xav[j] - xb[j * TB + tb];
        const double sc = use_pvec ? pinv[col] : sg[j];
        out[(int64_t)a * ld + col] = varK * (((-2.0 * th[j] * r * k1) * sr) * sc);
      }
    }
    if (sa < 0) continue;
    // ---- gradient rows
    for (int i = 0; i < d; i++) {
      const int row = n + i * ng + sa;
      const double ri = xav[i] - xb[i * TB + tb];
      const double sr = use_pvec ? pinv[row] : sg[i];
      const double ui = th[i] * ri;
      double* orow = out + (int64_t)row * ld;
      // gradient-value: K_i0 = 2 th_i r_i f1  (SqExp: -2 th_i r_i k)
      {
        const double sc = use_pvec ? pinv[b] : 1.0;
        orow[b] = varK * (((2.0 * ui * k1) * sr) * sc);
      }
      if (sb < 0) continue;
      const int jmax = lower_only ? i : d - 1;
      for (int j = 0; j <= jmax; j++) {
        if (lower_only && j == i && a < b) continue;
        const int col = n + j * ng + sb;
        const double rj = xav[j] - xb[j * TB + tb];
        double v;
        if (j == i) v = -2.0 * th[i] * k1 - 4.0 * (ui * ui) * k2;   // SqExp: (2 th_i - 4 th_i^2 r_i^2) k
        else v = -4.0 * (ui * (th[j] * rj)) * k2;                   // SqExp: -4 th_i th_j r_i r_j k
        const double sc = use_pvec ? pinv[col] : sg[j];
        double dadd = 0.0;
        if (same && j == i) {
          if (noise) v += noise_at(ns, z, row);
          dadd = (mode == GEGP_MODE_PRECON_COV) ? eta * v : eta;
        }
        orow[col] = varK * ((v * sr) * sc + dadd);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Fast builder for the common case (every point carries a gradient, n even).  Same contract as
// build_cov_kernel, restructured so that the inner loop costs ~5 instructions per stored element instead of
// ~55 and every store is a 16-byte st.global.v2.f64 (each thread owns two neighbouring b points; a warp writes
// one contiguous 512-byte row segment per instruction):
//   * exp(-sum theta r^2) once per pair, folded with varK;
//   * every gradient-gradient entry is a product  c_i(a,b) * w_j(a,b)  of a row factor c_i = -4 w_i k and a
//     column factor w_j = theta_j s_j r_j, so the (i, j) loop is: 3 LDS, 2 DADD, 4 DMUL, 1 STG.128 per two entries;
//   * the diagonal corrections (2 theta_i s_i^2 k on block (i,i); noise and nugget on the matrix diagonal) are
//     applied by separate fix-up stores of the owning thread after the bulk stores.
// PVEC: per-row scales P^-1 (preconditioned matrix with observation noise) instead of one scale per dimension.
// ------------------------------------------------------------------------------------------------
constexpr int FTA = 8;    // a-points per CTA (8 thread rows x 1): many small CTAs balance the triangular work (32: -20 %)
constexpr int FTB = 64;   // b-points per CTA (32 threads x 2); 128 measured slightly slower

template <bool PVEC>
__global__ void __launch_bounds__(BUILD_THREADS)
build_cov_fast_kernel(Geom gm, const double* __restrict__ theta_all, int64_t strideTheta, NoiseSpec ns,
                      const double* __restrict__ pinv_all, int64_t strideP, int mode, double eta,
                      double* __restrict__ out_all, int64_t ld, int64_t strideOut, int lower_only) {
  extern __shared__ __align__(16) double sm[];
  const int d = gm.d, n = gm.n;
  double* xa = sm;                 // [FTA][d]
  double* xb = xa + FTA * d;       // [d][FTB]  (transposed: a thread reads its two b's with one LDS.128)
  double* th = xb + d * FTB;       // [d] theta
  double* ts = th + d;             // [d] theta_i * s_i  (s_i: gradient scale 1/sqrt(2 theta_i) for precon without noise)
  double* dg = ts + d;             // [d] 2 theta_i s_i^2

  const int tid = threadIdx.x;
  const int a0 = blockIdx.y * FTA, b0 = blockIdx.x * FTB;
  const int z = blockIdx.z;
  const double* theta = theta_all + z * strideTheta;
  const double* pinv = pinv_all ? pinv_all + z * strideP : nullptr;
  double* out = out_all + z * strideOut;
  const bool noise = (ns.noise != nullptr);
  const double varK = ns.varK_all ? ns.varK_all[z] : ns.varK;
  const bool precon = (mode == GEGP_MODE_PRECON);

  for (int e = tid; e < FTA * d; e += BUILD_THREADS) {
    const int a = e / d, i = e - a * d;
    xa[e] = (a0 + a < n) ? gm.X[(int64_t)(a0 + a) * d + i] : 0.0;
  }
  for (int e = tid; e < FTB * d; e += BUILD_THREADS) {
    const int b = e / d, i = e - b * d;
    xb[i * FTB + b] = (b0 + b < n) ? gm.X[(int64_t)(b0 + b) * d + i] : 0.0;
  }
  for (int e = tid; e < d; e += BUILD_THREADS) {
    const double t = theta[e];
    const double sgi = (precon && !PVEC) ? 1.0 / sqrt(2.0 * t) : 1.0;
    th[e] = t;
    ts[e] = t * sgi;
    dg[e] = 2.0 * t * sgi * sgi;
  }
  __syncthreads();

  constexpr int TXN = FTB / 2, TYN = BUILD_THREADS / TXN;
  const int tx = tid % TXN, ty = tid / TXN;
  const int b = b0 + 2 * tx;
  if (b >= n) return;                      // n is even: b + 1 < n as well
  const double2* xbp = reinterpret_cast<const double2*>(xb + 2 * tx);   // xbp[i * FTB / 2] = (x_b,i , x_{b+1},i)
  const int64_t nn = n;

#pragma unroll 1
  for (int q = 0; q < FTA / TYN; q++) {
    const int al = ty + TYN * q, a = a0 + al;
    if (a >= n) continue;
    const double* xav = xa + al * d;
    double e0 = 0.0, e1 = 0.0;
    for (int i = 0; i < d; i++) {
      const double2 xbv = xbp[i * (FTB / 2)];
      const double r0 = xav[i] - xbv.x, r1 = xav[i] - xbv.y;
      e0 -= th[i] * (r0 * r0);
      e1 -= th[i] * (r1 * r1);
    }
    const double k0 = varK * exp(e0), k1 = varK * exp(e1);
    const bool lo0 = !lower_only || a >= b, lo1 = !lower_only || a >= b + 1;   // lower-triangle membership of the pair
    // ---- value row a
    {
      double* orow = out + (int64_t)a * ld;
      double sra = 1.0, sc0 = 1.0, sc1 = 1.0;
      if (PVEC) { sra = pinv[a]; sc0 = pinv[b]; sc1 = pinv[b + 1]; }
      const double v0 = (k0 * sra) * sc0, v1 = (k1 * sra) * sc1;
      if (lo0 && lo1) *reinterpret_cast<double2*>(orow + b) = make_double2(v0, v1);
      else if (lo0) orow[b] = v0;
      if (!lower_only) {                       // value row, gradient columns: +2 theta_j r_j k
        double* op = orow + nn + b;
        for (int j = 0; j < d; j++, op += nn) {
          const double2 xbv = xbp[j * (FTB / 2)];
          double w0 = ts[j] * (xav[j] - xbv.x), w1 = ts[j] * (xav[j] - xbv.y);
          if (PVEC) { const double2 sc = *reinterpret_cast<const double2*>(pinv + nn + j * nn + b); w0 *= sc.x; w1 *= sc.y; }
          *reinterpret_cast<double2*>(op) = make_double2((2.0 * w0) * (k0 * sra), (2.0 * w1) * (k1 * sra));
        }
      }
    }
    // ---- gradient rows (i, a)
    for (int i = 0; i < d; i++) {
      const double2 xbi = xbp[i * (FTB / 2)];
      double wi0 = ts[i] * (xav[i] - xbi.x), wi1 = ts[i] * (xav[i] - xbi.y);   // row-scaled u_i
      double wc0 = wi0, wc1 = wi1;                                               // column-scaled u_i (block (i,i))
      double sc0 = 1.0, sc1 = 1.0, dgi0 = dg[i], dgi1 = dg[i];
      const int64_t row = nn + (int64_t)i * nn + a;
      if (PVEC) {
        const double sr = pinv[row];
        const double2 scd = *reinterpret_cast<const double2*>(pinv + nn + i * nn + b);
        sc0 = pinv[b]; sc1 = pinv[b + 1];
        wc0 = wi0 * scd.x; wc1 = wi1 * scd.y;
        wi0 *= sr; wi1 *= sr;
        dgi0 = dg[i] * sr * scd.x; dgi1 = dg[i] * sr * scd.y;
      }
      double* orow = out + row * ld;
      // gradient-value: -2 theta_i r_i k   (always in the lower triangle)
      *reinterpret_cast<double2*>(orow + b) = make_double2((-2.0 * wi0) * (k0 * sc0), (-2.0 * wi1) * (k1 * sc1));
      const double c0 = -4.0 * wi0 * k0, c1 = -4.0 * wi1 * k1;
      const int jend = lower_only ? i : d;
      double* op = orow + nn + b;
      for (int j = 0; j < jend; j++, op += nn) {
        if (j == i) continue;                   // only reachable when !lower_only
        const double2 xbv = xbp[j * (FTB / 2)];
        double w0 = ts[j] * (xav[j] - xbv.x), w1 = ts[j] * (xav[j] - xbv.y);
        if (PVEC) { const double2 sc = *reinterpret_cast<const double2*>(pinv + nn + j * nn + b); w0 *= sc.x; w1 *= sc.y; }
        *reinterpret_cast<double2*>(op) = make_double2(c0 * w0, c1 * w1);
      }
      // block (i, i): (2 theta_i - 4 theta_i^2 r_i^2) k, scaled
      {
        double* od = orow + nn + (int64_t)i * nn + b;
        const double v0 = dgi0 * k0 + c0 * wc0, v1 = dgi1 * k1 + c1 * wc1;
        if (lo0 && lo1) *reinterpret_cast<double2*>(od) = make_double2(v0, v1);
        else if (lo0) od[0] = v0;
      }
    }
    // ---- same point: noise and nugget on the matrix diagonal (after the bulk stores of this thread)
    if (a == b || a == b + 1) {
      const double sr = PVEC ? pinv[a] : 1.0;
      double vv = 1.0;
      if (noise) vv += noise_at(ns, z, a);
      out[(int64_t)a * ld + a] = varK * ((vv * sr) * sr + ((mode == GEGP_MODE_PRECON_COV) ? eta * vv : eta));
      for (int i = 0; i < d; i++) {
        const int64_t row = nn + (int64_t)i * nn + a;
        const double sg2 = PVEC ? pinv[row] * pinv[row] : dg[i] / (2.0 * th[i]);   // s_i^2
        double v = 2.0 * th[i];
        if (noise) v += noise_at(ns, z, (int)row);
        out[row * ld + row] = varK * (v * sg2 + ((mode == GEGP_MODE_PRECON_COV) ? eta * v : eta));
      }
    }
  }
}

// Cross covariance rows for prediction: Kx[x][col] = K(x*_x ; training datum col) * pinv[col]
// value columns: k ; gradient column (j, slot): 2 th_j r_j f1 (SqExp: -2 th_j r_j k) with r = x_train - x_test
// (eval/GpEvalModel.py:133-139 builds K(X, X*) and keeps its value columns; this is its transpose).
__global__ void __launch_bounds__(256)
cross_cov_kernel(Geom gm, const double* __restrict__ theta, const double* __restrict__ pinv,
                 const double* __restrict__ Xs, int nx, double* __restrict__ out, int64_t ld) {
  extern __shared__ double sm[];
  const int d = gm.d, n = gm.n, ng = gm.ng;
  double* xt = sm;            // [CX][d] test points of this CTA
  double* th = xt + 8 * d;    // [d]
  constexpr int CX = 8;
  const int tid = threadIdx.x;
  const int x0 = blockIdx.y * CX;
  for (int e = tid; e < CX * d; e += 256) {
    const int x = e / d, i = e % d;
    xt[e] = (x0 + x < nx) ? Xs[(int64_t)(x0 + x) * d + i] : 0.0;
  }
  for (int e = tid; e < d; e += 256) th[e] = theta[e];
  __syncthreads();
  const int b = blockIdx.x * 256 + tid;  // training point
  if (b >= n) return;
  const int sb = gm.slot ? gm.slot[b] : b;
  const double* xb = gm.X + (int64_t)b * d;
  for (int x = 0; x < CX && x0 + x < nx; x++) {
    const double* xv = xt + x * d;
    double e = 0.0;
    for (int i = 0; i < d; i++) {
      const double r = xb[i] - xv[i];
      e += th[i] * (r * r);
    }
    const RadialProfile ph = radial_profile(gm.ktype, gm.khp, e);
    double* orow = out + (int64_t)(x0 + x) * ld;
    orow[b] = ph.f0 * (pinv ? pinv[b] : 1.0);
    if (sb >= 0) {
      for (int j = 0; j < d; j++) {
        const int col = n + j * ng + sb;
        const double r = xb[j] - xv[j];
        orow[col] = (2.0 * th[j] * r * ph.f1) * (pinv ? pinv[col] : 1.0);
      }
    }
  }
}

// Cross covariance WITH its derivatives with respect to the test point (eval/GpEvalModel.py:133-139 keeps the
// test-gradient columns of K(X, X*) for calc_grad; kernel/KernelSqExp.py:392-408 gives the blocks).  Per test point
// x the output holds d + 1 consecutive rows: row 0 = k*(x) as cross_cov_kernel writes it, row 1 + j = d k*(x) / d x*_j:
//   value entry a      :  -2 th_j r_j f1                        (r = x_train - x_test; SqExp: +2 th_j r_j k)
//   gradient entry (i,a): -2 th_i delta_ij f1 - 4 th_i th_j r_i r_j f2   (SqExp: (2 th_i delta_ij - 4 th_i th_j r_i r_j) k)
// every entry scaled by pinv of its training row.
__global__ void __launch_bounds__(256)
cross_cov_dx_kernel(Geom gm, const double* __restrict__ theta, const double* __restrict__ pinv,
                    const double* __restrict__ Xs, int nx, double* __restrict__ out, int64_t ld) {
  extern __shared__ double sm[];
  const int d = gm.d, n = gm.n, ng = gm.ng;
  double* xv = sm;          // [d] the test point of this CTA row
  double* th = xv + d;      // [d]
  const int tid = threadIdx.x, x = blockIdx.y;
  for (int e = tid; e < d; e += 256) { xv[e] = Xs[(int64_t)x * d + e]; th[e] = theta[e]; }
  __syncthreads();
  const int b = blockIdx.x * 256 + tid;  // training point
  if (b >= n) return;
  const int sb = gm.slot ? gm.slot[b] : b;
  const double* xb = gm.X + (int64_t)b * d;
  double e = 0.0;
  for (int i = 0; i < d; i++) {
    const double r = xb[i] - xv[i];
    e += th[i] * (r * r);
  }
  const RadialProfile ph = radial_profile(gm.ktype, gm.khp, e);
  const double k = ph.f0, k1 = ph.f1, k2 = ph.f2;
  double* base = out + (int64_t)x * (d + 1) * ld;
  const double pb = pinv ? pinv[b] : 1.0;
  base[b] = k * pb;
  for (int j = 0; j < d; j++) {
    const double rj = xb[j] - xv[j];
    base[(int64_t)(1 + j) * ld + b] = (-2.0 * th[j] * rj * k1) * pb;
  }
  if (sb >= 0) {
    for (int i = 0; i < d; i++) {
      const int col = n + i * ng + sb;
      const double pc = pinv ? pinv[col] : 1.0;
      const double ri = xb[i] - xv[i];
      const double ui = th[i] * ri;
      base[col] = (2.0 * ui * k1) * pc;
      for (int j = 0; j < d; j++) {
        const double rj = xb[j] - xv[j];
        const double v = ((i == j) ? -2.0 * th[i] * k1 : 0.0) - 4.0 * ui * th[j] * rj * k2;
        base[(int64_t)(1 + j) * ld + col] = v * pc;
      }
    }
  }
}

// rows[0] = pinv .* y ; rows[1] = pinv .* H  (H = [1_n ; 0], eval/GpMeanFun.py:172-191)
__global__ void append_rhs_kernel(int N, int n, const double* __restrict__ y, const double* __restrict__ pinv,
                                  int64_t strideP, double* __restrict__ rows, int64_t ld, int64_t strideRows) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  const double s = pinv ? pinv[blockIdx.z * strideP + i] : 1.0;
  double* r = rows + blockIdx.z * strideRows;
  r[i] = y[i] * s;
  r[ld + i] = (i < n) ? s : 0.0;
}

// row = pinv .* (y - beta H)
__global__ void append_res_kernel(int N, int n, const double* __restrict__ y, double beta,
                                  const double* __restrict__ pinv, double* __restrict__ row) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  row[i] = (y[i] - (i < n ? beta : 0.0)) * (pinv ? pinv[i] : 1.0);
}

int launch_append_res(const Ctx& ctx, int N, int n, const double* y, double beta, const double* pinv, double* row) {
  append_res_kernel<<<(N + 255) / 256, 256, 0, ctx.stream>>>(N, n, y, beta, pinv, row);
  GEGP_CHECK_LAUNCH();
  return 0;
}

int launch_prep_p(const Ctx& ctx, const Geom& gm, const double* theta, int64_t strideTheta, NoiseSpec ns, int mode,
                  double* p, double* pinv, int64_t strideP) {
  prep_p_kernel<<<dim3((gm.N + 255) / 256, 1, ctx.batch), 256, 0, ctx.stream>>>(gm, theta, strideTheta, ns, mode, p,
                                                                             pinv, strideP);
  GEGP_CHECK_LAUNCH();
  return 0;
}

int launch_build_cov(const Ctx& ctx, const Geom& gm, const double* theta, int64_t strideTheta, NoiseSpec ns,
                     const double* pinv, int64_t strideP, int mode, double eta, double* out, int64_t ld,
                     int64_t strideOut, int lower_only) {
  // fast path: all points carry gradients, even n (16-byte aligned column blocks), aligned even-stride output
  const size_t fsmem = (size_t)(FTA * gm.d + gm.d * FTB + 3 * gm.d) * sizeof(double);
  const bool use_pvec = (mode == GEGP_MODE_PRECON) && ns.noise != nullptr;
  if (gm.ktype == GEGP_KERNEL_SQEXP && gm.slot == nullptr && gm.ng == gm.n && (gm.n & 1) == 0 && (ld & 1) == 0 &&
      (strideOut & 1) == 0 &&
      (reinterpret_cast<uintptr_t>(out) & 15) == 0 && fsmem <= 200 * 1024 &&
      (!use_pvec || ((strideP & 1) == 0 && (reinterpret_cast<uintptr_t>(pinv) & 15) == 0))) {
    if (fsmem > 48 * 1024) {   // opt in once per device to the largest size any d can ask for
      if (use_pvec) GEGP_SET_SMEM(build_cov_fast_kernel<true>, GEGP_MAX_DYN_SMEM);
      else GEGP_SET_SMEM(build_cov_fast_kernel<false>, GEGP_MAX_DYN_SMEM);
    }
    dim3 grid((gm.n + FTB - 1) / FTB, (gm.n + FTA - 1) / FTA, ctx.batch);
    timeline_begin(ctx.stream, "build", gm.N, lower_only);
    if (use_pvec)
      build_cov_fast_kernel<true><<<grid, BUILD_THREADS, fsmem, ctx.stream>>>(gm, theta, strideTheta, ns, pinv, strideP, mode,
                                                                            eta, out, ld, strideOut, lower_only);
    else
      build_cov_fast_kernel<false><<<grid, BUILD_THREADS, fsmem, ctx.stream>>>(gm, theta, strideTheta, ns, pinv, strideP, mode,
                                                                             eta, out, ld, strideOut, lower_only);
    timeline_end(ctx.stream);
    GEGP_CHECK_LAUNCH();
    return 0;
  }
  const size_t smem = (size_t)(TA * gm.d + gm.d * TB + 2 * gm.d) * sizeof(double) + (TA + TB) * sizeof(int);
  if (smem > GEGP_MAX_DYN_SMEM) return -907;
  if (smem > 48 * 1024) GEGP_SET_SMEM(build_cov_kernel, GEGP_MAX_DYN_SMEM);
  dim3 grid((gm.n + TB - 1) / TB, (gm.n + TA - 1) / TA, ctx.batch);
  build_cov_kernel<<<grid, BUILD_THREADS, smem, ctx.stream>>>(gm, theta, strideTheta, ns, pinv, strideP, mode, eta, out,
                                                              ld, strideOut, lower_only);
  GEGP_CHECK_LAUNCH();
  return 0;
}

// Both cross-covariance kernels put test points on gridDim.y, which is limited to 65535.  A small training set lets
// the prediction chunk hold far more test points than that (n = 20, d = 2: ~700k gradient points per GiB), so the
// launch is issued in slices of at most MAX_GRID_Y grid rows, each with Xs and out advanced to its first point.  Every
// test point is computed by the same thread arithmetic whichever slice it lands in.
constexpr int MAX_GRID_Y = 65535;

int launch_cross_cov(const Ctx& ctx, const Geom& gm, const double* theta, const double* pinv, const double* Xs, int nx,
                     double* out, int64_t ld) {
  const size_t smem = (size_t)(8 * gm.d + gm.d) * sizeof(double);
  constexpr int SLICE = 8 * MAX_GRID_Y;   // 8 test points per CTA row
  for (int x0 = 0; x0 < nx; x0 += SLICE) {
    const int cx = (nx - x0 < SLICE) ? nx - x0 : SLICE;
    dim3 grid((gm.n + 255) / 256, (cx + 7) / 8, 1);
    cross_cov_kernel<<<grid, 256, smem, ctx.stream>>>(gm, theta, pinv, Xs + (int64_t)x0 * gm.d, cx,
                                                      out + (int64_t)x0 * ld, ld);
    GEGP_CHECK_LAUNCH();
  }
  return 0;
}

int launch_cross_cov_dx(const Ctx& ctx, const Geom& gm, const double* theta, const double* pinv, const double* Xs, int nx,
                        double* out, int64_t ld) {
  const size_t smem = (size_t)(2 * gm.d) * sizeof(double);
  for (int x0 = 0; x0 < nx; x0 += MAX_GRID_Y) {   // one test point (d + 1 output rows) per CTA row
    const int cx = (nx - x0 < MAX_GRID_Y) ? nx - x0 : MAX_GRID_Y;
    dim3 grid((gm.n + 255) / 256, cx, 1);
    cross_cov_dx_kernel<<<grid, 256, smem, ctx.stream>>>(gm, theta, pinv, Xs + (int64_t)x0 * gm.d, cx,
                                                         out + (int64_t)x0 * (gm.d + 1) * ld, ld);
    GEGP_CHECK_LAUNCH();
  }
  return 0;
}

int launch_append_rhs(const Ctx& ctx, int N, int n, const double* y, const double* pinv, int64_t strideP, double* rows,
                      int64_t ld, int64_t strideRows) {
  append_rhs_kernel<<<dim3((N + 255) / 256, 1, ctx.batch), 256, 0, ctx.stream>>>(N, n, y, pinv, strideP, rows, ld,
                                                                              strideRows);
  GEGP_CHECK_LAUNCH();
  return 0;
}

}  // namespace gegp
