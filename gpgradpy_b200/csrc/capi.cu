// extern "C" entry points of libgegp.so (see include/gegp.h for the contract and the reference mapping).
#include "kernels.h"
#include "linalg.h"
#include <algorithm>
#include <cstdlib>
#include <cstring>

#include <vector>

using namespace gegp;

namespace gegp {
static Prof g_prof;
static std::vector<cudaEvent_t> g_ev;   // begin/end pairs around every GEMM launch while profiling
static size_t g_ev_used = 0;
Prof& prof() { return g_prof; }
static cudaEvent_t next_event() {
  if (g_ev_used == g_ev.size()) {
    cudaEvent_t e;
    cudaEventCreate(&e);
    g_ev.push_back(e);
  }
  return g_ev[g_ev_used++];
}
void prof_gemm_begin(cudaStream_t s) {
  if (g_prof.on) cudaEventRecord(next_event(), s);
}
void prof_gemm_end(cudaStream_t s, double flops) {
  if (!g_prof.on) return;
  cudaEventRecord(next_event(), s);
  g_prof.gemm_flops += flops;
  g_prof.gemm_launches++;
}

struct TlMark { cudaEvent_t b, e; cudaStream_t s; char label[48]; };
static std::vector<TlMark> g_tl;
static int g_tl_state = -1;   // -1 unknown, 0 off, 1 on
bool timeline_on() {
  if (g_tl_state < 0) g_tl_state = getenv("GEGP_TIMELINE") ? 1 : 0;
  return g_tl_state == 1;
}
void timeline_begin(cudaStream_t s, const char* label, int a, int b, int c, double mflop) {
  if (!timeline_on()) return;
  TlMark m{};
  cudaEventCreate(&m.b);
  cudaEventCreate(&m.e);
  m.s = s;
  snprintf(m.label, sizeof(m.label), "%s:%d:%d:%d:%.0f", label, a, b, c, mflop);
  cudaEventRecord(m.b, s);
  g_tl.push_back(m);
}
void timeline_end(cudaStream_t s) {
  if (!timeline_on() || g_tl.empty()) return;
  cudaEventRecord(g_tl.back().e, s);
}
static void timeline_dump() {
  if (!timeline_on() || g_tl.empty()) return;
  cudaDeviceSynchronize();
  FILE* f = fopen(getenv("GEGP_TIMELINE"), "w");
  if (f) {
    for (const TlMark& m : g_tl) {
      float t0 = 0.f, t1 = 0.f;
      cudaEventElapsedTime(&t0, g_tl[0].b, m.b);
      cudaEventElapsedTime(&t1, g_tl[0].b, m.e);
      fprintf(f, "%s %p %.1f %.1f\n", m.label, (void*)m.s, t0 * 1e3, t1 * 1e3);
    }
    fclose(f);
  }
  for (TlMark& m : g_tl) { cudaEventDestroy(m.b); cudaEventDestroy(m.e); }
  g_tl.clear();
}
static int g_lookahead = -1;
int& lookahead_enabled() {
  if (g_lookahead < 0) g_lookahead = getenv("GEGP_NO_LOOKAHEAD") ? 0 : 1;
  return g_lookahead;
}
}  // namespace gegp

namespace {

inline int64_t round_up(int64_t v, int64_t q) { return (v + q - 1) / q * q; }

struct LmlLayout {
  int64_t ld;          // leading dimension of every N-column matrix
  size_t A, P, W, D, U, Kinv, Part;  // per-candidate element (double) offsets
  size_t per_cand_doubles;
};

LmlLayout lml_layout(int n, int d, int N, bool grad) {
  LmlLayout L{};
  L.ld = gegp_ld(N);
  size_t off = 0;
  L.A = off;    off += (size_t)(N + 2) * L.ld;
  L.P = off;    off += (size_t)2 * L.ld;
  L.W = off;    off += (size_t)2 * L.ld;   // w = L^-1 P^-1 res, then the preconditioned alpha = L^-T w
  L.D = off;    off += (size_t)dinv_doubles(N);
  if (grad) {
    L.U = off;    off += (size_t)N * L.ld;
    L.Kinv = off; off += (size_t)N * L.ld;
    L.Part = off; off += round_up((int64_t)lml_grad_partial_doubles(n, d), 2);
  }
  L.per_cand_doubles = off;
  return L;
}

// the workspace starts with one int per candidate (Cholesky info), padded to 256 bytes
size_t info_header_bytes(int B) { return (size_t)round_up((int64_t)B * (int64_t)sizeof(int), 256); }

bool bad_geom(int n, int n_g, int d) { return n <= 0 || d <= 0 || n_g < 0 || n_g > n; }

// kernel family + extra hyper-parameter: the rational-quadratic alpha must be positive, the others ignore it
bool bad_kernel(int kernel, double kernel_hp) {
  if (kernel < GEGP_KERNEL_SQEXP || kernel > GEGP_KERNEL_RATQUAD) return true;
  return kernel == GEGP_KERNEL_RATQUAD && !(kernel_hp > 0.0);
}

Geom make_geom(int n, int n_g, int d, const double* X, const int32_t* grad_slot, int kernel, double kernel_hp,
               const double* kernel_hp_batch = nullptr) {
  return Geom{n, n_g, d, n + n_g * d, X, (n_g == n) ? nullptr : grad_slot, kernel, kernel_hp, kernel_hp_batch};
}

// The factored training set that gegp_predict_setup leaves behind, as the posterior entry points read it.
struct Posterior {
  Geom gm;
  const double* theta;
  const double* A;      // factor L (lower), ld lda
  int64_t lda;
  const double* dinv;   // inverted diagonal blocks of L
  const double* pinv;   // P^-1
  const double* w;      // row N of A: L^-1 P^-1 (y - H beta)
};

// The arguments every posterior entry point starts with, checked in order: -1 geometry, -50 kernel, -4 X, -5 grad_slot,
// -6 theta, -7 A, -8 lda, -9 dinv, -10 p.
int posterior_args(int n, int n_g, int d, const double* X, const int32_t* grad_slot, const double* theta, int kernel,
                   double kernel_hp, const double* A, int64_t lda, const double* dinv, const double* p, Posterior* ps) {
  if (bad_geom(n, n_g, d)) return -1;
  if (bad_kernel(kernel, kernel_hp)) return -50;
  if (!X) return -4;
  if (n_g != n && !grad_slot) return -5;
  if (!theta) return -6;
  if (!A) return -7;
  const int N = n + n_g * d;
  if (lda < N || (lda & 1)) return -8;
  if (!dinv) return -9;
  if (!p) return -10;
  *ps = Posterior{make_geom(n, n_g, d, X, grad_slot, kernel, kernel_hp), theta, A, lda, dinv, p + N, A + (int64_t)N * lda};
  return 0;
}

// Test points x0 .. x0 + cx - 1 of Xs: their cross covariances k* (and dk*/dx when dmu is given: d + 1 rows per point)
// into Z, the forward solve Z := L^-1 P^-1 Z in place, then mu, sig, sig2 (and dmu, dsig) of those points.
int posterior_chunk(const Ctx& ctx, const Posterior& ps, double beta, double varK, const double* Xs, int x0, int cx,
                    double* Z, int64_t ldz, double* mu, double* sig, double* sig2, double* dmu, double* dsig,
                    int* n_negative) {
  const int d = ps.gm.d, N = ps.gm.N, dr = dmu ? d : 0;
  const double* xs = Xs + (int64_t)x0 * d;
  int rc = dmu ? launch_cross_cov_dx(ctx, ps.gm, ps.theta, ps.pinv, xs, cx, Z, ldz)
               : launch_cross_cov(ctx, ps.gm, ps.theta, ps.pinv, xs, cx, Z, ldz);
  if (rc) return rc;
  rc = trsm_right_rec(ctx, ps.A, ps.lda, 0, ps.dinv, 0, 0, Z, ldz, 0, cx * (dr + 1), N);
  if (rc) return rc;
  return launch_predict_grad_rows(ctx, N, dr, Z, ldz, cx, ps.w, beta, varK, mu + x0, sig + x0, sig2 ? sig2 + x0 : nullptr,
                                  dmu ? dmu + (int64_t)x0 * d : nullptr, dsig ? dsig + (int64_t)x0 * d : nullptr,
                                  n_negative);
}

}  // namespace

extern "C" {

int gegp_abi_version(void) { return GEGP_ABI_VERSION; }

void gegp_profile_begin(int time_gemm) {
  g_prof.launches = 0;
  g_prof.gemm_flops = 0.0;
  g_prof.gemm_launches = 0;
  g_prof.on = (time_gemm != 0);
  g_ev_used = 0;
}

int gegp_profile_end(long* launches, long* gemm_launches, double* gemm_ms, double* gemm_flops) {
  double ms = 0.0;
  if (g_prof.on) {
    if (cudaDeviceSynchronize() != cudaSuccess) return -1;
    for (size_t i = 0; i + 1 < g_ev_used; i += 2) {
      float t = 0.f;
      cudaEventElapsedTime(&t, g_ev[i], g_ev[i + 1]);
      ms += t;
    }
  }
  if (launches) *launches = g_prof.launches;
  if (gemm_launches) *gemm_launches = g_prof.gemm_launches;
  if (gemm_ms) *gemm_ms = ms;
  if (gemm_flops) *gemm_flops = g_prof.gemm_flops;
  g_prof.on = false;
  g_ev_used = 0;
  timeline_dump();
  return 0;
}

int64_t gegp_ld(int N) { return round_up(N, 16); }

int gegp_set_option(int key, int value) {
  if (key == GEGP_OPT_TMA_MIN_TILES) {
    if (value < 1) return -2;
    const int old = tma_min_tiles();
    tma_min_tiles() = value;
    return old;
  }
  if (key == GEGP_OPT_SMALL_TILE_MAX) {
    if (value < 0) return -2;
    const int old = small_tile_max();
    small_tile_max() = value;
    return old;
  }
  if (key == GEGP_OPT_CHAIN_CLUSTER) {
    if (value != 0 && value != 1 && value != 2 && value != 4) return -2;
    const int old = chain_cluster();
    chain_cluster() = value;
    return old;
  }
  if (key == GEGP_OPT_INV_EARLY) {
    if (value < 0 || value > 3) return -2;
    const int old = inv_early_option();
    inv_early_option() = value;
    return old;
  }
  if (key == GEGP_OPT_LOOKAHEAD) {
    const int old = lookahead_enabled();
    lookahead_enabled() = value ? 1 : 0;
    return old;
  }
  return -1;
}

size_t gegp_workspace_bytes(int op, int n, int n_g, int d, int arg) {
  if (bad_geom(n, n_g, d) || arg <= 0) return 0;
  const int N = n + n_g * d;
  if (op == GEGP_OP_LML || op == GEGP_OP_LML_GRAD) {
    LmlLayout L = lml_layout(n, d, N, op == GEGP_OP_LML_GRAD);
    return info_header_bytes(arg) + L.per_cand_doubles * sizeof(double) * (size_t)arg;
  }
  if (op == GEGP_OP_PREDICT) return (size_t)arg * gegp_ld(N) * sizeof(double);
  return 0;
}

int gegp_build_cov(int n, int n_g, int d, const double* X, const int32_t* grad_slot, const double* theta, int kernel, double kernel_hp,
                   const double* noise, int mode, double eta, double varK, double* K_out, int64_t ldk, double* p_out,
                   int uplo, void* stream) {
  if (bad_geom(n, n_g, d)) return -1;
  if (bad_kernel(kernel, kernel_hp)) return -50;
  if (!X) return -4;
  if (!theta) return -6;
  if (mode < GEGP_MODE_BASE || mode > GEGP_MODE_PRECON_COV) return -8;
  if (!K_out) return -11;
  const int N = n + n_g * d;
  if (ldk < N) return -12;
  if (mode == GEGP_MODE_PRECON && !p_out) return -13;
  if (n_g != n && !grad_slot) return -5;  // gradient-free GP (n_g == 0): pass a slot array of -1
  Ctx ctx{(cudaStream_t)stream, 1};
  const Geom gm = make_geom(n, n_g, d, X, grad_slot, kernel, kernel_hp);
  NoiseSpec ns{noise, 0, nullptr, varK, 0};
  int rc = 0;
  if (p_out) {
    rc = launch_prep_p(ctx, gm, theta, 0, ns, mode, p_out, p_out + N, 0);
    if (rc) return rc;
  }
  return launch_build_cov(ctx, gm, theta, 0, ns, p_out ? p_out + N : nullptr, 0, mode, eta, K_out, ldk, 0, uplo ? 1 : 0);
}

int gegp_build_cov_batch(int B, const double* theta_batch, const double* varK_batch, int kernel,
                         const double* kernel_hp_batch, int n, int n_g, int d, const double* X, const int32_t* grad_slot,
                         const double* noise, int mode, double eta, double* K_out, int64_t ldk, int64_t strideK,
                         double* p_out, int64_t strideP, int uplo, void* stream) {
  if (B <= 0 || B > 65535) return -1;
  if (!theta_batch) return -2;
  if (kernel < GEGP_KERNEL_SQEXP || kernel > GEGP_KERNEL_RATQUAD) return -50;
  if (kernel == GEGP_KERNEL_RATQUAD && !kernel_hp_batch) return -50;
  if (bad_geom(n, n_g, d)) return -6;
  if (!X) return -9;
  if (n_g != n && !grad_slot) return -10;
  if (mode < GEGP_MODE_BASE || mode > GEGP_MODE_PRECON_COV) return -12;
  if (!K_out) return -14;
  const int N = n + n_g * d;
  if (ldk < N) return -15;
  if (strideK < 0) return -16;
  if (mode == GEGP_MODE_PRECON && !p_out) return -17;
  if (p_out && strideP < 2 * (int64_t)N) return -18;
  Ctx ctx{(cudaStream_t)stream, B};
  const Geom gm = make_geom(n, n_g, d, X, grad_slot, kernel, 0.0, kernel_hp_batch);
  NoiseSpec ns{noise, 0, varK_batch, 1.0, (noise && varK_batch) ? 1 : 0};
  int rc = 0;
  if (p_out) {
    rc = launch_prep_p(ctx, gm, theta_batch, d, ns, mode, p_out, p_out + N, strideP);
    if (rc) return rc;
  }
  return launch_build_cov(ctx, gm, theta_batch, d, ns, p_out ? p_out + N : nullptr, strideP, mode, eta, K_out, ldk, strideK,
                          uplo ? 1 : 0);
}

int gegp_cross_cov(int n, int n_g, int d, const double* X, const int32_t* grad_slot, const double* Xs, int nx,
                   const double* theta, int kernel, double kernel_hp, const double* pinv, double* Kx, int64_t ld, void* stream) {
  if (bad_geom(n, n_g, d)) return -1;
  if (bad_kernel(kernel, kernel_hp)) return -50;
  if (!X) return -4;
  if (!Xs || nx < 0) return -6;
  if (!theta) return -8;
  if (!Kx) return -10;
  const int N = n + n_g * d;
  if (ld < N) return -11;
  if (n_g != n && !grad_slot) return -5;
  if (nx == 0) return 0;
  Ctx ctx{(cudaStream_t)stream, 1};
  const Geom gm = make_geom(n, n_g, d, X, grad_slot, kernel, kernel_hp);
  return launch_cross_cov(ctx, gm, theta, pinv, Xs, nx, Kx, ld);
}

int64_t gegp_dinv_doubles(int N) { return N > 0 ? dinv_doubles(N) : 0; }

int gegp_potrf(int N, int n_extra, double* A, int64_t lda, double* dinv, int* info_dev, void* stream) {
  if (N <= 0) return -1;
  if (n_extra < 0) return -2;
  if (!A || (reinterpret_cast<uintptr_t>(A) & 15)) return -3;
  if (lda < N || (lda & 1)) return -4;
  if (!dinv || (reinterpret_cast<uintptr_t>(dinv) & 15)) return -5;
  if (!info_dev) return -6;
  Ctx ctx{(cudaStream_t)stream, 1};
  const int rc = chol_trap(ctx, A, lda, 0, N + n_extra, N, 0, info_dev, dinv, 0);
  if (rc) return rc;
  return leaf_dinv_assemble(ctx, A, lda, 0, dinv, 0, N);   // hand out a complete factor (A, dinv)
}

int gegp_trsm_rows(int N, const double* L, int64_t ldl, const double* dinv, double* B, int64_t ldb, int r,
                   void* stream) {
  if (N <= 0) return -1;
  if (!L) return -2;
  if (ldl < N || (ldl & 1)) return -3;
  if (!dinv) return -4;
  if (!B || (reinterpret_cast<uintptr_t>(B) & 15)) return -5;
  if (ldb < N || (ldb & 1)) return -6;
  if (r < 0) return -7;
  Ctx ctx{(cudaStream_t)stream, 1};
  return trsm_right_rec(ctx, L, ldl, 0, dinv, 0, 0, B, ldb, 0, r, N);
}

int gegp_potri(int N, const double* L, int64_t ldl, const double* dinv, double* U, int64_t ldu, double* Kinv,
               int64_t ldk, void* stream) {
  if (N <= 0) return -1;
  if (!L) return -2;
  if (ldl < N || (ldl & 1)) return -3;
  if (!dinv) return -4;
  if (!U || (reinterpret_cast<uintptr_t>(U) & 15)) return -5;
  if (ldu < N || (ldu & 1)) return -6;
  if (!Kinv || (reinterpret_cast<uintptr_t>(Kinv) & 15)) return -7;
  if (ldk < N || (ldk & 1)) return -8;
  Ctx ctx{(cudaStream_t)stream, 1};
  return chol_inverse(ctx, L, ldl, 0, dinv, 0, U, ldu, 0, Kinv, ldk, 0, N);
}

int gegp_dgemm(int transb, int M, int N, int K, double alpha, const double* A, int64_t lda, const double* B,
               int64_t ldb, double beta, double* C, int64_t ldc, void* stream) {
  if (M < 0) return -2;
  if (N < 0) return -3;
  if (K < 0) return -4;
  if (!A || lda < K) return -6;
  if (!B || ldb < (transb ? K : N)) return -8;
  if (!C || ldc < N) return -11;
  Ctx ctx{(cudaStream_t)stream, 1};
  return gemm_f64(ctx, gemm_args(A, lda, B, ldb, C, ldc, M, N, K, alpha, beta, transb != 0));
}

int gegp_lml_eval(int B, const double* theta_batch, const double* varK_batch, int kernel,
                  const double* kernel_hp_batch, int n, int n_g, int d, const double* X,
                  const int32_t* grad_slot, const double* y, const double* noise, int mode, double eta, int noisy,
                  double pnlt_grad, int want_grad, double* out, double* alpha_out, void* work, size_t work_bytes,
                  void* stream) {
  if (B <= 0) return -1;
  if (!theta_batch) return -2;
  if (noisy && !varK_batch) return -3;
  if (kernel < GEGP_KERNEL_SQEXP || kernel > GEGP_KERNEL_RATQUAD) return -50;
  if (kernel == GEGP_KERNEL_RATQUAD && !kernel_hp_batch) return -50;
  if (bad_geom(n, n_g, d)) return -4;
  if (!X) return -7;
  if (n_g != n && !grad_slot) return -8;
  if (!y) return -9;
  if (noisy && !noise) return -10;
  if (mode != GEGP_MODE_BASE && mode != GEGP_MODE_PRECON) return -11;
  if (!out) return -16;
  if (!work || (reinterpret_cast<uintptr_t>(work) & 15)) return -18;
  const int N = n + n_g * d;
  const LmlLayout L = lml_layout(n, d, N, want_grad != 0);
  const size_t per = L.per_cand_doubles * sizeof(double);
  const size_t header = info_header_bytes(B);
  if (work_bytes < header + per) return -19;
  const int chunk = (int)std::min<size_t>((size_t)B, (work_bytes - header) / per);
  cudaStream_t st = (cudaStream_t)stream;
  int* info = reinterpret_cast<int*>(work);
  double* wk = reinterpret_cast<double*>(reinterpret_cast<char*>(work) + header);
  const int64_t sC = (int64_t)L.per_cand_doubles;  // candidate stride of every workspace array
  const int outlen = GEGP_OUT_LEN(d);

  for (int b0 = 0; b0 < B; b0 += chunk) {
    const int nb = std::min(chunk, B - b0);
    Ctx ctx{st, nb};
    const Geom gm = make_geom(n, n_g, d, X, grad_slot, kernel, 0.0, kernel_hp_batch ? kernel_hp_batch + b0 : nullptr);
    const double* theta = theta_batch + (int64_t)b0 * d;
    const double* varK = noisy ? varK_batch + b0 : nullptr;
    double* A = wk + L.A;
    double* P = wk + L.P;
    double* pinv = P + L.ld;
    double* W = wk + L.W;
    double* outb = out + (int64_t)b0 * outlen;
    {
      cudaError_t e = cudaMemsetAsync(info, 0, sizeof(int) * nb, st);
      if (e != cudaSuccess) return -1000 - (int)e;
    }
    NoiseSpec ns{noisy ? noise : nullptr, 0, varK, 1.0, 1};
    int rc = launch_prep_p(ctx, gm, theta, d, ns, mode, P, pinv, sC);
    if (rc) return rc;
    rc = launch_build_cov(ctx, gm, theta, d, ns, pinv, sC, mode, eta, A, L.ld, sC, 1);
    if (rc) return rc;
    rc = launch_append_rhs(ctx, N, n, y, pinv, sC, A + (int64_t)N * L.ld, L.ld, sC);
    if (rc) return rc;
    double* D = wk + L.D;
    if (want_grad) rc = chol_trap_inverse(ctx, A, L.ld, sC, N + 2, N, info, D, sC, wk + L.U, L.ld, sC, wk + L.Kinv, L.ld, sC);
    else rc = chol_trap(ctx, A, L.ld, sC, N + 2, N, 0, info, D, sC);
    if (rc) return rc;
    rc = launch_lml_finalize(ctx, N, A, L.ld, sC, pinv, sC, noisy, varK, W, sC, outb, outlen, info, want_grad ? 0 : d);
    if (rc) return rc;
    double* alpha_t = W;  // preconditioned alpha = L^-T w
    if (want_grad) {
      double* U = wk + L.U;
      double* Kinv = wk + L.Kinv;
      alpha_t = W + L.ld;
      rc = trmv_upper(ctx, U, L.ld, sC, W, sC, alpha_t, sC, N);  // U = L^-T is already there: no substitution
      if (rc) return rc;
      rc = launch_lml_grad(ctx, gm, theta, d, Kinv, L.ld, sC, alpha_t, sC, pinv, sC, mode, eta, noisy, varK, pnlt_grad,
                           wk + L.Part, sC, outb, outlen);
      if (rc) return rc;
    } else if (alpha_out) {
      rc = leaf_dinv_assemble(ctx, A, L.ld, sC, D, sC, N);
      if (rc) return rc;
      rc = trsv_lower_trans(ctx, A, L.ld, sC, D, sC, W, L.ld, sC, N, 1);
      if (rc) return rc;
    }
    if (alpha_out) {
      rc = launch_scale_vec(ctx, N, alpha_t, sC, pinv, sC, alpha_out + (int64_t)b0 * N, N);
      if (rc) return rc;
    }
  }
  return 0;
}

int gegp_lml_layout(int n, int n_g, int d, int want_grad, int B, int64_t* out8) {
  if (bad_geom(n, n_g, d)) return -1;
  if (B <= 0) return -5;
  if (!out8) return -6;
  const int N = n + n_g * d;
  const LmlLayout L = lml_layout(n, d, N, want_grad != 0);
  out8[0] = (int64_t)info_header_bytes(B);
  out8[1] = L.ld;
  out8[2] = (int64_t)L.per_cand_doubles;
  out8[3] = (int64_t)L.A;
  out8[4] = (int64_t)L.P;
  out8[5] = (int64_t)L.D;
  out8[6] = want_grad ? (int64_t)L.U : -1;
  out8[7] = want_grad ? (int64_t)L.Kinv : -1;
  return 0;
}

int gegp_symv(int N, const double* M, int64_t ld, const double* x, double* y, void* stream) {
  if (N <= 0) return -1;
  if (!M || (reinterpret_cast<uintptr_t>(M) & 15)) return -2;
  if (ld < N || (ld & 1)) return -3;
  if (!x || (reinterpret_cast<uintptr_t>(x) & 15)) return -4;
  if (!y) return -5;
  Ctx ctx{(cudaStream_t)stream, 1};
  return symv_full(ctx, N, M, ld, 0, x, 0, y, 0, nullptr);
}

int gegp_symv_batch(int B, int N, const double* M, int64_t ld, int64_t strideM, const double* x, int64_t strideX,
                    double* y, int64_t strideY, const int32_t* active, void* stream) {
  if (B <= 0 || B > 65535) return -1;
  if (N <= 0) return -2;
  if (!M || (reinterpret_cast<uintptr_t>(M) & 15)) return -3;
  if (ld < N || (ld & 1)) return -4;
  if (strideM < 0 || (strideM & 1)) return -5;
  if (!x || (reinterpret_cast<uintptr_t>(x) & 15)) return -6;
  if (strideX < 0 || (strideX & 1)) return -7;
  if (!y) return -8;
  if (strideY < 0) return -9;
  Ctx ctx{(cudaStream_t)stream, B};
  return symv_full(ctx, N, M, ld, strideM, x, strideX, y, strideY, active);
}

int gegp_row_abs_sum(int N, const double* M, int64_t ld, double* out, void* stream) {
  if (N <= 0) return -1;
  if (!M || (reinterpret_cast<uintptr_t>(M) & 15)) return -2;
  if (ld < N || (ld & 1)) return -3;
  if (!out) return -4;
  Ctx ctx{(cudaStream_t)stream, 1};
  return row_abs_sum(ctx, N, M, ld, out);
}

int gegp_row_sq_sum(int N, const double* M, int64_t ld, double* out, void* stream) {
  if (N <= 0) return -1;
  if (!M || (reinterpret_cast<uintptr_t>(M) & 15)) return -2;
  if (ld < N || (ld & 1)) return -3;
  if (!out) return -4;
  Ctx ctx{(cudaStream_t)stream, 1};
  return row_abs_sum(ctx, N, M, ld, out, true);
}

int gegp_lanczos_step(int N, int j, double* V, int64_t ldv, double* w, double* alpha, double* beta, void* stream) {
  if (N <= 0) return -1;
  if (j < 0 || j >= 255) return -2;
  if (!V) return -3;
  if (ldv < N) return -4;
  if (!w) return -5;
  if (!alpha) return -6;
  if (!beta) return -7;
  Ctx ctx{(cudaStream_t)stream, 1};
  return lanczos_step(ctx, N, j, V, ldv, 0, w, 0, alpha, beta, 0, nullptr);
}

int gegp_lanczos_step_batch(int B, int N, int j, double* V, int64_t ldv, int64_t strideV, double* w, int64_t strideW,
                            double* alpha, double* beta, int64_t strideAB, const int32_t* active, void* stream) {
  if (B <= 0) return -1;
  if (N <= 0) return -2;
  if (j < 0 || j >= 255) return -3;
  if (!V) return -4;
  if (ldv < N) return -5;
  if (strideV < 0) return -6;
  if (!w) return -7;
  if (strideW < 0) return -8;
  if (!alpha) return -9;
  if (!beta) return -10;
  if (strideAB < 0) return -11;
  Ctx ctx{(cudaStream_t)stream, B};
  return lanczos_step(ctx, N, j, V, ldv, strideV, w, strideW, alpha, beta, strideAB, active);
}

int gegp_lincomb(int N, int k, const double* V, int64_t ldv, const double* coef, double* out, void* stream) {
  if (N <= 0) return -1;
  if (k < 1 || k > 256) return -2;
  if (!V) return -3;
  if (ldv < N) return -4;
  if (!coef) return -5;
  if (!out) return -6;
  Ctx ctx{(cudaStream_t)stream, 1};
  return lincomb_rows(ctx, N, k, nullptr, V, ldv, 0, coef, 0, out, 0, nullptr);
}

int gegp_lincomb_batch(int B, int N, int k, const int32_t* ks, const double* V, int64_t ldv, int64_t strideV,
                       const double* coef, int64_t strideCoef, double* out, int64_t strideOut, const int32_t* active,
                       void* stream) {
  if (B <= 0) return -1;
  if (N <= 0) return -2;
  if (k < 1 || k > 256) return -3;
  if (!V) return -5;
  if (ldv < N) return -6;
  if (strideV < 0) return -7;
  if (!coef) return -8;
  if (strideCoef < 0) return -9;
  if (!out) return -10;
  if (strideOut < 0) return -11;
  Ctx ctx{(cudaStream_t)stream, B};
  return lincomb_rows(ctx, N, k, ks, V, ldv, strideV, coef, strideCoef, out, strideOut, active);
}

size_t gegp_quad_grad_work_bytes(int n, int n_g, int d) { return gegp_quad_grad_batch_work_bytes(1, n, n_g, d); }

size_t gegp_quad_grad_batch_work_bytes(int B, int n, int n_g, int d) {
  if (bad_geom(n, n_g, d) || B <= 0) return 0;
  const int N = n + n_g * d;
  return ((size_t)round_up(N, 2) + (size_t)B * (size_t)round_up((int64_t)lml_grad_partial_doubles(n, d), 2)) *
         sizeof(double);
}

}  // extern "C"

namespace {
// v_z^T (dKcov/dhp) v_z for ctx.batch vectors at once: rank-one weights (quad 1) of the LML-gradient contraction,
// p^-1 = 1 (base mode) shared by every candidate, one partial table per candidate behind it in `work`.
int quad_grad_rows(const Ctx& ctx, const Geom& gm, const double* theta, int64_t strideTheta, const double* v,
                   int64_t strideV, double eta, int noisy, const double* varK, double* out, void* work) {
  double* ones = reinterpret_cast<double*>(work);
  double* partial = ones + round_up(gm.N, 2);
  NoiseSpec ns{nullptr, 0, nullptr, 1.0, 0};
  int rc = launch_prep_p(Ctx{ctx.stream, 1}, gm, theta, 0, ns, GEGP_MODE_BASE, nullptr, ones, 0);
  if (rc) return rc;
  return launch_lml_grad(ctx, gm, theta, strideTheta, nullptr, 0, 0, v, strideV, ones, 0, GEGP_MODE_BASE, eta, noisy,
                         varK, 0.0, partial, round_up((int64_t)lml_grad_partial_doubles(gm.n, gm.d), 2), out,
                         GEGP_OUT_LEN(gm.d), 1);
}
}  // namespace

extern "C" {

int gegp_quad_grad(int n, int n_g, int d, const double* X, const int32_t* grad_slot, const double* theta, int kernel, double kernel_hp,
                   const double* v, int mode, double eta, int noisy, const double* varK_dev, double* out, void* work,
                   size_t work_bytes, void* stream) {
  if (bad_geom(n, n_g, d)) return -1;
  if (bad_kernel(kernel, kernel_hp)) return -50;
  if (!X) return -4;
  if (n_g != n && !grad_slot) return -5;
  if (!theta) return -6;
  if (!v) return -7;
  if (mode != GEGP_MODE_BASE) return -8;
  if (noisy && !varK_dev) return -11;
  if (!out) return -12;
  if (!work || (reinterpret_cast<uintptr_t>(work) & 15)) return -13;
  if (work_bytes < gegp_quad_grad_work_bytes(n, n_g, d)) return -14;
  Ctx ctx{(cudaStream_t)stream, 1};
  return quad_grad_rows(ctx, make_geom(n, n_g, d, X, grad_slot, kernel, kernel_hp), theta, 0, v, 0, eta, noisy, varK_dev,
                        out, work);
}

int gegp_quad_grad_batch(int B, const double* theta_batch, const double* varK_batch, int kernel,
                         const double* kernel_hp_batch, int n, int n_g, int d, const double* X, const int32_t* grad_slot,
                         const double* V, int64_t ldv, int mode, double eta, int noisy, double* out, void* work,
                         size_t work_bytes, void* stream) {
  if (B <= 0 || B > 65535) return -1;
  if (!theta_batch) return -2;
  if (noisy && !varK_batch) return -3;
  if (kernel < GEGP_KERNEL_SQEXP || kernel > GEGP_KERNEL_RATQUAD) return -50;
  if (kernel == GEGP_KERNEL_RATQUAD && !kernel_hp_batch) return -50;
  if (bad_geom(n, n_g, d)) return -6;
  if (!X) return -9;
  if (n_g != n && !grad_slot) return -10;
  if (!V) return -11;
  if (ldv < n + n_g * d) return -12;
  if (mode != GEGP_MODE_BASE) return -13;
  if (!out) return -16;
  if (!work || (reinterpret_cast<uintptr_t>(work) & 15)) return -17;
  if (work_bytes < gegp_quad_grad_batch_work_bytes(B, n, n_g, d)) return -18;
  Ctx ctx{(cudaStream_t)stream, B};
  const Geom gm = make_geom(n, n_g, d, X, grad_slot, kernel, 0.0, kernel_hp_batch);
  return quad_grad_rows(ctx, gm, theta_batch, d, V, ldv, eta, noisy, varK_batch, out, work);
}

int gegp_weighted_grad(int n, int n_g, int d, const double* X, const int32_t* grad_slot, const double* theta, int kernel, double kernel_hp,
                       const double* W, int64_t ldw, int mode, double eta, int noisy, const double* varK_dev, double* out,
                       void* work, size_t work_bytes, void* stream) {
  if (bad_geom(n, n_g, d)) return -1;
  if (bad_kernel(kernel, kernel_hp)) return -50;
  if (!X) return -4;
  if (n_g != n && !grad_slot) return -5;
  if (!theta) return -6;
  if (!W) return -7;
  const int N = n + n_g * d;
  if (ldw < N) return -8;
  if (mode != GEGP_MODE_BASE) return -9;
  if (noisy && !varK_dev) return -12;
  if (!out) return -13;
  if (!work || (reinterpret_cast<uintptr_t>(work) & 15)) return -14;
  if (work_bytes < gegp_quad_grad_work_bytes(n, n_g, d) + (size_t)round_up(N, 2) * sizeof(double)) return -15;
  Ctx ctx{(cudaStream_t)stream, 1};
  const Geom gm = make_geom(n, n_g, d, X, grad_slot, kernel, kernel_hp);
  double* ones = reinterpret_cast<double*>(work);
  double* zeros = ones + round_up(N, 2);                     // alpha := 0 (no rank-one part)
  double* partial = zeros + round_up(N, 2);
  NoiseSpec ns{nullptr, 0, nullptr, 1.0, 0};
  int rc = launch_prep_p(ctx, gm, theta, 0, ns, GEGP_MODE_BASE, nullptr, ones, 0);
  if (rc) return rc;
  cudaError_t e = cudaMemsetAsync(zeros, 0, (size_t)round_up(N, 2) * sizeof(double), ctx.stream);
  if (e != cudaSuccess) return -1000 - (int)e;
  return launch_lml_grad(ctx, gm, theta, 0, W, ldw, 0, zeros, 0, ones, 0, mode, eta, noisy, varK_dev, 0.0, partial, 0, out,
                         0, 2);
}

int gegp_predict_setup(int n, int n_g, int d, const double* X, const int32_t* grad_slot, const double* theta, int kernel, double kernel_hp,
                       const double* noise, int mode, double eta, const double* y, double beta, double* A, int64_t lda,
                       double* dinv, double* p_out, double* alpha_out, int* info_dev, void* stream) {
  if (bad_geom(n, n_g, d)) return -1;
  if (bad_kernel(kernel, kernel_hp)) return -50;
  if (!X) return -4;
  if (n_g != n && !grad_slot) return -5;
  if (!theta) return -6;
  if (mode != GEGP_MODE_BASE && mode != GEGP_MODE_PRECON) return -8;
  if (!y) return -10;
  if (!A) return -12;
  const int N = n + n_g * d;
  if (lda < N || (lda & 1)) return -13;
  if (!dinv) return -14;
  if (!p_out) return -15;
  if (!info_dev) return -17;
  Ctx ctx{(cudaStream_t)stream, 1};
  const Geom gm = make_geom(n, n_g, d, X, grad_slot, kernel, kernel_hp);
  NoiseSpec ns{noise, 0, nullptr, 1.0, 0};
  double* pinv = p_out + N;
  int rc = launch_prep_p(ctx, gm, theta, 0, ns, mode, p_out, pinv, 0);
  if (rc) return rc;
  rc = launch_build_cov(ctx, gm, theta, 0, ns, pinv, 0, mode, eta, A, lda, 0, 1);
  if (rc) return rc;
  double* row = A + (int64_t)N * lda;
  rc = launch_append_res(ctx, N, n, y, beta, pinv, row);
  if (rc) return rc;
  rc = chol_trap(ctx, A, lda, 0, N + 1, N, 0, info_dev, dinv, 0);
  if (rc) return rc;
  rc = leaf_dinv_assemble(ctx, A, lda, 0, dinv, 0, N);
  if (rc) return rc;
  if (alpha_out) {
    cudaError_t e = cudaMemcpyAsync(alpha_out, row, (size_t)N * sizeof(double), cudaMemcpyDeviceToDevice, ctx.stream);
    if (e != cudaSuccess) return -1000 - (int)e;
    rc = trsv_lower_trans(ctx, A, lda, 0, dinv, 0, alpha_out, N, 0, N, 1);
    if (rc) return rc;
    rc = launch_scale_vec(ctx, N, alpha_out, 0, pinv, 0, alpha_out, 0);
    if (rc) return rc;
  }
  return 0;
}

int gegp_predict(int n, int n_g, int d, const double* X, const int32_t* grad_slot, const double* theta, int kernel, double kernel_hp, const double* A,
                 int64_t lda, const double* dinv, const double* p, int mode, double beta, double varK, const double* Xs,
                 int nx, double* mu,
                 double* sig, double* sig2_out, int* n_negative_dev, void* work, size_t work_bytes, void* stream) {
  Posterior ps;
  int rc = posterior_args(n, n_g, d, X, grad_slot, theta, kernel, kernel_hp, A, lda, dinv, p, &ps);
  if (rc) return rc;
  if (!Xs || nx < 0) return -14;
  if (!mu) return -16;
  if (!sig) return -17;
  if (!work || (reinterpret_cast<uintptr_t>(work) & 15)) return -20;
  (void)mode;
  const int64_t ldz = gegp_ld(ps.gm.N);
  const int chunk = (int)std::min<size_t>((size_t)nx, work_bytes / (ldz * sizeof(double)));
  if (nx > 0 && chunk < 1) return -21;
  Ctx ctx{(cudaStream_t)stream, 1};
  double* Z = reinterpret_cast<double*>(work);
  for (int x0 = 0; x0 < nx; x0 += chunk) {
    rc = posterior_chunk(ctx, ps, beta, varK, Xs, x0, std::min(chunk, nx - x0), Z, ldz, mu, sig, sig2_out, nullptr,
                         nullptr, n_negative_dev);
    if (rc) return rc;
  }
  return 0;
}

int gegp_predict_grad(int n, int n_g, int d, const double* X, const int32_t* grad_slot, const double* theta, int kernel, double kernel_hp,
                      const double* A, int64_t lda, const double* dinv, const double* p, int mode, double beta,
                      double varK, const double* Xs, int nx, double* mu, double* sig, double* sig2_out, double* dmudx,
                      double* dsigdx, int* n_negative_dev, void* work, size_t work_bytes, void* stream) {
  Posterior ps;
  int rc = posterior_args(n, n_g, d, X, grad_slot, theta, kernel, kernel_hp, A, lda, dinv, p, &ps);
  if (rc) return rc;
  if (!Xs || nx < 0) return -14;
  if (!mu) return -16;
  if (!sig) return -17;
  if (!dmudx) return -19;
  if (!dsigdx) return -20;
  if (!work || (reinterpret_cast<uintptr_t>(work) & 15)) return -22;
  (void)mode;
  const int64_t ldz = gegp_ld(ps.gm.N);
  const size_t per_x = (size_t)(d + 1) * ldz * sizeof(double);
  const int chunk = (int)std::min<size_t>((size_t)nx, work_bytes / per_x);
  if (nx > 0 && chunk < 1) return -23;
  Ctx ctx{(cudaStream_t)stream, 1};
  double* Z = reinterpret_cast<double*>(work);
  for (int x0 = 0; x0 < nx; x0 += chunk) {
    rc = posterior_chunk(ctx, ps, beta, varK, Xs, x0, std::min(chunk, nx - x0), Z, ldz, mu, sig, sig2_out, dmudx, dsigdx,
                         n_negative_dev);
    if (rc) return rc;
  }
  return 0;
}

int gegp_predict_hess(int n, int n_g, int d, const double* X, const int32_t* grad_slot, const double* theta, int kernel, double kernel_hp,
                      const double* A, int64_t lda, const double* dinv, const double* p, const double* alpha, int mode,
                      double beta, double varK, const double* xs, double* mu, double* sig, double* sig2_out,
                      double* dmudx, double* dsigdx, double* hess3, int* n_negative_dev, void* work, size_t work_bytes,
                      void* stream) {
  Posterior ps;
  int rc = posterior_args(n, n_g, d, X, grad_slot, theta, kernel, kernel_hp, A, lda, dinv, p, &ps);
  if (rc) return rc;
  if (!alpha) return -11;
  if (!xs) return -15;
  if (!mu) return -16;
  if (!sig) return -17;
  if (!dmudx) return -19;
  if (!dsigdx) return -20;
  if (!hess3) return -21;
  if (!work || (reinterpret_cast<uintptr_t>(work) & 15)) return -23;
  (void)mode;
  const int N = ps.gm.N;
  const int64_t ldz = gegp_ld(N);
  if (work_bytes < (size_t)(d + 2) * ldz * sizeof(double)) return -24;
  Ctx ctx{(cudaStream_t)stream, 1};
  double* Z = reinterpret_cast<double*>(work);
  double* bt = Z + (int64_t)(d + 1) * ldz;             // L^-T z0 (K^-1 k* = P^-1 bt)
  rc = posterior_chunk(ctx, ps, beta, varK, xs, 0, 1, Z, ldz, mu, sig, sig2_out, dmudx, dsigdx, n_negative_dev);
  if (rc) return rc;
  cudaError_t e = cudaMemcpyAsync(bt, Z, (size_t)N * sizeof(double), cudaMemcpyDeviceToDevice, ctx.stream);
  if (e != cudaSuccess) return -1000 - (int)e;
  // one row: a single trsv launch per leaf, where trsm_right_lower_rec would issue several
  rc = trsv_lower_trans(ctx, A, lda, 0, dinv, 0, bt, ldz, 0, N, 1);
  if (rc) return rc;
  return launch_predict_hess_batch(ctx, ps.gm, theta, xs, 1, alpha, bt, ldz, ps.pinv, Z, ldz, hess3);
}

int gegp_predict_hess_batch(int n, int n_g, int d, const double* X, const int32_t* grad_slot, const double* theta, int kernel,
                            double kernel_hp, const double* A, int64_t lda, const double* dinv, const double* p,
                            const double* alpha, int mode, double beta, double varK, const double* Xs, int nx, double* mu,
                            double* sig, double* sig2_out, double* dmudx, double* dsigdx, double* hess3, int* n_negative_dev,
                            void* work, size_t work_bytes, void* stream) {
  if (!bad_geom(n, n_g, d) && hess_batch_tile_height(d) == 0) return -3;   // the contraction's tiles exceed shared memory
  Posterior ps;
  int rc = posterior_args(n, n_g, d, X, grad_slot, theta, kernel, kernel_hp, A, lda, dinv, p, &ps);
  if (rc) return rc;
  if (!alpha) return -11;
  if (!Xs) return -15;
  if (nx < 0) return -16;
  if (!mu) return -17;
  if (!sig) return -18;
  if (!dmudx) return -20;
  if (!dsigdx) return -21;
  if (!hess3) return -22;
  if (!work || (reinterpret_cast<uintptr_t>(work) & 15)) return -24;
  (void)mode;
  const int N = ps.gm.N;
  const int64_t ldz = gegp_ld(N);
  const size_t fixed = (size_t)dinv_doubles(N) * sizeof(double);
  const size_t per_x = ((size_t)(d + 1) * ldz + LEAF) * sizeof(double);
  const int chunk = work_bytes > fixed ? (int)std::min<size_t>((size_t)nx, (work_bytes - fixed) / per_x) : 0;
  if (nx > 0 && chunk < 1) return -25;
  if (nx == 0) return 0;
  Ctx ctx{(cudaStream_t)stream, 1};
  double* Lt = reinterpret_cast<double*>(work);                 // transposed diagonal blocks of the factor
  double* Z = Lt + dinv_doubles(N);                              // (d + 1) solved rows per point
  double* T = Z + (int64_t)chunk * (d + 1) * ldz;                // leaf scratch of the back substitution, chunk x LEAF
  const int64_t ldb = (int64_t)(d + 1) * ldz;                    // row 0 of every point: z0, then b~ = L^-T z0 in place
  rc = stage_leaf_lt(ctx, A, lda, Lt, N);
  if (rc) return rc;
  for (int x0 = 0; x0 < nx; x0 += chunk) {
    const int cx = std::min(chunk, nx - x0);
    rc = posterior_chunk(ctx, ps, beta, varK, Xs, x0, cx, Z, ldz, mu, sig, sig2_out, dmudx, dsigdx, n_negative_dev);
    if (rc) return rc;
    rc = trsm_right_lower_rec(ctx, A, lda, dinv, Lt, 0, Z, ldb, cx, N, T);
    if (rc) return rc;
    rc = launch_predict_hess_batch(ctx, ps.gm, theta, Xs + (int64_t)x0 * d, cx, alpha, Z, ldb, ps.pinv, Z, ldz,
                                   hess3 + (int64_t)x0 * 3 * d * d);
    if (rc) return rc;
  }
  return 0;
}

}  // extern "C"

namespace {
// hh = z_h . z_h ( = H^T K^-1 H ) and aH = sum_{i < n} pinv_i alpha~_i ( = H^T K^-1 (y - H beta) ), one CTA
__global__ void __launch_bounds__(256)
direct_scalars_kernel(int N, int n, const double* __restrict__ zh, const double* __restrict__ alpha_t,
                      const double* __restrict__ pinv, double* __restrict__ out2) {
  __shared__ double sh[32];
  double hh = 0.0, aH = 0.0;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    const double z = zh[i];
    hh += z * z;
    if (i < n) aH += pinv[i] * alpha_t[i];
  }
  hh = block_sum(hh, sh);
  aH = block_sum(aH, sh);
  if (threadIdx.x == 0) { out2[0] = hh; out2[1] = aH; }
}
// vp = a + h, vm = a - h, zero = 0
__global__ void direct_vectors_kernel(int N, const double* __restrict__ a, const double* __restrict__ h,
                                      double* __restrict__ vp, double* __restrict__ vm, double* __restrict__ zero) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  vp[i] = a[i] + h[i];
  vm[i] = a[i] - h[i];
  zero[i] = 0.0;
}
}  // namespace

extern "C" int gegp_lml_direct_terms(int n, int n_g, int d, const double* X, const int32_t* grad_slot, const double* theta,
                                     int kernel, double kernel_hp, int mode, double eta, int noisy, const double* varK_dev,
                                     void* work, size_t work_bytes, double* scratch, double* out, void* stream) {
  if (bad_geom(n, n_g, d)) return -1;
  if (bad_kernel(kernel, kernel_hp)) return -50;
  if (!X) return -4;
  if (n_g != n && !grad_slot) return -5;
  if (!theta) return -6;
  if (mode != GEGP_MODE_BASE && mode != GEGP_MODE_PRECON) return -7;
  if (noisy && !varK_dev) return -10;
  if (!work || (reinterpret_cast<uintptr_t>(work) & 15)) return -11;
  const int N = n + n_g * d;
  const LmlLayout L = lml_layout(n, d, N, true);
  const size_t header = info_header_bytes(1);
  if (work_bytes < header + L.per_cand_doubles * sizeof(double)) return -12;
  if (!scratch || (reinterpret_cast<uintptr_t>(scratch) & 15)) return -13;
  if (!out) return -14;
  double* wk = reinterpret_cast<double*>(reinterpret_cast<char*>(work) + header);
  const double* A = wk + L.A;
  const double* pinv = wk + L.P + L.ld;
  const double* alpha_t = wk + L.W + L.ld;          // preconditioned alpha = L^-T w of the evaluation
  const double* U = wk + L.U;
  const double* Kinv = wk + L.Kinv;
  double* part = wk + L.Part;
  const double* zh = A + (int64_t)(N + 1) * L.ld;   // L^-1 P^-1 H, second appended row of the trapezoid
  double* h_t = scratch;                             // preconditioned h = L^-T z_h  (K^-1 H = P^-1 h_t)
  double* vp = scratch + L.ld, *vm = scratch + 2 * L.ld, *zero = scratch + 3 * L.ld;
  const int outlen = GEGP_OUT_LEN(d);
  Ctx ctx{(cudaStream_t)stream, 1};
  const Geom gm = make_geom(n, n_g, d, X, grad_slot, kernel, kernel_hp);
  int rc = trmv_upper(ctx, U, L.ld, 0, zh, 0, h_t, 0, N);
  if (rc) return rc;
  direct_vectors_kernel<<<(N + 255) / 256, 256, 0, ctx.stream>>>(N, alpha_t, h_t, vp, vm, zero);
  GEGP_CHECK_LAUNCH();
  direct_scalars_kernel<<<1, 256, 0, ctx.stream>>>(N, n, zh, alpha_t, pinv, out + 4 * (int64_t)outlen);
  GEGP_CHECK_LAUNCH();
  {
    cudaError_t e = cudaMemsetAsync(out, 0, sizeof(double) * 4 * (size_t)outlen, ctx.stream);
    if (e != cudaSuccess) return -1000 - (int)e;
  }
  const double* vecs[3] = {alpha_t, vp, vm};
  for (int q = 0; q < 3; q++) {      // rows 0..2: v^T (dKcov/dhp) v for v = alpha, alpha + h, alpha - h
    rc = launch_lml_grad(ctx, gm, theta, 0, nullptr, 0, 0, vecs[q], 0, pinv, 0, mode, eta, noisy, varK_dev, 0.0, part, 0,
                         out + (int64_t)q * outlen, 0, 1);
    if (rc) return rc;
  }
  // row 3: sum(K^-1 .* dKcov/dhp) = tr(K^-1 dKcov/dhp)
  return launch_lml_grad(ctx, gm, theta, 0, Kinv, L.ld, 0, zero, 0, pinv, 0, mode, eta, noisy, varK_dev, 0.0, part, 0,
                         out + 3 * (int64_t)outlen, 0, 2);
}
