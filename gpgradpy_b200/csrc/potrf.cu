// Blocked fp64 algorithms built on the DMMA GEMM engine: recursive trapezoid Cholesky, recursive
// right-side triangular solve, and the explicit inverse K^-1 = L^-T L^-1 needed by the trace terms
// of the LML gradient (reference: scipy cho_factor / cho_solve at kernel/Kernel.py:251,
// optz/CalcLkd.py:154,174).
#include "linalg.h"
#include <algorithm>
#include <cstdlib>
#include <mutex>
#include <vector>

namespace gegp {

// GEGP_OPT_INV_EARLY / env GEGP_INV_EARLY: 0 = off, 1, 2 = forced level, 3 = by problem size (default)
static int g_inv_early = -1;
int& inv_early_option() {
  if (g_inv_early < 0) g_inv_early = getenv("GEGP_INV_EARLY") ? atoi(getenv("GEGP_INV_EARLY")) : 3;
  return g_inv_early;
}

static inline int split_point(int k) {
  // split k into k1 + k2 with k1 a multiple of LEAF, k1 >= k2
  int h = (k + 1) / 2;
  int k1 = ((h + LEAF - 1) / LEAF) * LEAF;
  if (k1 >= k) k1 = ((k - 1) / LEAF) * LEAF;
  return k1;
}

static const double* dinv_block(const double* Dinv, int col0) { return Dinv + (int64_t)(col0 / LEAF) * LEAF * LEAF; }

int trsm_right_rec(const Ctx& ctx, const double* L, int64_t ldl, int64_t strideL, const double* Dinv, int64_t strideD,
                   int col0, double* B, int64_t ldb, int64_t strideB, int r, int k) {
  if (r <= 0 || k <= 0) return 0;
  if (k <= LEAF) return leaf_trsm(ctx, L, ldl, strideL, dinv_block(Dinv, col0), strideD, B, ldb, strideB, r, k);
  // X = [X1 X2], L = [[L11 0],[L21 L22]]:  X1 = B1 L11^-T ; B2 -= X1 L21^T ; X2 = B2 L22^-T
  const int k1 = split_point(k);
  int rc = trsm_right_rec(ctx, L, ldl, strideL, Dinv, strideD, col0, B, ldb, strideB, r, k1);
  if (rc) return rc;
  GemmArgs g = gemm_args(B, ldb, L + (int64_t)k1 * ldl, ldl, B + k1, ldb, r, k - k1, k1, -1.0, 1.0, true);
  rc = gemm_f64(ctx, batched(ctx, g, strideB, strideL, strideB));
  if (rc) return rc;
  return trsm_right_rec(ctx, L + (int64_t)k1 * ldl + k1, ldl, strideL, Dinv, strideD, col0 + k1, B + k1, ldb, strideB, r,
                        k - k1);
}

// Lt block b (LEAF x LEAF, row-major, ld LEAF) <- L_bb^T with explicit zeros below the diagonal and outside a ragged last
// block: the K-contiguous form of L_bb for the residual product of the leaf refinement below (the strict upper part of
// the factor's diagonal blocks is never written by the factorisation, so it cannot be read as zeros).
__global__ void __launch_bounds__(256)
stage_leaf_lt_kernel(const double* __restrict__ L, int64_t ldl, double* __restrict__ Lt, int N) {
  const int b0 = blockIdx.x * LEAF;
  const int k = min(LEAF, N - b0);
  double* dst = Lt + (int64_t)blockIdx.x * LEAF * LEAF;
  for (int e = threadIdx.x; e < LEAF * LEAF; e += blockDim.x) {
    const int i = e / LEAF, j = e % LEAF;   // dst[i][j] = L[b0 + j][b0 + i] for j >= i
    dst[e] = (j >= i && j < k) ? L[(int64_t)(b0 + j) * ldl + b0 + i] : 0.0;
  }
}

int stage_leaf_lt(const Ctx& ctx, const double* L, int64_t ldl, double* Lt, int N) {
  if (N <= 0) return 0;
  stage_leaf_lt_kernel<<<(N + LEAF - 1) / LEAF, 256, 0, ctx.stream>>>(L, ldl, Lt, N);
  GEGP_CHECK_LAUNCH();
  return 0;
}

// B (r x k) <- B * L^-1 for one leaf (k <= LEAF), with the explicit inverse L^-1 = Dinv^T and one refinement step:
//   X1 = B Dinv^T ;  R = B - X1 L ;  X = X1 + R Dinv^T
// T (r x LEAF, ld LEAF) is scratch; B holds R between the second and the third product and X at the end.
static int leaf_trsm_lower_right(const Ctx& ctx, const double* Dinv, const double* Lt, double* B, int64_t ldb, int r, int k,
                                 double* T) {
  int rc = gemm_f64(ctx, gemm_args(B, ldb, Dinv, LEAF, T, LEAF, r, k, k, 1.0, 0.0, true));          // X1
  if (rc) return rc;
  rc = gemm_f64(ctx, gemm_args(T, LEAF, Lt, LEAF, B, ldb, r, k, k, -1.0, 1.0, true));               // R
  if (rc) return rc;
  rc = gemm_f64(ctx, gemm_args(B, ldb, Dinv, LEAF, T, LEAF, r, k, k, 1.0, 1.0, true));              // X1 + R Dinv^T
  if (rc) return rc;
  const cudaError_t e = cudaMemcpy2DAsync(B, (size_t)ldb * sizeof(double), T, LEAF * sizeof(double), (size_t)k * sizeof(double),
                                          (size_t)r, cudaMemcpyDeviceToDevice, ctx.stream);
  return e == cudaSuccess ? 0 : -1000 - (int)e;
}

int trsm_right_lower_rec(const Ctx& ctx, const double* L, int64_t ldl, const double* Dinv, const double* Lt, int col0,
                         double* B, int64_t ldb, int r, int k, double* T) {
  if (r <= 0 || k <= 0) return 0;
  if (k <= LEAF)
    return leaf_trsm_lower_right(ctx, dinv_block(Dinv, col0), dinv_block(Lt, col0), B, ldb, r, k, T);
  // X = [X1 X2], L = [[L11 0],[L21 L22]]:  X2 = B2 L22^-1 ; B1 -= X2 L21 ; X1 = B1 L11^-1
  const int k1 = split_point(k);
  int rc = trsm_right_lower_rec(ctx, L + (int64_t)k1 * ldl + k1, ldl, Dinv, Lt, col0 + k1, B + k1, ldb, r, k - k1, T);
  if (rc) return rc;
  rc = gemm_f64(ctx, gemm_args(B + k1, ldb, L + (int64_t)k1 * ldl, ldl, B, ldb, r, k1, k - k1, -1.0, 1.0, false));
  if (rc) return rc;
  return trsm_right_lower_rec(ctx, L, ldl, Dinv, Lt, col0, B, ldb, r, k1, T);
}

// ---- the products of the explicit inverse ----
// U = L^-T (upper) and, while U is built, W = U^T = L^-1 in the lower triangle of T (the Kinv buffer); each builder
// returns the GEMM over the ctx.batch problems of the call (U, L and T of one problem sU, sL and sT doubles apart).
// A pair is a = [r, r+m), b = [r+m, r+m+n) on the diagonal:  U_ab = -(U_aa L_ba^T) U_bb.

// first product of a pair: T_ab = U_aa L_ba^T, staged in the upper triangle of T at the coordinates of U_ab.  U_aa is upper
// triangular (k >= i): k clipped below by the row tile.
static GemmArgs pair_first(const Ctx& ctx, const double* L, int64_t ldl, int64_t sL, const double* U, int64_t ldu,
                           int64_t sU, double* T, int64_t ldt, int64_t sT, int r, int m, int n) {
  GemmArgs g = gemm_args(U + (int64_t)r * ldu + r, ldu, L + (int64_t)(r + m) * ldl + r, ldl, T + (int64_t)r * ldt + r + m,
                         ldt, m, n, m, 1.0, 0.0, true);
  g.klo_mode = KLO_M0;
  return batched(ctx, g, sU, sL, sT);
}
// second product: U_ab = -T_ab W_bb^T, W_bb = L_bb^-1 (lower: element (j, k) nonzero for k <= j, read from the lower
// triangle of T; k clipped above by the column tile), only the columns [c_from, n) of U_ab: the rows [c_from, n) of
// W_bb, whose k range starts c_from columns earlier.  store_w: U_ab^T is stored a second time, as W_ba in T.
static GemmArgs pair_second(const Ctx& ctx, double* U, int64_t ldu, int64_t sU, double* T, int64_t ldt, int64_t sT, int r,
                            int m, int n, int c_from, bool store_w) {
  GemmArgs g = gemm_args(T + (int64_t)r * ldt + r + m, ldt, T + (int64_t)(r + m + c_from) * ldt + r + m, ldt,
                         U + (int64_t)r * ldu + r + m + c_from, ldu, m, n - c_from, n, -1.0, 0.0, true);
  g.khi_mode = KHI_N0;
  g.khi_off = c_from;
  if (store_w) { g.Ct = T + (int64_t)(r + m + c_from) * ldt + r; g.ldct = ldt; g.sCto = sT; }
  return batched(ctx, g, sT, sT, sU);
}
// K^-1 = U U^T on the n x n diagonal block that starts at U and Kinv: U upper, so the sum runs over k >= max(i, j); the
// lower tiles are computed and mirrored to the upper half.
static GemmArgs kinv_from_u(const Ctx& ctx, const double* U, int64_t ldu, int64_t sU, double* Kinv, int64_t ldk,
                            int64_t sK, int n) {
  GemmArgs g = gemm_args(U, ldu, U, ldu, Kinv, ldk, n, n, n, 1.0, 0.0, true);
  g.klo_mode = KLO_MAXMN;
  g.cmode = C_LOWER_MIRROR;
  return batched(ctx, g, sU, sU, sK);
}
// Kinv_aa += U_a,x U_a,x^T for a = [0, m) and the columns x = [c0, c1) of U (lower tiles, mirrored)
static GemmArgs kinv_add_cols(const Ctx& ctx, const double* U, int64_t ldu, int64_t sU, double* Kinv, int64_t ldk,
                              int64_t sK, int m, int c0, int c1) {
  GemmArgs g = gemm_args(U + c0, ldu, U + c0, ldu, Kinv, ldk, m, m, c1 - c0, 1.0, 1.0, true);
  g.cmode = C_LOWER_MIRROR;
  return batched(ctx, g, sU, sU, sK);
}

// U = L^-T by levels: diagonal LEAF blocks first, then for block size bs = LEAF, 2*LEAF, ... every pair
// (a = [s, s+bs), b = [s+bs, s+2bs)):  U_ab = -(U_aa * L_ba^T) * U_bb.  The product in parentheses is staged in the
// upper triangle of T (the Kinv buffer, same coordinates as U_ab).  The LOWER triangle of T meanwhile collects
// W = U^T = L^-1, so the second product is written  -(T_ab) * (W_bb)^T  with the K-contiguous lower-triangular W_bb:
// both products are A * B^T and run on the TMA kernel; each U_ab is stored a second time, transposed, as W_ba.
static int inverse_transposed(const Ctx& ctx, const double* L, int64_t ldl, int64_t strideL, const double* Dinv,
                              int64_t strideD, double* U, int64_t ldu, int64_t strideU, double* T, int64_t ldt,
                              int64_t strideT, int N) {
  int rc = leaf_scatter_dinv(ctx, Dinv, strideD, U, ldu, strideU, T, ldt, strideT, N);
  if (rc) return rc;
  for (int bs = LEAF; bs < N; bs *= 2) {
    const int npairs_full = N / (2 * bs);  // pairs whose b block is full
    for (int pass = 0; pass < 2; pass++) {
      // pass 0: all full pairs in one batched launch; pass 1: the ragged last pair (if any)
      int s, bsz, inner;
      if (pass == 0) { if (npairs_full == 0) continue; s = 0; bsz = bs; inner = npairs_full; }
      else {
        s = npairs_full * 2 * bs; bsz = N - s - bs; inner = 1;
        if (bsz <= 0) continue;
      }
      // the inner batch: pair i + 1 lies 2 bs rows and columns further down the diagonal of every operand
      auto pairs = [&](GemmArgs g) {
        const int64_t step = 2 * bs;
        g.inner = inner;
        g.sAi = step * (g.lda + 1); g.sBi = step * (g.ldb + 1); g.sCi = step * (g.ldc + 1);
        if (g.Ct) g.sCti = step * (g.ldct + 1);
        g.inner_steps = true; g.iAr = g.iAc = g.iBr = g.iBc = 2 * bs;
        return g;
      };
      rc = gemm_f64(ctx, pairs(pair_first(ctx, L, ldl, strideL, U, ldu, strideU, T, ldt, strideT, s, bs, bsz)));
      if (rc) return rc;
      rc = gemm_f64(ctx, pairs(pair_second(ctx, U, ldu, strideU, T, ldt, strideT, s, bs, bsz, 0, true)));
      if (rc) return rc;
    }
  }
  return 0;
}


// ------------------------------------------------------------------------------------------------
// Look-ahead.  The factorisation's critical path is the chain
//     leaf factor (one CTA)  ->  solve of the NEXT leaf's 128-row block row + K = 128 update of its diagonal block
//                                (chain_prep_kernel, one small cluster)  ->  next leaf factor  -> ...
// It runs on its own HIGHEST-priority stream (`hi`, forked from and re-joined to the caller's stream), so that its
// CTAs take the next free SM ahead of queued GEMM tiles.  Everything else is dealt out so that the chain never does
// more than that:
//   * the rows below the next leaf's block row are solved against a leaf on stream `col` (high priority), beside the
//     next chain step: nothing on the chain reads them;
//   * the rows below the diagonal block in the next leaf's block column, updated with the LAST leaf's panel only
//     (K = LEAF)                                                                     -> stream `col` as well;
//   * the columns right of it, updated with the whole left child's panel, cut into pieces along the left spine of
//     the right child, plus the block column of the leaf that FOLLOWS the node       -> streams `bulk[depth]` (lowest
//     priority); a piece is joined only when the chain reaches a fork or leaf that touches its columns.
// See chol_node_la for the induction that every (source leaf, target block column) pair is applied exactly once.
// The summation order of an element differs from the single-stream schedule (same terms, grouped by update), so the
// two schedules agree to rounding, not bit for bit; within one schedule results are reproducible and independent of
// the batch size.  Fork/join is by events only and is capturable in a CUDA graph.
//
// Re-entrancy: the streams, events and piece table of one factorisation live in a LookAhead object taken from a
// per-device pool for the duration of the (host-side, asynchronous) call, so concurrent calls from several host
// threads or on several caller streams never share mutable state.
// ------------------------------------------------------------------------------------------------
namespace {
// a trailing update with fewer 128 x 128 tiles than this is cut into just-in-time pieces (env GEGP_SPLIT_TILES)
int split_max_tiles() {
  static const int v = getenv("GEGP_SPLIT_TILES") ? atoi(getenv("GEGP_SPLIT_TILES")) : 2500;
  return v;
}
// width of the look-ahead window: the columns right behind a node that receive its panels as early as they exist
// (env GEGP_LA_WINDOW, multiple of LEAF; LEAF = the next leaf only)
int la_window() {
  static const int v = [] {
    int x = getenv("GEGP_LA_WINDOW") ? atoi(getenv("GEGP_LA_WINDOW")) : 256;
    x = (x / LEAF) * LEAF;
    return x < LEAF ? LEAF : x;
  }();
  return v;
}
constexpr int MAX_PIECES = 256;
constexpr int MAX_DEV = 32;

// Explicit inverse interleaved with the factorisation (chol_trap_inverse): U receives L^-T (upper), T (the Kinv buffer)
// L^-1 (lower) and scratch.  A subtree of at most `unit_max` columns is inverted as one unit (diagonal blocks + block
// doubling, inverse_transposed) as soon as the factorisation has left it; above that size a node X contributes
// U_ab = -(U_aa L_ba^T) U_bb for its two children a, b: the first product as soon as a is inverted and factored rows of
// b exist, the second once b is inverted.  Everything goes to one lowest-priority stream in post-order, so the
// dependencies among the inverse tasks are its FIFO order.
struct InvHook {
  double* U; int64_t ldu, sU;
  double* T; int64_t ldt, sT;
  double* A0; int64_t lda, sA;        // the factor (global row/column 0)
  double* Dinv; int64_t sD;
  int unit_max;
};
// subtrees up to this many columns are inverted as one unit (env GEGP_INV_UNIT; 0 switches the interleaving off)
int inv_unit_max() {
  static const int v = getenv("GEGP_INV_UNIT") ? atoi(getenv("GEGP_INV_UNIT")) : 1024;
  return v;
}
// Parts of K^-1 = U U^T and of the root's pair product that only need the LEFT part of the factor are issued while the
// chain is still running (inv_root_early_aa / inv_root_early_pair / finish_inverse_split).  Levels: 0 = off, 1 = Kinv_aa
// only, 2 = also the root pair's first columns.  Pays where the chain leaves the machine idle (measured on B200, LML +
// gradient: N = 5500 6.76 -> 6.60 ms; N = 11250 45.7 -> 45.9 ms and N = 21000 273.8 -> 274.7 ms, where the bulk work of
// the factorisation already fills it), so by default it is on up to N = 8192 -- a function of the shape of one problem
// only.  env GEGP_INV_EARLY forces a level.
int inv_early_level(int N) {
  const int forced = inv_early_option();
  if (forced >= 0 && forced <= 2) return forced;
  return N <= 8192 ? 2 : 0;
}
struct Piece { int c0, c1; cudaEvent_t done; cudaStream_t stream; bool live; };   // global column range a queued bulk GEMM writes
struct LookAhead {
  static constexpr int NBULK = 16;
  int dev = 0;
  static constexpr int NLANE = 3;
  // bulk[depth][lane]: pieces queued at one fork are needed one after the other; the first two get streams of their
  // own with a higher priority than the rest, so that they run beside (not behind) each other and ahead of older work
  cudaStream_t hi = nullptr, col = nullptr, late = nullptr, inv = nullptr, early = nullptr, bulk[NBULK][NLANE] = {};
  cudaEvent_t fork[40], ev_prep, ev_fac, ev_colupd, ev_solve, ev_inv, ev_early, ev_fin[3], begin, end;
  // early pieces of the explicit inverse (root node only): columns of the root's left child (0: none issued) and of the
  // right child's left child whose share of the root's pair product has been issued early (0: none)
  int early_k1 = 0, early_ba = 0, early_n = 0;   // early_n: columns of the root
  Piece piece[MAX_PIECES];
  bool colupd_pending = false;   // a K = LEAF block-column update is in flight on `col` (the next chain step reads its top rows)
  bool solve_pending = false;    // a leaf solve is in flight on `col` (bulk pieces read its rows)
  bool ok = false;
  // the chain must not touch columns [c0, c1) before every queued bulk piece that writes them has finished
  int join_columns(cudaStream_t chain, int c0, int c1) {
    for (int i = 0; i < MAX_PIECES; i++) {
      Piece& p = piece[i];
      if (!p.live || p.c1 <= c0 || p.c0 >= c1) continue;
      if (cudaStreamWaitEvent(chain, p.done, 0) != cudaSuccess) return -1100;
      p.live = false;
    }
    return 0;
  }
  Piece* free_piece() {
    for (int i = 0; i < MAX_PIECES; i++)
      if (!piece[i].live) return &piece[i];
    return nullptr;
  }
  bool create() {
    int lo = 0, hip = 0;
    cudaDeviceGetStreamPriorityRange(&lo, &hip);   // lo: numerically largest = lowest priority; hip: greatest
    const int mid = hip < lo ? hip + 1 : hip;
    ok = cudaStreamCreateWithPriority(&hi, cudaStreamNonBlocking, hip) == cudaSuccess &&
         cudaStreamCreateWithPriority(&col, cudaStreamNonBlocking, mid) == cudaSuccess &&
         cudaStreamCreateWithPriority(&late, cudaStreamNonBlocking, mid) == cudaSuccess &&
         cudaStreamCreateWithPriority(&inv, cudaStreamNonBlocking, lo) == cudaSuccess &&
         cudaStreamCreateWithPriority(&early, cudaStreamNonBlocking, lo) == cudaSuccess;
    for (int i = 0; i < NBULK && ok; i++)
      for (int j = 0; j < NLANE && ok; j++) {
        int pr = lo - (NLANE - 1 - j);               // lane 0: two levels above the lowest priority
        if (pr < mid + 1) pr = mid + 1 <= lo ? mid + 1 : lo;
        ok = cudaStreamCreateWithPriority(&bulk[i][j], cudaStreamNonBlocking, pr) == cudaSuccess;
      }
    auto mk = [&](cudaEvent_t* e) { return cudaEventCreateWithFlags(e, cudaEventDisableTiming) == cudaSuccess; };
    for (int i = 0; i < 40 && ok; i++) ok = mk(&fork[i]);
    for (int i = 0; i < MAX_PIECES && ok; i++) { ok = mk(&piece[i].done); piece[i].live = false; }
    ok = ok && mk(&ev_prep) && mk(&ev_fac) && mk(&ev_colupd) && mk(&ev_solve) && mk(&ev_inv) && mk(&begin) && mk(&end) &&
         mk(&ev_early) && mk(&ev_fin[0]) && mk(&ev_fin[1]) && mk(&ev_fin[2]);
    return ok;
  }
};

struct LaPool {
  std::mutex mu;
  std::vector<LookAhead*> idle[MAX_DEV];
};
LaPool& la_pool() {
  static LaPool* p = new LaPool();   // leaked on purpose: streams must outlive static destruction order
  return *p;
}
// One LookAhead per factorisation in flight on the host side; returned to the pool when the call has been enqueued
// (re-using its streams and events for a later call only adds stream-order dependencies).
LookAhead* la_acquire() {
  if (!lookahead_enabled()) return nullptr;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= MAX_DEV) return nullptr;
  LaPool& pool = la_pool();
  {
    std::lock_guard<std::mutex> lock(pool.mu);
    if (!pool.idle[dev].empty()) {
      LookAhead* la = pool.idle[dev].back();
      pool.idle[dev].pop_back();
      return la;
    }
  }
  LookAhead* la = new LookAhead();
  la->dev = dev;
  if (!la->create()) { delete la; return nullptr; }   // (partially created handles are leaked: this never happens in practice)
  return la;
}
void la_release(LookAhead* la) {
  LaPool& pool = la_pool();
  std::lock_guard<std::mutex> lock(pool.mu);
  pool.idle[la->dev].push_back(la);
}

// Single-stream recursion (look-ahead off): factor the left half, one trailing update, factor the right half.
int chol_node(const Ctx& ctx, double* A, int64_t lda, int64_t strideA, int m, int k, int row0, int* info, double* Dinv,
              int64_t strideD) {
  if (k <= 0) return 0;
  if (k <= LEAF) {
    int rc = leaf_potf2_inv(ctx, A, lda, strideA, k, row0, info, Dinv + (int64_t)(row0 / LEAF) * LEAF * LEAF, strideD);
    if (rc) return rc;
    return trsm_right_rec(ctx, A, lda, strideA, Dinv, strideD, row0, A + (int64_t)k * lda, lda, strideA, m - k, k);
  }
  const int k1 = split_point(k);
  int rc = chol_node(ctx, A, lda, strideA, m, k1, row0, info, Dinv, strideD);
  if (rc) return rc;
  // trailing update: C = A[k1:, k1:k] -= A[k1:, :k1] * A[k1:k, :k1]^T  (lower part of the square region)
  double* C = A + (int64_t)k1 * lda + k1;
  const double* P = A + (int64_t)k1 * lda;
  GemmArgs g = gemm_args(P, lda, P, lda, C, lda, m - k1, k - k1, k1, -1.0, 1.0, true);
  g.cmode = C_LOWER;
  rc = gemm_f64(ctx, batched(ctx, g, strideA, strideA, strideA));
  if (rc) return rc;
  return chol_node(ctx, C, lda, strideA, m - k1, k - k1, row0 + k1, info, Dinv, strideD);
}

// Look-ahead recursion.  `ext` is the width of the WINDOW that follows this node's columns (0: none): the node applies
// all of its leaves except its last one to the window columns [k, k+ext) as early as their panels exist; the caller
// applies that last leaf.  A window is at most la_window() columns wide and never ends inside a leaf.  After the left
// child (k1 columns, a multiple of LEAF; its last leaf is l; its window was E_w = the first ext_l = min(window, kc + ext)
// columns behind it, so E_w lacks nothing of the left child but l) the work is dealt out as
//   chain : block row f of l's panel solved against l, then the diagonal block of the next leaf f = [k1, k1+w) -= that
//           block row's square (one chain_prep launch, K = LEAF)
//   col   : the rows below f in l's panel solved against l (queued by leaf l itself, beside the chain step)
//   col   : the rows below the diagonal block in f's block column     -= l's panel (K = LEAF)
//   late  : the other window columns, E_w \ f, leaf by leaf           -= l's panel (K = LEAF)
//   bulk  : columns of the right child behind the window, [ext_l, kc), in just-in-time pieces
//                                                                     -= the whole left child's panel (K = k1)
//   bulk  : the part of this node's own window that E_w did not reach -= the whole left child's panel (K = k1)
// so that every update the chain waits for at a fork has K = LEAF.  By induction every (source leaf, target block
// column) pair is applied exactly once: by chain + col + late when the source is the last leaf of left(X) and the
// target lies in the window behind it, by the window pieces of the nodes on the right spine of left(X) for the other
// sources of such a target, and by the bulk piece of their lowest common ancestor X otherwise.  Pieces that write the
// same columns from different streams are serialised through their events; a piece is joined by the chain when it
// reaches a fork or leaf that touches its columns.  The bulk pieces read panel rows from k1+w on only (never block row
// f), all of which are produced on `col`: they wait for its last solve.
// inverse tasks of a node (see InvHook); `chain` is the stream the factorisation's chain is on
int inv_sync(LookAhead* la, cudaStream_t chain) {
  // everything the factorisation has produced so far: the chain up to here and the solves on `col`
  if (cudaEventRecord(la->ev_inv, chain) != cudaSuccess) return -1120;
  if (cudaStreamWaitEvent(la->inv, la->ev_inv, 0) != cudaSuccess) return -1120;
  if (la->solve_pending && cudaStreamWaitEvent(la->inv, la->ev_solve, 0) != cudaSuccess) return -1120;
  return 0;
}
int inv_unit(LookAhead* la, const InvHook* h, const Ctx& chain, int row0, int k) {
  int rc = inv_sync(la, chain.stream);
  if (rc) return rc;
  const Ctx ic{la->inv, chain.batch};
  double* Ln = h->A0 + (int64_t)row0 * (h->lda + 1);
  double* Dn = h->Dinv + (int64_t)(row0 / LEAF) * LEAF * LEAF;
  rc = leaf_dinv_assemble(ic, Ln, h->lda, h->sA, Dn, h->sD, k);
  if (rc) return rc;
  return inverse_transposed(ic, Ln, h->lda, h->sA, Dn, h->sD, h->U + (int64_t)row0 * (h->ldu + 1), h->ldu, h->sU,
                            h->T + (int64_t)row0 * (h->ldt + 1), h->ldt, h->sT, k);
}
// first product of the node's pair: T_ab = U_aa L_ba^T (a = [row0, row0+k1), b = the kc columns behind it), staged in
// the upper triangle of T at the coordinates of U_ab
int inv_pair_first(LookAhead* la, const InvHook* h, const Ctx& chain, int row0, int k1, int kc) {
  int rc = inv_sync(la, chain.stream);
  if (rc) return rc;
  const Ctx ic{la->inv, chain.batch};
  return gemm_f64(ic, pair_first(ic, h->A0, h->lda, h->sA, h->U, h->ldu, h->sU, h->T, h->ldt, h->sT, row0, k1, kc));
}
// second product: U_ab = -T_ab W_bb^T (W_bb = L_bb^-1 from the lower triangle of T), with the transposed copy W_ba.
// `c_from` > 0 (root only): the first c_from columns of U_ab have been produced early (inv_root_early_pair).
// The root's W_ba is never read (the root is nobody's right child), so no transposed copy is stored then.
int inv_pair_second(LookAhead* la, const InvHook* h, const Ctx& chain, int row0, int k1, int kc, int c_from = 0,
                    bool store_w = true) {
  int rc = inv_sync(la, chain.stream);
  if (rc) return rc;
  const Ctx ic{la->inv, chain.batch};
  return gemm_f64(ic, pair_second(ic, h->U, h->ldu, h->sU, h->T, h->ldt, h->sT, row0, k1, kc, c_from, store_w));
}

// ---- early pieces of K^-1 (root node only; a = the root's left child, b = its right child with children ba, bb) ----
// K^-1 = U U^T in blocks:  Kinv_aa = U_aa U_aa^T + U_ab U_ab^T,  Kinv_ab = U_ab U_bb^T,  Kinv_bb = U_bb U_bb^T.
// U_aa is complete half-way down the chain, and the left spine never reads its W = L^-1 again, so the aa block of the
// Kinv buffer is free from then on:  Kinv_aa = U_aa U_aa^T  goes to the lowest-priority stream `early` right away.
// All tasks a piece depends on precede the event on `inv` (FIFO, post-order).
int inv_root_early_aa(LookAhead* la, const InvHook* h, const Ctx& chain, int k1) {
  if (cudaEventRecord(la->ev_early, la->inv) != cudaSuccess) return -1130;
  if (cudaStreamWaitEvent(la->early, la->ev_early, 0) != cudaSuccess) return -1130;
  const Ctx ec{la->early, chain.batch};
  const int rc = gemm_f64(ec, kinv_from_u(ec, h->U, h->ldu, h->sU, h->T, h->ldt, h->sT, k1));
  if (!rc) la->early_k1 = k1;
  return rc;
}
// Once ba is inverted (three quarters down the chain) the first kba columns of the root's pair product are final:
//   U_a,ba = -T_a,ba U_ba,ba   (the second product restricted to the columns of ba)   and   Kinv_aa += U_a,ba U_a,ba^T.
int inv_root_early_pair(LookAhead* la, const InvHook* h, const Ctx& chain, int k1, int kba) {
  if (cudaEventRecord(la->ev_early, la->inv) != cudaSuccess) return -1131;
  if (cudaStreamWaitEvent(la->early, la->ev_early, 0) != cudaSuccess) return -1131;
  const Ctx ec{la->early, chain.batch};
  int rc = gemm_f64(ec, pair_second(ec, h->U, h->ldu, h->sU, h->T, h->ldt, h->sT, 0, k1, kba, 0, false));
  if (rc) return rc;
  rc = gemm_f64(ec, kinv_add_cols(ec, h->U, h->ldu, h->sU, h->T, h->ldt, h->sT, k1, k1, k1 + kba));
  if (!rc) la->early_ba = kba;
  return rc;
}
// What is left of K^-1 = U U^T after the early pieces, three independent products on three streams:
//   Kinv_bb = U_bb U_bb^T (hi),   Kinv_ab = U_ab U_bb^T with its mirror Kinv_ba (col),
//   Kinv_aa += U_a,x U_a,x^T over the columns x of b not yet accumulated (late).
// Called when everything has been joined into `hi`.
int finish_inverse_split(LookAhead* la, const InvHook* h, int batch, int N) {
  const int k1 = la->early_k1, kc = N - k1, off = la->early_ba;
  if (cudaEventRecord(la->ev_fin[0], la->hi) != cudaSuccess) return -1132;
  if (cudaStreamWaitEvent(la->col, la->ev_fin[0], 0) != cudaSuccess) return -1132;
  if (cudaStreamWaitEvent(la->late, la->ev_fin[0], 0) != cudaSuccess) return -1132;
  const double* Ubb = h->U + (int64_t)k1 * (h->ldu + 1);
  int rc;
  {  // the largest first: Kinv_ab (k1 x kc) = U_ab U_bb^T, U_bb upper: k >= column
    const Ctx c{la->col, batch};
    GemmArgs g = gemm_args(h->U + k1, h->ldu, Ubb, h->ldu, h->T + k1, h->ldt, k1, kc, kc, 1.0, 0.0, true);
    g.klo_mode = KLO_N0;
    g.Ct = h->T + (int64_t)k1 * h->ldt; g.ldct = h->ldt; g.sCto = h->sT;
    if ((rc = gemm_f64(c, batched(c, g, h->sU, h->sU, h->sT)))) return rc;
  }
  {  // Kinv_aa += U_a,x U_a,x^T
    const Ctx c{la->late, batch};
    if ((rc = gemm_f64(c, kinv_add_cols(c, h->U, h->ldu, h->sU, h->T, h->ldt, h->sT, k1, k1 + off, N)))) return rc;
  }
  {  // Kinv_bb = U_bb U_bb^T
    const Ctx c{la->hi, batch};
    if ((rc = gemm_f64(c, kinv_from_u(c, Ubb, h->ldu, h->sU, h->T + (int64_t)k1 * (h->ldt + 1), h->ldt, h->sT, kc))))
      return rc;
  }
  if (cudaEventRecord(la->ev_fin[1], la->col) != cudaSuccess || cudaEventRecord(la->ev_fin[2], la->late) != cudaSuccess ||
      cudaStreamWaitEvent(la->hi, la->ev_fin[1], 0) != cudaSuccess ||
      cudaStreamWaitEvent(la->hi, la->ev_fin[2], 0) != cudaSuccess)
    return -1133;
  return 0;
}

// role: 1 = the root of a factorisation with interleaved inverse, 2 = the root's right child, 0 = any other node
int chol_node_la(const Ctx& ctx, LookAhead* la, int depth, double* A, int64_t lda, int64_t strideA, int m, int k,
                 int row0, int ext, int* info, double* Dinv, int64_t strideD, const InvHook* hook = nullptr,
                 int role = 0) {
  if (k <= 0) return 0;
  int rc = 0;
  // a subtree small enough is inverted as one unit once it is factored: its descendants carry no hook
  const bool inv_unit_here = hook && k <= hook->unit_max;
  const InvHook* child_hook = inv_unit_here ? nullptr : hook;
  if (k <= LEAF) {
    if ((rc = la->join_columns(ctx.stream, row0, row0 + k))) return rc;
    rc = leaf_potf2_inv(ctx, A, lda, strideA, k, row0, info, Dinv + (int64_t)(row0 / LEAF) * LEAF * LEAF, strideD);
    if (rc) return rc;
    const int nxt = ext < LEAF ? ext : LEAF;   // the next leaf's block row is solved by the next chain step
    const int below = m - k - nxt;
    if (below > 0) {
      if (cudaEventRecord(la->ev_fac, ctx.stream) != cudaSuccess) return -1104;
      if (cudaStreamWaitEvent(la->col, la->ev_fac, 0) != cudaSuccess) return -1104;
      const Ctx cc{la->col, ctx.batch};
      rc = trsm_right_rec(cc, A, lda, strideA, Dinv, strideD, row0, A + (int64_t)(k + nxt) * lda, lda, strideA, below, k);
      if (rc) return rc;
      if (cudaEventRecord(la->ev_solve, la->col) != cudaSuccess) return -1104;
      la->solve_pending = true;
    }
    if (inv_unit_here) return inv_unit(la, hook, ctx, row0, k);
    return 0;
  }
  const int k1 = split_point(k);
  const int mc = m - k1, kc = k - k1;
  const int w = kc < LEAF ? kc : LEAF;
  const int ext_l = std::min(la_window(), kc + ext);   // the left child's window, in the right child's frame [0, ext_l)
  rc = chol_node_la(ctx, la, depth + 1, A, lda, strideA, m, k1, row0, ext_l, info, Dinv, strideD, child_hook);
  if (rc) return rc;
  double* C = A + (int64_t)k1 * lda + k1;
  const double* P = A + (int64_t)k1 * lda;        // rows k1.., all k1 columns of the left child
  double* Pl = A + (int64_t)k1 * lda + (k1 - LEAF);   // ... its last leaf only
  const int dq = depth < 40 ? depth : 39;
  // every queued piece that writes the next leaf's block column must have finished (the chain step and the column
  // update touch it right away; the other columns of the right child are only written by further pieces, which
  // order themselves behind the live ones through their events)
  if ((rc = la->join_columns(ctx.stream, row0 + k1, row0 + k1 + w))) return rc;
  if (cudaEventRecord(la->fork[dq], ctx.stream) != cudaSuccess) return -1101;
  {
    // block row f of the last leaf's panel has received that leaf's own K = LEAF column update on `col`
    if (la->colupd_pending) {
      if (cudaStreamWaitEvent(ctx.stream, la->ev_colupd, 0) != cudaSuccess) return -1105;
      la->colupd_pending = false;
    }
    const double* Lp = A + (int64_t)(k1 - LEAF) * (lda + 1);
    rc = leaf_chain_prep(ctx, Lp, lda, strideA, Dinv + (int64_t)((row0 + k1 - LEAF) / LEAF) * LEAF * LEAF, strideD, Pl, C, w);
    if (rc) return rc;
  }
  if (mc > w) {
    if (cudaEventRecord(la->ev_prep, ctx.stream) != cudaSuccess) return -1105;
    if (cudaStreamWaitEvent(la->col, la->ev_prep, 0) != cudaSuccess) return -1105;
    GemmArgs g1 = gemm_args(Pl + (int64_t)w * lda, lda, Pl, lda, C + (int64_t)w * lda, lda, mc - w, w, LEAF, -1.0, 1.0,
                            true);
    Ctx cc{la->col, ctx.batch};
    rc = gemm_f64(cc, batched(cc, g1, strideA, strideA, strideA));
    if (rc) return rc;
    if (cudaEventRecord(la->ev_colupd, la->col) != cudaSuccess) return -1106;
    la->colupd_pending = true;
  }
  cudaStream_t* lanes = la->bulk[depth < LookAhead::NBULK ? depth : LookAhead::NBULK - 1];
  cudaStream_t bs = lanes[LookAhead::NLANE - 1];
  // columns [a, b) of the right child's frame (may reach into this node's window) -= the last kk columns of the left
  // child's panel, on stream st
  auto queue_piece = [&](cudaStream_t st, int a, int b, int kk) -> int {
    if (b <= a || mc <= a) return 0;
    if (cudaStreamWaitEvent(st, la->fork[dq], 0) != cudaSuccess) return -1102;
    if (la->solve_pending && cudaStreamWaitEvent(st, la->ev_solve, 0) != cudaSuccess) return -1102;
    // older pieces for the same columns may still be running on other streams: this stream waits for them, the chain
    // does not (same-stream pieces are ordered anyway)
    for (int i = 0; i < MAX_PIECES; i++) {
      const Piece& p = la->piece[i];
      if (p.live && p.stream != st && p.c1 > row0 + k1 + a && p.c0 < row0 + k1 + b)
        if (cudaStreamWaitEvent(st, p.done, 0) != cudaSuccess) return -1112;
    }
    const double* Pa = P + (int64_t)a * lda + (k1 - kk);
    GemmArgs g2 = gemm_args(Pa, lda, Pa, lda, C + (int64_t)a * lda + a, lda, mc - a, b - a, kk, -1.0, 1.0, true);
    g2.cmode = C_LOWER;
    Ctx bc{st, ctx.batch};
    int r = gemm_f64(bc, batched(bc, g2, strideA, strideA, strideA));
    if (r) return r;
    Piece* pc = la->free_piece();
    if (!pc) return -1111;
    if (cudaEventRecord(pc->done, st) != cudaSuccess) return -1103;
    pc->c0 = row0 + k1 + a; pc->c1 = row0 + k1 + b; pc->stream = st; pc->live = true;
    return 0;
  };
  // the rest of the left child's window: only its last leaf is missing there (K = LEAF), leaf by leaf, next leaf first
  for (int a = w; a < ext_l; a += LEAF)
    if ((rc = queue_piece(la->late, a, std::min(a + LEAF, ext_l), LEAF))) return rc;
  if (kc > ext_l) {
    // A bulk that is itself latency-bound (too small for the TMA kernel) is cut along the left spine of the right
    // child -- the sibling of the first leaf, then the sibling of that pair, ... -- and queued smallest first.
    int cut[40];
    int ncut = 0;
    cut[ncut++] = kc;
    const long big_tiles = ((long)(mc - ext_l + 127) / 128) * ((kc - ext_l + 127) / 128);
    if (big_tiles < split_max_tiles()) {
      int sz = kc;
      while (sz > LEAF && ncut < 39) {
        sz = split_point(sz);
        if (sz <= ext_l) break;
        cut[ncut++] = sz;
      }
    }
    cut[ncut++] = ext_l;
    for (int i = ncut - 2, q = 0; i >= 0; i--, q++)
      if ((rc = queue_piece(lanes[q < LookAhead::NLANE ? q : LookAhead::NLANE - 1], cut[i + 1], cut[i], k1))) return rc;
  }
  // the part of this node's own window that the left child's window did not reach
  if (ext > 0 && kc + ext > ext_l)
    if ((rc = queue_piece(bs, std::max(kc, ext_l), kc + ext, k1))) return rc;
  // the left child is inverted and the rows of the right child in its panel are final once the solves queued so far
  // are done: the first product of this node's pair can start while the right child is being factored
  const int early = (child_hook && role != 0) ? inv_early_level(role == 1 ? k : la->early_n) : 0;
  // (the events of the early pieces are recorded BEFORE this node's first product is queued: they do not wait for it)
  if (role == 1) la->early_n = k;
  if (early >= 1 && role == 1 && (rc = inv_root_early_aa(la, child_hook, ctx, k1))) return rc;
  if (early >= 2 && role == 2 && la->early_k1 > 0 && (rc = inv_root_early_pair(la, child_hook, ctx, la->early_k1, k1)))
    return rc;
  if (child_hook && (rc = inv_pair_first(la, child_hook, ctx, row0, k1, kc))) return rc;
  rc = chol_node_la(ctx, la, depth + 1, C, lda, strideA, mc, kc, row0 + k1, ext, info, Dinv, strideD, child_hook,
                    role == 1 ? 2 : 0);
  if (rc) return rc;
  if (child_hook) {
    if (role == 1 && la->early_k1 > 0) return inv_pair_second(la, child_hook, ctx, row0, k1, kc, la->early_ba, false);
    return inv_pair_second(la, child_hook, ctx, row0, k1, kc);
  }
  if (inv_unit_here) return inv_unit(la, hook, ctx, row0, k);
  return 0;
}
}  // namespace

static int chol_trap_impl(const Ctx& ctx, double* A, int64_t lda, int64_t strideA, int m, int k, int row0, int* info,
                          double* Dinv, int64_t strideD, const InvHook* hook, int* inverse_done) {
  // *inverse_done: 0 = nothing of the inverse has been produced, 1 = U = L^-T is complete, 2 = Kinv is complete as well
  if (inverse_done) *inverse_done = 0;
  LookAhead* la = (k > LEAF) ? la_acquire() : nullptr;
  if (!la) return chol_node(ctx, A, lda, strideA, m, k, row0, info, Dinv, strideD);
  if (hook && (hook->unit_max < LEAF || row0 != 0)) hook = nullptr;
  for (int i = 0; i < MAX_PIECES; i++) la->piece[i].live = false;
  la->colupd_pending = la->solve_pending = false;
  la->early_k1 = la->early_ba = 0;
  int rc = 0;
  if (cudaEventRecord(la->begin, ctx.stream) != cudaSuccess) rc = -1107;
  if (!rc && (cudaStreamWaitEvent(la->hi, la->begin, 0) != cudaSuccess ||
              cudaStreamWaitEvent(la->col, la->begin, 0) != cudaSuccess ||
              (hook && cudaStreamWaitEvent(la->inv, la->begin, 0) != cudaSuccess))) rc = -1108;
  if (!rc) {
    const Ctx chain{la->hi, ctx.batch};
    rc = chol_node_la(chain, la, 0, A, lda, strideA, m, k, row0, 0, info, Dinv, strideD, hook, hook ? 1 : 0);
    if (!rc && hook && inverse_done) *inverse_done = 1;
  }
  // join everything back into the chain, then into the caller's stream (also after a failure, so that no work is left
  // un-joined inside a stream capture)
  cudaEventRecord(la->ev_solve, la->col);   // the tail of `col`: covers its last solve and column update
  cudaStreamWaitEvent(la->hi, la->ev_solve, 0);
  if (hook) {                               // ... and the tail of the inverse stream
    cudaEventRecord(la->ev_inv, la->inv);
    cudaStreamWaitEvent(la->hi, la->ev_inv, 0);
    if (la->early_k1 > 0) {
      cudaEventRecord(la->ev_early, la->early);
      cudaStreamWaitEvent(la->hi, la->ev_early, 0);
    }
  }
  la->join_columns(la->hi, 0, 1 << 30);
  la->colupd_pending = la->solve_pending = false;
  if (!rc && hook && la->early_k1 > 0) {   // early pieces of K^-1 were issued: the rest of it, split the same way
    rc = finish_inverse_split(la, hook, ctx.batch, k);
    if (!rc && inverse_done) *inverse_done = 2;
  }
  if (cudaEventRecord(la->end, la->hi) != cudaSuccess && !rc) rc = -1109;
  if (cudaStreamWaitEvent(ctx.stream, la->end, 0) != cudaSuccess && !rc) rc = -1110;
  la_release(la);
  return rc;
}

int chol_trap(const Ctx& ctx, double* A, int64_t lda, int64_t strideA, int m, int k, int row0, int* info, double* Dinv,
              int64_t strideD) {
  return chol_trap_impl(ctx, A, lda, strideA, m, k, row0, info, Dinv, strideD, nullptr, nullptr);
}

int chol_inverse(const Ctx& ctx, const double* L, int64_t ldl, int64_t strideL, const double* Dinv, int64_t strideD,
                 double* U, int64_t ldu, int64_t strideU, double* Kinv, int64_t ldk, int64_t strideK, int N);

// Factorisation AND explicit inverse, interleaved (see InvHook): on return (stream order) A holds L with the solved
// appended rows, Dinv the complete inverse-transposed diagonal blocks, U = L^-T and Kinv = (L L^T)^-1.
int chol_trap_inverse(const Ctx& ctx, double* A, int64_t lda, int64_t strideA, int m, int k, int* info, double* Dinv,
                      int64_t strideD, double* U, int64_t ldu, int64_t strideU, double* Kinv, int64_t ldk,
                      int64_t strideK) {
  const InvHook hook{U, ldu, strideU, Kinv, ldk, strideK, A, lda, strideA, Dinv, strideD, inv_unit_max()};
  const bool interleave = inv_unit_max() >= LEAF;
  int done = 0;
  int rc = chol_trap_impl(ctx, A, lda, strideA, m, k, 0, info, Dinv, strideD, interleave ? &hook : nullptr, &done);
  if (rc) return rc;
  if (done == 2) return 0;
  if (!done) {   // single-stream schedule or interleaving switched off: the inverse follows the factorisation
    rc = leaf_dinv_assemble(ctx, A, lda, strideA, Dinv, strideD, k);
    if (rc) return rc;
    return chol_inverse(ctx, A, lda, strideA, Dinv, strideD, U, ldu, strideU, Kinv, ldk, strideK, k);
  }
  return gemm_f64(ctx, kinv_from_u(ctx, U, ldu, strideU, Kinv, ldk, strideK, k));
}

int chol_inverse(const Ctx& ctx, const double* L, int64_t ldl, int64_t strideL, const double* Dinv, int64_t strideD,
                 double* U, int64_t ldu, int64_t strideU, double* Kinv, int64_t ldk, int64_t strideK, int N) {
  if (N <= 0) return 0;
  // Only the upper triangle of U (plus the zero lower parts of its diagonal blocks, which come with Dinv) is ever
  // read, and only the lower triangle of W = L^-1 inside Kinv (plus the zero upper parts of its diagonal blocks):
  // every GEMM below clips its k range at tile granularity and tiles nest inside the LEAF blocks.
  int rc = inverse_transposed(ctx, L, ldl, strideL, Dinv, strideD, U, ldu, strideU, Kinv, ldk, strideK, N);
  if (rc) return rc;
  return gemm_f64(ctx, kinv_from_u(ctx, U, ldu, strideU, Kinv, ldk, strideK, N));
}

}  // namespace gegp
