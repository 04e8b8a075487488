// Internal dense fp64 linear-algebra engine (row-major, lower-triangular convention).
// All routines are asynchronous on ctx.stream and batched over ctx.batch problems (blockIdx.z).
#pragma once
#include "common.cuh"

namespace gegp {

enum KLo { KLO_ZERO = 0, KLO_M0 = 1, KLO_N0 = 2, KLO_MAXMN = 3 };
enum KHi { KHI_K = 0, KHI_N0 = 2 };
enum CMode { C_FULL = 0, C_LOWER = 1, C_LOWER_MIRROR = 2 };

struct GemmArgs {
  const double* A;  // element (m,k) at A[m*lda + k]
  const double* B;  // b_kcont: element (n,k) at B[n*ldb + k]; else element (k,n) at B[k*ldb + n]
  double* C;        // element (m,n) at C[m*ldc + n]
  int64_t lda, ldb, ldc;
  int M, N, K;
  double alpha, beta;     // C = alpha * A*op(B) + beta * C
  bool b_kcont;
  int klo_mode, khi_mode; // triangular-operand clipping of the k range per output tile
  int khi_off;            // KHI_N0 only: the k range of column tile n0 ends at khi_off + n0 + BN (B is a row slice of a
                          // lower-triangular matrix that starts khi_off rows below its first row)
  int cmode;
  // batching: z = zo*inner + zi ; pointer offset = zo*s?o + zi*s?i (elements)
  int inner;
  int64_t sAo, sBo, sCo, sAi, sBi, sCi;
  int outer;
  bool inner_steps;        // iAr..iBc below are valid (needed by the TMA kernel when inner > 1)
  int iAr, iAc, iBr, iBc;  // inner-batch steps of A and B as (rows, columns): sAi == iAr*lda + iAc, sBi likewise
  // optional second, transposed destination: Ct[col * ldct + row] = value for every stored C(row, col)
  double* Ct;
  int64_t ldct, sCto, sCti;
};

GemmArgs gemm_args(const double* A, int64_t lda, const double* B, int64_t ldb, double* C, int64_t ldc,
                   int M, int N, int K, double alpha, double beta, bool b_kcont);
// g over the ctx.batch problems of a call, whose A, B and C lie sA, sB and sC doubles after those of the previous one
inline GemmArgs batched(const Ctx& ctx, GemmArgs g, int64_t sA, int64_t sB, int64_t sC) {
  g.outer = ctx.batch; g.inner = 1;
  g.sAo = sA; g.sBo = sB; g.sCo = sC;
  return g;
}

// C = alpha*A*op(B) + beta*C on fp64 tensor cores (DMMA). Returns 0 or a negative launch error.
int gemm_f64(const Ctx& ctx, GemmArgs g);
// TMA + mbarrier warp-specialised kernel for the K-contiguous (A * B^T) case and large tiles.
// 0: launched; 1: not covered (use the cp.async engine); < 0: launch error.
int gemm_tma_nt(const Ctx& ctx, const GemmArgs& g);
double gemm_useful_flops(const GemmArgs& g);
// smallest number of 128 x 128 output tiles (of one problem) for which the TMA kernel is chosen (tuning knob)
int& tma_min_tiles();
// largest number of 64 x 64 output tiles (of one problem) for which the 32 x 32-tile kernel is chosen (tuning knob)
int& small_tile_max();

// --- leaves (<= LEAF wide) ---
// Every factor carries the inverse-transposed diagonal blocks Dinv: block b (rows/cols [b*LEAF, (b+1)*LEAF)) is
// the LEAF x LEAF row-major (ld LEAF) upper-triangular matrix L_bb^-T at Dinv + b*LEAF*LEAF.
inline int64_t dinv_doubles(int N) { return (int64_t)((N + LEAF - 1) / LEAF) * LEAF * LEAF; }

// In-place Cholesky of the k x k lower block at A (k <= LEAF) and Dinv <- L^-T; the first non-positive pivot is
// recorded in info[z] (1-based global index row0+i+1) if info[z] was 0.
int leaf_potf2_inv(const Ctx& ctx, double* A, int64_t lda, int64_t strideA, int k, int row0, int* info, double* Dinv,
                   int64_t strideD);
// After leaf_potf2_inv only the 32 x 32 diagonal inverses of each Dinv block are valid (enough for leaf_trsm);
// this completes every block to the full 128 x 128 L_bb^-T (needed by chol_inverse and trsv_lower_trans).
int leaf_dinv_assemble(const Ctx& ctx, const double* L, int64_t ldl, int64_t strideL, double* Dinv, int64_t strideD,
                       int N);
// B (r x k) <- B * L^-T for one factored leaf block (k <= LEAF): fused block substitution on the tensor cores with
// the 32 x 32 diagonal inverses taken from Dinv and one refinement step each (as accurate as a substitution).
int leaf_trsm(const Ctx& ctx, const double* L, int64_t ldl, int64_t strideL, const double* Dinv, int64_t strideD,
              double* B, int64_t ldb, int64_t strideB, int r, int k);
// Chain step between two leaf factorisations: B (kc x LEAF, the block row right below the factored leaf Lp) <- B Lp^-T
// in place, then E (kc x kc, lower: the next leaf's diagonal block) -= B B^T.  One small thread-block cluster.
int leaf_chain_prep(const Ctx& ctx, const double* Lp, int64_t lda, int64_t strideA, const double* Dinv, int64_t strideD,
                    double* B, double* E, int kc);
// cluster size of that step (0: automatic; 1, 2, 4) -- tuning knob, same results for every value
int& chain_cluster();
// early pieces of the explicit inverse (chol_trap_inverse): 0 off, 1 / 2 forced level, 3 by problem size (default)
int& inv_early_option();
// Diagonal blocks of the N x N buffer U <- Dinv blocks (upper triangular), diagonal blocks of W <- their transposes
// (lower triangular); the rest of both buffers is left untouched.
int leaf_scatter_dinv(const Ctx& ctx, const double* Dinv, int64_t strideD, double* U, int64_t ldu, int64_t strideU,
                      double* W, int64_t ldw, int64_t strideW, int N);

// --- blocked algorithms ---
// Trapezoid Cholesky: A is m x k (m >= k), lower. Factors the leading k x k block in place (L) and
// overwrites rows k..m-1 with A21 * L^-T (so appended right-hand-side rows come out forward-solved).
// row0 (multiple of LEAF) is the global index of the first row/column; Dinv is indexed by global block.
int chol_trap(const Ctx& ctx, double* A, int64_t lda, int64_t strideA, int m, int k, int row0, int* info, double* Dinv,
              int64_t strideD);
// chol_trap followed by chol_inverse, with the triangular inverse interleaved with the factorisation: each subtree is
// inverted on a lowest-priority stream as soon as the chain has left it, so the SMs the latency-bound chain leaves idle
// do the inverse's GEMMs.  Same results as the two calls in sequence up to the summation order inside U (the pairs
// follow the factorisation's tree instead of aligned power-of-two blocks).  Dinv comes back complete.
int chol_trap_inverse(const Ctx& ctx, double* A, int64_t lda, int64_t strideA, int m, int k, int* info, double* Dinv,
                      int64_t strideD, double* U, int64_t ldu, int64_t strideU, double* Kinv, int64_t ldk,
                      int64_t strideK);
// B (r x k) <- B * L^-T for an already factored k x k lower L (col0: global index of L's first column).
int trsm_right_rec(const Ctx& ctx, const double* L, int64_t ldl, int64_t strideL, const double* Dinv, int64_t strideD,
                   int col0, double* B, int64_t ldb, int64_t strideB, int r, int k);
// Lt[dinv_doubles(N)] <- the transposed diagonal blocks L_bb^T of a factor (row-major, ld LEAF, zeros elsewhere).
int stage_leaf_lt(const Ctx& ctx, const double* L, int64_t ldl, double* Lt, int N);
// B (r x k) <- B * L^-1 (rows against the lower factor, not transposed) for an already factored k x k lower L: the mirror
// of trsm_right_rec (right block first, then the GEMM update of the left block).  Leaves multiply with the full Dinv blocks
// and take one refinement step against the staged Lt blocks; T is r x LEAF scratch.
int trsm_right_lower_rec(const Ctx& ctx, const double* L, int64_t ldl, const double* Dinv, const double* Lt, int col0,
                         double* B, int64_t ldb, int r, int k, double* T);
// Kinv (full symmetric N x N) = L^-T L^-1. U (N x N) receives L^-T in its upper triangle (its strictly lower part
// outside the diagonal blocks is never written nor read).  Kinv doubles as scratch: while U is built its lower triangle
// holds the transpose L^-1, so that every product of the inverse is an A * B^T with K-contiguous operands (TMA kernel).
int chol_inverse(const Ctx& ctx, const double* L, int64_t ldl, int64_t strideL, const double* Dinv, int64_t strideD,
                 double* U, int64_t ldu, int64_t strideU, double* Kinv, int64_t ldk, int64_t strideK, int N);
// x <- L^-T x (blocked back substitution with the Dinv blocks), nrhs vectors x[r*ldx + i].
int trsv_lower_trans(const Ctx& ctx, const double* L, int64_t ldl, int64_t strideL, const double* Dinv, int64_t strideD,
                     double* x, int64_t ldx, int64_t strideX, int N, int nrhs);
// y = U x with U upper triangular (N x N, row-major).
int trmv_upper(const Ctx& ctx, const double* U, int64_t ldu, int64_t strideU, const double* x, int64_t strideX,
               double* y, int64_t strideY, int N);


// --- extreme eigenpairs (Lanczos building blocks, csrc/eig.cu) ---
// Each takes ctx.batch candidates at once: candidate z's arrays sit `stride` doubles after candidate 0's, and the
// optional int32 list `active` names the candidate of each of the ctx.batch launch rows (nullptr: rows 0 .. batch-1).
// The arithmetic for one candidate does not depend on the batch.
// y = M x for a dense row-major N x ld matrix.
int symv_full(const Ctx& ctx, int N, const double* M, int64_t ld, int64_t strideM, const double* x, int64_t strideX,
              double* y, int64_t strideY, const int* active);
// out[row] = sum_c |M[row, c]| (Gershgorin row sums for the variable nugget) or sum_c M[row, c]^2 (Frobenius norm).
int row_abs_sum(const Ctx& ctx, int N, const double* M, int64_t ld, double* out, bool squares = false);
// One Lanczos step with full re-orthogonalisation: V rows 0..j orthonormal, w = M v_j on entry; writes alpha[j],
// beta[j] (device) and V row j+1 (j < 255).
int lanczos_step(const Ctx& ctx, int N, int j, double* V, int64_t ldv, int64_t strideV, double* w, int64_t strideW,
                 double* alpha, double* beta, int64_t strideAB, const int* active);
// out = normalised sum_i coef[i] V_i (k <= 256, coef on the device); ks (optional, device): each candidate's own k,
// clamped to 1 .. k.
int lincomb_rows(const Ctx& ctx, int N, int k, const int* ks, const double* V, int64_t ldv, int64_t strideV,
                 const double* coef, int64_t strideCoef, double* out, int64_t strideOut, const int* active);

}  // namespace gegp
