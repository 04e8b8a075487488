// Pieces shared by the GEMM kernels of gemm.cu and gemm_tma.cu: the k range of an output tile, the longest-first tile
// order, the epilogue store and the launch bookkeeping.
#pragma once
#include "linalg.h"

namespace gegp {

// k range [kb, ke) of the output tile at (m0, n0), clipped by the triangular operands; kb rounded down to a k-tile of
// BK, `tiles` k-tiles of BK (the last one may be ragged).
struct KRange { int kb, ke, tiles; };
template <int BN, int BK>
__device__ __forceinline__ KRange tile_k_range(const GemmArgs& g, int m0, int n0) {
  int kb = 0;
  if (g.klo_mode == KLO_M0) kb = m0;
  else if (g.klo_mode == KLO_N0) kb = n0;
  else if (g.klo_mode == KLO_MAXMN) kb = max(m0, n0);
  const int ke = g.khi_mode == KHI_N0 ? min(g.K, g.khi_off + n0 + BN) : g.K;
  kb = (kb / BK) * BK;
  return {kb, ke, ke > kb ? (ke - kb + BK - 1) / BK : 0};
}

// k range clipped above by the column tile (KHI_N0): the work of a tile grows with its column.  CTAs are dispatched
// in linear blockIdx order, so the tiles are re-mapped to longest-processing-time-first: all tiles of the last
// (longest) column, then the one before, ...  (list-scheduling simulation of the 32 x 32-tile product of the inverse on
// 592 CTA slots: makespan 1.73x the ideal in row-major order, 1.10x in this order; ncu showed the SMs idle a third of
// the kernel before.)
__device__ __forceinline__ void longest_first(int& bx, int& by) {
  const int lin = blockIdx.y * gridDim.x + blockIdx.x;
  bx = (int)gridDim.x - 1 - lin / (int)gridDim.y;
  by = lin % (int)gridDim.y;
}

// Epilogue of one output pair: C(row, col .. col+1) = alpha * (a0, a1) + beta * C, col even, row < M.  A lower-
// triangular output (cmode != C_FULL) stores only on and below the diagonal, C_LOWER_MIRROR stores every strictly lower
// element a second time at its mirror position, and a non-null Ct receives every stored element transposed.  vec_ok: C
// and ldc allow 16-byte stores.
__device__ __forceinline__ void store_pair(const GemmArgs& g, double* __restrict__ C, double* __restrict__ Ct,
                                           bool vec_ok, int row, int col, double a0, double a1) {
  if (col >= g.N) return;
  double* cp = C + (int64_t)row * g.ldc + col;
  double v0 = g.alpha * a0, v1 = g.alpha * a1;
  const bool has1 = (col + 1 < g.N);
  bool st0 = true, st1 = has1;
  if (g.cmode != C_FULL) { st0 = (col <= row); st1 = has1 && (col + 1 <= row); }
  if (g.beta != 0.0) {
    if (st0) v0 += g.beta * cp[0];
    if (st1) v1 += g.beta * cp[1];
  }
  if (st0 && st1 && vec_ok) {
    *reinterpret_cast<double2*>(cp) = make_double2(v0, v1);
  } else {
    if (st0) cp[0] = v0;
    if (st1) cp[1] = v1;
  }
  if (g.cmode == C_LOWER_MIRROR) {
    if (st0 && col < row) C[(int64_t)col * g.ldc + row] = v0;
    if (st1 && col + 1 < row) C[(int64_t)(col + 1) * g.ldc + row] = v1;
  }
  if (Ct) {
    if (st0) Ct[(int64_t)col * g.ldct + row] = v0;
    if (st1) Ct[(int64_t)(col + 1) * g.ldct + row] = v1;
  }
}

// Launches one GEMM kernel: opts it in to `smem` bytes of dynamic shared memory, counts the launch and its useful
// flops in prof() and marks it on the debug timeline as "label a b c" (tools/timeline.py and tools/tl_eval.py parse it).
template <auto KERNEL, class... Params>
static int launch_gemm(const Ctx& ctx, const GemmArgs& g, dim3 grid, int threads, size_t smem, const char* label, int a,
                       int b, int c, const Params&... params) {
  GEGP_SET_SMEM(KERNEL, smem);
  prof_gemm_begin(ctx.stream);
  timeline_begin(ctx.stream, label, a, b, c, timeline_on() ? gemm_useful_flops(g) * 1e-6 : 0.0);
  KERNEL<<<grid, threads, smem, ctx.stream>>>(params...);
  timeline_end(ctx.stream);
  if (prof().on) prof_gemm_end(ctx.stream, gemm_useful_flops(g));
  GEGP_CHECK_LAUNCH();
  return 0;
}

}  // namespace gegp
