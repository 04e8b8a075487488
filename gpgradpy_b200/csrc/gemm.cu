// fp64 tensor-core GEMM engine:  C = alpha * A * op(B) + beta * C   (row-major, DMMA.8x8x4).
//
// Every O(N^3) step of the gradient-enhanced GP hot path (Cholesky trailing updates, triangular
// solves against many right-hand sides, the explicit inverse for the trace terms) is expressed on this
// kernel.  CTA tile BM x BN x 16, multi-stage cp.async pipeline into padded shared memory whose row
// strides (20 / BN+4 doubles) make every DMMA fragment load bank-conflict free, warp tile WM x WN built
// from m8n8k4 fp64 MMAs.  Triangular operands are exploited by clipping the k range per output tile.
#include "gemm_tile.cuh"
#include <cstdlib>

namespace gegp {

constexpr int BK = 16;
constexpr int KPAD = BK + 4;  // 20 doubles: 4 consecutive rows land on 4 disjoint 8-bank groups

template <int BM, int BN, int WM, int WN, int STAGES, bool B_KCONT>
struct GemmCfg {
  static constexpr int WARPS_M = BM / WM, WARPS_N = BN / WN;
  static constexpr int THREADS = WARPS_M * WARPS_N * 32;
  static constexpr int MI = WM / 8, NI = WN / 8;
  static constexpr int A_STAGE = BM * KPAD;
  static constexpr int B_LD = B_KCONT ? KPAD : (BN + 4);
  static constexpr int B_STAGE = B_KCONT ? BN * KPAD : BK * (BN + 4);
  static constexpr size_t SMEM = (size_t)STAGES * (A_STAGE + B_STAGE) * sizeof(double);
};

template <int BM, int BN, int WM, int WN, int STAGES, bool B_KCONT>
__global__ void __launch_bounds__(GemmCfg<BM, BN, WM, WN, STAGES, B_KCONT>::THREADS)
gemm_f64_kernel(const GemmArgs g) {
  using Cfg = GemmCfg<BM, BN, WM, WN, STAGES, B_KCONT>;
  constexpr int T = Cfg::THREADS;
  extern __shared__ __align__(16) double smem[];
  double* sA = smem;
  double* sB = smem + STAGES * Cfg::A_STAGE;

  int bx = blockIdx.x, by = blockIdx.y;
  if (g.khi_mode == KHI_N0) longest_first(bx, by);
  const int m0 = by * BM, n0 = bx * BN;
  if (g.cmode != C_FULL && n0 >= m0 + BM) return;  // tile entirely above the diagonal

  const int zo = blockIdx.z / g.inner, zi = blockIdx.z - zo * g.inner;
  const double* __restrict__ A = g.A + zo * g.sAo + zi * g.sAi;
  const double* __restrict__ B = g.B + zo * g.sBo + zi * g.sBi;
  double* __restrict__ C = g.C + zo * g.sCo + zi * g.sCi;
  double* __restrict__ Ct = g.Ct ? g.Ct + zo * g.sCto + zi * g.sCti : nullptr;

  const KRange kr = tile_k_range<BN, BK>(g, m0, n0);
  const int kb = kr.kb, ke = kr.ke, ktiles = kr.tiles;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wm0 = (warp / Cfg::WARPS_N) * WM, wn0 = (warp % Cfg::WARPS_N) * WN;
  const int lr = lane >> 2, lk = lane & 3;

  // Per-thread copy state, computed once: every thread owns the same 16-byte column chunk `ck` of NA rows of
  // the A tile and NB rows of the B tile (K-contiguous B), or NB (k-row, column-chunk) slots (row-major B), so
  // that issuing one k-tile costs a handful of instructions per cp.async and no index arithmetic.
  constexpr int CPR = BK / 2;                  // 16-byte chunks per K-contiguous tile row
  constexpr int NA = BM * CPR / T;
  constexpr int RSTEP = T / CPR;               // tile rows between two chunks of one thread
  static_assert(BM * CPR % T == 0 && T % CPR == 0, "tile/thread mismatch");
  const int ck = tid % CPR, r0 = tid / CPR;
  const double* a_src[NA];
  bool a_ok[NA];
#pragma unroll
  for (int i = 0; i < NA; i++) {
    const int gr = m0 + r0 + i * RSTEP;
    a_ok[i] = gr < g.M;
    a_src[i] = A + (int64_t)(a_ok[i] ? gr : 0) * g.lda + kb + 2 * ck;
  }
  const int a_dst = r0 * KPAD + 2 * ck;
  constexpr int NBK = B_KCONT ? BN * CPR / T : BK * (BN / 2) / T;
  const double* b_src[NBK];
  bool b_ok[NBK];
  int b_dst, b_bytes = 16, b_row0 = 0;
  if (B_KCONT) {
#pragma unroll
    for (int i = 0; i < NBK; i++) {
      const int gr = n0 + r0 + i * RSTEP;
      b_ok[i] = gr < g.N;
      b_src[i] = B + (int64_t)(b_ok[i] ? gr : 0) * g.ldb + kb + 2 * ck;
    }
    b_dst = r0 * KPAD + 2 * ck;
  } else {
    constexpr int CPRB = BN / 2;               // chunks per k-row of the row-major B tile
    constexpr int KSTEP = T / CPRB;
    static_assert(T % CPRB == 0, "tile/thread mismatch");
    const int cn = tid % CPRB;
    b_row0 = tid / CPRB;
    const int gn = n0 + 2 * cn;
    b_bytes = min(16, max(0, (g.N - gn) * 8));
#pragma unroll
    for (int i = 0; i < NBK; i++) {
      b_ok[i] = true;
      b_src[i] = B + (int64_t)(kb + b_row0 + i * KSTEP) * g.ldb + (b_bytes ? gn : 0);
    }
    b_dst = b_row0 * (BN + 4) + 2 * cn;
  }

  auto load_tile = [&](int stage, int kt) {
    const int k0 = kb + kt * BK;
    double* a_s = sA + stage * Cfg::A_STAGE + a_dst;
    double* b_s = sB + stage * Cfg::B_STAGE + b_dst;
    const int kbytes = min(16, max(0, (ke - k0 - 2 * ck) * 8));   // 16 except in a ragged last k-tile
#pragma unroll
    for (int i = 0; i < NA; i++) {
      cp_async16(a_s + i * RSTEP * KPAD, a_src[i], a_ok[i] ? kbytes : 0);
      a_src[i] += BK;
    }
    if (B_KCONT) {
#pragma unroll
      for (int i = 0; i < NBK; i++) {
        cp_async16(b_s + i * RSTEP * KPAD, b_src[i], b_ok[i] ? kbytes : 0);
        b_src[i] += BK;
      }
    } else {
      constexpr int KSTEP = T / (BN / 2);
#pragma unroll
      for (int i = 0; i < NBK; i++) {
        const bool kok = k0 + b_row0 + i * KSTEP < ke;
        cp_async16(b_s + i * KSTEP * (BN + 4), kok ? b_src[i] : B, kok ? b_bytes : 0);
        b_src[i] += (int64_t)BK * g.ldb;
      }
    }
  };

  double acc[Cfg::MI][Cfg::NI][2];
#pragma unroll
  for (int i = 0; i < Cfg::MI; i++)
#pragma unroll
    for (int j = 0; j < Cfg::NI; j++) acc[i][j][0] = acc[i][j][1] = 0.0;

#pragma unroll
  for (int s = 0; s < STAGES - 1; s++) {
    if (s < ktiles) load_tile(s, s);
    cp_async_commit();
  }

  for (int kt = 0; kt < ktiles; kt++) {
    cp_async_wait<STAGES - 2>();
    __syncthreads();
    {
      const int nk = kt + STAGES - 1;
      if (nk < ktiles) load_tile(nk % STAGES, nk);
      cp_async_commit();
    }
    const double* a_s = sA + (kt % STAGES) * Cfg::A_STAGE;
    const double* b_s = sB + (kt % STAGES) * Cfg::B_STAGE;
#pragma unroll
    for (int kk = 0; kk < BK; kk += 4) {
      double af[Cfg::MI], bf[Cfg::NI];
#pragma unroll
      for (int i = 0; i < Cfg::MI; i++) af[i] = a_s[(wm0 + i * 8 + lr) * KPAD + kk + lk];
#pragma unroll
      for (int j = 0; j < Cfg::NI; j++) {
        if (B_KCONT) bf[j] = b_s[(wn0 + j * 8 + lr) * KPAD + kk + lk];
        else bf[j] = b_s[(kk + lk) * (BN + 4) + wn0 + j * 8 + lr];
      }
#pragma unroll
      for (int i = 0; i < Cfg::MI; i++)
#pragma unroll
        for (int j = 0; j < Cfg::NI; j++) dmma884(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
    }
  }
  cp_async_wait<0>();

  const bool vec_ok = ((g.ldc & 1) == 0) && ((reinterpret_cast<uintptr_t>(C) & 15) == 0);
#pragma unroll
  for (int i = 0; i < Cfg::MI; i++) {
    const int row = m0 + wm0 + i * 8 + lr;
    if (row >= g.M) continue;
#pragma unroll
    for (int j = 0; j < Cfg::NI; j++)
      store_pair(g, C, Ct, vec_ok, row, n0 + wn0 + j * 8 + 2 * lk, acc[i][j][0], acc[i][j][1]);
  }
}

// useful flops: triangular output halves the tile count, triangular operands halve the k range
double gemm_useful_flops(const GemmArgs& g) {
  double f = 2.0 * g.M * (double)g.N * g.K * g.outer * g.inner;
  if (g.cmode != C_FULL) f *= 0.5 * (g.M >= g.N ? (2.0 - (double)g.N / g.M) : 1.0);
  if (g.klo_mode == KLO_MAXMN) f *= 1.0 / 3.0;  // sum_{i>=j} (N - i) / (N^2/2 * N)
  else if (g.khi_mode == KHI_N0 && g.khi_off > 0) f *= (g.khi_off + 0.5 * g.N) / g.K;
  else if (g.klo_mode != KLO_ZERO || g.khi_mode != KHI_K) f *= 0.5;
  return f;
}

template <int BM, int BN, int WM, int WN, int STAGES, bool B_KCONT>
static int launch_cfg(const Ctx& ctx, const GemmArgs& g) {
  using Cfg = GemmCfg<BM, BN, WM, WN, STAGES, B_KCONT>;
  const dim3 grid((g.N + BN - 1) / BN, (g.M + BM - 1) / BM, g.outer * g.inner);
  const char* label = BM == 32 ? "gemm32" : (BM == 64 ? (STAGES == 2 ? "gemm64s2" : "gemm64s4") : "gemm128");
  return launch_gemm<gemm_f64_kernel<BM, BN, WM, WN, STAGES, B_KCONT>>(ctx, g, grid, Cfg::THREADS, Cfg::SMEM, label, g.M,
                                                                       g.N, g.K, g);
}


// ------------------------------------------------------------------------------------------------
// Panel update with K = LEAF:  C (M x N, N <= 128) = alpha * A (M x 128) * B (N x 128)^T + beta * C.
// This is the shape of every K = 128 update beside the factorisation's chain (the block column below the next leaf
// and the other columns of the look-ahead window get the last leaf's panel): tall, 128 wide, and so shallow that the
// generic kernel's k-pipeline (8 k-tiles, a barrier each) is all ramp.  Here a CTA owns BM rows and ALL N columns,
// brings its whole A strip and the whole B block into shared memory with one wave of cp.async (a single wait, a
// single barrier) and then issues its 32 k-steps of DMMA back to back.  8 warps: BM / 16 row groups x 8 / (BM / 16)
// column groups, 16 rows per warp.  Same k order per output element as the generic kernels (k = 0 .. 127 in steps of 4).
// ------------------------------------------------------------------------------------------------
constexpr int K128 = 128;
constexpr int K128_LD = K128 + 4;   // == 4 (mod 16): conflict-free fragment loads

template <int BM>
__global__ void __launch_bounds__(256, 1)
gemm_k128_kernel(const GemmArgs g) {
  constexpr int RG = BM / 16;            // row groups (warps along M)
  constexpr int CG = 8 / RG;             // column groups (warps along N)
  constexpr int WN = 128 / CG;           // columns per warp
  constexpr int NI = WN / 8;
  extern __shared__ __align__(16) double smem[];
  double* sA = smem;                     // [BM][K128_LD]
  double* sB = smem + BM * K128_LD;      // [128][K128_LD]
  const int zo = blockIdx.z;
  const double* __restrict__ A = g.A + zo * g.sAo;
  const double* __restrict__ B = g.B + zo * g.sBo;
  double* __restrict__ C = g.C + zo * g.sCo;
  const int m0 = blockIdx.x * BM;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int lr = lane >> 2, lk = lane & 3;
  // one wave of 16-byte copies: rows outside the operands are zero-filled
  for (int e = tid; e < BM * (K128 / 2); e += 256) {
    const int r = e >> 6, c = (e & 63) * 2;
    const bool ok = m0 + r < g.M;
    cp_async16(sA + r * K128_LD + c, A + (int64_t)(ok ? m0 + r : 0) * g.lda + c, ok ? 16 : 0);
  }
  for (int e = tid; e < 128 * (K128 / 2); e += 256) {
    const int r = e >> 6, c = (e & 63) * 2;
    const bool ok = r < g.N;
    cp_async16(sB + r * K128_LD + c, B + (int64_t)(ok ? r : 0) * g.ldb + c, ok ? 16 : 0);
  }
  cp_async_commit();
  const int wr = warp / CG, wc = warp % CG;
  const int r0 = wr * 16, c0 = wc * WN;
  if (g.cmode != C_FULL && c0 >= m0 + r0 + 16) {   // this warp's tile lies entirely above the diagonal
    cp_async_wait<0>();
    __syncthreads();
    return;
  }
  double acc[2][NI][2];
#pragma unroll
  for (int i = 0; i < 2; i++)
#pragma unroll
    for (int j = 0; j < NI; j++) acc[i][j][0] = acc[i][j][1] = 0.0;
  cp_async_wait<0>();
  __syncthreads();
  const double* a0 = sA + (r0 + lr) * K128_LD + lk;
  const double* b0 = sB + (c0 + lr) * K128_LD + lk;
#pragma unroll 4
  for (int kq = 0; kq < 32; kq++) {
    const double af0 = a0[4 * kq], af1 = a0[8 * K128_LD + 4 * kq];
    double bf[NI];
#pragma unroll
    for (int j = 0; j < NI; j++) bf[j] = b0[j * 8 * K128_LD + 4 * kq];
#pragma unroll
    for (int j = 0; j < NI; j++) {
      dmma884(acc[0][j][0], acc[0][j][1], af0, bf[j]);
      dmma884(acc[1][j][0], acc[1][j][1], af1, bf[j]);
    }
  }
  const bool vec_ok = ((g.ldc & 1) == 0) && ((reinterpret_cast<uintptr_t>(C) & 15) == 0);
#pragma unroll
  for (int i = 0; i < 2; i++) {
    const int row = m0 + r0 + i * 8 + lr;
    if (row >= g.M) continue;
#pragma unroll
    for (int j = 0; j < NI; j++)
      store_pair(g, C, nullptr, vec_ok, row, c0 + j * 8 + 2 * lk, acc[i][j][0], acc[i][j][1]);
  }
}

template <int BM>
static int launch_k128(const Ctx& ctx, const GemmArgs& g) {
  const size_t smem = (size_t)(BM + 128) * K128_LD * sizeof(double);
  return launch_gemm<gemm_k128_kernel<BM>>(ctx, g, dim3((g.M + BM - 1) / BM, 1, g.outer), 256, smem, "gemm_k128", g.M,
                                           g.N, BM, g);
}

// rows per CTA: the smallest of 16 / 32 / 64 that still gives every CTA an SM of its own (one wave), else 64
static int gemm_k128(const Ctx& ctx, const GemmArgs& g) {
  const long rows_total = (long)g.M * g.outer;
  if (rows_total <= 148L * 16) return launch_k128<16>(ctx, g);
  if (rows_total <= 148L * 32) return launch_k128<32>(ctx, g);
  return launch_k128<64>(ctx, g);
}

static int g_tma_min_tiles = -1;
int& tma_min_tiles() {
  if (g_tma_min_tiles < 0) g_tma_min_tiles = getenv("GEGP_BIG_TILES") ? atoi(getenv("GEGP_BIG_TILES")) : 400;
  return g_tma_min_tiles;
}

static int g_small_tile_max = -1;
int& small_tile_max() {
  if (g_small_tile_max < 0) g_small_tile_max = getenv("GEGP_SMALL_TILES") ? atoi(getenv("GEGP_SMALL_TILES")) : 36;
  return g_small_tile_max;
}

GemmArgs gemm_args(const double* A, int64_t lda, const double* B, int64_t ldb, double* C, int64_t ldc,
                   int M, int N, int K, double alpha, double beta, bool b_kcont) {
  GemmArgs g{};
  g.A = A; g.B = B; g.C = C; g.lda = lda; g.ldb = ldb; g.ldc = ldc;
  g.M = M; g.N = N; g.K = K; g.alpha = alpha; g.beta = beta; g.b_kcont = b_kcont;
  g.klo_mode = KLO_ZERO; g.khi_mode = KHI_K; g.cmode = C_FULL; g.khi_off = 0;
  g.inner = 1; g.outer = 1;
  g.inner_steps = false; g.iAr = g.iAc = g.iBr = g.iBc = 0;
  g.Ct = nullptr; g.ldct = 0; g.sCto = g.sCti = 0;
  g.sAo = g.sBo = g.sCo = g.sAi = g.sBi = g.sCi = 0;
  return g;
}

// output tiles of one M x N problem in tile x tile tiles; a lower-triangular output skips those strictly above the diagonal
static long tiles(int M, int N, int tile, int cmode) {
  const long rt = (M + tile - 1) / tile, ct = (N + tile - 1) / tile;
  long t = rt * ct;
  if (cmode != C_FULL) {
    const long sq = rt < ct ? rt : ct;
    t -= sq * (sq - 1) / 2 + (ct > rt ? (ct - rt) * rt : 0);
  }
  return t;
}

int gemm_f64(const Ctx& ctx, GemmArgs g) {
  if (g.M <= 0 || g.N <= 0 || g.outer * g.inner <= 0) return 0;
  if (g.K <= 0 && g.beta == 1.0) return 0;
  // operands must allow 16-byte cp.async: even leading dimensions and 16-byte aligned bases
  if ((g.lda & 1) || (g.ldb & 1) || (reinterpret_cast<uintptr_t>(g.A) & 15) || (reinterpret_cast<uintptr_t>(g.B) & 15) ||
      (g.sAo & 1) || (g.sAi & 1) || (g.sBo & 1) || (g.sBi & 1))
    return -900;
  // Large tile when one problem still fills the machine with it, small tile otherwise.  The choice depends on the
  // shape of ONE problem only, never on the batch count: a candidate evaluated alone, in a batch, or on another rank
  // of a sharded batch goes through the same kernels and gives bit-identical results.
  const long tiles_big = tiles(g.M, g.N, 128, g.cmode) * g.inner;
  // Measured on B200 (d=10, n=500 and d=20, n=1000 evaluations): with fewer than ~400 tiles of 128 x 128 per problem
  // the TMA kernel loses more to wave quantisation than it gains over the 64 x 64 cp.async kernel; between 400 and 1000
  // the two are equal, above the TMA kernel wins (measured with 128 x 64 tiles on 296 CTA slots; re-checked at both sizes
  // with the 128 x 128 tiles / 148 slots the kernel has now: 150 ... 400 give the same evaluation times).
  const bool big = tiles_big >= tma_min_tiles() && g.M >= 128 && g.N >= 128;
  // K = LEAF panel updates (tall, at most 128 wide): the single-wave kernel; BM (rows per CTA) only changes which CTA
  // owns a row, not the arithmetic of an element.
  // Only while one wave of whole-SM CTAs covers the panel (M <= 148 * 64): beyond that the problem is throughput-bound and
  // the generic kernels, which share an SM with the bulk GEMM CTAs, are the better neighbours (measured at N = 21000).
  // It accumulates every element in the same k order as the generic kernels (bit-identical results, tested), which is why
  // this choice -- like the 32 x 32 one below -- may look at the batch count.
  if (g.b_kcont && g.K == K128 && g.N <= 128 && g.klo_mode == KLO_ZERO && g.khi_mode == KHI_K && !g.Ct && g.inner == 1 &&
      (long)g.M * g.outer <= 148L * 64)
    return gemm_k128(ctx, g);
  if (g.b_kcont && big) {
    const int rc = gemm_tma_nt(ctx, g);
    if (rc <= 0) return rc;
  }
  if (g.b_kcont) {
    if (big) return launch_cfg<128, 128, 64, 32, 4, true>(ctx, g);
    // A product with only a handful of 64 x 64 tiles (the diagonal-block updates on the factorisation's critical
    // path: 128 x 128 x K, lower) is bound by the latency of ONE CTA walking K; 32 x 32 tiles put it on 4x as many
    // SMs.  Same k order per output element, so the result does not depend on the tile size (tested bit for bit),
    // which is why this choice -- unlike the TMA one -- may look at the batch count.
    const long ctas = tiles(g.M, g.N, 64, g.cmode) * g.inner * g.outer;   // of 64 x 64 tiles
    if (ctas <= small_tile_max()) return launch_cfg<32, 32, 16, 16, 4, true>(ctx, g);
    // skinny and deep (one block column updated by a long panel: the just-in-time pieces of the factorisation that the
    // critical path reaches first): less than one 64 x 64 tile per SM, each walking a long K -- 32 x 32 tiles again
    if (g.N <= 128 && g.K >= 512 && ctas <= 148) return launch_cfg<32, 32, 16, 16, 4, true>(ctx, g);
    // 64 x 64 tiles: with enough CTAs to give every SM several, a 2-stage ring (41 KB, 4 CTAs = 16 warps per SM)
    // beats the 4-stage one (82 KB, 2 CTAs per SM) by 10-15 % (measured: 2048^3 32.5 vs 28.2 TFLOP/s, the batched
    // N=1200 scan +12 %); with few CTAs the deeper prefetch of the 4-stage ring wins.  Same arithmetic either way.
    if (ctas >= 4 * 148) return launch_cfg<64, 64, 32, 32, 2, true>(ctx, g);
    return launch_cfg<64, 64, 32, 32, 4, true>(ctx, g);
  } else {
    if (big) return launch_cfg<128, 128, 64, 32, 4, false>(ctx, g);
    return launch_cfg<64, 64, 32, 32, 4, false>(ctx, g);
  }
}

}  // namespace gegp
