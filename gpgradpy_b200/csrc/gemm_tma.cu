// fp64 tensor-core GEMM, TMA-staged and warp-specialised:  C = alpha * A * B^T + beta * C
// (row-major, A is M x K and B is N x K, both K-contiguous -- the shape of every Cholesky trailing update,
// of the first half of the triangular inverse and of K^-1 = U U^T).
//
// One CTA per 128 x 128 output tile, ONE CTA per SM, which it has to itself (see TmaCfg).  A producer warp streams
// [rows x 16 doubles] boxes of A and B into a 6-deep shared-memory ring with cp.async.bulk.tensor (TMA, 128-byte swizzle,
// zero fill outside the operand), signalling one mbarrier per stage; eight consumer warps (64 x 32 warp tiles) wait on
// that barrier, feed DMMA.8x8x4 from the swizzled tiles and release the stage through a second mbarrier.  There is no
// CTA-wide barrier and no address arithmetic in the math warps, so the fp64 tensor pipe is the only busy unit.
//
// Shared-memory reads are bank-conflict free without padding: a tile row is one 128-byte line whose 16-byte
// chunks are XOR-swizzled with (row & 7) by the TMA unit.  The k index inside a 16-wide k-tile is a summation
// index, so each DMMA step s may pick any 4 of the 16 k values as long as A and B pick the same ones: lanes with
// (lane & 3) < 2 read chunk s, the others chunk s + 4, which makes the 16 lanes of a half-warp touch all eight
// chunk positions of the line exactly once.
#include "gemm_tile.cuh"
#include <cuda.h>
#include <cstring>
#include <mutex>
#include <unordered_map>

namespace gegp {

namespace {

constexpr int TBK = 16;
constexpr int TWM = 64, TWN = 32;                  // warp tile
constexpr int TMI = TWM / 8, TNI = TWN / 8;

// CTA tile TBM x TBN (multiples of the 64 x 32 warp tile), TSTAGES-deep ring, one CTA per SM: the CTA asks for ALL the
// shared memory a block may have (227 KB, SOLO), so that no other CTA -- of this grid, of another kernel of this library
// or of a foreign kernel on another stream -- can share its SM.
struct TmaCfg {
  static constexpr int TBM = 128, TBN = 128, TSTAGES = 6;
  static constexpr int CONSUMERS = (TBM / TWM) * (TBN / TWN);
  static constexpr int THREADS = (CONSUMERS + 1) * 32;    // + 1 producer warp
  static constexpr uint32_t A_BYTES = TBM * TBK * sizeof(double);
  static constexpr uint32_t B_BYTES = TBN * TBK * sizeof(double);
  static constexpr uint32_t STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr size_t USED = (size_t)TSTAGES * STAGE_BYTES + 2 * TSTAGES * sizeof(uint64_t) + 1024;  // + alignment slack
  static constexpr size_t SMEM = GEGP_MAX_DYN_SMEM;
  static_assert(USED <= (size_t)GEGP_MAX_DYN_SMEM, "ring does not fit");
};
// WHY SOLO.  With the 128 x 64 tile / two CTAs per SM this kernel was first built with (35.2 TFLOP/s at 8192^3), an
// evaluation was NOT reproducible whenever CTAs of this kernel shared SMs with CTAs of other kernels: beside foreign cuBLAS DGEMMs on another stream 18 of 30 factorisations at N = 21000 came out wrong (a few tiles of a product,
// up to NaN), and with this library's own inverse running beside the factorisation 3 to 5 of 24 evaluations at
// N = 41000 / 51000 deviated by up to 1e-7 (tools/repro_probe.py; profiles/r02/repro_tma_shared_sm.log).  The cp.async
// kernels never deviated under the same load, nor did this kernel once it had the SM to itself; tensor maps in global
// memory, unswizzled tiles, the .shared::cta form of the copy and a producer warp that outlives the consumers did not
// help (each tried).  The mechanism was not found -- every dependency of the ring is on an mbarrier and the protocol is
// the textbook one -- so the kernel simply no longer shares an SM: 128 x 128 tile, 8 math warps + 1 producer warp,
// 6 stages, the whole 227 KB.  Same k order per element as before (bit-identical results), same speed at N = 5500 and
// 21000.  The two-CTA configuration is in the history of this file (git show 815988e:gpgradpy_b200/csrc/gemm_tma.cu).

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(bar),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
      ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(bar)
      : "memory");
}

__global__ void __launch_bounds__(TmaCfg::THREADS, 1)
gemm_tma_nt_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                   const __grid_constant__ GemmArgs g) {
  constexpr int TBM = TmaCfg::TBM, TBN = TmaCfg::TBN, TSTAGES = TmaCfg::TSTAGES, TCONSUMERS = TmaCfg::CONSUMERS;
  constexpr uint32_t TILE_BYTES = TmaCfg::A_BYTES, STAGE_BYTES = TmaCfg::STAGE_BYTES;
  extern __shared__ uint8_t smem_raw[];
  int bx = blockIdx.x, by = blockIdx.y;
  if (g.khi_mode == KHI_N0) {
    longest_first(bx, by);
  } else {
    // Grouped raster: CTAs are dispatched in linear block order, so walk the tiles in bands of RASTER_ROWS row tiles,
    // down the rows of a band first.  The ~296 CTAs in flight then cover RASTER_ROWS A panels x ~37 B panels instead
    // of one A panel x 296 B panels, and every k-slice a CTA streams is read from DRAM once per band instead of once
    // per tile (ncu at N = 21000, K^-1 = U U^T: 95 GB of DRAM reads for 5.3 GB of operands in row-major order).  Long
    // tiles (small row index when k is clipped below) still come first.
    constexpr int RASTER_ROWS = 8;
    const int lin = blockIdx.y * gridDim.x + blockIdx.x;
    const int per_band = RASTER_ROWS * (int)gridDim.x;
    const int band = lin / per_band, within = lin - band * per_band;
    const int rows = min(RASTER_ROWS, (int)gridDim.y - band * RASTER_ROWS);
    by = band * RASTER_ROWS + within % rows;
    bx = within / rows;
  }
  const int m0 = by * TBM, n0 = bx * TBN;
  if (g.cmode != C_FULL && n0 >= m0 + TBM) return;  // tile entirely above the diagonal

  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;  // 128B-swizzled TMA tiles need 1024-byte alignment
  const uint8_t* tiles = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t bar_full = base + TSTAGES * STAGE_BYTES;
  const uint32_t bar_empty = bar_full + TSTAGES * 8;

  const int zo = blockIdx.z / g.inner, zi = blockIdx.z - zo * g.inner;

  const KRange kr = tile_k_range<TBN, TBK>(g, m0, n0);
  const int kb = kr.kb, ktiles = kr.tiles;
  const bool k_down = g.klo_mode != KLO_ZERO && g.khi_mode == KHI_K;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) {
    for (int s = 0; s < TSTAGES; s++) {
      mbar_init(bar_full + 8 * s, 1);
      mbar_init(bar_empty + 8 * s, TCONSUMERS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  if (warp == TCONSUMERS) {
    // ===== producer warp: one lane issues the TMA loads =====
    if (lane == 0) {
      const int ca = zi * g.iAc, ra = zi * g.iAr + m0;
      const int cb = zi * g.iBc, rb = zi * g.iBr + n0;
      for (int kt = 0; kt < ktiles; kt++) {
        const int s = kt % TSTAGES;
        if (kt >= TSTAGES) mbar_wait(bar_empty + 8 * s, ((kt / TSTAGES) - 1) & 1);
        const uint32_t full = bar_full + 8 * s;
        mbar_expect_tx(full, STAGE_BYTES);
        // k clipped below (triangular operand): every tile ends at k = K but starts at its own row, so the tiles walk k
        // DOWNWARDS -- CTAs dispatched together then stream the same k-slices at the same time and the slices of a
        // B panel are shared through L2 by all rows of a band (upwards, row r lags row r - 1 by 128 k and finds them evicted)
        const int k0 = kb + (k_down ? ktiles - 1 - kt : kt) * TBK;
        tma_load_3d(base + s * STAGE_BYTES, &tmA, ca + k0, ra, zo, full);
        tma_load_3d(base + s * STAGE_BYTES + TILE_BYTES, &tmB, cb + k0, rb, zo, full);
      }
    }
    return;
  }

  // ===== consumer warps =====
  const int wm0 = (warp / (TBN / TWN)) * TWM, wn0 = (warp % (TBN / TWN)) * TWN;
  const int lr = lane >> 2, lk = lane & 3;
  // byte offsets inside a tile: row * 128 + ((chunk ^ (row & 7)) << 4) + (k & 1) * 8, chunk = s + 4 * (lk >> 1)
  const uint32_t a_row = (uint32_t)(wm0 + lr) * 128u + (uint32_t)(lk & 1) * 8u;
  const uint32_t b_row = TILE_BYTES + (uint32_t)(wn0 + lr) * 128u + (uint32_t)(lk & 1) * 8u;
  uint32_t sw[4];
#pragma unroll
  for (int s = 0; s < 4; s++) sw[s] = (uint32_t)(((s + 4 * (lk >> 1)) ^ lr) << 4);

  double acc[TMI][TNI][2];
#pragma unroll
  for (int i = 0; i < TMI; i++)
#pragma unroll
    for (int j = 0; j < TNI; j++) acc[i][j][0] = acc[i][j][1] = 0.0;

  for (int kt = 0; kt < ktiles; kt++) {
    const int s = kt % TSTAGES;
    mbar_wait(bar_full + 8 * s, (kt / TSTAGES) & 1);
    const uint8_t* st = tiles + s * STAGE_BYTES;
#pragma unroll
    for (int q = 0; q < 4; q++) {
      double af[TMI], bf[TNI];
      const uint8_t* pa = st + a_row + sw[q];
      const uint8_t* pb = st + b_row + sw[q];
#pragma unroll
      for (int i = 0; i < TMI; i++) af[i] = *reinterpret_cast<const double*>(pa + i * 1024);
#pragma unroll
      for (int j = 0; j < TNI; j++) bf[j] = *reinterpret_cast<const double*>(pb + j * 1024);
#pragma unroll
      for (int i = 0; i < TMI; i++)
#pragma unroll
        for (int j = 0; j < TNI; j++) dmma884(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(bar_empty + 8 * s);
  }

  // ===== epilogue =====
  double* __restrict__ C = g.C + zo * g.sCo + zi * g.sCi;
  double* __restrict__ Ct = g.Ct ? g.Ct + zo * g.sCto + zi * g.sCti : nullptr;
  const bool vec_ok = ((g.ldc & 1) == 0) && ((reinterpret_cast<uintptr_t>(C) & 15) == 0);
#pragma unroll
  for (int i = 0; i < TMI; i++) {
    const int row = m0 + wm0 + i * 8 + lr;
    if (row >= g.M) continue;
#pragma unroll
    for (int j = 0; j < TNI; j++)
      store_pair(g, C, Ct, vec_ok, row, n0 + wn0 + j * 8 + 2 * lk, acc[i][j][0], acc[i][j][1]);
  }
}

// ---- host side: tensor maps (encoded through the driver entry point, cached per operand) ----
using EncodeFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                              const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                              CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeFn encode_fn() {
  static EncodeFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    return reinterpret_cast<EncodeFn>(p);
  }();
  return fn;
}

struct MapKey {
  const void* ptr;
  uint64_t d0, d1, d2, ld, s2, box;
  bool operator==(const MapKey& o) const {
    return ptr == o.ptr && d0 == o.d0 && d1 == o.d1 && d2 == o.d2 && ld == o.ld && s2 == o.s2 && box == o.box;
  }
};
struct MapKeyHash {
  size_t operator()(const MapKey& k) const {
    uint64_t h = reinterpret_cast<uint64_t>(k.ptr) * 0x9E3779B97F4A7C15ull;
    for (uint64_t v : {k.d0, k.d1, k.d2, k.ld, k.s2, k.box}) h = (h ^ v) * 0x9E3779B97F4A7C15ull + (h >> 29);
    return (size_t)h;
  }
};

// [d2 problems] x [d1 rows] x [d0 K-contiguous doubles], row stride ld, problem stride s2 (elements)
bool get_map(const double* ptr, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t ld, uint64_t s2, uint32_t box_rows,
             CUtensorMap* out) {
  static std::unordered_map<MapKey, CUtensorMap, MapKeyHash> cache;
  static std::mutex mu;
  const MapKey key{ptr, d0, d1, d2, ld, s2, box_rows};
  std::lock_guard<std::mutex> lock(mu);
  auto it = cache.find(key);
  if (it != cache.end()) { *out = it->second; return true; }
  EncodeFn enc = encode_fn();
  if (!enc) return false;
  if (cache.size() > 8192) cache.clear();
  const cuuint64_t dims[3] = {d0, d1, d2};
  const cuuint64_t strides[2] = {ld * sizeof(double), (d2 > 1 ? s2 : ld * d1) * sizeof(double)};
  const cuuint32_t box[3] = {TBK, box_rows, 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  CUtensorMap m;
  const CUresult r = enc(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, const_cast<double*>(ptr), dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return false;
  cache.emplace(key, m);
  *out = m;
  return true;
}

}  // namespace

// Returns 0 on launch, 1 when this GEMM is outside what the TMA kernel covers (caller falls back to the
// cp.async engine), negative on a launch error.
int gemm_tma_nt(const Ctx& ctx, const GemmArgs& g) {
  if (!g.b_kcont) return 1;
  if (g.M < 1 || g.N < 1) return 1;
  if (g.inner > 1 && !g.inner_steps) return 1;
  if ((g.sAo & 1) || (g.sBo & 1)) return 1;
  const int inner = g.inner;
  const uint64_t a_d0 = (uint64_t)(inner - 1) * g.iAc + g.K, a_d1 = (uint64_t)(inner - 1) * g.iAr + g.M;
  const uint64_t b_d0 = (uint64_t)(inner - 1) * g.iBc + g.K, b_d1 = (uint64_t)(inner - 1) * g.iBr + g.N;
  if (g.K < 1 || a_d0 > (uint64_t)g.lda || b_d0 > (uint64_t)g.ldb) return 1;
  CUtensorMap tmA, tmB;
  if (!get_map(g.A, a_d0, a_d1, g.outer, g.lda, g.sAo, TmaCfg::TBM, &tmA)) return 1;
  if (!get_map(g.B, b_d0, b_d1, g.outer, g.ldb, g.sBo, TmaCfg::TBN, &tmB)) return 1;
  const dim3 grid((g.N + TmaCfg::TBN - 1) / TmaCfg::TBN, (g.M + TmaCfg::TBM - 1) / TmaCfg::TBM, g.outer * g.inner);
  return launch_gemm<gemm_tma_nt_kernel>(ctx, g, grid, TmaCfg::THREADS, TmaCfg::SMEM, "gemm_tma", g.M, g.N, g.K, tmA, tmB,
                                         g);
}

}  // namespace gegp
