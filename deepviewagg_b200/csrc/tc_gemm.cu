// Hand-written tcgen05 projection GEMMs of the pool MLPs (E_mod / E_mix / E_main; reference
// core/common_modules/base_modules.py:42 `nn.Linear(bias=False)` over ALL views, pooling.py:239-261).
//
//   rows kernel  (forward and dX):  D[M, N] = X[M, K] . W[N, K]^T      M = views (millions), N, K <= 512
//   dw kernel    (weight gradient): D[N, K] = dZ[M, N]^T . X[M, K]      contraction over the M rows
//
// Precision: 3xTF32.  Every fp32 operand is split x = hi + lo with hi = tf32(x) and lo = tf32(x - hi)
// (both rounded to nearest here -- the tensor core itself would truncate, a biased error that grows
// linearly with K); the tensor cores accumulate lo.hi + hi.lo + hi.hi in fp32 (the dropped lo.lo term is
// 2^-22 relative): fp32-grade results (~1e-6 of the result's max at K = 128, measured against fp64) at
// three TF32 MMAs per product instead of nine BF16 ones.
//
// Shape of the rows kernel (HBM-bound for K, N <= 128: 4 (MK + MN) bytes against 6 K N flops per row):
//   * the OUTPUT is computed transposed: UMMA "A" (the M = 128 TMEM lanes) is the weight tile
//     [128 output columns, K], UMMA "B" (N = 128 TMEM columns) is a tile of 128 rows of X.  A thread of
//     the epilogue then owns one output COLUMN: a tcgen05.ld gives it that column's values for 32
//     consecutive rows, so (a) a warp-wide store of register j writes 32 consecutive floats of row j --
//     one fully coalesced 128-byte line per instruction, no shared-memory staging -- and (b) the
//     BatchNorm batch statistics of the layer (column sum and sum of squares, base_modules.py:44) are a
//     thread-local accumulation over registers, free of shuffles;
//   * warp roles (320 threads, 1 CTA / SM, persistent over row tiles): warp 0 = TMA producer (one lane),
//     warp 1 = MMA issuer (one lane; allocates TMEM), warps 2-5 = split warps (read the fp32 tile TMA
//     landed, write hi in place and lo next to it, same swizzled offsets), warps 6-9 = epilogue;
//   * shared memory: X tiles are [128 rows x 32 fp32] = 128-byte rows in the SWIZZLE_128B K-major
//     canonical layout (what TMA writes and UMMA reads); 3 stages of {X_hi, X_lo} (96 KB); the weight
//     (hi and lo, pre-split by a tiny prep kernel) stays resident for the whole kernel when K <= 128 and
//     N <= 128 (2 x 64 KB), else it is streamed per k-block next to X;
//   * TMEM: two 128-column fp32 accumulators (epilogue of tile i overlaps the MMAs of tile i + 1).
//
// SASS: UTMALDG (TMA loads), UTCHMMA (tcgen05.mma), LDTM (tcgen05.ld), UTCBAR (tcgen05.commit).
#include <cuda.h>

#include "dva_common.cuh"

namespace dva {
namespace tc {

constexpr int kTile = 128;                 // rows of X per tile (UMMA N) and output columns per tile (UMMA M)
constexpr int kBK = 32;                    // fp32 per k-block: one 128-byte swizzle row
constexpr int kTileBytes = kTile * kBK * 4;  // 16 KB
constexpr int kStages = 3;                 // stages of the streamed-weight rows kernel and of the dw kernel
constexpr int kStagesT = 6;                // stages of the rows kernel with the weight in tensor memory
constexpr int kThreads = 320;
constexpr int kSplitThreads = 128;
constexpr int kThreadsAll = kThreads + kSplitThreads;   // + a second set of split warps (warps 10-13)
constexpr uint32_t kTmemCols = 256;        // two 128-column accumulators
constexpr uint32_t kTmemColsW = 512;       // + weight hi at column 256, weight lo at column 384 (K <= 128 each)

// ---- PTX wrappers (tcgen05, TMA tensor copies; the generic async-copy ones are in dva_common.cuh) ----------
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
      ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar) : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// D[tmem] (+)= A[smem desc] . B[smem desc]^T, TF32 inputs, fp32 accumulate; issued by ONE thread
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// same with the A operand (the weight tile: 128 lanes x K tf32 columns) read from tensor memory
__device__ __forceinline__ void umma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, {%5, %5, %5, %5}, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(0u) : "memory");
}
// 32 registers per thread -> 32 TMEM lanes (this warp's quadrant) x 32 consecutive columns
__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]),
        "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]),
        "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// mbarrier arrive once every MMA issued so far by this thread has completed (implies fence::before_thread_sync)
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// 32 TMEM lanes (this warp's quadrant) x 32 consecutive fp32 columns -> 32 registers per thread
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// Shared-memory matrix descriptor, K-major operand in the SWIZZLE_128B canonical layout: rows of 128
// bytes, 8-row swizzle atoms of 1024 bytes (SBO), descriptor version 1 (sm_100), layout type 2.
__device__ __forceinline__ uint64_t smem_desc_k_sw128(uint32_t addr) {
  return (uint64_t)((addr >> 4) & 0x3fffu) | (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
// kind::tf32, fp32 accumulate, both operands K-major, M = N = 128
constexpr uint32_t kIdescTf32 = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(kTile >> 3) << 17) | ((uint32_t)(kTile >> 4) << 24);

__device__ __forceinline__ float tf32_rna(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

__device__ __forceinline__ float tf32_trunc(float x) { return __uint_as_float(__float_as_uint(x) & 0xffffe000u); }

// ---- weight preparation: W [N, K] (or its transpose) -> hi / lo, rows zero-padded to a multiple of 128 ----
// transpose = 0: Wp[n, k] = W[n * ldw + k]      (forward: output column n, reduction k)
// transpose = 1: Wp[n, k] = W[k * ldw + n]      (dX: output column n = input channel, reduction k = out channel)
__global__ void __launch_bounds__(256)
split_weight_kernel(const float* __restrict__ W, float* __restrict__ hi, float* __restrict__ lo, int n_out,
                    int n_pad, int k_red, int64_t ldw, int transpose) {
  const int64_t total = (int64_t)n_pad * k_red;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int n = (int)(t / k_red), k = (int)(t - (int64_t)n * k_red);
    float w = 0.f;
    if (n < n_out) w = transpose ? W[(int64_t)k * ldw + n] : W[(int64_t)n * ldw + k];
    const float h = tf32_rna(w);
    hi[t] = h;
    lo[t] = tf32_rna(w - h);     // rounded here: the tensor core would truncate (biased)
  }
}

// ---- rows kernel --------------------------------------------------------------------------------------------
struct RowsParams {
  const float *w_hi, *w_lo;   // split weight [n_pad, k_red] row-major (read directly by the WTMEM variant)
  int k_red;
  float* out;            // [M, n_out] row-major, leading dimension ldo
  float* col_stats;      // nullptr or [gridDim.x, 3, 128] per-CTA (sum (v - shift), sum (v - shift)^2, shift) per column
  int64_t M;
  int n_out, n_tiles, k_blocks, ldo;
  int64_t m_tiles;
  int rep_cols;          // 128, or 32 / 64: narrow layer with the weight replicated over the TMEM lane quadrants (below)
};

// Narrow layers (n_out <= 64, weight in tensor memory): with lane = output column, a 32-wide layer would leave the
// whole epilogue of a 128-row tile (4 tcgen05.ld, 128 row stores, the statistics) to the ONE warp that may read
// lane quadrant 0 -- ~1.2 us per tile, the kernel's pace.  The M = 128 MMA computes all 128 lanes anyway, so the
// weight rows are REPLICATED over the quadrants (lane l holds output column l % rep_cols) and quadrant j's warp
// stores rows [rep_cols * j', ...) of the tile: same tensor work, the epilogue spread over 4 (2) warps.
static inline int rows_rep_cols(int64_t n_out, int64_t k_red) {
  const bool resident = n_out <= kTile && k_red <= 4 * kBK;
  if (!resident || n_out > 64) return kTile;
  return n_out <= 32 ? 32 : 64;
}

// WTMEM = true : K <= 128 and one column tile: the weight (hi, lo) lives in TENSOR MEMORY for the whole kernel
//                (tcgen05.mma with the A operand from TMEM): shared memory only carries the X stages (6 x 32 KB)
//                and the tensor core's operand reads from shared memory are halved -- the N = 128 MMA at full
//                rate would otherwise eat the whole 128 B/clk of shared-memory bandwidth by itself;
// WTMEM = false: wider layers: weight k-blocks are streamed through shared memory next to X (3 x 64 KB).
template <bool WTMEM>
__global__ void __launch_bounds__(kThreadsAll, 1)
tc_rows_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_whi,
               const __grid_constant__ CUtensorMap map_wlo, const RowsParams p) {
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment: swizzle atoms are addressed relative to 1024-byte boundaries
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int KB = p.k_blocks;
  constexpr int NS = WTMEM ? kStagesT : kStages;
  // stage: X_hi, X_lo (, W_hi, W_lo); then the barriers
  constexpr uint32_t kStageBytes = (WTMEM ? 2u : 4u) * kTileBytes;
  uint8_t* st_base = smem;
  uint64_t* bars = reinterpret_cast<uint64_t*>(st_base + NS * kStageBytes);
  // barriers: full_tma[NS] full_cvt[NS] empty[NS] tmem_full[2] tmem_empty[2] w_full[1]; then the TMEM base word
  const uint32_t bar0 = smem_u32(bars);
  auto full_tma = [&](int s) { return bar0 + 8u * s; };
  auto full_cvt = [&](int s) { return bar0 + 8u * (NS + s); };
  auto empty = [&](int s) { return bar0 + 8u * (2 * NS + s); };
  auto tmem_full = [&](int a) { return bar0 + 8u * (3 * NS + a); };
  auto tmem_empty = [&](int a) { return bar0 + 8u * (3 * NS + 2 + a); };
  const uint32_t w_full = bar0 + 8u * (3 * NS + 4);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * NS + 5);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t tiles = p.m_tiles * p.n_tiles;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_x);
    if (!WTMEM) { tma_prefetch_desc(&map_whi); tma_prefetch_desc(&map_wlo); }
    for (int s = 0; s < NS; ++s) { mbar_init(full_tma(s), 1); mbar_init(full_cvt(s), kSplitThreads / 32); mbar_init(empty(s), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(tmem_full(a), 1); mbar_init(tmem_empty(a), 4); }
    mbar_init(w_full, 4);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(smem_u32(tmem_slot), WTMEM ? kTmemColsW : kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int s = 0; uint32_t ph = 0;
      for (int64_t t = blockIdx.x; t < tiles; t += gridDim.x) {
        const int64_t mt = t / p.n_tiles;
        const int nt = (int)(t - mt * p.n_tiles);
        for (int kb = 0; kb < KB; ++kb) {
          mbar_wait(empty(s), ph ^ 1u);
          uint8_t* st = st_base + (size_t)s * kStageBytes;
          mbar_expect_tx(full_tma(s), WTMEM ? kTileBytes : 3u * kTileBytes);
          tma_load_2d(smem_u32(st), &map_x, kb * kBK, (int)(mt * kTile), full_tma(s));
          if (!WTMEM) {
            tma_load_2d(smem_u32(st + 2 * kTileBytes), &map_whi, kb * kBK, nt * kTile, full_tma(s));
            tma_load_2d(smem_u32(st + 3 * kTileBytes), &map_wlo, kb * kBK, nt * kTile, full_tma(s));
          }
          if (++s == NS) { s = 0; ph ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      if (WTMEM) { mbar_wait(w_full, 0); tc_fence_after(); }
      int s = 0; uint32_t ph = 0; int acc = 0; uint32_t aph = 0;
      for (int64_t t = blockIdx.x; t < tiles; t += gridDim.x) {
        mbar_wait(tmem_empty(acc), aph ^ 1u);
        tc_fence_after();
        const uint32_t d = tmem_base + (uint32_t)acc * kTile;
        for (int kb = 0; kb < KB; ++kb) {
          mbar_wait(full_tma(s), ph);
          mbar_wait(full_cvt(s), ph);
          tc_fence_after();
          uint8_t* st = st_base + (size_t)s * kStageBytes;
          const uint64_t x_hi = smem_desc_k_sw128(smem_u32(st));
          const uint64_t x_lo = smem_desc_k_sw128(smem_u32(st + kTileBytes));
          if (WTMEM) {
            const uint32_t w_hi = tmem_base + 256u + (uint32_t)kb * kBK, w_lo = tmem_base + 384u + (uint32_t)kb * kBK;
#pragma unroll
            for (int k = 0; k < kBK / 8; ++k) {         // UMMA_K = 8 tf32: 8 TMEM columns of W, 32 bytes of X
              const uint64_t o = (uint64_t)(2 * k);
              umma_tf32_ts(d, w_lo + 8u * k, x_hi + o, kIdescTf32, (uint32_t)((kb | k) != 0));
              umma_tf32_ts(d, w_hi + 8u * k, x_lo + o, kIdescTf32, 1u);
              umma_tf32_ts(d, w_hi + 8u * k, x_hi + o, kIdescTf32, 1u);
            }
          } else {
            const uint64_t w_hi = smem_desc_k_sw128(smem_u32(st + 2 * kTileBytes));
            const uint64_t w_lo = smem_desc_k_sw128(smem_u32(st + 3 * kTileBytes));
#pragma unroll
            for (int k = 0; k < kBK / 8; ++k) {         // UMMA_K = 8 tf32 = 32 bytes: +2 in the 16-byte address field
              const uint64_t o = (uint64_t)(2 * k);
              umma_tf32(d, w_lo + o, x_hi + o, kIdescTf32, (uint32_t)((kb | k) != 0));
              umma_tf32(d, w_hi + o, x_lo + o, kIdescTf32, 1u);
              umma_tf32(d, w_hi + o, x_hi + o, kIdescTf32, 1u);
            }
          }
          umma_commit(empty(s));                         // stage reusable once these MMAs have read it
          if (kb == KB - 1) umma_commit(tmem_full(acc)); // accumulator complete
          if (++s == NS) { s = 0; ph ^= 1u; }
        }
        if (++acc == 2) { acc = 0; aph ^= 1u; }
      }
    }
  } else if (warp < 2 + kSplitThreads / 32 || warp >= kThreads / 32) {
    // ===================== split warps: X -> (hi in place, lo next to it) =====================
    // two sets of four warps (2-5 and 10-13) take the k-blocks alternately: the chain wait -> LDS -> split ->
    // STS -> proxy fence -> arrive of one block overlaps the next block's
    const int set = warp >= kThreads / 32 ? 1 : 0;
    const int tid = threadIdx.x - (set ? kThreads : 64);
    int s = 0; uint32_t ph = 0, cnt = 0;
    for (int64_t t = blockIdx.x; t < tiles; t += gridDim.x) {
      for (int kb = 0; kb < KB; ++kb, ++cnt) {
        if ((int)(cnt & 1u) != set) {
          if (++s == NS) { s = 0; ph ^= 1u; }
          continue;
        }
        mbar_wait(full_tma(s), ph);
        float4* hi = reinterpret_cast<float4*>(st_base + (size_t)s * kStageBytes);
        float4* lo = reinterpret_cast<float4*>(st_base + (size_t)s * kStageBytes + kTileBytes);
#pragma unroll
        for (int i = 0; i < kTileBytes / 16 / kSplitThreads; ++i) {
          const int e = i * kSplitThreads + tid;
          // hi is the landed fp32 tile itself: kind::tf32 reads the upper 19 bits of each word (truncation), so
          // lo = tf32(x - trunc(x)) completes the split exactly and the 16 KB hi write-back is saved
          const float4 v = hi[e];
          float4 l;
          l.x = tf32_rna(v.x - tf32_trunc(v.x)); l.y = tf32_rna(v.y - tf32_trunc(v.y));
          l.z = tf32_rna(v.z - tf32_trunc(v.z)); l.w = tf32_rna(v.w - tf32_trunc(v.w));
          lo[e] = l;
        }
        fence_proxy_async();                             // generic-proxy writes -> visible to the tensor core (async proxy)
        __syncwarp();
        if (lane == 0) mbar_arrive(full_cvt(s));
        if (++s == NS) { s = 0; ph ^= 1u; }
      }
    }
  } else {
    // ===================== epilogue: TMEM -> registers -> coalesced global stores =====================
    const int q = warp & 3;                              // TMEM lane quadrant this warp may access
    const int col = q * 32 + lane;                       // TMEM lane
    const int rep = WTMEM ? p.rep_cols : kTile;
    const int part = col / rep;                          // which slice of the tile's rows this lane stores
    const int src_col = col - part * rep;                // output column within the tile
    if (WTMEM) {
      // the weight tile into tensor memory: lane = output column (mod rep_cols), TMEM column = k (row-major prep
      // buffers [128, K], zero padded rows); 32 columns per tcgen05.st
      const float* whi = p.w_hi + (int64_t)src_col * p.k_red;
      const float* wlo = p.w_lo + (int64_t)src_col * p.k_red;
      for (int c0 = 0; c0 < KB * kBK; c0 += 32) {
        uint32_t rh[32], rl[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const bool ok = c0 + j < p.k_red;
          rh[j] = ok ? __float_as_uint(whi[c0 + j]) : 0u;
          rl[j] = ok ? __float_as_uint(wlo[c0 + j]) : 0u;
        }
        tmem_st_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + 256u + (uint32_t)c0, rh);
        tmem_st_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + 384u + (uint32_t)c0, rl);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(w_full);
    }
    // BatchNorm column statistics (single n tile only): sums of (v - shift) and (v - shift)^2, shifted by
    // the first value this thread sees (no catastrophic cancellation in the variance); every CTA has its
    // own shift, bn_stats_finalize_kernel recombines them in fp64
    float s1 = 0.f, s2 = 0.f, shift = 0.f;
    bool have_shift = false;
    int acc = 0; uint32_t aph = 0;
    for (int64_t t = blockIdx.x; t < tiles; t += gridDim.x) {
      const int64_t mt = t / p.n_tiles;
      const int nt = (int)(t - mt * p.n_tiles);
      const int n = nt * kTile + src_col;
      const bool col_ok = n < p.n_out;
      const bool warp_ok = rep < kTile || nt * kTile + q * 32 < p.n_out;
      mbar_wait(tmem_full(acc), aph);
      tc_fence_after();
      if (warp_ok) {
        const int64_t row0 = mt * kTile;
#pragma unroll 1
        for (int c0 = part * rep; c0 < (part + 1) * rep; c0 += 32) {
          if (row0 + c0 >= p.M) break;
          uint32_t r[32];
          tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * kTile + c0), r);
          float* o = p.out + (row0 + c0) * (int64_t)p.ldo + n;
          const int rows = (int)((p.M - row0 - c0) < 32 ? (p.M - row0 - c0) : 32);
          if (col_ok) {
            if (rows == 32) {
#pragma unroll
              for (int j = 0; j < 32; ++j) o[(int64_t)j * p.ldo] = __uint_as_float(r[j]);
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (j < rows) o[(int64_t)j * p.ldo] = __uint_as_float(r[j]);
            }
            if (p.col_stats != nullptr) {
              if (!have_shift) { shift = __uint_as_float(r[0]); have_shift = true; }
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                const float dv = __uint_as_float(r[j]) - shift;
                if (rows == 32 || j < rows) { s1 += dv; s2 = fmaf(dv, dv, s2); }
              }
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tmem_empty(acc));
      if (++acc == 2) { acc = 0; aph ^= 1u; }
    }
    if (p.col_stats != nullptr && p.n_tiles == 1) {
      p.col_stats[((int64_t)blockIdx.x * 3 + 0) * kTile + col] = s1;
      p.col_stats[((int64_t)blockIdx.x * 3 + 1) * kTile + col] = s2;
      p.col_stats[((int64_t)blockIdx.x * 3 + 2) * kTile + col] = shift;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, WTMEM ? kTmemColsW : kTmemCols);
  }
}

// ---- dw kernel: D[n_out, k_in] = sum over rows v of dZ[v, n_out] * X[v, k_in] --------------------------------
// Both operands are "MN-major" for the tensor core: the contraction index v is the SLOW dimension of the
// row-major [V, C] matrices.  For 32-bit (tf32) MN-major operands the only swizzled shared-memory layout
// the tensor core reads is SWIZZLE_128B with 32-byte atoms (descriptor layout type 1; TMA mode
// CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B): rows of 128 bytes whose 32-byte chunks are XOR-ed with (row % 4),
// swizzle atoms of 4 rows = 512 bytes.  A TMA box of [32 rows x 32 columns] lands as 32 such rows; the
// canonical layout strings boxes together: LBO = distance between two 32-column groups (one box each,
// 4096 bytes), SBO = distance between two 4-row atoms (512 bytes); one tcgen05.mma consumes 8 rows
// (UMMA_K = 8 tf32), i.e. two atoms = 1024 bytes per group.
// One CTA = one (128 x 128 output tile, slice of the rows): it accumulates its slice in TMEM and writes a
// partial tile; dw_reduce_kernel adds the slices in a fixed order (deterministic, no atomics).
constexpr int kDwRows = 32;                      // contraction rows per stage
constexpr int kGroupBytes = kDwRows * 128;       // one [32 x 32] box
constexpr int kDwMaxStages = 6;                  // tensor memory: 128 accumulator columns + 64 per stage <= 512
constexpr size_t kDwSmemBudget = 200 * 1024;
constexpr uint32_t kDwTmemCols = 512;            // accumulator [0,128) + per stage dZ_hi | dZ_lo (32 + 32 columns)
constexpr int kDwThreads = kThreadsAll;            // the second set of split warps (10-13) takes the odd row blocks

__device__ __forceinline__ uint64_t smem_desc_mn_sw128(uint32_t addr) {
  return (uint64_t)((addr >> 4) & 0x3fffu) | ((uint64_t)(kGroupBytes >> 4) << 16) | ((uint64_t)(512 >> 4) << 32) |
         (1ull << 46) | (1ull << 61);
}
// A (dZ^T) from tensor memory: K-major by construction; B (X) MN-major in shared memory
constexpr uint32_t kIdescTf32TsMN = kIdescTf32 | (1u << 16);

struct DwParams {
  float* partial;        // [splits, n_pad, k_pad]
  int64_t V, blocks_total, blocks_per_split;
  int n_out, k_in, n_pad, k_pad, k_tiles, splits;
  int stages;            // 4 .. kDwMaxStages: as many as shared memory (compact stages) and tensor memory (64 columns each) hold
  uint32_t a_bytes, b_bytes;   // per stage: dZ boxes (4 KB per 32 output rows), X boxes (4 KB per 32 columns; hi and lo each)
};

// The dZ operand never goes back to shared memory: split warp g (TMEM lane quadrant g = output rows 32 g ..)
// reads column n = 32 g + lane of the landed [32 x 128] tile row by row (a warp-wide LDS of one 128-byte row:
// conflict-free whatever the swizzle), splits it and stores hi / lo TRANSPOSED into tensor memory with one
// tcgen05.st each -- lane = output row, 32 columns = the 32 contraction rows of the stage.  The tensor core
// then reads A from TMEM and only X from shared memory: 144 KB instead of 224 KB of shared-memory traffic
// per 32 KB of HBM traffic (the all-shared-memory version was bound by the 128 B/clk of shared memory).
__global__ void __launch_bounds__(kDwThreads, 1)
tc_dw_kernel(const __grid_constant__ CUtensorMap map_dz, const __grid_constant__ CUtensorMap map_x, const DwParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  // The per-stage chain TMA -> split -> MMA -> empty is ~3 us long whatever the width, so the stage count sets the
  // pace (0.84 us per 32 rows with 4): narrow layers pack their stages (only the boxes they use) and get up to 6.
  const int NS = p.stages;
  const uint32_t kStageBytes = p.a_bytes + 2u * p.b_bytes;    // dZ (raw), X_hi, X_lo
  const uint32_t x_hi_off = p.a_bytes, x_lo_off = p.a_bytes + p.b_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)NS * kStageBytes);
  const uint32_t bar0 = smem_u32(bars);
  auto full_tma = [&](int s) { return bar0 + 8u * s; };
  auto full_cvt = [&](int s) { return bar0 + 8u * (NS + s); };
  auto empty = [&](int s) { return bar0 + 8u * (2 * NS + s); };
  const uint32_t tmem_full = bar0 + 8u * (3 * NS);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * NS + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int split = blockIdx.x % p.splits, tile = blockIdx.x / p.splits;
  const int nt = tile / p.k_tiles, kt = tile - nt * p.k_tiles;
  const int64_t b0 = (int64_t)split * p.blocks_per_split;
  int64_t b1 = b0 + p.blocks_per_split;
  if (b1 > p.blocks_total) b1 = p.blocks_total;
  const int64_t nblk = b1 > b0 ? b1 - b0 : 0;
  int a_groups = (p.n_out - nt * kTile + 31) / 32; if (a_groups > 4) a_groups = 4;
  int b_groups = (p.k_in - kt * kTile + 31) / 32; if (b_groups > 4) b_groups = 4;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_dz); tma_prefetch_desc(&map_x);
    for (int s = 0; s < NS; ++s) { mbar_init(full_tma(s), 1); mbar_init(full_cvt(s), kSplitThreads / 32); mbar_init(empty(s), 1); }
    mbar_init(tmem_full, 1);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(smem_u32(tmem_slot), kDwTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      int s = 0; uint32_t ph = 0;
      for (int64_t b = 0; b < nblk; ++b) {
        mbar_wait(empty(s), ph ^ 1u);
        uint8_t* st = smem + (size_t)s * kStageBytes;
        mbar_expect_tx(full_tma(s), (uint32_t)(a_groups + b_groups) * kGroupBytes);
        const int row = (int)((b0 + b) * kDwRows);
        for (int g = 0; g < a_groups; ++g)
          tma_load_2d(smem_u32(st + g * kGroupBytes), &map_dz, nt * kTile + g * 32, row, full_tma(s));
        for (int g = 0; g < b_groups; ++g)
          tma_load_2d(smem_u32(st + x_hi_off + g * kGroupBytes), &map_x, kt * kTile + g * 32, row, full_tma(s));
        if (++s == NS) { s = 0; ph ^= 1u; }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      int s = 0; uint32_t ph = 0;
      for (int64_t b = 0; b < nblk; ++b) {
        mbar_wait(full_tma(s), ph);
        mbar_wait(full_cvt(s), ph);
        tc_fence_after();
        uint8_t* st = smem + (size_t)s * kStageBytes;
        const uint32_t a_hi = tmem_base + 128u + (uint32_t)s * 64u, a_lo = a_hi + 32u;
        const uint64_t x_hi = smem_desc_mn_sw128(smem_u32(st + x_hi_off));
        const uint64_t x_lo = smem_desc_mn_sw128(smem_u32(st + x_lo_off));
        // UMMA N = the X columns this tile really has (32 per box): packed stages hold no more than that
        const uint32_t idesc = (kIdescTf32TsMN & ~(0x3fu << 17)) | ((uint32_t)(b_groups * 32 >> 3) << 17);
#pragma unroll
        for (int k = 0; k < kDwRows / 8; ++k) {          // 8 contraction rows: 8 TMEM columns of dZ^T, two 512-byte atoms of X
          const uint64_t o = (uint64_t)(k * (1024 >> 4));
          umma_tf32_ts(tmem_base, a_lo + 8u * k, x_hi + o, idesc, (uint32_t)((b | k) != 0));
          umma_tf32_ts(tmem_base, a_hi + 8u * k, x_lo + o, idesc, 1u);
          umma_tf32_ts(tmem_base, a_hi + 8u * k, x_hi + o, idesc, 1u);
        }
        umma_commit(empty(s));
        if (b == nblk - 1) umma_commit(tmem_full);
        if (++s == NS) { s = 0; ph ^= 1u; }
      }
    }
  } else if (warp < 2 + kSplitThreads / 32 || warp >= kThreads / 32) {
    // Two sets of four split warps take the row blocks alternately (set 0 = warps 2-5: even blocks, set 1 = warps
    // 10-13: odd ones): the chain wait -> 32 LDS -> split -> tcgen05.st -> wait::st -> X split -> fence -> arrive
    // of one block overlaps the next block's (8 M x 128 x 128: 1.77 -> 1.54 ms).
    const int set = warp >= kThreads / 32 ? 1 : 0;
    const int tid = threadIdx.x - (set ? kThreads : 64);
    const int g = warp & 3;                              // TMEM lane quadrant = dZ column group of this warp
    int s = 0; uint32_t ph = 0;
    for (int64_t b = 0; b < nblk; ++b) {
      if ((int)(b & 1) != set) {
        if (++s == NS) { s = 0; ph ^= 1u; }
        continue;
      }
      mbar_wait(full_tma(s), ph);
      uint8_t* st = smem + (size_t)s * kStageBytes;
      if (g < a_groups) {
        // dZ column n = 32 g + lane over the 32 rows of the stage -> TMEM (hi, lo); 128B / 32-byte-atom swizzle:
        // the 32-byte chunk index is XOR-ed with (row & 3)
        const uint8_t* grp = st + g * kGroupBytes + (lane & 7) * 4;
        uint32_t rh[32], rl[32];
#pragma unroll
        for (int v = 0; v < 32; ++v) {
          const float x = *reinterpret_cast<const float*>(grp + v * 128 + ((((lane >> 3) ^ (v & 3)) & 3) << 5));
          const float h = tf32_rna(x);
          rh[v] = __float_as_uint(h);
          rl[v] = __float_as_uint(tf32_rna(x - h));
        }
        const uint32_t ta = tmem_base + ((uint32_t)(g * 32) << 16) + 128u + (uint32_t)s * 64u;
        tmem_st_32x32(ta, rh);
        tmem_st_32x32(ta + 32u, rl);
        tmem_st_wait();
      }
      {
        float4* hi = reinterpret_cast<float4*>(st + x_hi_off);
        float4* lo = reinterpret_cast<float4*>(st + x_lo_off);
        for (int i = 0; i < b_groups * (kGroupBytes / 16) / kSplitThreads; ++i) {
          const int e = i * kSplitThreads + tid;
          // hi is the landed fp32 tile itself: kind::tf32 reads the upper 19 bits of each word (truncation), so
          // lo = tf32(x - trunc(x)) completes the split exactly and the 16 KB hi write-back is saved
          const float4 v = hi[e];
          float4 l;
          l.x = tf32_rna(v.x - tf32_trunc(v.x)); l.y = tf32_rna(v.y - tf32_trunc(v.y));
          l.z = tf32_rna(v.z - tf32_trunc(v.z)); l.w = tf32_rna(v.w - tf32_trunc(v.w));
          lo[e] = l;
        }
      }
      fence_proxy_async();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(full_cvt(s));
      if (++s == NS) { s = 0; ph ^= 1u; }
    }
  } else {
    // epilogue: lane = output row (n_out index), 32 consecutive k_in columns per tcgen05.ld
    const int q = warp & 3;
    const int m = nt * kTile + q * 32 + lane;
    float* dst = p.partial + ((int64_t)split * p.n_pad + m) * p.k_pad + kt * kTile;
    if (nblk > 0) {
      mbar_wait(tmem_full, 0);
      tc_fence_after();
    }
#pragma unroll 1
    for (int c0 = 0; c0 < kTile; c0 += 32) {
      uint32_t r[32];
      if (nblk > 0) {
        tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, r);
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) r[j] = 0u;
      }
#pragma unroll
      for (int j = 0; j < 32; j += 4)
        *reinterpret_cast<uint4*>(dst + c0 + j) = make_uint4(r[j], r[j + 1], r[j + 2], r[j + 3]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kDwTmemCols);
  }
}

__global__ void __launch_bounds__(256)
dw_reduce_kernel(const float* __restrict__ partial, float* __restrict__ out, int n_out, int k_in, int n_pad,
                 int k_pad, int splits, int64_t ldo) {
  const int64_t total = (int64_t)n_out * k_in;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int n = (int)(t / k_in), k = (int)(t - (int64_t)n * k_in);
    float acc = 0.f;
    for (int s = 0; s < splits; ++s) acc += partial[((int64_t)s * n_pad + n) * k_pad + k];   // fixed order
    out[(int64_t)n * ldo + k] = acc;
  }
}

// ---- BatchNorm statistics from the rows kernel's per-CTA partials (base_modules.py:44, nn.BatchNorm1d) ------
// One warp per column; lanes stride over the CTAs in a fixed order, fp64 combine:
//   sum_b = s_b + n_b sh_b,   sumsq_b = q_b + 2 sh_b s_b + n_b sh_b^2,   n_b = rows CTA b processed.
__global__ void __launch_bounds__(128)
bn_stats_finalize_kernel(const float* __restrict__ col_stats, int ctas, int64_t M, int64_t m_tiles, int C, int rep,
                         float eps, float momentum, float* __restrict__ mean, float* __restrict__ invstd,
                         float* __restrict__ running_mean, float* __restrict__ running_var) {
  const int lane = threadIdx.x & 31;
  const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (c >= C) return;
  double S = 0.0, Q = 0.0;
  const int parts = kTile / rep;                       // slot part * rep + c: column c over rows [part * rep, + rep) of each tile
  const int64_t rem = M - (m_tiles - 1) * kTile;       // rows of the globally last tile
  for (int e = lane; e < ctas * parts; e += 32) {
    const int b = e / parts, part = e - b * parts;
    // tiles b, b + ctas, ...: all full except possibly the globally last one
    const int64_t nt = b < m_tiles ? (m_tiles - 1 - b) / ctas + 1 : 0;
    int64_t nb = nt * rep;
    if (nt > 0 && b + (nt - 1) * ctas == m_tiles - 1) {
      int64_t last = rem - (int64_t)part * rep;
      last = last < 0 ? 0 : (last > rep ? rep : last);
      nb += last - rep;
    }
    const int slot = part * rep + c;
    const double s = (double)col_stats[((int64_t)b * 3 + 0) * kTile + slot];
    const double q = (double)col_stats[((int64_t)b * 3 + 1) * kTile + slot];
    const double sh = (double)col_stats[((int64_t)b * 3 + 2) * kTile + slot];
    S += s + (double)nb * sh;
    Q += q + 2.0 * sh * s + (double)nb * sh * sh;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { S += __shfl_xor_sync(0xffffffffu, S, o); Q += __shfl_xor_sync(0xffffffffu, Q, o); }
  if (lane != 0) return;
  const double n = (double)M, mu = S / n;
  double var = Q / n - mu * mu;
  if (var < 0.0) var = 0.0;
  mean[c] = (float)mu;
  invstd[c] = (float)(1.0 / sqrt(var + (double)eps));
  if (running_mean != nullptr) {
    const double unbiased = M > 1 ? var * n / (n - 1.0) : var;
    running_mean[c] = (float)((1.0 - momentum) * running_mean[c] + momentum * mu);
    running_var[c] = (float)((1.0 - momentum) * running_var[c] + momentum * unbiased);
  }
}

// ---- host side ---------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      f = nullptr;
    return (EncodeTiledFn)f;
  }();
  return fn;
}

// 2-D fp32 tensor [rows, cols] with leading dimension ld (elements); box = [box_rows x 32 columns], 128B swizzle
static int make_map(CUtensorMap* m, const float* base, int64_t rows, int64_t cols, int64_t ld, int box_rows,
                    CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(DVA_EUNSUPPORTED, "tc_gemm: cuTensorMapEncodeTiled not available from the driver");
  const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
  const cuuint32_t box[2] = {(cuuint32_t)kBK, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return failf(DVA_EINVAL, "tc_gemm: cuTensorMapEncodeTiled failed (%d)", (int)r);
  return DVA_OK;
}

static inline int n_pad_of(int64_t n_out) { return (int)((n_out + kTile - 1) / kTile) * kTile; }

}  // namespace tc
}  // namespace dva

using namespace dva;

// workspace of the rows kernel: split weight (hi | lo), rows padded to a multiple of 128
extern "C" size_t dva_tc_rows_workspace_bytes(int64_t n_out, int64_t k_red) {
  return (size_t)2 * tc::n_pad_of(n_out) * (size_t)k_red * 4 + 256;
}

extern "C" int dva_tc_rows_supported(int64_t M, int64_t n_out, int64_t k_red) {
  return M >= 1 && n_out >= 1 && k_red >= 4 && k_red % 4 == 0 && n_out <= 65536 && k_red <= 65536 && M < (1ll << 40);
}

// D[M, n_out] = X[M, k_red] . Wp^T with Wp[n, k] = transpose ? W[k, n] : W[n, k]   (W row-major, leading dimension ldw)
// col_stats: nullptr, or [148, 3, 128] floats receiving the per-CTA shifted column statistics of D (n_out <= 128)
extern "C" int dva_tc_rows_gemm(const float* X, const float* W, float* D, int64_t M, int64_t n_out, int64_t k_red,
                                int64_t ldx, int64_t ldw, int64_t ldo, int transpose_w, float* col_stats,
                                int* stats_ctas, void* workspace, size_t workspace_bytes, void* stream) {
  if (M == 0) return DVA_OK;
  if (!dva_tc_rows_supported(M, n_out, k_red)) return fail(DVA_EUNSUPPORTED, "tc_rows_gemm: unsupported shape");
  if (!X || !W || !D || !workspace) return fail(DVA_EINVAL, "tc_rows_gemm: null pointer");
  if (!aligned16(X) || !aligned16(workspace) || ldx % 4 != 0) return fail(DVA_EALIGN, "tc_rows_gemm: X rows must be 16-byte aligned");
  if (workspace_bytes < dva_tc_rows_workspace_bytes(n_out, k_red)) return fail(DVA_EINVAL, "tc_rows_gemm: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  const int n_pad = tc::n_pad_of(n_out);
  float* whi = reinterpret_cast<float*>(workspace);
  float* wlo = whi + (size_t)n_pad * k_red;
  {
    const int64_t total = (int64_t)n_pad * k_red;
    const int grid = (int)((total + 255) / 256 > 592 ? 592 : (total + 255) / 256);
    tc::split_weight_kernel<<<grid, 256, 0, st>>>(W, whi, wlo, (int)n_out, n_pad, (int)k_red, ldw, transpose_w);
    int rc = check_launch("split_weight");
    if (rc) return rc;
  }
  CUtensorMap mx, mh, ml;
  int rc = tc::make_map(&mx, X, M, k_red, ldx, tc::kTile);
  if (rc) return rc;
  rc = tc::make_map(&mh, whi, n_pad, k_red, k_red, tc::kTile);
  if (rc) return rc;
  rc = tc::make_map(&ml, wlo, n_pad, k_red, k_red, tc::kTile);
  if (rc) return rc;
  tc::RowsParams p;
  p.w_hi = whi; p.w_lo = wlo; p.k_red = (int)k_red;
  p.out = D; p.col_stats = col_stats; p.M = M; p.n_out = (int)n_out; p.n_tiles = n_pad / tc::kTile;
  p.k_blocks = (int)((k_red + tc::kBK - 1) / tc::kBK); p.ldo = (int)ldo; p.m_tiles = (M + tc::kTile - 1) / tc::kTile;
  const bool resident = p.n_tiles == 1 && p.k_blocks <= 4;
  p.rep_cols = tc::rows_rep_cols(n_out, k_red);
  if (col_stats && p.n_tiles != 1) return fail(DVA_EUNSUPPORTED, "tc_rows_gemm: column statistics need n_out <= 128");
  const int64_t tiles = p.m_tiles * p.n_tiles;
  const int grid = (int)(tiles < kNumSMs ? tiles : kNumSMs);
  if (stats_ctas) *stats_ctas = grid;
  const size_t smem = 1024 + (resident ? (size_t)tc::kStagesT * 2 : (size_t)tc::kStages * 4) * tc::kTileBytes + 256;
  cudaError_t e;
  if (resident) {
    e = cudaFuncSetAttribute(tc::tc_rows_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail((int)e, "tc_rows_gemm: cannot reserve shared memory");
    tc::tc_rows_kernel<true><<<grid, tc::kThreadsAll, smem, st>>>(mx, mh, ml, p);
  } else {
    e = cudaFuncSetAttribute(tc::tc_rows_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail((int)e, "tc_rows_gemm: cannot reserve shared memory");
    tc::tc_rows_kernel<false><<<grid, tc::kThreadsAll, smem, st>>>(mx, mh, ml, p);
  }
  return check_launch("tc_rows_gemm");
}

// ---- dW -------------------------------------------------------------------------------------------------------
static void dw_plan(int64_t V, int64_t n_out, int64_t k_in, int* n_tiles, int* k_tiles, int* splits, int64_t* bps,
                    int64_t* blocks) {
  *n_tiles = (int)((n_out + tc::kTile - 1) / tc::kTile);
  *k_tiles = (int)((k_in + tc::kTile - 1) / tc::kTile);
  *blocks = (V + tc::kDwRows - 1) / tc::kDwRows;
  int sp = kNumSMs / (*n_tiles * *k_tiles);
  if (sp < 1) sp = 1;
  if ((int64_t)sp > *blocks) sp = (int)(*blocks < 1 ? 1 : *blocks);
  *splits = sp;
  *bps = (*blocks + sp - 1) / sp;
}

extern "C" size_t dva_tc_dw_workspace_bytes(int64_t V, int64_t n_out, int64_t k_in) {
  int nt, kt, sp; int64_t bps, blocks;
  dw_plan(V, n_out, k_in, &nt, &kt, &sp, &bps, &blocks);
  return (size_t)sp * nt * tc::kTile * (size_t)kt * tc::kTile * 4 + 256;
}

// D[n_out, k_in] = dZ[V, n_out]^T . X[V, k_in]   (row-major, leading dimensions ldz / ldx / ldo)
extern "C" int dva_tc_dw_gemm(const float* dZ, const float* X, float* D, int64_t V, int64_t n_out, int64_t k_in,
                              int64_t ldz, int64_t ldx, int64_t ldo, void* workspace, size_t workspace_bytes,
                              void* stream) {
  if (n_out < 1 || k_in < 1 || V < 0 || n_out > 65536 || k_in > 65536) return fail(DVA_EUNSUPPORTED, "tc_dw_gemm: unsupported shape");
  if (!D || (V > 0 && (!dZ || !X)) || !workspace) return fail(DVA_EINVAL, "tc_dw_gemm: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (V == 0) {
    for (int64_t n = 0; n < n_out; ++n) {
      cudaError_t e = cudaMemsetAsync(D + n * ldo, 0, (size_t)k_in * 4, st);
      if (e != cudaSuccess) return fail((int)e, "tc_dw_gemm: memset failed");
    }
    return DVA_OK;
  }
  if (!aligned16(dZ) || !aligned16(X) || !aligned16(workspace) || ldz % 4 != 0 || ldx % 4 != 0)
    return fail(DVA_EALIGN, "tc_dw_gemm: operand rows must be 16-byte aligned");
  if (workspace_bytes < dva_tc_dw_workspace_bytes(V, n_out, k_in)) return fail(DVA_EINVAL, "tc_dw_gemm: workspace too small");
  tc::DwParams p;
  int nt, kt, sp; int64_t bps, blocks;
  dw_plan(V, n_out, k_in, &nt, &kt, &sp, &bps, &blocks);
  p.partial = reinterpret_cast<float*>(workspace);
  p.V = V; p.blocks_total = blocks; p.blocks_per_split = bps; p.n_out = (int)n_out; p.k_in = (int)k_in;
  p.n_pad = nt * tc::kTile; p.k_pad = kt * tc::kTile; p.k_tiles = kt; p.splits = sp;
  CUtensorMap mz, mx;
  int rc = tc::make_map(&mz, dZ, V, n_out, ldz, tc::kDwRows, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B);
  if (rc) return rc;
  rc = tc::make_map(&mx, X, V, k_in, ldx, tc::kDwRows, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B);
  if (rc) return rc;
  const int ag = (int)(n_out >= tc::kTile ? 4 : (n_out + 31) / 32), bg = (int)(k_in >= tc::kTile ? 4 : (k_in + 31) / 32);
  p.a_bytes = (uint32_t)ag * tc::kGroupBytes; p.b_bytes = (uint32_t)bg * tc::kGroupBytes;
  const size_t stage_bytes = p.a_bytes + 2 * (size_t)p.b_bytes;
  p.stages = (int)(tc::kDwSmemBudget / stage_bytes);
  if (p.stages > tc::kDwMaxStages) p.stages = tc::kDwMaxStages;
  const size_t smem = 1024 + (size_t)p.stages * stage_bytes + 256;
  cudaError_t e = cudaFuncSetAttribute(tc::tc_dw_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return fail((int)e, "tc_dw_gemm: cannot reserve shared memory");
  tc::tc_dw_kernel<<<nt * kt * sp, tc::kDwThreads, smem, st>>>(mz, mx, p);
  rc = check_launch("tc_dw_gemm");
  if (rc) return rc;
  const int64_t total = n_out * k_in;
  tc::dw_reduce_kernel<<<(int)((total + 255) / 256 > 1184 ? 1184 : (total + 255) / 256), 256, 0, st>>>(
      p.partial, D, (int)n_out, (int)k_in, p.n_pad, p.k_pad, sp, ldo);
  return check_launch("tc_dw_reduce");
}

// Forward of one MLP layer's Linear with the BatchNorm batch statistics taken in the GEMM epilogue:
// D = X . W^T and mean / invstd (+ momentum update of the running buffers) of D's columns, without the
// separate statistics pass over D.  n_out <= 128 (one column tile) and not a skinny shape.
extern "C" size_t dva_linear_bnstats_workspace_bytes(int64_t n_out, int64_t k_red) {
  return dva_tc_rows_workspace_bytes(n_out, k_red) + (size_t)kNumSMs * 3 * tc::kTile * 4;
}

extern "C" int dva_linear_bnstats_supported(int64_t M, int64_t n_out, int64_t k_red) {
  return dva_tc_rows_supported(M, n_out, k_red) && n_out <= tc::kTile && n_out % 4 == 0 && n_out >= 32 && k_red >= 8;
}

extern "C" int dva_linear_bnstats_fwd(const float* X, const float* W, float* D, int64_t M, int64_t n_out,
                                      int64_t k_red, float eps, float momentum, float* mean, float* invstd,
                                      float* running_mean, float* running_var, void* workspace,
                                      size_t workspace_bytes, void* stream) {
  if (!dva_linear_bnstats_supported(M, n_out, k_red)) return fail(DVA_EUNSUPPORTED, "linear_bnstats_fwd: unsupported shape");
  if (!mean || !invstd) return fail(DVA_EINVAL, "linear_bnstats_fwd: null pointer");
  if (workspace_bytes < dva_linear_bnstats_workspace_bytes(n_out, k_red)) return fail(DVA_EINVAL, "linear_bnstats_fwd: workspace too small");
  const size_t wbytes = dva_tc_rows_workspace_bytes(n_out, k_red);
  float* stats = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(workspace) + wbytes);
  int ctas = 0;
  int rc = dva_tc_rows_gemm(X, W, D, M, n_out, k_red, k_red, k_red, n_out, 0, stats, &ctas, workspace, wbytes, stream);
  if (rc) return rc;
  tc::bn_stats_finalize_kernel<<<(int)((n_out + 3) / 4), 128, 0, (cudaStream_t)stream>>>(
      stats, ctas, M, (M + tc::kTile - 1) / tc::kTile, (int)n_out, tc::rows_rep_cols(n_out, k_red), eps, momentum, mean,
      invstd, running_mean, running_var);
  return check_launch("bn_stats_finalize");
}
