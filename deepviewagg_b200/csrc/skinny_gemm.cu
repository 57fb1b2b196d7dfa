// Skinny projections of the pool MLPs (base_modules.py:42 -- Linear(bias=False) inside every MLP
// layer of DeepSetFeat / E_mod / E_mix, pooling.py:239-261, 645-656): [rows, K] x [N, K]^T with
// K, N <= 64 and millions of rows (one per view).  linear_api.cu sends here the shapes the tcgen05
// kernels of tc_gemm.cu do not take: odd widths, K < 8 or N < 32, and dW unless both widths exceed 32.
// 3xTF32 split operands on mma.sync (fp32-grade accuracy), weights resident in shared memory, every
// global access a coalesced 16-byte vector through a shared staging tile:
//   layouts 0/1  skinny_rows_mma_kernel : D[M,OUT] = A[M,RED] . Wt[RED,OUT]
//   layout  2    skinny_dw_mma_kernel   : D[N,K]   = A[M,N]^T . B[M,K]   (the rows are the MMA k
//                dimension; per-CTA partials reduced in a fixed order by skinny_dw_reduce_cols_kernel)
#include "dva_common.cuh"

namespace dva {

constexpr int kSkTile = 128;       // rows per CTA tile
constexpr int kSkMax = 64;         // largest K / N served here

// rows [row0, row0 + kSkTile) x cols of a row-major [M, cols] matrix -> dst[r * dst_stride + c];
// rows past M become zero.  vec: 16-byte cp.async (LDGSTS) -- every copy of the tile is in flight
// at once and no register waits on it; the caller commits / waits.  Otherwise plain scalar loads.
__device__ __forceinline__ void sk_load_tile(float* __restrict__ dst, int dst_stride, const float* __restrict__ src,
                                             int64_t row0, int64_t M, int cols, bool vec) {
  const int nthreads = blockDim.x;
  if (vec) {
    const int c4 = cols >> 2;
    const uint32_t d0 = smem_u32(dst);
    if (nthreads % c4 == 0) {                        // the usual case: a thread keeps its column, rows advance by a constant
      const int c = ((int)threadIdx.x % c4) << 2, rstep = nthreads / c4;
      for (int r = threadIdx.x / c4; r < kSkTile; r += rstep) {
        const bool in = row0 + r < M;
        const float* g = src + (in ? (row0 + r) * cols + c : 0);
        const int bytes = in ? 16 : 0;               // src-size 0: the 16 destination bytes are zero-filled
        cp_async16_zfill(d0 + (uint32_t)(r * dst_stride + c) * 4, g, bytes);
      }
    } else {
      for (int e = threadIdx.x; e < kSkTile * c4; e += nthreads) {
        const int r = e / c4, c = (e - r * c4) << 2;
        const bool in = row0 + r < M;
        const float* g = src + (in ? (row0 + r) * cols + c : 0);
        const int bytes = in ? 16 : 0;
        cp_async16_zfill(d0 + (uint32_t)(r * dst_stride + c) * 4, g, bytes);
      }
    }
  } else {
    for (int e = threadIdx.x; e < kSkTile * cols; e += nthreads) {
      const int r = e / cols, c = e - r * cols;
      dst[r * dst_stride + c] = (row0 + r < M) ? __ldg(src + (row0 + r) * cols + c) : 0.f;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Rows kernel: 3xTF32 (a = a_hi + a_lo, w = w_hi + w_lo in TF32; a.w ~ a_lo.w_hi + a_hi.w_lo +
// a_hi.w_hi accumulated in fp32 -> fp32-grade accuracy) on mma.sync.m16n8k8.  4 warps per CTA, a
// warp owns 32 rows x all columns of the 128-row tile: per k-step of 8 it loads 8 A values per lane
// (bank-conflict-free: tile stride = 4 mod 8 words), splits them, and issues 6 MMAs per 8-column
// block.  ~3.8x fewer instructions than the same tiles on FFMA, which ran at the fp32-pipe limit
// (61-72 % issue slots, 60-70 % of them FFMA).
// ---------------------------------------------------------------------------------------------
template <bool TRANS, int NT /* 8-column blocks: OUT <= 8 * NT */>
__global__ void __launch_bounds__(128)
skinny_rows_mma_kernel(const float* __restrict__ A, const float* __restrict__ W, float* __restrict__ D,
                       int64_t M, int RED, int OUT, int avec, int dvec) {
  extern __shared__ __align__(16) float sk_smem[];
  const int RED8 = (RED + 7) & ~7;
  const int REDP = RED8 + 4;                        // A tile stride: fragment loads hit 32 distinct banks
  constexpr int WS = ((NT * 8 + 31) / 32) * 32 + 8;  // weight / output tile stride (= 8 mod 32)
  uint32_t* wHi = reinterpret_cast<uint32_t*>(sk_smem);          // [RED8][WS]
  uint32_t* wLo = wHi + RED8 * WS;
  float* tbuf = reinterpret_cast<float*>(wLo + RED8 * WS);         // 2 x (A tile [kSkTile][REDP], then output tile [kSkTile][WS])
  const int tile_floats = kSkTile * (REDP > WS ? REDP : WS);
  for (int e = threadIdx.x; e < RED8 * WS; e += blockDim.x) {
    const int k = e / WS, n = e - k * WS;
    float v = 0.f;
    if (k < RED && n < OUT) v = TRANS ? __ldg(W + (int64_t)n * RED + k) : __ldg(W + (int64_t)k * OUT + n);
    const uint32_t hi = to_tf32(v);
    wHi[e] = hi;
    wLo[e] = to_tf32(v - __uint_as_float(hi));
  }
  for (int e = threadIdx.x; e < 2 * tile_floats; e += blockDim.x) tbuf[e] = 0.f;   // padding columns stay zero
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, tq = lane & 3;
  const int64_t tiles = (M + kSkTile - 1) / kSkTile;
  if (blockIdx.x < tiles) sk_load_tile(tbuf, REDP, A, (int64_t)blockIdx.x * kSkTile, M, RED, avec != 0);
  cp_async_commit();
  int cur = 0;
  for (int64_t t = blockIdx.x; t < tiles; t += gridDim.x, cur ^= 1) {
    const int64_t row0 = t * kSkTile;
    float* tS = tbuf + cur * tile_floats;
    float* oS = tS;                                  // the output tile replaces the A tile once it is consumed
    __syncthreads();                                 // the other buffer's output has been stored
    if (t + gridDim.x < tiles)
      sk_load_tile(tbuf + (cur ^ 1) * tile_floats, REDP, A, (t + gridDim.x) * kSkTile, M, RED, avec != 0);
    cp_async_commit();
    cp_async_wait<1>();                                    // tile t has landed
    if (RED8 != RED) {                               // padding columns of the k-loop (an output tile lived here before)
      for (int e = threadIdx.x; e < kSkTile * (RED8 - RED); e += blockDim.x) {
        const int r = e / (RED8 - RED), c = RED + e % (RED8 - RED);
        tS[r * REDP + c] = 0.f;
      }
    }
    __syncthreads();
    float acc[2][NT][4];
#pragma unroll
    for (int m = 0; m < 2; ++m)
#pragma unroll
      for (int n = 0; n < NT; ++n)
#pragma unroll
        for (int q = 0; q < 4; ++q) acc[m][n][q] = 0.f;
    const float* ar = tS + (warp * 32 + g) * REDP + tq;
    for (int k0 = 0; k0 < RED8; k0 += 8) {
      uint32_t ahi[2][4], alo[2][4];
#pragma unroll
      for (int m = 0; m < 2; ++m) {
        const float* p = ar + (m * 16) * REDP + k0;
        const float v[4] = {p[0], p[8 * REDP], p[4], p[8 * REDP + 4]};   // (g,t) (g+8,t) (g,t+4) (g+8,t+4)
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          ahi[m][q] = to_tf32(v[q]);
          alo[m][q] = to_tf32(v[q] - __uint_as_float(ahi[m][q]));
        }
      }
      const uint32_t* bh = wHi + (k0 + tq) * WS + g;
      const uint32_t* bl = wLo + (k0 + tq) * WS + g;
      // the three products of one output tile depend on each other through its accumulator: issue
      // them across 2 column blocks x 2 row blocks so that dependent MMAs are 4 apart (small terms first)
      constexpr int NB = NT >= 2 ? 2 : 1;
#pragma unroll
      for (int n = 0; n < NT; n += NB) {
        uint32_t h0[NB], h1[NB], l0[NB], l1[NB];
#pragma unroll
        for (int j = 0; j < NB; ++j) {
          h0[j] = bh[(n + j) * 8]; h1[j] = bh[4 * WS + (n + j) * 8];
          l0[j] = bl[(n + j) * 8]; l1[j] = bl[4 * WS + (n + j) * 8];
        }
#pragma unroll
        for (int j = 0; j < NB; ++j)
#pragma unroll
          for (int m = 0; m < 2; ++m) mma_tf32(acc[m][n + j], alo[m], h0[j], h1[j]);
#pragma unroll
        for (int j = 0; j < NB; ++j)
#pragma unroll
          for (int m = 0; m < 2; ++m) mma_tf32(acc[m][n + j], ahi[m], l0[j], l1[j]);
#pragma unroll
        for (int j = 0; j < NB; ++j)
#pragma unroll
          for (int m = 0; m < 2; ++m) mma_tf32(acc[m][n + j], ahi[m], h0[j], h1[j]);
      }
    }
    __syncthreads();                                 // every warp is done reading the A tile
    // C fragment: c0 (g, 2t) c1 (g, 2t+1) c2 (g+8, 2t) c3 (g+8, 2t+1)
#pragma unroll
    for (int m = 0; m < 2; ++m)
#pragma unroll
      for (int n = 0; n < NT; ++n) {
        float* o = oS + (warp * 32 + m * 16 + g) * WS + n * 8 + 2 * tq;
        *reinterpret_cast<float2*>(o) = make_float2(acc[m][n][0], acc[m][n][1]);
        *reinterpret_cast<float2*>(o + 8 * WS) = make_float2(acc[m][n][2], acc[m][n][3]);
      }
    __syncthreads();
    if (dvec && (int)blockDim.x % (OUT >> 2) == 0) {
      const int c4 = OUT >> 2, c = ((int)threadIdx.x % c4) << 2, rstep = (int)blockDim.x / c4;
      for (int r = threadIdx.x / c4; r < kSkTile; r += rstep)
        if (row0 + r < M)
          *reinterpret_cast<float4*>(D + (row0 + r) * OUT + c) = *reinterpret_cast<const float4*>(oS + r * WS + c);
    } else {
      for (int e = threadIdx.x; e < kSkTile * OUT; e += blockDim.x) {
        const int r = e / OUT, c = e - r * OUT;
        if (row0 + r < M) D[(row0 + r) * OUT + c] = oS[r * WS + c];
      }
    }
  }
}

template <bool TRANS, int NT>
static int sk_launch_rows_mma(const float* A, const float* B, float* D, int64_t M, int RED, int OUT, cudaStream_t st) {
  const int RED8 = (RED + 7) & ~7, REDP = RED8 + 4;
  constexpr int WS = ((NT * 8 + 31) / 32) * 32 + 8;
  const size_t smem = (size_t)(2 * RED8 * WS + 2 * kSkTile * (REDP > WS ? REDP : WS)) * sizeof(float);
  auto kern = skinny_rows_mma_kernel<TRANS, NT>;
  if (smem > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  const int avec = (RED % 4 == 0) && aligned16(A), dvec = (OUT % 4 == 0) && aligned16(D);
  const int64_t tiles = (M + kSkTile - 1) / kSkTile;
  const int64_t cap = (int64_t)kNumSMs * 5;
  const int grid = (int)(tiles < cap ? tiles : cap);
  kern<<<grid, 128, smem, st>>>(A, B, D, M, RED, OUT, avec, dvec);
  return check_launch("skinny_gemm(rows, 3xTF32 mma)");
}
template <bool TRANS>
static int sk_rows_mma(const float* A, const float* B, float* D, int64_t M, int RED, int OUT, cudaStream_t st) {
  const int nt = (OUT + 7) / 8;
  if (nt <= 1) return sk_launch_rows_mma<TRANS, 1>(A, B, D, M, RED, OUT, st);
  if (nt <= 2) return sk_launch_rows_mma<TRANS, 2>(A, B, D, M, RED, OUT, st);
  if (nt <= 4) return sk_launch_rows_mma<TRANS, 4>(A, B, D, M, RED, OUT, st);
  return sk_launch_rows_mma<TRANS, 8>(A, B, D, M, RED, OUT, st);
}

// ---------------------------------------------------------------------------------------------
// Tensor-core dW: partial[cta][N x kcols] = sum_rows A[r][n] * B[r][kofs + k] with the ROWS as the
// MMA k-dimension (m16n8k8: m = 16 outputs n, n = 8 outputs k, k = 8 rows), 3xTF32 split operands.
// 4 warps per CTA, 64-row tiles: a warp owns 16 rows (two k-steps) and the whole MT x NT block of
// output tiles in registers (MT * NT <= 16); the four warps' accumulators meet in shared memory
// once, after the CTA's last tile.
// ---------------------------------------------------------------------------------------------
constexpr int kSkDwRows = 64;
template <int MT, int NT>
__global__ void __launch_bounds__(128)
skinny_dw_mma_kernel(const float* __restrict__ A, const float* __restrict__ B, float* __restrict__ partial,
                     int64_t M, int N, int K /* row length of B */, int kofs, int kcols, int avec, int bvec) {
  extern __shared__ __align__(16) float sk_smem[];
  constexpr int NP = MT * 16 + 8, KP = NT * 8 + 8;   // tile strides: fragment loads spread over the banks
  constexpr int pair_floats = kSkDwRows * (NP + KP);
  float* rS = sk_smem;                               // cross-warp reduction, after the last tile
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, tq = lane & 3;
  float acc[MT][NT][4];
#pragma unroll
  for (int m = 0; m < MT; ++m)
#pragma unroll
    for (int n = 0; n < NT; ++n)
#pragma unroll
      for (int q = 0; q < 4; ++q) acc[m][n][q] = 0.f;
  for (int e = threadIdx.x; e < 2 * pair_floats; e += blockDim.x) sk_smem[e] = 0.f;   // padding columns stay zero
  __syncthreads();
  // tile loader: 64 rows of A (N columns) and of B (kcols columns starting at kofs)
  auto load = [&](float* buf, int64_t row0) {
    const uint32_t a0 = smem_u32(buf), b0 = a0 + kSkDwRows * NP * 4;
    if (avec) {
      const int c4 = N >> 2;
      if ((int)blockDim.x % c4 == 0) {               // the usual widths: a thread keeps its chunk, rows advance by a constant (no division in the loop)
        const int c = ((int)threadIdx.x % c4) << 2, rstep = (int)blockDim.x / c4;
        for (int r = threadIdx.x / c4; r < kSkDwRows; r += rstep) {
          const bool in = row0 + r < M;
          cp_async16_zfill(a0 + (uint32_t)(r * NP + c) * 4, A + (in ? (row0 + r) * N + c : 0), in ? 16 : 0);
        }
      } else {
        for (int e = threadIdx.x; e < kSkDwRows * c4; e += blockDim.x) {
          const int r = e / c4, c = (e - r * c4) << 2;
          const bool in = row0 + r < M;
          cp_async16_zfill(a0 + (uint32_t)(r * NP + c) * 4, A + (in ? (row0 + r) * N + c : 0), in ? 16 : 0);
        }
      }
    } else {
      for (int e = threadIdx.x; e < kSkDwRows * N; e += blockDim.x) {
        const int r = e / N, c = e - r * N;
        buf[r * NP + c] = (row0 + r < M) ? __ldg(A + (row0 + r) * N + c) : 0.f;
      }
    }
    float* bb = buf + kSkDwRows * NP;
    if (bvec) {
      const int c4 = kcols >> 2;
      if ((int)blockDim.x % c4 == 0) {
        const int c = ((int)threadIdx.x % c4) << 2, rstep = (int)blockDim.x / c4;
        for (int r = threadIdx.x / c4; r < kSkDwRows; r += rstep) {
          const bool in = row0 + r < M;
          cp_async16_zfill(b0 + (uint32_t)(r * KP + c) * 4, B + (in ? (row0 + r) * K + kofs + c : 0), in ? 16 : 0);
        }
      } else {
        for (int e = threadIdx.x; e < kSkDwRows * c4; e += blockDim.x) {
          const int r = e / c4, c = (e - r * c4) << 2;
          const bool in = row0 + r < M;
          cp_async16_zfill(b0 + (uint32_t)(r * KP + c) * 4, B + (in ? (row0 + r) * K + kofs + c : 0), in ? 16 : 0);
        }
      }
    } else {
      for (int e = threadIdx.x; e < kSkDwRows * kcols; e += blockDim.x) {
        const int r = e / kcols, c = e - r * kcols;
        bb[r * KP + c] = (row0 + r < M) ? __ldg(B + (row0 + r) * K + kofs + c) : 0.f;
      }
    }
  };
  const int64_t tiles = (M + kSkDwRows - 1) / kSkDwRows;
  if (blockIdx.x < tiles) load(sk_smem, (int64_t)blockIdx.x * kSkDwRows);
  cp_async_commit();
  int cur = 0;
  for (int64_t t = blockIdx.x; t < tiles; t += gridDim.x, cur ^= 1) {
    const float* aS = sk_smem + cur * pair_floats;
    const float* bS = aS + kSkDwRows * NP;
    __syncthreads();                                 // every warp is done with the other buffer
    if (t + gridDim.x < tiles) load(sk_smem + (cur ^ 1) * pair_floats, (t + gridDim.x) * kSkDwRows);
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
#pragma unroll
    for (int ks = 0; ks < 2; ++ks) {                 // this warp's 16 rows = two k-steps of 8 rows
      const int r0 = warp * 16 + ks * 8;
      const float* ap = aS + (r0 + tq) * NP + g;     // A fragment (n, row): a0 (g,t) a1 (g+8,t) a2 (g,t+4) a3 (g+8,t+4)
      const float* bp = bS + (r0 + tq) * KP + g;     // B fragment (row, k): b0 (t,g) b1 (t+4,g)
      uint32_t ahi[MT][4], alo[MT][4];
#pragma unroll
      for (int m = 0; m < MT; ++m) {
        const float v[4] = {ap[m * 16], ap[m * 16 + 8], ap[4 * NP + m * 16], ap[4 * NP + m * 16 + 8]};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          ahi[m][q] = to_tf32(v[q]);
          alo[m][q] = to_tf32(v[q] - __uint_as_float(ahi[m][q]));
        }
      }
      constexpr int NB = (NT >= 2 && MT <= 2) ? 2 : 1;   // dependent MMAs at least 4 apart
#pragma unroll
      for (int n = 0; n < NT; n += NB) {
        uint32_t h0[NB], h1[NB], l0[NB], l1[NB];
#pragma unroll
        for (int j = 0; j < NB; ++j) {
          const float w0 = bp[(n + j) * 8], w1 = bp[4 * KP + (n + j) * 8];
          h0[j] = to_tf32(w0); h1[j] = to_tf32(w1);
          l0[j] = to_tf32(w0 - __uint_as_float(h0[j])); l1[j] = to_tf32(w1 - __uint_as_float(h1[j]));
        }
#pragma unroll
        for (int j = 0; j < NB; ++j)
#pragma unroll
          for (int m = 0; m < MT; ++m) mma_tf32(acc[m][n + j], alo[m], h0[j], h1[j]);
#pragma unroll
        for (int j = 0; j < NB; ++j)
#pragma unroll
          for (int m = 0; m < MT; ++m) mma_tf32(acc[m][n + j], ahi[m], l0[j], l1[j]);
#pragma unroll
        for (int j = 0; j < NB; ++j)
#pragma unroll
          for (int m = 0; m < MT; ++m) mma_tf32(acc[m][n + j], ahi[m], h0[j], h1[j]);
      }
    }
  }
  __syncthreads();                                   // tiles are dead: their memory becomes rS [4][MT*16][NT*8]
  constexpr int OW = NT * 8;
#pragma unroll
  for (int m = 0; m < MT; ++m)
#pragma unroll
    for (int n = 0; n < NT; ++n) {
      float* o = rS + (warp * MT * 16 + m * 16 + g) * OW + n * 8 + 2 * tq;   // c0 (g,2t) c1 (g,2t+1) c2 (g+8,2t) c3 (g+8,2t+1)
      o[0] = acc[m][n][0]; o[1] = acc[m][n][1];
      o[8 * OW] = acc[m][n][2]; o[8 * OW + 1] = acc[m][n][3];
    }
  __syncthreads();
  float* out = partial + (int64_t)blockIdx.x * N * kcols;
  for (int e = threadIdx.x; e < N * kcols; e += blockDim.x) {
    const int n = e / kcols, k = e - n * kcols;
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < 4; ++w) s += rS[(w * MT * 16 + n) * OW + k];
    out[e] = s;
  }
}

// D[n][kofs + k] = sum_cta partial[cta][n * kcols + k]
__global__ void __launch_bounds__(256)
skinny_dw_reduce_cols_kernel(const float* __restrict__ partial, float* __restrict__ D, int ctas, int N, int K,
                             int kofs, int kcols) {
  const int lane = threadIdx.x & 31;
  const int e = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (e >= N * kcols) return;
  float s = 0.f;
  for (int c = lane; c < ctas; c += 32) s += partial[(int64_t)c * N * kcols + e];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) D[(e / kcols) * K + kofs + e % kcols] = s;
}

}  // namespace dva

using namespace dva;

// Served here: both small dimensions <= 64 (any values, multiples of 4 take the vector loads).
extern "C" int dva_skinny_gemm_supported(int64_t M, int64_t N, int64_t K, int layout) {
  (void)layout;
  return M >= 1 && N >= 1 && K >= 1 && N <= kSkMax && K <= kSkMax;
}

extern "C" size_t dva_skinny_gemm_workspace_bytes(int64_t M, int64_t N, int64_t K, int layout) {
  if (layout != 2) return 16;
  const int64_t t64 = (M + kSkDwRows - 1) / kSkDwRows, cap = (int64_t)kNumSMs * 4;
  const size_t ctas = (size_t)(t64 < cap ? t64 : cap);
  return ctas * (size_t)N * (size_t)K * sizeof(float) + 16;
}

// layout 0: D[M,N] = A[M,K] . B[N,K]^T;  1: D[M,N] = A[M,K] . B[K,N];  2: D[N,K] = A[M,N]^T . B[M,K]
extern "C" int dva_skinny_gemm(const float* A, const float* B, float* D, int64_t M, int64_t N, int64_t K,
                               int layout, void* workspace, size_t workspace_bytes, void* stream) {
  if (M == 0) return DVA_OK;
  if (!dva_skinny_gemm_supported(M, N, K, layout)) return fail(DVA_EUNSUPPORTED, "skinny_gemm: N and K must be <= 64");
  if (!A || !B || !D) return fail(DVA_EINVAL, "skinny_gemm: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (layout == 0 || layout == 1)
    return layout == 0 ? sk_rows_mma<true>(A, B, D, M, (int)K, (int)N, st) : sk_rows_mma<false>(A, B, D, M, (int)K, (int)N, st);
  if (layout != 2) return fail(DVA_EINVAL, "skinny_gemm: bad layout");
  // output N x K in column blocks of at most 32 (64 when N <= 32) so that MT * NT <= 16 register tiles
  const int MT = N <= 32 ? 2 : 4;
  const int kblk = (MT == 2) ? 64 : 32;
  const int64_t tiles = (M + kSkDwRows - 1) / kSkDwRows;
  const int64_t cap = (int64_t)kNumSMs * 4;
  const int grid = (int)(tiles < cap ? tiles : cap);
  if (!workspace || workspace_bytes < (size_t)grid * N * K * sizeof(float))
    return fail(DVA_EINVAL, "skinny_gemm: workspace too small");
  float* partial = reinterpret_cast<float*>(workspace);
  const int avec = (N % 4 == 0) && aligned16(A);
  for (int kofs = 0; kofs < (int)K; kofs += kblk) {
    const int kcols = ((int)K - kofs < kblk) ? (int)K - kofs : kblk;
    const int NT = kcols <= 8 ? 1 : (kcols <= 32 ? 4 : 8);
    const int bvec = (K % 4 == 0) && (kofs % 4 == 0) && (kcols % 4 == 0) && aligned16(B);
    const int NP = MT * 16 + 8, KP = NT * 8 + 8;
    size_t smem = (size_t)2 * kSkDwRows * (NP + KP) * sizeof(float);
    const size_t red = (size_t)4 * MT * 16 * NT * 8 * sizeof(float);
    if (smem < red) smem = red;
#define SK_DW(MTv, NTv)                                                                            \
    do {                                                                                           \
      auto kern = skinny_dw_mma_kernel<MTv, NTv>;                                                  \
      if (smem > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
      kern<<<grid, 128, smem, st>>>(A, B, partial, M, (int)N, (int)K, kofs, kcols, avec, bvec);    \
    } while (0)
    if (MT == 2) { if (NT == 1) SK_DW(2, 1); else if (NT == 4) SK_DW(2, 4); else SK_DW(2, 8); }
    else { if (NT == 1) SK_DW(4, 1); else SK_DW(4, 4); }
#undef SK_DW
    if (int rc = check_launch("skinny_gemm(dw, 3xTF32 mma)")) return rc;
    skinny_dw_reduce_cols_kernel<<<((int)N * kcols + 7) / 8, 256, 0, st>>>(partial, D, grid, (int)N, (int)K, kofs, kcols);
    if (int rc = check_launch("skinny_gemm(dw reduce)")) return rc;
  }
  return DVA_OK;
}
