// Backward of one narrow MLP layer  a = LeakyReLU(BatchNorm1d(x . W^T))  (base_modules.py:38-48; the layers of
// DeepSetFeat / MLPSetFeat, pooling.py:645-656: 8 / 32 / 64 -> 32 on one row per view) in TWO passes over the
// rows instead of four:
//   pass 1 (bn_act.cu)   sums of g and g * zhat over the rows, g = dA * act'(.)          reads dA, z
//   pass 2 (this file)   dz = gamma invstd (g - mean(g) - zhat mean(g zhat)) per element, kept on chip;
//                        dX = dz . W  and  dW += dz^T . x  from the same tile            reads dA, z, x; writes dX
// Before: BN-apply (2 R + 1 W), dX GEMM (1 R + 1 W), dW GEMM (2 R) = 5 R + 2 W passes and three launches after
// the reduction; now 3 R + 1 W and one launch.  3xTF32 split operands on mma.sync.m16n8k8 (fp32-grade accuracy,
// the arithmetic of skinny_gemm.cu).  Measured at 1.28 M x 32 x 32: 0.106 ms inside a training step (inputs partly
// L2-resident), 0.155 ms cold under ncu, against 0.100 ms of HBM time; the first version, with integer divisions by
// the run-time row width in the copy loops, took 0.137 / 0.200 ms (issue-bound: 1 500 instructions per tile).
//
// A WARP is its own pipeline: 16-row tiles (dA, z, x) double-buffered with cp.async in the warp's private shared
// memory, no CTA-wide barrier inside the loop; the dW accumulators (N x K, 32 .. 64 registers per lane) live in
// registers for the whole kernel and meet in shared memory once at the end; per-CTA partial tiles are summed in
// a fixed order by mlp_dw_reduce_kernel (deterministic, no atomics).
#include "dva_common.cuh"

namespace dva {

constexpr int kMlWarps = 4;
constexpr int kMlRows = 16;          // rows per warp tile (one m16 block of dX, two k8 steps of dW)
constexpr int kMlNP = 36;            // stride of the dA -> dz tile and of the z tile (32 columns + 4: row fragments conflict-free)
constexpr int kMlN = 32;             // widest layer output served here

struct MlParams {
  const float *dA, *Z, *X, *W, *gamma, *beta, *mean, *invstd, *sums;
  float *dX, *partial;
  int64_t M;
  int N, K;
  float slope, inv_m;
};

template <int NT /* 8-column blocks of x: K <= 8 NT */>
__global__ void __launch_bounds__(kMlWarps * 32)
mlp_layer_bwd_kernel(const MlParams p) {
  extern __shared__ __align__(16) float ml_smem[];
  constexpr int KP = NT * 8 + 8;                     // x tile / dX staging stride and weight stride
  constexpr int stage_floats = kMlRows * (2 * kMlNP + KP);
  uint32_t* wHi = reinterpret_cast<uint32_t*>(ml_smem);          // [32][KP]: W[n][k], zero outside N x K
  uint32_t* wLo = wHi + kMlN * KP;
  float* coef = reinterpret_cast<float*>(wLo + kMlN * KP);       // [6][32]: sc, sh, mu, invstd, mean(g), mean(g zhat)
  float* tiles = coef + 6 * kMlN;                                // [warps][2][stage_floats]
  const int N = p.N, K = p.K;
  for (int e = threadIdx.x; e < kMlN * KP; e += blockDim.x) {
    const int n = e / KP, k = e - n * KP;
    const float v = (n < N && k < K) ? __ldg(p.W + (int64_t)n * K + k) : 0.f;
    const uint32_t hi = to_tf32(v);
    wHi[e] = hi;
    wLo[e] = to_tf32(v - __uint_as_float(hi));
  }
  for (int c = threadIdx.x; c < kMlN; c += blockDim.x) {
    float sc = 0.f, sh = 0.f, mu = 0.f, is = 0.f, k0 = 0.f, k1 = 0.f;
    if (c < N) {
      mu = p.mean[c]; is = p.invstd[c];
      sc = (p.gamma ? p.gamma[c] : 1.f) * is;
      sh = (p.beta ? p.beta[c] : 0.f) - mu * sc;
      k0 = p.sums[c] * p.inv_m; k1 = p.sums[N + c] * p.inv_m;
    }
    coef[c] = sc; coef[kMlN + c] = sh; coef[2 * kMlN + c] = mu; coef[3 * kMlN + c] = is;
    coef[4 * kMlN + c] = k0; coef[5 * kMlN + c] = k1;
  }
  for (int e = threadIdx.x; e < kMlWarps * 2 * stage_floats; e += blockDim.x) tiles[e] = 0.f;   // padding columns stay zero
  __syncthreads();

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, tq = lane & 3;
  float* my = tiles + warp * 2 * stage_floats;
  const int nc4 = N >> 2, kc4 = K >> 2;
  const bool want_dx = p.dX != nullptr;
  const int64_t tiles_total = (p.M + kMlRows - 1) / kMlRows;
  const int64_t t0 = (int64_t)blockIdx.x * kMlWarps + warp, tstep = (int64_t)gridDim.x * kMlWarps;

  // the lane's fixed column group in the element-wise step: columns 4 (lane % 8) .. + 3
  const int cc = (lane & 7) << 2;
  float c_sc[4], c_sh[4], c_mu[4], c_is[4], c_k0[4], c_k1[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    c_sc[j] = coef[cc + j]; c_sh[j] = coef[kMlN + cc + j]; c_mu[j] = coef[2 * kMlN + cc + j];
    c_is[j] = coef[3 * kMlN + cc + j]; c_k0[j] = coef[4 * kMlN + cc + j]; c_k1[j] = coef[5 * kMlN + cc + j];
  }

  // fixed lane -> (row, 16-byte chunk) map, no divisions: lane owns chunk c4 = lane % 8 (and c4 + 8 of x when
  // K > 32) of rows lane / 8 + 4 i
  const int c4 = lane & 7, rr = lane >> 3;
  constexpr int XH = (NT + 3) / 4;                   // 8-chunk column blocks of x: 2 for K > 32
  auto load = [&](float* buf, int64_t t) {
    const int64_t row0 = t * kMlRows;
    const uint32_t s0 = smem_u32(buf);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = rr + 4 * i;
      const bool in = row0 + r < p.M;
      if (c4 < nc4) {
        const int64_t off = in ? (row0 + r) * N + c4 * 4 : 0;
        cp_async16_zfill(s0 + (uint32_t)(r * kMlNP + c4 * 4) * 4, p.dA + off, in ? 16 : 0);
        cp_async16_zfill(s0 + (uint32_t)(kMlRows * kMlNP + r * kMlNP + c4 * 4) * 4, p.Z + off, in ? 16 : 0);
      }
#pragma unroll
      for (int h = 0; h < XH; ++h) {
        const int cx = c4 + 8 * h;
        if (cx < kc4)
          cp_async16_zfill(s0 + (uint32_t)(2 * kMlRows * kMlNP + r * KP + cx * 4) * 4,
                           p.X + (in ? (row0 + r) * K + cx * 4 : 0), in ? 16 : 0);
      }
    }
  };

  float acc_w[2][NT][4];
#pragma unroll
  for (int m = 0; m < 2; ++m)
#pragma unroll
    for (int n = 0; n < NT; ++n)
#pragma unroll
      for (int q = 0; q < 4; ++q) acc_w[m][n][q] = 0.f;

  if (t0 < tiles_total) load(my, t0);
  cp_async_commit();
  int cur = 0;
  for (int64_t t = t0; t < tiles_total; t += tstep, cur ^= 1) {
    float* gS = my + cur * stage_floats;             // dA, then dz
    float* zS = gS + kMlRows * kMlNP;
    float* xS = zS + kMlRows * kMlNP;                // x, then the dX staging tile
    if (t + tstep < tiles_total) load(my + (cur ^ 1) * stage_floats, t + tstep);
    cp_async_commit();
    cp_async_wait<1>();
    __syncwarp();
    const int64_t row0 = t * kMlRows;
    // ---- dz in place of dA: 16 x 32 elements, one float4 per lane and step -------------------------------
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = (lane >> 3) + 4 * i;
      float4 gv = *reinterpret_cast<const float4*>(gS + r * kMlNP + cc);
      const float4 zv = *reinterpret_cast<const float4*>(zS + r * kMlNP + cc);
      float gq[4] = {gv.x, gv.y, gv.z, gv.w};
      const float zq[4] = {zv.x, zv.y, zv.z, zv.w};
      const bool in = row0 + r < p.M;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float a = fmaf(zq[j], c_sc[j], c_sh[j]);   // the forward's own expression: same sign decision
        const float gg = a > 0.f ? gq[j] : gq[j] * p.slope;
        const float zh = (zq[j] - c_mu[j]) * c_is[j];
        gq[j] = in ? c_sc[j] * (gg - c_k0[j] - zh * c_k1[j]) : 0.f;
      }
      *reinterpret_cast<float4*>(gS + r * kMlNP + cc) = make_float4(gq[0], gq[1], gq[2], gq[3]);
    }
    __syncwarp();
    // ---- dX[16, K] = dz[16, N] . W[N, K] ------------------------------------------------------------------
    float acc_x[NT][4];
    if (want_dx) {
#pragma unroll
      for (int n = 0; n < NT; ++n)
#pragma unroll
        for (int q = 0; q < 4; ++q) acc_x[n][q] = 0.f;
#pragma unroll
      for (int ks = 0; ks < kMlN / 8; ++ks) {
        if (ks * 8 < N) {
          const float* ap = gS + g * kMlNP + ks * 8 + tq;
          const float v[4] = {ap[0], ap[8 * kMlNP], ap[4], ap[8 * kMlNP + 4]};   // (g,t) (g+8,t) (g,t+4) (g+8,t+4)
          uint32_t ahi[4], alo[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            ahi[q] = to_tf32(v[q]);
            alo[q] = to_tf32(v[q] - __uint_as_float(ahi[q]));
          }
          const uint32_t* bh = wHi + (ks * 8 + tq) * KP + g;
          const uint32_t* bl = wLo + (ks * 8 + tq) * KP + g;
          uint32_t h0[NT], h1[NT], l0[NT], l1[NT];
#pragma unroll
          for (int j = 0; j < NT; ++j) {
            h0[j] = bh[j * 8]; h1[j] = bh[4 * KP + j * 8];
            l0[j] = bl[j * 8]; l1[j] = bl[4 * KP + j * 8];
          }
          // the three products of one output block depend on each other through its accumulator: small terms
          // first, dependent MMAs NT apart
#pragma unroll
          for (int j = 0; j < NT; ++j) mma_tf32(acc_x[j], alo, h0[j], h1[j]);
#pragma unroll
          for (int j = 0; j < NT; ++j) mma_tf32(acc_x[j], ahi, l0[j], l1[j]);
#pragma unroll
          for (int j = 0; j < NT; ++j) mma_tf32(acc_x[j], ahi, h0[j], h1[j]);
        }
      }
    }
    // ---- dW[N, K] += dz^T[N, 16] . x[16, K]: the rows are the MMA k dimension ------------------------------
#pragma unroll
    for (int ks = 0; ks < 2; ++ks) {
      const float* ap = gS + (ks * 8 + tq) * kMlNP + g;   // A fragment (n, row): a0 (g,t) a1 (g+8,t) a2 (g,t+4) a3 (g+8,t+4)
      const float* bp = xS + (ks * 8 + tq) * KP + g;      // B fragment (row, k): b0 (t,g) b1 (t+4,g)
      uint32_t ahi[2][4], alo[2][4];
#pragma unroll
      for (int m = 0; m < 2; ++m) {
        const float v[4] = {ap[m * 16], ap[m * 16 + 8], ap[4 * kMlNP + m * 16], ap[4 * kMlNP + m * 16 + 8]};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          ahi[m][q] = to_tf32(v[q]);
          alo[m][q] = to_tf32(v[q] - __uint_as_float(ahi[m][q]));
        }
      }
#pragma unroll
      for (int j = 0; j < NT; ++j) {
        const float w0 = bp[j * 8], w1 = bp[4 * KP + j * 8];
        const uint32_t h0 = to_tf32(w0), h1 = to_tf32(w1);
        const uint32_t l0 = to_tf32(w0 - __uint_as_float(h0)), l1 = to_tf32(w1 - __uint_as_float(h1));
#pragma unroll
        for (int m = 0; m < 2; ++m) mma_tf32(acc_w[m][j], alo[m], h0, h1);
#pragma unroll
        for (int m = 0; m < 2; ++m) mma_tf32(acc_w[m][j], ahi[m], l0, l1);
#pragma unroll
        for (int m = 0; m < 2; ++m) mma_tf32(acc_w[m][j], ahi[m], h0, h1);
      }
    }
    // ---- dX tile through the (dead) x tile: coalesced 16-byte stores ----------------------------------------
    if (want_dx) {
      __syncwarp();
#pragma unroll
      for (int j = 0; j < NT; ++j) {   // C fragment: c0 (g, 2t) c1 (g, 2t+1) c2 (g+8, 2t) c3 (g+8, 2t+1)
        float* o = xS + g * KP + j * 8 + 2 * tq;
        *reinterpret_cast<float2*>(o) = make_float2(acc_x[j][0], acc_x[j][1]);
        *reinterpret_cast<float2*>(o + 8 * KP) = make_float2(acc_x[j][2], acc_x[j][3]);
      }
      __syncwarp();
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int r = rr + 4 * i;
#pragma unroll
        for (int h = 0; h < XH; ++h) {
          const int cx = c4 + 8 * h;
          if (cx < kc4 && row0 + r < p.M)
            *reinterpret_cast<float4*>(p.dX + (row0 + r) * K + cx * 4) = *reinterpret_cast<const float4*>(xS + r * KP + cx * 4);
        }
      }
    }
    __syncwarp();                                    // the stage may be refilled two iterations from now
  }
  cp_async_wait<0>();
  __syncthreads();                                   // every warp is out of its loop: the tiles become rS [4][32][NT*8]
  constexpr int OW = NT * 8;
  float* rS = tiles;
#pragma unroll
  for (int m = 0; m < 2; ++m)
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      float* o = rS + (warp * kMlN + m * 16 + g) * OW + j * 8 + 2 * tq;
      o[0] = acc_w[m][j][0]; o[1] = acc_w[m][j][1];
      o[8 * OW] = acc_w[m][j][2]; o[8 * OW + 1] = acc_w[m][j][3];
    }
  __syncthreads();
  float* out = p.partial + (int64_t)blockIdx.x * N * K;
  for (int e = threadIdx.x; e < N * K; e += blockDim.x) {
    const int n = e / K, k = e - n * K;
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < kMlWarps; ++w) s += rS[(w * kMlN + n) * OW + k];
    out[e] = s;
  }
}

// dW[e] = sum over CTAs of partial[cta][e]: one warp per element, lanes stride over the CTAs, fixed-order
// butterfly at the end -> deterministic
__global__ void __launch_bounds__(256)
mlp_dw_reduce_kernel(const float* __restrict__ partial, float* __restrict__ D, int ctas, int NK) {
  const int lane = threadIdx.x & 31;
  const int e = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (e >= NK) return;
  float s = 0.f;
  for (int c = lane; c < ctas; c += 32) s += partial[(int64_t)c * NK + e];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) D[e] = s;
}

static int ml_nt(int64_t K) { return K <= 8 ? 1 : K <= 16 ? 2 : K <= 32 ? 4 : 8; }
static size_t ml_smem_bytes(int nt) {
  const int KP = nt * 8 + 8;
  return (size_t)(2 * kMlN * KP + 6 * kMlN + kMlWarps * 2 * kMlRows * (2 * kMlNP + KP)) * sizeof(float);
}
static int ml_grid(int64_t M, int nt) {
  const int64_t tiles = (M + kMlRows - 1) / kMlRows;
  const int64_t want = (tiles + kMlWarps - 1) / kMlWarps;
  const int64_t cap = (int64_t)kNumSMs * (nt == 8 ? 2 : 3);   // shared memory: 92 KB (K = 64) / 67 KB (K = 32) per CTA
  return (int)(want < cap ? (want < 1 ? 1 : want) : cap);
}
static size_t ml_round256(size_t b) { return (b + 255) & ~(size_t)255; }

template <int NT>
static int ml_launch(const MlParams& p, int grid, cudaStream_t st) {
  const size_t smem = ml_smem_bytes(NT);
  auto kern = mlp_layer_bwd_kernel<NT>;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return failf((int)e, "mlp_layer_bwd: %s", cudaGetErrorString(e));
  }
  kern<<<grid, kMlWarps * 32, smem, st>>>(p);
  return check_launch("mlp_layer_bwd");
}

}  // namespace dva

using namespace dva;

extern "C" int dva_mlp_layer_bwd_supported(int64_t M, int64_t N, int64_t K) {
  return M >= 1 && N >= 4 && N <= kMlN && N % 4 == 0 && K >= 4 && K <= 64 && K % 4 == 0;
}

extern "C" size_t dva_mlp_layer_bwd_workspace_bytes(int64_t M, int64_t N, int64_t K) {
  if (!dva_mlp_layer_bwd_supported(M, N, K)) return 0;
  return ml_round256(dva_bn_workspace_bytes(M, N)) + (size_t)ml_grid(M, ml_nt(K)) * N * K * sizeof(float);
}

extern "C" int dva_mlp_layer_bwd(const float* dA, const float* Z, const float* X, const float* W, const float* gamma,
                                 const float* beta, const float* mean, const float* invstd, float* dX, float* dW,
                                 float* dgamma_dbeta, int64_t M, int64_t N, int64_t K, float slope, void* workspace,
                                 size_t workspace_bytes, void* stream) {
  if (!dva_mlp_layer_bwd_supported(M, N, K)) return fail(DVA_EUNSUPPORTED, "mlp_layer_bwd: N <= 32, K <= 64, multiples of 4, M >= 1");
  if (!dA || !Z || !X || !W || !mean || !invstd || !dW || !dgamma_dbeta) return fail(DVA_EINVAL, "mlp_layer_bwd: null pointer");
  if (!aligned16(dA) || !aligned16(Z) || !aligned16(X) || (dX && !aligned16(dX)))
    return fail(DVA_EINVAL, "mlp_layer_bwd: row pointers must be 16-byte aligned");
  if (!workspace || workspace_bytes < dva_mlp_layer_bwd_workspace_bytes(M, N, K)) return fail(DVA_EINVAL, "mlp_layer_bwd: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  // pass 1: dgamma_dbeta = [sum g ; sum g zhat] (bn_act.cu; dz = nullptr stops after the reduction)
  const size_t bn_bytes = ml_round256(dva_bn_workspace_bytes(M, N));
  int rc = dva_bn_act_bwd(dA, Z, gamma, beta, mean, invstd, nullptr, dgamma_dbeta, M, N, slope, 1, DVA_F32, workspace,
                          bn_bytes, stream);
  if (rc) return rc;
  const int nt = ml_nt(K), grid = ml_grid(M, nt);
  MlParams p;
  p.dA = dA; p.Z = Z; p.X = X; p.W = W; p.gamma = gamma; p.beta = beta; p.mean = mean; p.invstd = invstd;
  p.sums = dgamma_dbeta; p.dX = dX;
  p.partial = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(workspace) + bn_bytes);
  p.M = M; p.N = (int)N; p.K = (int)K; p.slope = slope; p.inv_m = 1.f / (float)M;
  switch (nt) {
    case 1: rc = ml_launch<1>(p, grid, st); break;
    case 2: rc = ml_launch<2>(p, grid, st); break;
    case 4: rc = ml_launch<4>(p, grid, st); break;
    default: rc = ml_launch<8>(p, grid, st); break;
  }
  if (rc) return rc;
  const int NK = (int)(N * K);
  mlp_dw_reduce_kernel<<<(NK + 7) / 8, 256, 0, st>>>(p.partial, dW, grid, NK);
  return check_launch("mlp_dw_reduce");
}
