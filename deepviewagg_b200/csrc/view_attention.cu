// Fused CSR-gather + ragged group softmax + attention-weighted sum + gating (fwd and bwd).
//
// Replaces, in one pass over HBM, the reference chain
//   modules.py:518              x_mod = cat(x_mod)[idx_sorting]            (row gather, [V,C] copy)
//   pooling.py:285-286 / 515    a = segment_softmax_csr(compat, csr, scaling)
//   pooling.py:289-291 / 519    y = segment_csr(x_mod * expand_group_feat(a), csr, 'sum')
//   pooling.py:293-300 / 523    out = y * expand_group_feat(Gating(segment_csr(compat,'max')))
// which materialises >= 4 [V,C] temporaries in the reference.
//
// Work decomposition: one warp owns one point (CSR segment) at a time; CTAs are persistent
// (148 SMs x occupancy) and stride over the points.  A feature row of C channels is split into
// 16-byte chunks; LPR lanes cover one row (LPR*CPL chunks), so a warp reads 32/LPR rows per step
// with every lane issuing one LDG.128 -- for C=128 fp32 a row is exactly one 512 B warp-wide
// load, kUnroll of them in flight per lane.  Scores live in the flat (view,group) order of
// `compat` so that lane l always owns group l%G; per-group max / sum are xor-shuffle reductions
// over the lanes of equal l%G.  Per view the inner loop is: LDS row id, IMAD.WIDE address,
// LDG.128, LDS attention, VEC FFMAs -- the kernels are sized to stay below the ~90 warp
// instructions per 512 B that the issue slots allow at full HBM bandwidth.
//
// HBM bytes per launch (s = sizeof(T)):
//   fwd: V*(C*s + 4 + 4G) + N*(8 + C*s) (+ N*12G saved statistics when training)
//   bwd: V*(2*C*s + 4 + 8G) + N*(8 + C*s + 12G)
#include "view_attention.cuh"
#include <stdlib.h>

namespace dva {

#ifndef DVA_FWD_UNROLL
#define DVA_FWD_UNROLL 8
#endif
#ifndef DVA_BWD_UNROLL
#define DVA_BWD_UNROLL 4
#endif
#ifndef DVA_FWD_MINB
#define DVA_FWD_MINB 4
#endif
#ifndef DVA_BWD_MINB
#define DVA_BWD_MINB 4
#endif
constexpr int kWarps = 8;          // warps per CTA
constexpr int kUnroll = DVA_FWD_UNROLL;     // fwd: row loads in flight per lane (x CPL)
constexpr int kUnrollBwd = DVA_BWD_UNROLL;  // bwd: row loads in flight per lane (x CPL)

// A row chunk in flight: the raw 16 bytes (or one scalar) -- unpacked to fp32 only at use so
// that kUnroll loads cost 4 registers each whatever the storage type.
template <typename T, int VEC> struct Chunk {
  uint4 raw;
  __device__ __forceinline__ void load(const void* p) { raw = ldg_stream16(p); }
  __device__ __forceinline__ void zero() { raw = make_uint4(0u, 0u, 0u, 0u); }
  __device__ __forceinline__ void get(float (&f)[VEC]) const { unpack16<T, VEC>(raw, f); }
};
template <typename T> struct Chunk<T, 1> {
  T raw;
  __device__ __forceinline__ void load(const void* p) { raw = __ldg(reinterpret_cast<const T*>(p)); }
  __device__ __forceinline__ void zero() { raw = Cvt<T>::from_f(0.f); }
  __device__ __forceinline__ void get(float (&f)[1]) const { f[0] = Cvt<T>::to_f(raw); }
};
template <typename T, int VEC>
__device__ __forceinline__ void load_chunk(const void* p, float (&f)[VEC]) {
  Chunk<T, VEC> c; c.load(p); c.get(f);
}
template <typename T, int VEC>
__device__ __forceinline__ void store_chunk(void* p, const float (&f)[VEC]) {
  if constexpr (VEC == 1) {
    *reinterpret_cast<T*>(p) = Cvt<T>::from_f(f[0]);
  } else {
    stg_stream16(p, pack16<T, VEC>(f));
  }
}

// byte address of row `row`: one IMAD.WIDE.U32 (row and row_bytes are 32-bit)
__device__ __forceinline__ const char* row_addr(const char* base, uint32_t row, uint32_t row_bytes) {
  return base + (uint64_t)row * row_bytes;
}
__device__ __forceinline__ char* row_addr(char* base, uint32_t row, uint32_t row_bytes) {
  return base + (uint64_t)row * row_bytes;
}

// Per-point softmax statistics over the flat (view, group) scores of one segment.
// Lane l owns elements e = l, l+32, ... (all of group l % G).  The first kCache elements per lane
// stay in registers between the max pass and the exp pass.  `park`: segments of <= 32 views
// leave their e-values in the [G][33] tile so the row loop needs no second exp pass.
constexpr int kCache = 4;
struct SegStats { float m, den; int am; };

__device__ __forceinline__ SegStats seg_softmax_stats(const float* __restrict__ cp, int nG, int G,
                                                      int lane, float inv_sq, bool park,
                                                      float* __restrict__ tile) {
  float c[kCache];
  float m = -INFINITY; int am = 0x7fffffff;
#pragma unroll
  for (int j = 0; j < kCache; ++j) {
    const int e = lane + 32 * j;
    c[j] = (e < nG) ? __ldg(cp + e) : -INFINITY;
    if (c[j] > m) { m = c[j]; am = e; }
  }
  for (int e = lane + 32 * kCache; e < nG; e += 32) {
    const float v = __ldg(cp + e);
    if (v > m) { m = v; am = e; }
  }
  for (int off = 16; off >= G; off >>= 1) {
    const float om = __shfl_xor_sync(0xffffffffu, m, off);
    const int oa = __shfl_xor_sync(0xffffffffu, am, off);
    if (om > m || (om == m && oa < am)) { m = om; am = oa; }
  }
  const int gl = lane % G;
  float den = 0.f;
#pragma unroll
  for (int j = 0; j < kCache; ++j) {
    const int e = lane + 32 * j;
    if (e < nG) {
      const float ev = expf((c[j] - m) * inv_sq);
      den += ev;
      if (park) tile[gl * kTileStride + e / G] = ev;
    }
  }
  for (int e = lane + 32 * kCache; e < nG; e += 32) {
    const float ev = expf((__ldg(cp + e) - m) * inv_sq);
    den += ev;
    if (park) tile[gl * kTileStride + e / G] = ev;
  }
  den = group_lane_sum(den, G);
  SegStats r; r.m = m; r.den = den; r.am = am;   // am: flat element index e = v*G + g
  return r;
}

// ---------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------
template <typename T, int VEC, int LPR, int CPL, int MINB>
__global__ void __launch_bounds__(kWarps * 32, MINB)
view_attention_fwd_kernel(const VAParams P) {
  constexpr int RPI = 32 / LPR;              // rows per warp step
  constexpr int TILE_C = VEC * LPR * CPL;    // channels per pass
  constexpr int U = (kUnroll / CPL) > 0 ? (kUnroll / CPL) : 1;  // row steps in flight
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int C = P.C, G = P.G;
  float* att_s = reinterpret_cast<float*>(smem_raw) + warp * (G * kTileStride);
  uint32_t* row_s = reinterpret_cast<uint32_t*>(smem_raw + (size_t)kWarps * G * kTileStride * sizeof(float)) + warp * 32;
  const int sg = lane / LPR, lir = lane % LPR;
  const char* __restrict__ xb = reinterpret_cast<const char*>(P.x);
  char* __restrict__ ob = reinterpret_cast<char*>(P.out);
  const uint32_t row_bytes = (uint32_t)C * sizeof(T);
  const int gl = lane % G;                   // group owned by this lane in the flat score order
  const bool gating = P.gate_w != nullptr;
  const float gw = gating ? P.gate_w[gl] : 0.f, gb = gating ? P.gate_b[gl] : 0.f;
  const bool single_tile = C <= TILE_C;
  const bool has_idx = P.idx != nullptr;

  // Per-lane chunk geometry of tile 0, hoisted out of the point loop.  Lanes past the end of
  // the row load a clamped (valid) chunk and simply never store.
  int gk0[CPL]; uint32_t off0[CPL]; bool live0[CPL];
#pragma unroll
  for (int k = 0; k < CPL; ++k) {
    const int c0 = (lir + LPR * k) * VEC;
    live0[k] = c0 < C;
    const int cc = live0[k] ? c0 : 0;
    gk0[k] = group_of_channel(cc, C, G);      // VEC>1: host guarantees chunks never straddle groups
    off0[k] = (uint32_t)cc * sizeof(T);
  }

  const int64_t warps_total = (int64_t)gridDim.x * kWarps;
  for (int64_t i = (int64_t)blockIdx.x * kWarps + warp; i < P.N; i += warps_total) {
    const int64_t p0 = P.ptr[i];
    const int n = (int)(P.ptr[i + 1] - p0);
    __syncwarp();                            // att_s / row_s of the previous point are free
    if (n == 0) {                            // unseen point: exact zeros (segment_csr of nothing)
      if (lane < G && P.seg_max != nullptr) {
        P.seg_max[i * G + lane] = 0.f; P.seg_den[i * G + lane] = P.eps; P.seg_arg[i * G + lane] = -1;
      }
      if (sg == 0) {
        float z[VEC];
#pragma unroll
        for (int j = 0; j < VEC; ++j) z[j] = 0.f;
        for (int c0 = lir * VEC; c0 < C; c0 += LPR * VEC)
          store_chunk<T, VEC>(ob + i * (int64_t)row_bytes + (size_t)c0 * sizeof(T), z);
      }
      continue;
    }
    const int nG = n * G;
    const float* __restrict__ cp = P.compat + p0 * G;
    // reference: (c - max) / sqrt(n) (pooling.py:792-801); one reciprocal per point instead
    const float inv_sq = P.group_scaling ? rsqrtf((float)n) : 1.f;
    const bool one_chunk = n <= 32;
    const SegStats st = seg_softmax_stats(cp, nG, G, lane, inv_sq, one_chunk, att_s);
    const float den = st.den + P.eps;
    const float t = gating ? tanhf(fmaxf(fmaf(gw, st.m, gb), 0.f)) : 1.f;
    if (lane < G && P.seg_max != nullptr) {
      P.seg_max[i * G + lane] = st.m;
      P.seg_den[i * G + lane] = den;
      P.seg_arg[i * G + lane] = (int32_t)(p0 + st.am / G);
    }
    const float inv_den = 1.f / den;
    const float scale = t * inv_den;         // applied once per output channel instead of per view

    for (int ct = 0; ct < C; ct += TILE_C) {
      float acc[CPL][VEC];
      int gk[CPL]; uint32_t off[CPL]; bool live[CPL];
#pragma unroll
      for (int k = 0; k < CPL; ++k) {
#pragma unroll
        for (int j = 0; j < VEC; ++j) acc[k][j] = 0.f;
        if (single_tile) {
          gk[k] = gk0[k]; off[k] = off0[k]; live[k] = live0[k];
        } else {
          const int c0 = ct + (lir + LPR * k) * VEC;
          live[k] = c0 < C;
          const int cc = live[k] ? c0 : 0;
          gk[k] = group_of_channel(cc, C, G);
          off[k] = (uint32_t)cc * sizeof(T);
        }
      }

      for (int vs = 0; vs < n; vs += 32) {
        const int nc = min(32, n - vs);
        if (!one_chunk) {                    // long segments: e-values of this chunk
          __syncwarp();
          for (int e = lane; e < nc * G; e += 32)
            att_s[gl * kTileStride + e / G] = expf((__ldg(cp + vs * G + e) - st.m) * inv_sq);
        }
        if (lane < nc)
          row_s[lane] = has_idx ? (uint32_t)load_idx(P.idx, P.idx64, p0 + vs + lane)
                                : (uint32_t)(p0 + vs + lane);
        __syncwarp();

        const uint32_t* rs = row_s + sg;     // this sub-group's row of each step
        const float* as[CPL];
        const char* xk[CPL];                 // per-lane base pointers: row address = 1 IMAD.WIDE
#pragma unroll
        for (int k = 0; k < CPL; ++k) { as[k] = att_s + gk[k] * kTileStride + sg; xk[k] = xb + off[k]; }
        int v0 = 0;
        // ---- main loop: U full row steps, no predicates
        for (; v0 + RPI * U <= nc; v0 += RPI * U) {
          Chunk<T, VEC> f[U][CPL];
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const uint32_t srow = rs[v0 + u * RPI];
#pragma unroll
            for (int k = 0; k < CPL; ++k) f[u][k].load(row_addr(xk[k], srow, row_bytes));
          }
#pragma unroll
          for (int u = 0; u < U; ++u) {
#pragma unroll
            for (int k = 0; k < CPL; ++k) {
              float fv[VEC];
              f[u][k].get(fv);
              const float a = as[k][v0 + u * RPI];
#pragma unroll
              for (int j = 0; j < VEC; ++j) acc[k][j] = fmaf(a, fv[j], acc[k][j]);
            }
          }
        }
        // ---- tail: the remaining < U row steps, all loads issued before the first use
        if (v0 < nc) {
          Chunk<T, VEC> f[U][CPL];
          bool ok[U];
#pragma unroll
          for (int u = 0; u < U; ++u) {
            ok[u] = v0 + u * RPI + sg < nc;
            if (v0 + u * RPI < nc) {           // warp-uniform: skip whole row steps past the end
              const uint32_t srow = rs[ok[u] ? v0 + u * RPI : 0 - sg];   // idle sub-group: row 0
#pragma unroll
              for (int k = 0; k < CPL; ++k) f[u][k].load(row_addr(xk[k], srow, row_bytes));
            } else {
#pragma unroll
              for (int k = 0; k < CPL; ++k) f[u][k].zero();
            }
          }
#pragma unroll
          for (int u = 0; u < U; ++u) {
#pragma unroll
            for (int k = 0; k < CPL; ++k) {
              float fv[VEC];
              f[u][k].get(fv);
              const float a = ok[u] ? as[k][v0 + u * RPI] : 0.f;
#pragma unroll
              for (int j = 0; j < VEC; ++j) acc[k][j] = fmaf(a, fv[j], acc[k][j]);
            }
          }
        }
      }

      // combine the RPI row sub-groups, apply gating and 1/den, store
#pragma unroll
      for (int k = 0; k < CPL; ++k) {
        const float sc = __shfl_sync(0xffffffffu, scale, gk[k]);
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
          float a = acc[k][j];
#pragma unroll
          for (int o = LPR; o < 32; o <<= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
          acc[k][j] = a * sc;
        }
      }
      if (sg == 0) {
#pragma unroll
        for (int k = 0; k < CPL; ++k)
          if (live[k]) store_chunk<T, VEC>(ob + i * (int64_t)row_bytes + off[k], acc[k]);
      }
    }

    if (P.att != nullptr) {                  // save_last tap / autograd: normalised attentions
      float* __restrict__ ao = P.att + p0 * G;
      if (one_chunk) {
        for (int e = lane; e < nG; e += 32) ao[e] = att_s[gl * kTileStride + e / G] * inv_den;
      } else {
        for (int e = lane; e < nG; e += 32) ao[e] = expf((__ldg(cp + e) - st.m) * inv_sq) * inv_den;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// backward.  With gd = dO * t (gate folded into the upstream gradient):
//   s'_vg  = sum_{c in g} gd_c x_vc           (one dot product per view and group)
//   S'_g   = sum_v a_vg s'_vg                 (= t_g * dL/dt_g)
//   dx_vc  = a_vg gd_c
//   dc_vg  = a_vg (s'_vg - S'_g)/sqrt(n)  +  [v == argmax_g] (S'_g/t_g) (1-t_g^2) w_g 1[w q + b > 0]
//   dw_g  += (S'_g/t_g) (1-t^2) 1[.] q_g ;  db_g += (S'_g/t_g) (1-t^2) 1[.]
// (SURVEY Appendix A; the reference obtains the same through autograd over pooling.py:285-300.)
// ---------------------------------------------------------------------------------------------
// REG: all groups equally wide, a power-of-two number of chunks each (cpg), so the lanes of a group
// form aligned blocks -> log2(min(cpg,LPR)) shuffle steps.  !REG: arbitrary group_sizes(C,G)
// (pooling.py:737-745), one masked full-row reduction per group (scalar kernels only).
template <typename T, int VEC, int LPR, int CPL, int MINB, bool REG>
__global__ void __launch_bounds__(kWarps * 32, MINB)
view_attention_bwd_kernel(const VAParams P) {
  constexpr int RPI = 32 / LPR;
  constexpr int TILE_C = VEC * LPR * CPL;
  constexpr int U = (kUnrollBwd / CPL) > 0 ? (kUnrollBwd / CPL) : 1;
  constexpr int UT = U >= 2 ? 2 : 1;          // tail block width
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int C = P.C, G = P.G;
  const int tile = G * kTileStride;
  float* att_s = reinterpret_cast<float*>(smem_raw) + warp * tile;
  float* s_s = reinterpret_cast<float*>(smem_raw) + (kWarps + warp) * tile;
  uint32_t* row_s = reinterpret_cast<uint32_t*>(smem_raw + (size_t)2 * kWarps * tile * sizeof(float)) + warp * 64;
  uint32_t* orow_s = row_s + 32;             // destination row of dx (== row_s when scattering)
  float* gate_s = reinterpret_cast<float*>(smem_raw + (size_t)2 * kWarps * tile * sizeof(float) +
                                           (size_t)kWarps * 64 * sizeof(uint32_t));  // [kWarps][2][G]
  const int sg = lane / LPR, lir = lane % LPR;
  const char* __restrict__ xb = reinterpret_cast<const char*>(P.x);
  const char* __restrict__ gob = reinterpret_cast<const char*>(P.gout);
  char* __restrict__ gxb = reinterpret_cast<char*>(P.gx);
  const uint32_t row_bytes = (uint32_t)C * sizeof(T);
  const int gl = lane % G;
  const bool gating = P.gate_w != nullptr;
  const float gw = gating ? P.gate_w[gl] : 0.f, gb = gating ? P.gate_b[gl] : 0.f;
  float dw_acc = 0.f, db_acc = 0.f;
  const bool single_tile = C <= TILE_C;
  const bool has_idx = P.idx != nullptr;
  const bool scatter = P.scatter && has_idx;
  // cpg = chunks per group (host guarantees a power of two when REG); cpe = lanes of one row
  // step that share a group; a (view,group) slot of s_s is written once per tile iff cpg <= LPR.
  const int cpg = REG ? (C / G) / VEC : 0;
  const int cpe = cpg < LPR ? cpg : LPR;
  // CPL == 1 kernels always see the whole row in one tile and cpg <= LPR: plain assignment
  const bool assign_s = (REG && CPL == 1) || (REG && single_tile && cpg <= LPR);
  // butterfly step o contributes iff o < cpe: as a 0/1 multiplier (no predicates in the loop)
  float red_mask[5];
#pragma unroll
  for (int b = 0; b < 5; ++b) red_mask[b] = ((1 << b) < cpe) ? 1.f : 0.f;
  const bool leader = REG ? ((lir & (cpe - 1)) == 0) : (lir == 0);

  int gk0[CPL]; uint32_t off0[CPL]; bool live0[CPL];
#pragma unroll
  for (int k = 0; k < CPL; ++k) {
    const int c0 = (lir + LPR * k) * VEC;
    live0[k] = c0 < C;
    const int cc = live0[k] ? c0 : 0;
    gk0[k] = group_of_channel(cc, C, G);
    off0[k] = (uint32_t)cc * sizeof(T);
  }

  const int64_t warps_total = (int64_t)gridDim.x * kWarps;
  for (int64_t i = (int64_t)blockIdx.x * kWarps + warp; i < P.N; i += warps_total) {
    const int64_t p0 = P.ptr[i];
    const int n = (int)(P.ptr[i + 1] - p0);
    if (n == 0) continue;                     // no view: out == 0 and nothing flows back
    const int nG = n * G;
    const float* __restrict__ cp = P.compat + p0 * G;
    float* __restrict__ gc = P.gcompat + p0 * G;
    const float m = P.s_max[i * G + gl];
    const float inv_den = 1.f / P.s_den[i * G + gl];
    const int arg_v = P.s_arg[i * G + gl];
    const float inv_sq = P.group_scaling ? rsqrtf((float)n) : 1.f;
    const float z = fmaf(gw, m, gb);
    const float t = gating ? tanhf(fmaxf(z, 0.f)) : 1.f;
    const bool one_chunk = n <= 32;
    float S = 0.f;                            // sum_v a_vg s'_vg for g = lane%G (partial per lane)

    // gd = dO * t of this lane's channels (single channel tile: loaded once per point)
    float gd[CPL][VEC];
    int gk[CPL]; uint32_t off[CPL]; bool live[CPL];
    auto load_gd = [&](int ct) {
#pragma unroll
      for (int k = 0; k < CPL; ++k) {
        if (single_tile) {
          gk[k] = gk0[k]; off[k] = off0[k]; live[k] = live0[k];
        } else {
          const int c0 = ct + (lir + LPR * k) * VEC;
          live[k] = c0 < C;
          const int cc = live[k] ? c0 : 0;
          gk[k] = group_of_channel(cc, C, G);
          off[k] = (uint32_t)cc * sizeof(T);
        }
        const float tk = __shfl_sync(0xffffffffu, t, gk[k]);
        load_chunk<T, VEC>(gob + i * (int64_t)row_bytes + off[k], gd[k]);
#pragma unroll
        for (int j = 0; j < VEC; ++j) gd[k][j] = live[k] ? gd[k][j] * tk : 0.f;   // dead lanes add 0
      }
    };
    if (single_tile) load_gd(0);

    for (int vs = 0; vs < n; vs += 32) {
      const int nc = min(32, n - vs);
      __syncwarp();
      for (int e = lane; e < nc * G; e += 32) {
        const int slot = gl * kTileStride + e / G;
        att_s[slot] = expf((__ldg(cp + vs * G + e) - m) * inv_sq) * inv_den;
        if (!assign_s) s_s[slot] = 0.f;
      }
      if (lane < nc) {
        const uint32_t lin = (uint32_t)(p0 + vs + lane);
        const uint32_t r = has_idx ? (uint32_t)load_idx(P.idx, P.idx64, p0 + vs + lane) : lin;
        row_s[lane] = r;
        orow_s[lane] = scatter ? r : lin;
      }
      __syncwarp();

      for (int ct = 0; ct < C; ct += TILE_C) {
        if (!single_tile) load_gd(ct);
        const uint32_t* rs = row_s + sg;
        const uint32_t* os = orow_s + sg;
        const float* as[CPL]; float* ss[CPL];
        const char* xk[CPL]; char* ok_[CPL];     // per-lane base pointers: row address = 1 IMAD.WIDE
#pragma unroll
        for (int k = 0; k < CPL; ++k) {
          as[k] = att_s + gk[k] * kTileStride + sg;
          ss[k] = s_s + gk[k] * kTileStride + sg;
          xk[k] = xb + off[k];
          ok_[k] = gxb + off[k];
        }

        // one row step: x chunk(s) of view v0+sg -> dx store + per-group dot product into s_s
        auto consume = [&](int v0, const Chunk<T, VEC> (&f)[CPL], bool ok) {
          const uint32_t orow = os[v0];
#pragma unroll
          for (int k = 0; k < CPL; ++k) {
            float fv[VEC], dx[VEC];
            f[k].get(fv);
            const float a = as[k][v0];
            float dot = 0.f;
#pragma unroll
            for (int j = 0; j < VEC; ++j) {
              dot = fmaf(gd[k][j], fv[j], dot);
              dx[j] = a * gd[k][j];
            }
            const bool lv = ok && live[k];
            if (lv) store_chunk<T, VEC>(row_addr(ok_[k], orow, row_bytes), dx);
            if constexpr (REG) {              // groups = aligned blocks of cpe lanes
              float r = dot;
#pragma unroll
              for (int b = 0; (1 << b) < LPR; ++b)
                r = fmaf(__shfl_xor_sync(0xffffffffu, r, 1 << b), red_mask[b], r);
              if (lv && leader) {
                if (assign_s) ss[k][v0] = r; else ss[k][v0] += r;
              }
            } else {                          // irregular group sizes: one reduction per group
              for (int g = 0; g < G; ++g) {
                const bool mine = lv && (gk[k] == g);
                if (!__any_sync(0xffffffffu, mine)) continue;
                float r = mine ? dot : 0.f;
#pragma unroll
                for (int o = 1; o < LPR; o <<= 1) r += __shfl_xor_sync(0xffffffffu, r, o);
                if (ok && lir == 0) s_s[g * kTileStride + sg + v0] += r;
              }
            }
          }
        };

        // main loop: U full row steps, all loads issued before the first use, no predicates
        int v0 = 0;
        for (; v0 + RPI * U <= nc; v0 += RPI * U) {
          Chunk<T, VEC> f[U][CPL];
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const uint32_t srow = rs[v0 + u * RPI];
#pragma unroll
            for (int k = 0; k < CPL; ++k) f[u][k].load(row_addr(xk[k], srow, row_bytes));
          }
#pragma unroll
          for (int u = 0; u < U; ++u) consume(v0 + u * RPI, f[u], true);
        }
        // tail: predicated blocks of UT row steps (kept narrow: a U-wide tail spills at 64 registers);
        // idle sub-groups still join the shuffles of consume()
        for (; v0 < nc; v0 += RPI * UT) {
          Chunk<T, VEC> f[UT][CPL];
          bool okv[UT];
#pragma unroll
          for (int u = 0; u < UT; ++u) {
            okv[u] = v0 + u * RPI + sg < nc;
            if (v0 + u * RPI < nc) {           // warp-uniform
              const uint32_t srow = okv[u] ? rs[v0 + u * RPI] : row_s[0];   // idle sub-group: a valid row
#pragma unroll
              for (int k = 0; k < CPL; ++k) f[u][k].load(row_addr(xk[k], srow, row_bytes));
            }
          }
#pragma unroll
          for (int u = 0; u < UT; ++u)
            if (v0 + u * RPI < nc) consume(okv[u] ? v0 + u * RPI : 0 - sg, f[u], okv[u]);   // warp-uniform guard
        }
        __syncwarp();
      }

      // S partial; raw s' -> grad_compat for long segments (finalised below once S is complete)
      for (int e = lane; e < nc * G; e += 32) {
        const int slot = gl * kTileStride + e / G;
        const float sv = s_s[slot];
        S = fmaf(att_s[slot], sv, S);
        if (!one_chunk) gc[vs * G + e] = sv;
      }
    }

    S = group_lane_sum(S, G);
    const float one_m_t2 = 1.f - t * t;
    const float dLdt = (t != 0.f) ? S / t : 0.f;
    const bool open = gating && z > 0.f;
    const float dq = open ? dLdt * one_m_t2 * gw : 0.f;
    if (open && lane < G) {
      dw_acc += dLdt * one_m_t2 * m;
      db_acc += dLdt * one_m_t2;
    }
    for (int e = lane; e < nG; e += 32) {
      float a, sv;
      if (one_chunk) { const int slot = gl * kTileStride + e / G; a = att_s[slot]; sv = s_s[slot]; }
      else { a = expf((__ldg(cp + e) - m) * inv_sq) * inv_den; sv = gc[e]; }
      float d = a * (sv - S) * inv_sq;
      if (p0 + e / G == arg_v) d += dq;
      gc[e] = d;
    }
  }

  // ---- gate parameter gradients: warp -> block partial (deterministic), block -> workspace
  if (P.gate_partial != nullptr) {
    if (lane < G) {
      gate_s[(warp * 2 + 0) * G + lane] = dw_acc;
      gate_s[(warp * 2 + 1) * G + lane] = db_acc;
    }
    __syncthreads();
    if (threadIdx.x < 2 * G) {
      float acc = 0.f;
      for (int w = 0; w < kWarps; ++w) acc += gate_s[w * 2 * G + threadIdx.x];
      P.gate_partial[(int64_t)blockIdx.x * 2 * G + threadIdx.x] = acc;
    }
  }
}

// one warp per output (2G <= 64 outputs): lanes stride over the CTA partials in a fixed order
__global__ void gate_reduce_kernel(const float* __restrict__ partial, float* __restrict__ out,
                                   int blocks, int twoG) {
  const int lane = threadIdx.x & 31;
  for (int j = threadIdx.x >> 5; j < twoG; j += blockDim.x >> 5) {
    float acc = 0.f;
    for (int b = lane; b < blocks; b += 32) acc += partial[(int64_t)b * twoG + j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) out[j] = acc;
  }
}

// ---------------------------------------------------------------------------------------------
// host dispatch
// ---------------------------------------------------------------------------------------------
struct VAConfig { int vec, lpr, cpl; bool reg; };

template <typename T>
static VAConfig choose_config(const VAParams& P, const void* o1, const void* o2, bool need_regular) {
  constexpr int V16 = Vec16<T>::N;
  const int C = P.C, G = P.G;
  bool vec_ok = (C % V16 == 0) && aligned16(P.x) && aligned16(o1) && (o2 == nullptr || aligned16(o2));
  if (vec_ok) {  // every 16-byte chunk must sit inside one channel group
    for (int c0 = 0; c0 < C && vec_ok; c0 += V16)
      if (group_of_channel(c0, C, G) != group_of_channel(c0 + V16 - 1, C, G)) vec_ok = false;
  }
  // regular layout: equal groups made of a power-of-two number of chunks
  auto regular = [&](int vec) {
    if (C % G != 0 || (C / G) % vec != 0) return false;
    const int cpg = (C / G) / vec;
    return (cpg & (cpg - 1)) == 0;
  };
  if (vec_ok && need_regular && !regular(V16)) vec_ok = false;   // irregular: scalar bwd kernels
  VAConfig cfg;
  if (!vec_ok) { cfg.vec = 1; cfg.lpr = 32; cfg.cpl = (C > 32) ? 4 : 1; cfg.reg = regular(1); return cfg; }
  const int cv = C / V16;
  cfg.vec = V16; cfg.reg = true;
  if (cv <= 4) { cfg.lpr = 4; cfg.cpl = 1; }
  else if (cv <= 8) { cfg.lpr = 8; cfg.cpl = 1; }
  else if (cv <= 16) { cfg.lpr = 16; cfg.cpl = 1; }
  else if (cv <= 32) { cfg.lpr = 32; cfg.cpl = 1; }
  else if (cv <= 64) { cfg.lpr = 32; cfg.cpl = 2; }
  else { cfg.lpr = 32; cfg.cpl = 4; }
  return cfg;
}

// persistent grid: exactly the number of CTAs that are co-resident (148 SMs x occupancy), so the
// grid-stride point loop has no second wave; never more CTAs than there are point groups.
template <typename K>
static int va_grid(K kern, size_t smem, int64_t N) {
  int occ = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kWarps * 32, smem) != cudaSuccess || occ < 1) occ = 2;
  int64_t blocks = (int64_t)kNumSMs * occ;
  const int64_t need = (N + kWarps - 1) / kWarps;
  if (blocks > need) blocks = need;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

constexpr int kMinBlocksFwd = DVA_FWD_MINB;   // x 8 warps / SM
constexpr int kMinBlocksBwd = DVA_BWD_MINB;

static size_t fwd_smem(int G) {
  return (size_t)kWarps * G * kTileStride * sizeof(float) + (size_t)kWarps * 32 * sizeof(uint32_t);
}
static size_t bwd_smem(int G) {
  return (size_t)2 * kWarps * G * kTileStride * sizeof(float) + (size_t)kWarps * 64 * sizeof(uint32_t) +
         (size_t)kWarps * 2 * G * sizeof(float);
}

template <typename T, int VEC, int LPR, int CPL>
static int launch_fwd(const VAParams& P, cudaStream_t st) {
  const size_t smem = fwd_smem(P.G);
  auto kern = view_attention_fwd_kernel<T, VEC, LPR, CPL, (CPL >= 4 ? 2 : kMinBlocksFwd)>;
  if (smem > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  kern<<<va_grid(kern, smem, P.N), kWarps * 32, smem, st>>>(P);
  return check_launch("view_attention_fwd");
}

template <typename T, int VEC, int LPR, int CPL, bool REG>
static int launch_bwd_k(const VAParams& P, int* grid_out, cudaStream_t st) {
  const size_t smem = bwd_smem(P.G);
  auto kern = view_attention_bwd_kernel<T, VEC, LPR, CPL, (CPL >= 4 ? 2 : kMinBlocksBwd), REG>;
  if (smem > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  const int grid = va_grid(kern, smem, P.N);
  *grid_out = grid;
  kern<<<grid, kWarps * 32, smem, st>>>(P);
  return check_launch("view_attention_bwd");
}

template <typename T, int VEC, int LPR, int CPL>
static int launch_bwd(const VAParams& P, bool reg, int* grid_out, cudaStream_t st) {
  if constexpr (VEC == 1) {
    if (!reg) return launch_bwd_k<T, VEC, LPR, CPL, false>(P, grid_out, st);
  }
  return launch_bwd_k<T, VEC, LPR, CPL, true>(P, grid_out, st);
}

#define DVA_VA_DISPATCH(FN, T, cfg, ...)                                                   \
  do {                                                                                     \
    constexpr int V16 = Vec16<T>::N;                                                       \
    if (cfg.vec == 1) {                                                                    \
      if (cfg.cpl == 1) return FN<T, 1, 32, 1>(__VA_ARGS__);                               \
      return FN<T, 1, 32, 4>(__VA_ARGS__);                                                 \
    }                                                                                      \
    if (cfg.lpr == 4) return FN<T, V16, 4, 1>(__VA_ARGS__);                                \
    if (cfg.lpr == 8) return FN<T, V16, 8, 1>(__VA_ARGS__);                                \
    if (cfg.lpr == 16) return FN<T, V16, 16, 1>(__VA_ARGS__);                              \
    if (cfg.cpl == 1) return FN<T, V16, 32, 1>(__VA_ARGS__);                               \
    if (cfg.cpl == 2) return FN<T, V16, 32, 2>(__VA_ARGS__);                               \
    return FN<T, V16, 32, 4>(__VA_ARGS__);                                                 \
  } while (0)

template <typename T> static int fwd_typed(const VAParams& P, cudaStream_t st) {
  const VAConfig cfg = choose_config<T>(P, P.out, nullptr, false);
  DVA_VA_DISPATCH(launch_fwd, T, cfg, P, st);
}
template <typename T> static int bwd_typed(const VAParams& P, int* grid, cudaStream_t st) {
  const VAConfig cfg = choose_config<T>(P, P.gout, P.gx, true);
  DVA_VA_DISPATCH(launch_bwd, T, cfg, P, cfg.reg, grid, st);
}

static bool pow2_le32(int64_t g) { return g >= 1 && g <= 32 && (g & (g - 1)) == 0; }

// 0 = auto, 1 = streaming kernels, 2 = ring forward + lane backward, 3 = lane backward + streaming forward
// (each where applicable).  Process-wide tuning knob (dva_view_attention_set_path /
// DVA_VA_PATH=auto|stream|ring|lane, read once); results do not depend on it.
static std::atomic<int>& va_path() {
  static std::atomic<int> p{[] {
    const char* e = getenv("DVA_VA_PATH");
    if (e == nullptr) return 0;
    if (strcmp(e, "stream") == 0) return 1;
    if (strcmp(e, "ring") == 0) return 2;
    if (strcmp(e, "lane") == 0) return 3;
    return 0;
  }()};
  return p;
}

// Short segments: the per-point scalar work dominates, and the ring forward / lane backward give it a
// lane per point or per view.  Auto (measured on B200, tools/bench_shapes.py, profiles/r1_shapes_*.json,
// profiles/r2_shapes_*.json): both need at most DVA_RING_MAX_MEAN_VIEWS views per point on average.
#ifndef DVA_RING_MAX_MEAN_VIEWS
#define DVA_RING_MAX_MEAN_VIEWS 12
#endif
static bool use_ring_fwd(const VAParams& P, bool applicable) {
  if (!applicable) return false;
  const int path = va_path().load(std::memory_order_relaxed);
  if (path == 1 || path == 3) return false;
  if (path == 2) return true;
  return P.V <= (int64_t)DVA_RING_MAX_MEAN_VIEWS * P.N;
}

// backward: the lane-per-view kernel (view_attention_lane.cu); auto also needs rows of at most 256 bytes --
// with 512-byte rows the streaming backward is as fast (1 M x 8 x 128: 1.85 ms vs 1.99 ms)
static bool use_lane_bwd(const VAParams& P, int dtype, bool applicable) {
  if (!applicable) return false;
  const int path = va_path().load(std::memory_order_relaxed);
  if (path == 2 || path == 3) return true;
  if (path == 1) return false;
  const size_t esz = dtype == DVA_F32 ? 4 : 2;
  return P.V <= (int64_t)DVA_RING_MAX_MEAN_VIEWS * P.N && (size_t)P.C * esz <= 256;
}

}  // namespace dva

using namespace dva;

extern "C" int dva_view_attention_fwd(const void* x, const void* idx, int idx_is_i64,
                                      const float* compat, const int64_t* ptr,
                                      const float* gate_w, const float* gate_b, void* out,
                                      float* att, float* seg_max, float* seg_den,
                                      int32_t* seg_arg, int64_t N, int64_t V, int64_t R,
                                      int64_t C, int64_t G, int group_scaling, float eps,
                                      int dtype, void* stream) {
  if (N < 0 || V < 0 || R < 0 || C < 1 || G < 1) return fail(DVA_EINVAL, "view_attention_fwd: bad sizes");
  if (G > C) return fail(DVA_EINVAL, "view_attention_fwd: num_groups > channels");
  if (!pow2_le32(G)) return fail(DVA_EUNSUPPORTED, "view_attention_fwd: G must be a power of two <= 32");
  if (C > (1 << 20)) return fail(DVA_EUNSUPPORTED, "view_attention_fwd: C too large");
  if (R >= (1ll << 32) || V >= (1ll << 32)) return fail(DVA_EUNSUPPORTED, "view_attention_fwd: more than 2^32 rows");
  if (N == 0) return DVA_OK;
  if (!ptr || !out || (V > 0 && (!x || !compat))) return fail(DVA_EINVAL, "view_attention_fwd: null pointer");
  if ((gate_w == nullptr) != (gate_b == nullptr)) return fail(DVA_EINVAL, "view_attention_fwd: gate_w/gate_b must both be given");
  if ((seg_max != nullptr) && (!seg_den || !seg_arg)) return fail(DVA_EINVAL, "view_attention_fwd: seg_max/seg_den/seg_arg go together");
  if (idx == nullptr && R < V) return fail(DVA_EINVAL, "view_attention_fwd: identity idx needs R >= V");
  VAParams P{};
  P.x = x; P.idx = idx; P.idx64 = idx_is_i64; P.compat = compat; P.ptr = ptr;
  P.gate_w = gate_w; P.gate_b = gate_b; P.out = out; P.att = att;
  P.seg_max = seg_max; P.seg_den = seg_den; P.seg_arg = seg_arg;
  P.N = N; P.V = V; P.R = R; P.C = (int)C; P.G = (int)G; P.group_scaling = group_scaling; P.eps = eps;
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype != DVA_F32 && dtype != DVA_BF16 && dtype != DVA_F16) return fail(DVA_EINVAL, "view_attention_fwd: unknown dtype");
  if (use_ring_fwd(P, va_ring_fwd_applicable(P, dtype))) return va_ring_fwd(P, dtype, st);
  switch (dtype) {
    case DVA_F32: return fwd_typed<float>(P, st);
    case DVA_BF16: return fwd_typed<__nv_bfloat16>(P, st);
    case DVA_F16: return fwd_typed<__half>(P, st);
    default: return fail(DVA_EINVAL, "view_attention_fwd: unknown dtype");
  }
}

extern "C" int dva_view_attention_set_path(int path) {
  if (path < 0 || path > 3) return fail(DVA_EINVAL, "view_attention_set_path: 0 = auto, 1 = streaming, 2 = ring, 3 = lane");
  va_path().store(path, std::memory_order_relaxed);
  return DVA_OK;
}

extern "C" size_t dva_view_attention_bwd_workspace_bytes(int64_t G) {
  // one [2,G] partial per CTA of the persistent grid (at most 148 SMs x 8 co-resident CTAs)
  return (size_t)kNumSMs * 8 * 2 * (size_t)(G > 0 ? G : 1) * sizeof(float);
}

extern "C" int dva_view_attention_bwd(const void* x, const void* idx, int idx_is_i64,
                                      const float* compat, const int64_t* ptr,
                                      const float* gate_w, const float* gate_b,
                                      const void* grad_out, const float* seg_max,
                                      const float* seg_den, const int32_t* seg_arg,
                                      void* grad_x_rows, float* grad_compat, float* grad_gate,
                                      int scatter_rows, int64_t N, int64_t V, int64_t R,
                                      int64_t C, int64_t G, int group_scaling, int dtype,
                                      void* workspace, size_t workspace_bytes, void* stream) {
  if (N < 0 || V < 0 || R < 0 || C < 1 || G < 1) return fail(DVA_EINVAL, "view_attention_bwd: bad sizes");
  if (G > C) return fail(DVA_EINVAL, "view_attention_bwd: num_groups > channels");
  if (!pow2_le32(G)) return fail(DVA_EUNSUPPORTED, "view_attention_bwd: G must be a power of two <= 32");
  if (R >= (1ll << 32) || V >= (1ll << 32)) return fail(DVA_EUNSUPPORTED, "view_attention_bwd: more than 2^32 rows");
  const bool gating = gate_w != nullptr;
  if (gating != (gate_b != nullptr)) return fail(DVA_EINVAL, "view_attention_bwd: gate_w/gate_b must both be given");
  cudaStream_t st = (cudaStream_t)stream;
  if (N == 0 || V == 0) {
    if (gating && grad_gate) cudaMemsetAsync(grad_gate, 0, 2 * G * sizeof(float), st);
    return DVA_OK;
  }
  if (!x || !compat || !ptr || !grad_out || !seg_max || !seg_den || !seg_arg || !grad_x_rows || !grad_compat)
    return fail(DVA_EINVAL, "view_attention_bwd: null pointer");
  if (gating && (!grad_gate || !workspace || workspace_bytes < dva_view_attention_bwd_workspace_bytes(G)))
    return fail(DVA_EINVAL, "view_attention_bwd: gating needs grad_gate and workspace");
  VAParams P{};
  P.x = x; P.idx = idx; P.idx64 = idx_is_i64; P.compat = compat; P.ptr = ptr;
  P.gate_w = gate_w; P.gate_b = gate_b; P.gout = grad_out;
  P.s_max = seg_max; P.s_den = seg_den; P.s_arg = seg_arg;
  P.gx = grad_x_rows; P.gcompat = grad_compat; P.scatter = scatter_rows;
  P.gate_partial = gating ? reinterpret_cast<float*>(workspace) : nullptr;
  P.N = N; P.V = V; P.R = R; P.C = (int)C; P.G = (int)G; P.group_scaling = group_scaling;
  int grid = 1;
  int rc;
  if (dtype != DVA_F32 && dtype != DVA_BF16 && dtype != DVA_F16) return fail(DVA_EINVAL, "view_attention_bwd: unknown dtype");
  if (use_lane_bwd(P, dtype, va_lane_bwd_applicable(P, dtype))) {
    rc = va_lane_bwd(P, dtype, &grid, st);
  } else {
    switch (dtype) {
      case DVA_F32: rc = bwd_typed<float>(P, &grid, st); break;
      case DVA_BF16: rc = bwd_typed<__nv_bfloat16>(P, &grid, st); break;
      default: rc = bwd_typed<__half>(P, &grid, st); break;
    }
  }
  if (rc) return rc;
  if (gating) {
    gate_reduce_kernel<<<1, 1024, 0, st>>>(P.gate_partial, grad_gate, grid, 2 * (int)G);
    return check_launch("gate_reduce");
  }
  return DVA_OK;
}
