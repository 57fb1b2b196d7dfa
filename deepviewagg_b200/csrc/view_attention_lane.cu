// "Lane per view" backward of the fused view-attention pair for SHORT segments (the shapes every shipped
// config runs: S3DIS / ScanNet ~7 views per point, rows of 128 .. 512 bytes).  Same math and C ABI as
// view_attention.cu (reference chain: modules.py:518 row gather -> pooling.py:285-300 / 515-530, gradients
// SURVEY.md Appendix A); the short-segment backward next to the streaming kernels and the ring forward.
//
// Why.  ncu at the S3DIS step shape: the streaming backward spends a whole warp on one point at a time
// (836 warp instructions per point, issue-bound); a backward on the ring of view_attention_ring.cu halved the
// instruction count but its 29 KB of shared memory per warp left 8 warps per SM (21 % issue-active,
// latency-bound): 0.47 of the HBM peak.  Here a warp takes a GROUP of consecutive points holding at most 32
// views and gives every kind of work its natural SIMT shape, with registers and ~2.8 KB of shared memory per
// warp (32+ warps per SM):
//   phase 1  LANE PER VIEW: scores, row id, the point's saved statistics -> attentions a, gate t (32 views
//            per instruction; coalesced 16-byte score loads);
//   phase 1b EVERY VIEW LANE issues ONE bulk async copy (cp.async.bulk -> UBLKCP) of its own row into the
//            warp's shared-memory row buffer, completion on the warp's mbarrier: up to 32 rows in flight per
//            warp for one instruction slot each and no registers (the register-only first version had 40 KB
//            in flight per SM and sat at 0.54 of the peak, latency-bound; this one 0.63 / 0.76 at 160 k / 1 M
//            points x 7 views x 64 ch).  Tried and dropped: a second row buffer with the next group's copies
//            issued one group ahead -- twice the shared memory (12 instead of 20 warps per SM) and fewer
//            rows per step in flight made it 1.8x SLOWER;
//   phase 2  SUB-WARP PER ROW: LPR lanes own the 16-byte chunks of a row, 32 / LPR rows per step: x row out
//            of shared memory (LDS.128), grad_out row of the view's point through L1; dx = (a t) grad_out
//            stored once, raw dot <grad_out, x> per group to a tile;
//   phase 3  LANE PER POINT then LANE PER VIEW: S = sum_v a s', gate gradients; grad_compat stored as one
//            coalesced float4 per lane.
// A point with more than 32 views (never in the short-segment regime this kernel is dispatched for) is
// walked in chunks of 32 views with its raw s' parked in grad_compat.
// Requires G == 4 and the regular channel layout (a row is LPR = 4 * 2^k chunks of 16 bytes, <= 512 bytes).
// HBM bytes per launch: those of the streaming backward (V (2 C s + 4 + 8 G) + N (C s + 8 + 12 G)).
#include "view_attention.cuh"

namespace dva {

constexpr int kLaneWarps = 4;
constexpr uint32_t kFull = 0xffffffffu;

struct LaneSmem {            // per warp
  float wt[32][4];           // a * t per (view, group)
  float at[32][4];           // a
  float st[32][4];           // raw dot <grad_out, x> per (view, group)
  float Sp[32][4];           // per point: S
  float dq[32][4];           // per point: gate term routed to the arg-max view
  uint32_t ri[32];           // x row of the view
  uint32_t orow[32];         // dx row of the view
  uint32_t go[32];           // point of the view (grad_out row), relative to the group's first point
  uint64_t bar;              // completion of the group's row copies
  uint64_t pad;
};

template <typename T, int LPR>
__global__ void __launch_bounds__(kLaneWarps * 32, 5)
va_lane_bwd_kernel(const VAParams P, const int PR) {
  constexpr int VEC = Vec16<T>::N, RPI = 32 / LPR, CPE = LPR / 4, G = 4, U = 4, RS = LPR * 16;
  extern __shared__ __align__(128) unsigned char rows_all[];       // [kLaneWarps][32 rows][RS bytes]
  __shared__ LaneSmem sm_all[kLaneWarps];
  __shared__ float gate_s[kLaneWarps][8];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  LaneSmem& sm = sm_all[warp];
  unsigned char* rows_s = rows_all + (size_t)warp * 32 * RS;
  const uint32_t rows_u = smem_u32(rows_s), bar_u = smem_u32(&sm.bar);
  uint32_t uses = 0;                                              // completed uses of the barrier (parity)
  if (lane == 0) {
    mbar_init(bar_u, 1);
    fence_mbar_init();
  }
  __syncwarp();
  const int sg = lane / LPR, lir = lane % LPR, gk = lir / CPE;
  const uint32_t row_bytes = (uint32_t)P.C * sizeof(T);           // == RS (host checks C / VEC == LPR)
  const char* __restrict__ xbase = reinterpret_cast<const char*>(P.x);
  const char* __restrict__ gob = reinterpret_cast<const char*>(P.gout) + lir * 16;
  char* __restrict__ gxb = reinterpret_cast<char*>(P.gx) + lir * 16;
  const bool gating = P.gate_w != nullptr;
  float4 gw4 = make_float4(0.f, 0.f, 0.f, 0.f), gb4 = gw4;
  if (gating) {
    gw4 = make_float4(P.gate_w[0], P.gate_w[1], P.gate_w[2], P.gate_w[3]);
    gb4 = make_float4(P.gate_b[0], P.gate_b[1], P.gate_b[2], P.gate_b[3]);
  }
  float4 dw4 = make_float4(0.f, 0.f, 0.f, 0.f), db4 = dw4;         // gate gradients (lane partials)
  const bool scatter = P.scatter && P.idx != nullptr;

  // every view lane copies its own row into the warp's buffer; wait_rows() before the rows are read
  auto issue_rows = [&](int nv, uint32_t rid) {
    fence_proxy_async();                                     // earlier generic reads of the buffer come first
    __syncwarp();
    if (lane == 0) mbar_expect_tx(bar_u, (uint32_t)nv * row_bytes);
    __syncwarp();
    if (lane < nv) bulk_g2s(rows_u + (uint32_t)lane * RS, xbase + (uint64_t)rid * row_bytes, row_bytes, bar_u);
  };
  auto wait_rows = [&]() {
    mbar_wait(bar_u, uses & 1u);
    ++uses;
  };

  // rows of the views [0, nv) of the current tile: dx stores + raw dots -> sm.st
  auto rows_phase = [&](int nv, int64_t pg) {
    for (int u0 = 0; u0 < nv; u0 += RPI * U) {
      uint4 xr[U], gr[U];
      float w[U];
      uint32_t orow[U];
      bool ok[U];
#pragma unroll
      for (int q = 0; q < U; ++q) {
        const int u = u0 + q * RPI + sg;
        ok[q] = u < nv;
        const int uu = ok[q] ? u : 0;
        orow[q] = sm.orow[uu];
        w[q] = sm.wt[uu][gk];
        xr[q] = *reinterpret_cast<const uint4*>(rows_s + (size_t)uu * RS + lir * 16);
        gr[q] = *reinterpret_cast<const uint4*>(gob + (uint64_t)(pg + sm.go[uu]) * row_bytes);   // reused by the point's views: cached
      }
#pragma unroll
      for (int q = 0; q < U; ++q) {
        float fx[VEC], fg[VEC], dx[VEC];
        unpack16<T, VEC>(xr[q], fx);
        unpack16<T, VEC>(gr[q], fg);
        float dot = 0.f;
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
          dot = fmaf(fg[j], fx[j], dot);
          dx[j] = w[q] * fg[j];
        }
        if (ok[q]) stg_stream16(gxb + (uint64_t)orow[q] * row_bytes, pack16<T, VEC>(dx));
#pragma unroll
        for (int o = 1; o < CPE; o <<= 1) dot += __shfl_xor_sync(kFull, dot, o);
        if (ok[q] && (lir & (CPE - 1)) == 0) sm.st[u0 + q * RPI + sg][gk] = dot;
      }
    }
  };

  const int64_t n_ranges = (P.N + PR - 1) / PR;
  const int64_t warps_total = (int64_t)gridDim.x * kLaneWarps;
  for (int64_t r = (int64_t)blockIdx.x * kLaneWarps + warp; r < n_ranges; r += warps_total) {
    const int64_t pa = r * PR;
    const int64_t pb = (pa + PR < P.N) ? pa + PR : P.N;
    for (int64_t pg = pa; pg < pb;) {
      // ---- group: lane k looks at point pg + k
      const int64_t pk = pg + lane;
      const bool valid = pk < pb;
      const int64_t p0 = valid ? P.ptr[pk] : 0;
      const int cnt = valid ? (int)(P.ptr[pk + 1] - p0) : 0;
      int incl = cnt;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(kFull, incl, o);
        if (lane >= o) incl += t;
      }
      const int excl = incl - cnt;
      const unsigned fitm = __ballot_sync(kFull, valid && incl <= 32);
      const int kfit = (fitm == kFull) ? 32 : __ffs(~fitm) - 1;
      const int64_t gvb = __shfl_sync(kFull, p0, 0);                // first view of the group

      if (kfit == 0) {
        // ---- one point with more than 32 views: chunks of 32 views, raw s' parked in grad_compat
        const int n = __shfl_sync(kFull, cnt, 0);
        const float4 smx = reinterpret_cast<const float4*>(P.s_max)[pg];
        const float4 sdn = reinterpret_cast<const float4*>(P.s_den)[pg];
        const int4 sar = reinterpret_cast<const int4*>(P.s_arg)[pg];
        const float inv_sq = P.group_scaling ? rsqrtf((float)n) : 1.f;
        float4 z4 = make_float4(1.f, 1.f, 1.f, 1.f), t4 = z4;
        if (gating) {
          z4 = make_float4(fmaf(gw4.x, smx.x, gb4.x), fmaf(gw4.y, smx.y, gb4.y), fmaf(gw4.z, smx.z, gb4.z), fmaf(gw4.w, smx.w, gb4.w));
          t4 = make_float4(tanhf(fmaxf(z4.x, 0.f)), tanhf(fmaxf(z4.y, 0.f)), tanhf(fmaxf(z4.z, 0.f)), tanhf(fmaxf(z4.w, 0.f)));
        }
        float4 Sacc = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int c0 = 0; c0 < n; c0 += 32) {
          const int nv = (n - c0 < 32) ? n - c0 : 32;
          const int64_t v = gvb + c0 + lane;
          float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
          __syncwarp();
          const uint32_t rid_l = lane < nv ? load_row_id(P.idx, P.idx64, v) : 0u;
          issue_rows(nv, rid_l);
          if (lane < nv) {
            const float4 c = __ldg(reinterpret_cast<const float4*>(P.compat) + v);
            a = make_float4(__expf((c.x - smx.x) * inv_sq) / sdn.x, __expf((c.y - smx.y) * inv_sq) / sdn.y,
                            __expf((c.z - smx.z) * inv_sq) / sdn.z, __expf((c.w - smx.w) * inv_sq) / sdn.w);
            sm.ri[lane] = rid_l;
            sm.orow[lane] = scatter ? rid_l : (uint32_t)v;
            sm.go[lane] = 0u;
            *reinterpret_cast<float4*>(sm.wt[lane]) = make_float4(a.x * t4.x, a.y * t4.y, a.z * t4.z, a.w * t4.w);
          }
          __syncwarp();
          wait_rows();
          rows_phase(nv, pg);
          __syncwarp();
          if (lane < nv) {
            const float4 raw = *reinterpret_cast<const float4*>(sm.st[lane]);
            const float4 sp = make_float4(raw.x * t4.x, raw.y * t4.y, raw.z * t4.z, raw.w * t4.w);
            Sacc.x = fmaf(a.x, sp.x, Sacc.x); Sacc.y = fmaf(a.y, sp.y, Sacc.y);
            Sacc.z = fmaf(a.z, sp.z, Sacc.z); Sacc.w = fmaf(a.w, sp.w, Sacc.w);
            reinterpret_cast<float4*>(P.gcompat)[v] = sp;           // finalised below once S is complete
          }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          Sacc.x += __shfl_xor_sync(kFull, Sacc.x, o); Sacc.y += __shfl_xor_sync(kFull, Sacc.y, o);
          Sacc.z += __shfl_xor_sync(kFull, Sacc.z, o); Sacc.w += __shfl_xor_sync(kFull, Sacc.w, o);
        }
        float4 dq = make_float4(0.f, 0.f, 0.f, 0.f);
        if (gating) {
#define DVA_LGATE(c)                                                                       \
          if (z4.c > 0.f) {                                                                \
            const float dLdt = (t4.c != 0.f) ? Sacc.c / t4.c : 0.f;                         \
            const float uu = dLdt * (1.f - t4.c * t4.c);                                   \
            dq.c = uu * gw4.c;                                                             \
            if (lane == 0) { dw4.c += uu * smx.c; db4.c += uu; }                           \
          }
          DVA_LGATE(x) DVA_LGATE(y) DVA_LGATE(z) DVA_LGATE(w)
#undef DVA_LGATE
        }
        __syncwarp();
        for (int c0 = lane; c0 < n; c0 += 32) {
          const int64_t v = gvb + c0;
          const float4 c = __ldg(reinterpret_cast<const float4*>(P.compat) + v);
          const float4 sp = __ldcg(reinterpret_cast<const float4*>(P.gcompat) + v);
          float4 d;
          d.x = __expf((c.x - smx.x) * inv_sq) / sdn.x * (sp.x - Sacc.x) * inv_sq;
          d.y = __expf((c.y - smx.y) * inv_sq) / sdn.y * (sp.y - Sacc.y) * inv_sq;
          d.z = __expf((c.z - smx.z) * inv_sq) / sdn.z * (sp.z - Sacc.z) * inv_sq;
          d.w = __expf((c.w - smx.w) * inv_sq) / sdn.w * (sp.w - Sacc.w) * inv_sq;
          if ((int)v == sar.x) d.x += dq.x;
          if ((int)v == sar.y) d.y += dq.y;
          if ((int)v == sar.z) d.z += dq.z;
          if ((int)v == sar.w) d.w += dq.w;
          reinterpret_cast<float4*>(P.gcompat)[v] = d;
        }
        pg += 1;
        continue;
      }

      // ---- phase 1: lane u owns view gvb + u of the group (nv <= 32 views over kfit points)
      const int nv = __shfl_sync(kFull, incl, kfit - 1);
      int mp = 0;                                                   // point (relative to pg) of my view
      for (int k = 0; k < kfit; ++k) {
        const int s = __shfl_sync(kFull, excl, k), c = __shfl_sync(kFull, cnt, k);
        if (lane >= s && lane < s + c) mp = k;
      }
      const int cntp = __shfl_sync(kFull, cnt, mp);
      float4 a = make_float4(0.f, 0.f, 0.f, 0.f), t4 = make_float4(1.f, 1.f, 1.f, 1.f);
      float inv_sq = 1.f;
      int4 sar = make_int4(-1, -1, -1, -1);
      const int64_t v = gvb + lane;
      __syncwarp();                                                 // previous group's tiles are free
      const uint32_t rid_m = lane < nv ? load_row_id(P.idx, P.idx64, v) : 0u;
      if (nv > 0) issue_rows(nv, rid_m);                            // rows go in flight before anything else is loaded
      if (lane < nv) {
        const float4 c = __ldg(reinterpret_cast<const float4*>(P.compat) + v);
        const float4 smx = reinterpret_cast<const float4*>(P.s_max)[pg + mp];
        const float4 sdn = reinterpret_cast<const float4*>(P.s_den)[pg + mp];
        sar = reinterpret_cast<const int4*>(P.s_arg)[pg + mp];
        inv_sq = P.group_scaling ? rsqrtf((float)cntp) : 1.f;
        a = make_float4(__expf((c.x - smx.x) * inv_sq) / sdn.x, __expf((c.y - smx.y) * inv_sq) / sdn.y,
                        __expf((c.z - smx.z) * inv_sq) / sdn.z, __expf((c.w - smx.w) * inv_sq) / sdn.w);
        if (gating)
          t4 = make_float4(tanhf(fmaxf(fmaf(gw4.x, smx.x, gb4.x), 0.f)), tanhf(fmaxf(fmaf(gw4.y, smx.y, gb4.y), 0.f)),
                           tanhf(fmaxf(fmaf(gw4.z, smx.z, gb4.z), 0.f)), tanhf(fmaxf(fmaf(gw4.w, smx.w, gb4.w), 0.f)));
        sm.ri[lane] = rid_m;
        sm.orow[lane] = scatter ? rid_m : (uint32_t)v;
        sm.go[lane] = (uint32_t)mp;
        *reinterpret_cast<float4*>(sm.at[lane]) = a;
        *reinterpret_cast<float4*>(sm.wt[lane]) = make_float4(a.x * t4.x, a.y * t4.y, a.z * t4.z, a.w * t4.w);
      }
      __syncwarp();

      // ---- phase 2: rows
      if (nv > 0) wait_rows();
      rows_phase(nv, pg);
      __syncwarp();

      // ---- phase 3a: lane k owns point pg + k: S = sum_v a s', gate gradients
      if (lane < nv) {                                              // s' = t * raw dot, in place
        float4 raw = *reinterpret_cast<const float4*>(sm.st[lane]);
        raw.x *= t4.x; raw.y *= t4.y; raw.z *= t4.z; raw.w *= t4.w;
        *reinterpret_cast<float4*>(sm.st[lane]) = raw;
      }
      __syncwarp();
      if (lane < kfit) {
        float4 S = make_float4(0.f, 0.f, 0.f, 0.f), dq = S;
        for (int j = 0; j < cnt; ++j) {
          const float4 aa = *reinterpret_cast<const float4*>(sm.at[excl + j]);
          const float4 sv = *reinterpret_cast<const float4*>(sm.st[excl + j]);
          S.x = fmaf(aa.x, sv.x, S.x); S.y = fmaf(aa.y, sv.y, S.y); S.z = fmaf(aa.z, sv.z, S.z); S.w = fmaf(aa.w, sv.w, S.w);
        }
        if (gating && cnt > 0) {
          const float4 smx = reinterpret_cast<const float4*>(P.s_max)[pk];
#define DVA_LGATE(c)                                                                       \
          {                                                                                \
            const float z = fmaf(gw4.c, smx.c, gb4.c);                                     \
            if (z > 0.f) {                                                                 \
              const float t = tanhf(z);                                                    \
              const float dLdt = (t != 0.f) ? S.c / t : 0.f;                               \
              const float uu = dLdt * (1.f - t * t);                                       \
              dq.c = uu * gw4.c; dw4.c += uu * smx.c; db4.c += uu;                         \
            }                                                                              \
          }
          DVA_LGATE(x) DVA_LGATE(y) DVA_LGATE(z) DVA_LGATE(w)
#undef DVA_LGATE
        }
        *reinterpret_cast<float4*>(sm.Sp[lane]) = S;
        *reinterpret_cast<float4*>(sm.dq[lane]) = dq;
      }
      __syncwarp();
      // ---- phase 3b: lane per view: grad_compat
      if (lane < nv) {
        const float4 S = *reinterpret_cast<const float4*>(sm.Sp[mp]);
        const float4 dq = *reinterpret_cast<const float4*>(sm.dq[mp]);
        const float4 sv = *reinterpret_cast<const float4*>(sm.st[lane]);
        float4 d;
        d.x = a.x * (sv.x - S.x) * inv_sq; d.y = a.y * (sv.y - S.y) * inv_sq;
        d.z = a.z * (sv.z - S.z) * inv_sq; d.w = a.w * (sv.w - S.w) * inv_sq;
        if ((int)v == sar.x) d.x += dq.x;
        if ((int)v == sar.y) d.y += dq.y;
        if ((int)v == sar.z) d.z += dq.z;
        if ((int)v == sar.w) d.w += dq.w;
        reinterpret_cast<float4*>(P.gcompat)[v] = d;
      }
      pg += kfit;
    }
  }

  // ---- gate parameter gradients: lanes -> warp -> block partial (fixed order), block -> workspace
  if (P.gate_partial != nullptr) {
    float vv[8] = {dw4.x, dw4.y, dw4.z, dw4.w, db4.x, db4.y, db4.z, db4.w};
#pragma unroll
    for (int q = 0; q < 8; ++q) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) vv[q] += __shfl_xor_sync(kFull, vv[q], o);
    }
    if (lane == 0) {
#pragma unroll
      for (int q = 0; q < 8; ++q) gate_s[warp][q] = vv[q];
    }
    __syncthreads();
    if ((int)threadIdx.x < 2 * G) {
      float acc = 0.f;
      for (int w = 0; w < kLaneWarps; ++w) acc += gate_s[w][threadIdx.x];
      P.gate_partial[(int64_t)blockIdx.x * 2 * G + threadIdx.x] = acc;
    }
  }
}

template <typename T> static bool lane_bwd_ok(const VAParams& P) {
  constexpr int V16 = Vec16<T>::N;
  const int C = P.C;
  if (P.G != 4 || C % V16 != 0 || C / V16 > 32 || C / V16 < 4) return false;
  const int cv = C / V16;
  if ((cv & (cv - 1)) != 0) return false;                       // a row is exactly LPR = 4, 8, 16 or 32 chunks
  if (!aligned16(P.x) || !aligned16(P.gout) || !aligned16(P.gx) || !aligned16(P.compat) || !aligned16(P.gcompat)) return false;
  if (!aligned16(P.s_max) || !aligned16(P.s_den) || !aligned16(P.s_arg)) return false;
  if (P.V >= (1ll << 31) || P.R >= (1ll << 32)) return false;
  return true;
}

bool va_lane_bwd_applicable(const VAParams& P, int dtype) {
  switch (dtype) {
    case DVA_F32: return lane_bwd_ok<float>(P);
    case DVA_BF16: return lane_bwd_ok<__nv_bfloat16>(P);
    case DVA_F16: return lane_bwd_ok<__half>(P);
    default: return false;
  }
}

template <typename T, int LPR>
static int lane_bwd_launch(const VAParams& P, int* grid_out, cudaStream_t st) {
  auto kern = va_lane_bwd_kernel<T, LPR>;
  const size_t smem = (size_t)kLaneWarps * 32 * LPR * 16;          // row buffers: 32 rows per warp
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return fail((int)e, "va_lane_bwd: cannot reserve shared memory");
  int occ = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kLaneWarps * 32, smem) != cudaSuccess || occ < 1) occ = 1;
  if (occ > 8) occ = 8;                                          // gate partials: at most 148 x 8 CTAs
  int64_t grid = (int64_t)kNumSMs * occ;
  const int64_t warps = grid * kLaneWarps;
  int64_t pr = (P.N + warps * 4 - 1) / (warps * 4);              // ~4 ranges per warp: balances ragged counts
  if (pr < 8) pr = 8;
  const int64_t n_ranges = (P.N + pr - 1) / pr;
  const int64_t need = (n_ranges + kLaneWarps - 1) / kLaneWarps;
  if (grid > need) grid = need;
  if (grid < 1) grid = 1;
  kern<<<(unsigned)grid, kLaneWarps * 32, smem, st>>>(P, (int)pr);
  *grid_out = (int)grid;
  return check_launch("va_lane_bwd");
}

template <typename T>
static int lane_bwd_typed(const VAParams& P, int* grid_out, cudaStream_t st) {
  switch (P.C / Vec16<T>::N) {
    case 4: return lane_bwd_launch<T, 4>(P, grid_out, st);
    case 8: return lane_bwd_launch<T, 8>(P, grid_out, st);
    case 16: return lane_bwd_launch<T, 16>(P, grid_out, st);
    default: return lane_bwd_launch<T, 32>(P, grid_out, st);
  }
}

int va_lane_bwd(const VAParams& P, int dtype, int* grid_out, cudaStream_t st) {
  switch (dtype) {
    case DVA_F32: return lane_bwd_typed<float>(P, grid_out, st);
    case DVA_BF16: return lane_bwd_typed<__nv_bfloat16>(P, grid_out, st);
    default: return lane_bwd_typed<__half>(P, grid_out, st);
  }
}

}  // namespace dva
