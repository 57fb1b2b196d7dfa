// Ring forward of the fused view-attention pair (same math and C ABI as view_attention.cu;
// reference chain: modules.py:518 row gather -> pooling.py:285-300 / 515-530).
//
// Why a second forward.  ncu on the shipped-config shapes (S3DIS: 160 k points x ~8 views x 64 ch)
// shows the streaming kernels ISSUE-bound, not HBM-bound: ~590 warp instructions per point, of which
// only ~40 touch feature rows -- the rest is per-point scalar work (softmax statistics, gating,
// pointer chasing) executed by a whole warp for one point at a time.  Here the two kinds of work get
// the SIMT shape that suits them:
//
//   * a warp owns a contiguous RANGE of points = a contiguous range of views, and streams that
//     range's feature rows through a shared-memory ring as fixed-size BATCHES that ignore point
//     boundaries: one 16-byte cp.async (LDGSTS) per lane and row step, S-1 batches in flight, row
//     ids prefetched a batch ahead into one register per lane -- no load of the consumer sits on a
//     dependent-address chain;
//   * the consumer walks the range in GROUPS of up to 32 points (at most 256 views):
//       phase 1  LANE PER POINT: every lane computes the softmax statistics of its own point
//                (max, first arg-max, denominator, gate) from the fp32 scores and leaves the final
//                per-view weights e * t / den in a shared tile -- 32 points per instruction;
//       phase 2  WARP PER ROW STEP: per point, weighted sum of its rows out of the ring
//                (LDS.128 row chunk + LDS weight + VEC FFMA per row step), no arithmetic besides;
//   * a point with more views than a group holds (never in the shipped configs) takes a
//     warp-cooperative path: online softmax over the pieces of its segment.
//
// The backward of these shapes is the lane-per-view kernel (view_attention_lane.cu).
// Requires G == 4 (every shipped config), rows of whole 16-byte chunks and at most 512 bytes;
// everything else runs on the streaming kernels.  HBM bytes per launch are those of the streaming
// kernels (see view_attention.cu).  exp is ex2.approx-based here (relative error ~1e-6).
#include "view_attention.cuh"

namespace dva {

#ifndef DVA_RING_STAGES
#define DVA_RING_STAGES 3
#endif
#ifndef DVA_RING_WARPS
#define DVA_RING_WARPS 1
#endif
#ifndef DVA_RING_FWD_MINB
#define DVA_RING_FWD_MINB 12      // CTAs per SM the register budget is sized for (x kRingWarps warps)
#endif
#ifndef DVA_RING_CAPV_FWD
#define DVA_RING_CAPV_FWD 256     // views per point group (weight tile), multiple of 8
#endif
constexpr int kRingStages = DVA_RING_STAGES;
constexpr int kRingWarps = DVA_RING_WARPS;     // warps of a CTA never synchronise with each other
constexpr int kRG = 4;                          // groups
constexpr uint32_t FULL = 0xffffffffu;
#ifndef DVA_RING_P1_UNROLL
#define DVA_RING_P1_UNROLL 8
#endif
constexpr int kP1Unroll = DVA_RING_P1_UNROLL;   // score loads in flight per lane in the lane-per-point phases

// Batch size (measured, tools/bench_shapes.py): 16 rows per batch for 128/256-byte rows and more
// resident warps (2 KB batches) for 64- and 512-byte rows.
template <int LPR> struct RingGeom {
  static constexpr int RPI = 32 / LPR;                       // rows per warp step
  static constexpr int RS = LPR * 16;                        // row stride in the ring (bytes)
#ifdef DVA_RING_BATCH_BYTES
  static constexpr int BATCH = DVA_RING_BATCH_BYTES;
#else
  static constexpr int BATCH = LPR == 16 ? 4096 : 2048;
#endif
  static constexpr int RB = (BATCH / RS) < 32 ? (BATCH / RS) : 32;   // rows per batch
  static constexpr int STEPS = RB / RPI;                     // row steps per batch
  static constexpr int MINB = BATCH <= 2048 ? 16 : DVA_RING_FWD_MINB;
  static_assert(RB >= RPI && RB % RPI == 0 && (RB & (RB - 1)) == 0, "batch geometry");
};

__device__ __forceinline__ void prefetch_l2(const void* p) {
  asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
}

// the weight tile holds one float4 (4 groups) per view, 8 views per 36-float row: lanes
// that walk their own points at a stride of 8k views still hit distinct banks
__device__ __forceinline__ int tix(int u) { return (u + (u >> 3)) << 2; }
constexpr int tile_floats(int capv) { return (capv / 8) * 36; }

__device__ __forceinline__ float sel4(const float4& v, int g) {
  return g == 0 ? v.x : (g == 1 ? v.y : (g == 2 ? v.z : v.w));
}

// per-warp shared memory (bytes): the ring, the weight tile, the output scale per point of the group
template <int LPR> struct RingSmem {
  using Gm = RingGeom<LPR>;
  size_t rows, tile, tpt, total;
  __host__ __device__ RingSmem() {
    rows = (size_t)kRingStages * Gm::RB * Gm::RS;
    tile = (size_t)tile_floats(DVA_RING_CAPV_FWD) * sizeof(float);
    tpt = (size_t)32 * kRG * sizeof(float);
    total = rows + tile + tpt;
  }
};

// window of points [pg, pg + 32): lane k holds the range-relative first view and the view count
// of point pg + k (0 views past the end of the range)
__device__ __forceinline__ void load_window(const int64_t* __restrict__ ptr, int64_t pg, int64_t pb,
                                            int64_t vb, int lane, int& pl, int& cnt) {
  const int64_t q0 = (pg + lane < pb) ? pg + lane : pb;
  const int64_t q1 = (q0 + 1 < pb) ? q0 + 1 : pb;
  pl = (int)(ptr[q0] - vb);
  cnt = (int)(ptr[q1] - vb) - pl;
}

template <typename T, int LPR>
__global__ void __launch_bounds__(kRingWarps * 32, RingGeom<LPR>::MINB)
va_ring_fwd_kernel(const VAParams P, const int PR) {
  using Gm = RingGeom<LPR>;
  constexpr int VEC = Vec16<T>::N, RPI = Gm::RPI, RB = Gm::RB, RS = Gm::RS, S = kRingStages;
  constexpr int G = kRG, CAPV = DVA_RING_CAPV_FWD;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int C = P.C;
  const RingSmem<LPR> L;
  unsigned char* base = smem_raw + (size_t)warp * L.total;
  unsigned char* rows_s = base;
  float* wt = reinterpret_cast<float*>(base + L.rows);
  float* spt = reinterpret_cast<float*>(base + L.rows + L.tile);   // output scale per point of the group
  const uint32_t rows_u = smem_u32(rows_s);

  // dead chunks (lanes past the end of a row) are never copied: keep them zero for good
  for (int q = lane; q < (int)(L.rows / 16); q += 32) reinterpret_cast<uint4*>(rows_s)[q] = make_uint4(0u, 0u, 0u, 0u);
  __syncwarp();

  const int sg = lane / LPR, lir = lane % LPR;
  const bool live = lir * VEC < C;
  const int gk = group_of_channel(live ? lir * VEC : 0, C, G);   // chunks never straddle groups (host)
  const uint32_t row_bytes = (uint32_t)C * sizeof(T);
  const char* __restrict__ xb = reinterpret_cast<const char*>(P.x) + (live ? lir * 16 : 0);
  char* __restrict__ ob = reinterpret_cast<char*>(P.out) + (live ? lir * 16 : 0);
  const bool gating = P.gate_w != nullptr;
  float4 gw4 = make_float4(0.f, 0.f, 0.f, 0.f), gb4 = gw4;
  if (gating) {
    gw4 = make_float4(P.gate_w[0], P.gate_w[1], P.gate_w[2], P.gate_w[3]);
    gb4 = make_float4(P.gate_b[0], P.gate_b[1], P.gate_b[2], P.gate_b[3]);
  }
  const bool save = P.seg_max != nullptr;

  const int64_t n_ranges = (P.N + PR - 1) / PR;
  const int64_t warps_total = (int64_t)gridDim.x * kRingWarps;
  for (int64_t r = (int64_t)blockIdx.x * kRingWarps + warp; r < n_ranges; r += warps_total) {
    const int64_t pa = r * PR;
    const int64_t pb = (pa + PR < P.N) ? pa + PR : P.N;
    const int64_t vb = P.ptr[pa];
    const int nv = (int)(P.ptr[pb] - vb);           // views of this range (host: V < 2^31)
    uint32_t rid = (lane < RB && lane < nv) ? load_row_id(P.idx, P.idx64, vb + lane) : 0u;

    // batch bi of this range -> slot bi % S; then prefetch the row ids of batch bi + 1
    auto issue = [&](int bi) {
      const int slot = bi % S;
      const int v0 = bi * RB;
      const int nrows = (nv - v0 < RB) ? nv - v0 : RB;
      if (nrows > 0) {
        const uint32_t dst0 = rows_u + (uint32_t)(slot * RB) * RS + lir * 16;
#pragma unroll
        for (int st = 0; st < Gm::STEPS; ++st) {
          const int rr = st * RPI + sg;
          const uint32_t srow = __shfl_sync(FULL, rid, rr);
          if (rr < nrows && live) cp_async16(dst0 + rr * RS, xb + (uint64_t)srow * row_bytes);
        }
      }
      cp_async_commit();
      const int v1 = v0 + RB;
      rid = (lane < RB && v1 + lane < nv) ? load_row_id(P.idx, P.idx64, vb + v1 + lane) : 0u;
    };
    auto advance_to = [&](int b, int& cb) {         // make batch b resident; refill the freed slots
      while (cb < b) {
        __syncwarp();
        ++cb;
        issue(cb + S - 1);
        cp_async_wait<S - 1>();
        __syncwarp();
      }
    };
    // weighted sum of the rows of one piece (views [lo, lo+np) of batch slot) into acc
    auto piece_rows = [&](int slot, int lo, int np, int u0, float (&acc)[VEC]) {
      const unsigned char* rp = rows_s + (size_t)(slot * RB + lo) * RS + lir * 16;
#pragma unroll 4
      for (int v0 = sg; v0 < np + sg; v0 += RPI) {  // warp-uniform trip count; idle sub-groups add 0
        const bool ok = v0 < np;
        const int vv = ok ? v0 : 0;
        const uint4 raw = *reinterpret_cast<const uint4*>(rp + (size_t)vv * RS);
        const float a = ok ? wt[tix(u0 + vv) + gk] : 0.f;
        float fv[VEC];
        unpack16<T, VEC>(raw, fv);
#pragma unroll
        for (int j = 0; j < VEC; ++j) acc[j] = fmaf(a, fv[j], acc[j]);
      }
    };
    auto store_out = [&](int64_t i, float (&acc)[VEC], float sc) {
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        float a = acc[j];
#pragma unroll
        for (int o = LPR; o < 32; o <<= 1) a += __shfl_xor_sync(FULL, a, o);
        acc[j] = a * sc;
      }
      if (sg == 0 && live) stg_stream16(ob + i * (int64_t)row_bytes, pack16<T, VEC>(acc));
    };

#pragma unroll
    for (int bi = 0; bi < S - 1; ++bi) issue(bi);
    int cb = -1;                                    // newest batch known to be resident
    int pl, cnt;
    load_window(P.ptr, pa, pb, vb, lane, pl, cnt);

    for (int64_t pg = pa; pg < pb;) {
      // group = longest prefix of the window with at most CAPV views
      const int gs0 = __shfl_sync(FULL, pl, 0);
      const bool fits = (pg + lane < pb) && (pl + cnt - gs0 <= CAPV);
      const unsigned fm = __ballot_sync(FULL, fits);
      const int kmax = (fm == FULL) ? 32 : __ffs(~fm) - 1;

      if (kmax == 0) {
        // ---- one point with more views than the tile holds: warp-cooperative online softmax
        const int n = __shfl_sync(FULL, cnt, 0);
        const int s = gs0;
        const int64_t i = pg;
        int pl_n, cnt_n;
        load_window(P.ptr, pg + 1, pb, vb, lane, pl_n, cnt_n);
        const float inv_sq = P.group_scaling ? rsqrtf((float)n) : 1.f;
        const int gl = lane & (G - 1);
        const float* __restrict__ cp = P.compat + (vb + s) * G;
        float m_run = -INFINITY, den = 0.f;
        int am = -1;
        float acc[VEC];
#pragma unroll
        for (int j = 0; j < VEC; ++j) acc[j] = 0.f;
        const int vend = s + n;
        for (int v = s; v < vend;) {
          const int b = v / RB, lo = v % RB;
          const int np = (RB - lo < vend - v) ? RB - lo : vend - v;
          advance_to(b, cb);
          const float* cs = cp + (size_t)(v - s) * G;
          const int npG = np * G;
          float pm = -INFINITY; int pe = 0x7fffffff;
          for (int e = lane; e < npG; e += 32) {
            const float c = __ldg(cs + e);
            if (c > pm) { pm = c; pe = e; }
          }
          for (int off = 16; off >= G; off >>= 1) {
            const float om = __shfl_xor_sync(FULL, pm, off);
            const int oe = __shfl_xor_sync(FULL, pe, off);
            if (om > pm || (om == pm && oe < pe)) { pm = om; pe = oe; }
          }
          if (pm > m_run) am = (int)(vb + v) + pe / G;
          const float m_new = fmaxf(m_run, pm);
          const float alpha = __expf((m_run - m_new) * inv_sq);   // first piece: exp(-inf) = 0
          m_run = m_new;
          den *= alpha;
          __syncwarp();                             // readers of the previous piece's weights are done
          for (int e = lane; e < npG; e += 32) {
            const float ev = __expf((__ldg(cs + e) - m_new) * inv_sq);
            den += ev;
            wt[tix(e / G) + gl] = ev;
          }
          __syncwarp();
          const float ak = __shfl_sync(FULL, alpha, gk);
#pragma unroll
          for (int j = 0; j < VEC; ++j) acc[j] *= ak;
          piece_rows(b % S, lo, np, 0, acc);
          v += np;
        }
        den = group_lane_sum(den, G) + P.eps;
        const float gwl = sel4(gw4, gl), gbl = sel4(gb4, gl);
        const float t = gating ? tanhf(fmaxf(fmaf(gwl, m_run, gbl), 0.f)) : 1.f;
        if (lane < G && save) {
          P.seg_max[i * G + lane] = m_run; P.seg_den[i * G + lane] = den; P.seg_arg[i * G + lane] = am;
        }
        const float inv_den = 1.f / den;
        store_out(i, acc, __shfl_sync(FULL, t * inv_den, gk));
        if (P.att != nullptr) {
          float* __restrict__ ao = P.att + (vb + s) * G;
          for (int e = lane; e < n * G; e += 32) ao[e] = __expf((__ldg(cp + e) - m_run) * inv_sq) * inv_den;
        }
        __syncwarp();
        pg += 1; pl = pl_n; cnt = cnt_n;
        continue;
      }

      int pl_n = 0, cnt_n = 0;                      // next window: loaded a group early
      if (pg + kmax < pb) {
        load_window(P.ptr, pg + kmax, pb, vb, lane, pl_n, cnt_n);
        // warm the next group's scores in L2: 32 lanes x 128 bytes = the next 256 views
        const int64_t pv = vb + __shfl_sync(FULL, pl + cnt, kmax - 1) + lane * 8;
        if (pv < P.V) prefetch_l2(P.compat + pv * G);
      }

      // ---- phase 1: lane k owns point pg + k: statistics and gate; e-values -> tile, scale -> spt
      {
        float4 sc = make_float4(0.f, 0.f, 0.f, 0.f);
        if (lane < kmax) {
          const int64_t i = pg + lane;
          const int n = cnt, u0 = pl - gs0;
          float4 mx = make_float4(0.f, 0.f, 0.f, 0.f), dn = make_float4(P.eps, P.eps, P.eps, P.eps);
          int4 ar = make_int4(-1, -1, -1, -1);
          if (n > 0) {
            const float4* __restrict__ cp = reinterpret_cast<const float4*>(P.compat + (vb + pl) * G);
            mx = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
            int a0 = 0, a1 = 0, a2 = 0, a3 = 0;
            for (int j0 = 0; j0 < n; j0 += kP1Unroll) {   // kP1Unroll score loads in flight per lane
              float4 c[kP1Unroll];
#pragma unroll
              for (int u = 0; u < kP1Unroll; ++u)
                c[u] = (j0 + u < n) ? __ldg(cp + j0 + u) : make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
#pragma unroll
              for (int u = 0; u < kP1Unroll; ++u) {
                const int j = j0 + u;
                if (c[u].x > mx.x) { mx.x = c[u].x; a0 = j; }
                if (c[u].y > mx.y) { mx.y = c[u].y; a1 = j; }
                if (c[u].z > mx.z) { mx.z = c[u].z; a2 = j; }
                if (c[u].w > mx.w) { mx.w = c[u].w; a3 = j; }
                if (j < n) *reinterpret_cast<float4*>(wt + tix(u0 + j)) = c[u];
              }
            }
            const int v0g = (int)(vb + pl);
            ar = make_int4(v0g + a0, v0g + a1, v0g + a2, v0g + a3);
            const float inv_sq = P.group_scaling ? rsqrtf((float)n) : 1.f;
            float4 d = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
            for (int j = 0; j < n; ++j) {
              float4* w = reinterpret_cast<float4*>(wt + tix(u0 + j));
              const float4 c = *w;
              float4 e;
              e.x = __expf((c.x - mx.x) * inv_sq); e.y = __expf((c.y - mx.y) * inv_sq);
              e.z = __expf((c.z - mx.z) * inv_sq); e.w = __expf((c.w - mx.w) * inv_sq);
              d.x += e.x; d.y += e.y; d.z += e.z; d.w += e.w;
              *w = e;
            }
            dn = make_float4(d.x + P.eps, d.y + P.eps, d.z + P.eps, d.w + P.eps);
            sc = make_float4(1.f / dn.x, 1.f / dn.y, 1.f / dn.z, 1.f / dn.w);
            if (P.att != nullptr) {
              float4* __restrict__ ao = reinterpret_cast<float4*>(P.att + (vb + pl) * G);
#pragma unroll 4
              for (int j = 0; j < n; ++j) {
                const float4 e = *reinterpret_cast<const float4*>(wt + tix(u0 + j));
                ao[j] = make_float4(e.x * sc.x, e.y * sc.y, e.z * sc.z, e.w * sc.w);
              }
            }
            if (gating) {
              sc.x *= tanhf(fmaxf(fmaf(gw4.x, mx.x, gb4.x), 0.f));
              sc.y *= tanhf(fmaxf(fmaf(gw4.y, mx.y, gb4.y), 0.f));
              sc.z *= tanhf(fmaxf(fmaf(gw4.z, mx.z, gb4.z), 0.f));
              sc.w *= tanhf(fmaxf(fmaf(gw4.w, mx.w, gb4.w), 0.f));
            }
          }
          if (save) {
            reinterpret_cast<float4*>(P.seg_max)[i] = mx;
            reinterpret_cast<float4*>(P.seg_den)[i] = dn;
            reinterpret_cast<int4*>(P.seg_arg)[i] = ar;
          }
        }
        reinterpret_cast<float4*>(spt)[lane] = sc;   // per-point, per-group output scale t / den
      }
      __syncwarp();

      // ---- phase 2: per point, weighted sum of its rows out of the ring
      for (int k = 0; k < kmax; ++k) {
        const int s = __shfl_sync(FULL, pl, k);
        const int n = __shfl_sync(FULL, cnt, k);
        float acc[VEC];
#pragma unroll
        for (int j = 0; j < VEC; ++j) acc[j] = 0.f;
        const int vend = s + n;
        for (int v = s; v < vend;) {
          const int b = v / RB, lo = v % RB;
          const int np = (RB - lo < vend - v) ? RB - lo : vend - v;
          advance_to(b, cb);
          piece_rows(b % S, lo, np, v - gs0, acc);
          v += np;
        }
        store_out(pg + k, acc, spt[k * G + gk]);     // unseen point: exact zeros
      }
      __syncwarp();                                 // the tile is rewritten by the next group
      pg += kmax; pl = pl_n; cnt = cnt_n;
    }
    cp_async_wait<0>();                             // only empty groups can be left; then reuse the ring
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
template <typename T> static int ring_lpr(const VAParams& P) {
  const int cv = P.C / Vec16<T>::N;                 // 16-byte chunks per row
  if (cv <= 4) return 4;
  if (cv <= 8) return 8;
  if (cv <= 16) return 16;
  return 32;
}

template <typename T> static bool ring_fwd_ok(const VAParams& P) {
  constexpr int V16 = Vec16<T>::N;
  const int C = P.C, G = P.G;
  if (G != kRG) return false;
  if (C % V16 != 0 || C / V16 > 32) return false;   // rows of at most 512 bytes, whole 16-byte chunks
  if (!aligned16(P.x) || !aligned16(P.out) || !aligned16(P.compat)) return false;
  if (P.att != nullptr && !aligned16(P.att)) return false;
  if (P.seg_max != nullptr && (!aligned16(P.seg_max) || !aligned16(P.seg_den) || !aligned16(P.seg_arg))) return false;
  if (P.V >= (1ll << 31) || P.R >= (1ll << 32)) return false;
  for (int c0 = 0; c0 < C; c0 += V16)               // chunks never straddle channel groups
    if (group_of_channel(c0, C, G) != group_of_channel(c0 + V16 - 1, C, G)) return false;
  return true;
}
bool va_ring_fwd_applicable(const VAParams& P, int dtype) {
  switch (dtype) {
    case DVA_F32: return ring_fwd_ok<float>(P);
    case DVA_BF16: return ring_fwd_ok<__nv_bfloat16>(P);
    case DVA_F16: return ring_fwd_ok<__half>(P);
    default: return false;
  }
}

// grid = co-resident CTAs (148 SMs x occupancy); PR = points per range (one range per warp when
// the problem is large enough, never fewer than 8 points)
template <typename T, int LPR>
static int ring_fwd_launch(const VAParams& P, cudaStream_t st) {
  const RingSmem<LPR> L;
  const size_t smem = L.total * kRingWarps;
  auto kern = va_ring_fwd_kernel<T, LPR>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return failf((int)e, "view_attention ring: %zu bytes of shared memory: %s", smem, cudaGetErrorString(e));
  int occ = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kRingWarps * 32, smem) != cudaSuccess || occ < 1) occ = 1;
  if (occ > 32) occ = 32;
  int64_t grid = (int64_t)kNumSMs * occ;
  const int64_t warps = grid * kRingWarps;
  int64_t pr = (P.N + warps - 1) / warps;
  if (pr < 8) pr = 8;
  const int64_t n_ranges = (P.N + pr - 1) / pr;
  const int64_t need = (n_ranges + kRingWarps - 1) / kRingWarps;
  if (grid > need) grid = need;
  if (grid < 1) grid = 1;
  kern<<<(int)grid, kRingWarps * 32, smem, st>>>(P, (int)pr);
  return check_launch("view_attention_fwd(ring)");
}
template <typename T> static int ring_fwd_typed(const VAParams& P, cudaStream_t st) {
  switch (ring_lpr<T>(P)) {
    case 4: return ring_fwd_launch<T, 4>(P, st);
    case 8: return ring_fwd_launch<T, 8>(P, st);
    case 16: return ring_fwd_launch<T, 16>(P, st);
    default: return ring_fwd_launch<T, 32>(P, st);
  }
}
int va_ring_fwd(const VAParams& P, int dtype, cudaStream_t st) {
  switch (dtype) {
    case DVA_F32: return ring_fwd_typed<float>(P, st);
    case DVA_BF16: return ring_fwd_typed<__nv_bfloat16>(P, st);
    case DVA_F16: return ring_fwd_typed<__half>(P, st);
    default: return fail(DVA_EINVAL, "view_attention_fwd: unknown dtype");
  }
}

}  // namespace dva
