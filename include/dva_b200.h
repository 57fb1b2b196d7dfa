/*
 * dva_b200.h -- C ABI of libdva_b200.so: the B200 (sm_100a) multi-view aggregation hot path.
 *
 * Every entry point replaces one operator (or a fused chain of operators) on the reference's
 * path  ImageMapping gather -> per-point ragged attention over views -> softmax-weighted reduce
 * (DeepViewAgg, torch_points3d/modules/multimodal + torch_points3d/core/multimodal).  The
 * "replaces" line of each declaration cites the reference file:line (relative to the reference
 * repository root) whose behaviour the entry point reproduces.
 *
 * Conventions (all entry points)
 *   - extern "C", plain pointers and sizes; no torch / C++ types.
 *   - all data pointers are DEVICE pointers owned by the caller (workspace included); the
 *     library never allocates or frees device memory and keeps no global mutable state.
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); no internal
 *     synchronisation, never the legacy default stream unless the caller passes it.
 *   - row-major contiguous tensors. CSR pointers are int64 (the reference dtype,
 *     core/multimodal/csr.py:54). Row indices are int32 or int64 (`idx_is_i64`).
 *   - `dtype` selects the storage type of feature tensors (DVA_F32 / DVA_BF16 / DVA_F16);
 *     scores, softmax statistics and all accumulation are fp32.
 *   - return value: 0 = OK; <0 = DVA_E* argument error (nothing was launched);
 *     >0 = cudaError_t of the failed launch.  dva_last_error() gives a thread-local message.
 */
#ifndef DVA_B200_H_
#define DVA_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DVA_ABI_VERSION 1

enum { DVA_OK = 0, DVA_EINVAL = -1, DVA_EALIGN = -2, DVA_EUNSUPPORTED = -3 };
enum { DVA_F32 = 0, DVA_BF16 = 1, DVA_F16 = 2 };
/* reduce codes follow BimodalCSRPool._POOLING_MODES order-independent names (pooling.py:36) */
enum { DVA_SUM = 0, DVA_MEAN = 1, DVA_MAX = 2, DVA_MIN = 3 };

int dva_abi_version(void);
const char* dva_last_error(void);
/* number of kernels this library has launched in this process since load (all threads:
 * autograd runs backward from a worker thread); bench.py reports it as gpu_launches. */
int64_t dva_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * T1 / P1  segment_csr                      replaces torch_scatter.segment_csr as used at
 *   pooling.py:63 (BimodalCSRPool), :289,:295,:519,:525 (pools), :628 (DeepSetFeat.f_pool),
 *   :787,:807 (segment_softmax_csr), :851 (segment_gather_csr); image.py:1767.
 *   out[i,:] = reduce_{p in [ptr[i],ptr[i+1])} src[p,:];  EMPTY segment -> 0 for every reduce
 *   (pooling.py:870).  mean divides by max(count,1).  For max/min `arg` (nullable, int64
 *   [n_seg,K]) receives the FIRST arg-max/min row in segment order, or n_items for empty
 *   segments (torch_scatter convention); backward routes the gradient to that row only.
 * ------------------------------------------------------------------------------------------ */
int dva_segment_csr_fwd(const void* src, const int64_t* ptr, void* out, int64_t* arg,
                        int64_t n_seg, int64_t n_items, int64_t K, int reduce, int dtype,
                        void* stream);
/* grad_src[n_items,K] fully written (zeros where no gradient flows). */
int dva_segment_csr_bwd(const void* grad_out, const int64_t* ptr, const int64_t* arg,
                        void* grad_src, int64_t n_seg, int64_t n_items, int64_t K, int reduce,
                        int dtype, void* stream);

/* P8  gather_csr                            replaces pooling.py:813-841
 *   out[p,:] = src[i,:] for p in [ptr[i],ptr[i+1]).  Its backward is segment_csr(sum). */
int dva_gather_csr(const void* src, const int64_t* ptr, void* out, int64_t n_seg,
                   int64_t n_items, int64_t K, int dtype, void* stream);

/* P7  segment_softmax_csr                   replaces pooling.py:758-810
 *   m = segment max (0 if empty); z = (src-m)/(sqrt(count) if scaling); e = exp(z);
 *   out = e / (segment_sum(e) + eps).   src/out [n_items,K]. */
int dva_segment_softmax_csr_fwd(const void* src, const int64_t* ptr, void* out, int64_t n_seg,
                                int64_t n_items, int64_t K, float eps, int scaling, int dtype,
                                void* stream);
/* grad_src = out * (grad_out - sum_seg(out*grad_out)) / (sqrt(count) if scaling) */
int dva_segment_softmax_csr_bwd(const void* out, const void* grad_out, const int64_t* ptr,
                                void* grad_src, int64_t n_seg, int64_t n_items, int64_t K,
                                int scaling, int dtype, void* stream);

/* ------------------------------------------------------------------------------------------
 * P3 / P4 core: fused CSR-gather + ragged group softmax + weighted sum + gating.
 *   replaces the chain  modules.py:518 (x_mod[idx_sorting] row gather)  ->
 *   pooling.py:285-300 (GroupBimodalCSRPool)  /  pooling.py:515-530 (QKVBimodalCSRPool):
 *     a    = segment_softmax_csr(compat, ptr, scaling=group_scaling)          [V,G]
 *     y    = segment_csr(x[idx] * expand_group_feat(a, G, C), ptr, 'sum')     [N,C]
 *     t    = tanh(relu(gate_w * segment_csr(compat, ptr, 'max') + gate_b))    [N,G]  (if gating)
 *     out  = y * expand_group_feat(t, G, C)
 *   x      [R,C] feature rows (dtype); idx [V] row of x for view v (nullable: identity, R==V)
 *   compat [V,G] fp32; ptr [N+1] int64; gate_w/gate_b [G] fp32 (both null: no gating)
 *   out    [N,C] (dtype)
 *   saved for backward / save_last taps (all nullable except in training):
 *     att [V,G] fp32 attention a;  seg_max [N,G] fp32;  seg_den [N,G] fp32 (sum e + eps);
 *     seg_arg [N,G] int32 = first arg-max view (absolute view id, -1 if empty)
 *   channel->group map: group_sizes(C,G) of pooling.py:737-755 (first C%G groups one wider).
 *   G must be a power of two <= 32 (all shipped configs use 4); otherwise DVA_EUNSUPPORTED and
 *   the host composes the unfused entry points above.
 * ------------------------------------------------------------------------------------------ */
int dva_view_attention_fwd(const void* x, const void* idx, int idx_is_i64, const float* compat,
                           const int64_t* ptr, const float* gate_w, const float* gate_b,
                           void* out, float* att, float* seg_max, float* seg_den,
                           int32_t* seg_arg, int64_t N, int64_t V, int64_t R, int64_t C,
                           int64_t G, int group_scaling, float eps, int dtype, void* stream);

/* Implementation choice of the fused pair (tuning / test knob, process-wide; results are the same
 * up to fp32 summation order): 0 = auto (default; also DVA_VA_PATH=auto|stream|ring|lane in the
 * environment), 1 = streaming kernels for both passes (rows in registers, one point per warp at a
 * time), 2 = ring forward (rows staged in shared memory by async copies across point boundaries,
 * softmax statistics one lane per point; G == 4, rows of whole 16-byte chunks, <= 512 bytes) and
 * lane-per-view backward (groups of <= 32 views per warp: lane per view for the scores, sub-warp per
 * row for the features; G == 4, rows of 4 / 8 / 16 / 32 chunks), 3 = streaming forward and
 * lane-per-view backward.  A pass whose kernel does not apply to the shape runs on the streaming
 * kernel whatever the setting.
 * TEST / TUNING ONLY: production callers leave it at 0; the choice is a pure function of the shape. */
int dva_view_attention_set_path(int path);

/* Backward of the chain above.
 *   grad_out [N,C] (dtype) -> grad_x_rows [V,C] (dtype; row v is d/d(x[idx[v]]); when
 *   scatter_rows!=0 and idx!=null it is written to row idx[v] of a [R,C] buffer instead, which
 *   requires idx to be injective, as view_cat_sorting is, image.py:1549-1574),
 *   grad_compat [V,G] fp32 (softmax path + gating arg-max path),
 *   grad_gate [2,G] fp32 (d gate_w ; d gate_b), nullable when no gating.
 *   workspace: dva_view_attention_bwd_workspace_bytes(G) bytes (per-block partials). */
size_t dva_view_attention_bwd_workspace_bytes(int64_t G);
int dva_view_attention_bwd(const void* x, const void* idx, int idx_is_i64, const float* compat,
                           const int64_t* ptr, const float* gate_w, const float* gate_b,
                           const void* grad_out, const float* seg_max, const float* seg_den,
                           const int32_t* seg_arg, void* grad_x_rows, float* grad_compat,
                           float* grad_gate, int scatter_rows, int64_t N, int64_t V, int64_t R,
                           int64_t C, int64_t G, int group_scaling, int dtype, void* workspace,
                           size_t workspace_bytes, void* stream);

/* P4  ragged per-group Q.K scores           replaces pooling.py:499-512
 *   compat[v,g] = scale * sum_d keys[v,g*D+d] * queries[i(v),g*D+d]   (i(v): point of view v;
 *   the reference materialises repeat_interleave(queries), pooling.py:500).  fp32 I/O. */
int dva_qk_scores_fwd(const float* keys, const float* queries, const int64_t* ptr, float* compat,
                      int64_t N, int64_t V, int64_t G, int64_t D, float scale, void* stream);
int dva_qk_scores_bwd(const float* keys, const float* queries, const int64_t* ptr,
                      const float* grad_compat, float* grad_keys, float* grad_queries, int64_t N,
                      int64_t V, int64_t G, int64_t D, float scale, void* stream);

/* P2  HeuristicBimodalCSRPool               replaces pooling.py:129-152
 *   j_i = first arg-max/min over the segment of x_map[:,feat]; out[i,:] = x_mod[j_i,:] or 0.
 *   arg [N] int64 (n_items when empty). */
int dva_heuristic_pool_fwd(const void* x_mod, const float* x_map, int64_t map_stride,
                           int64_t feat, const int64_t* ptr, void* out, int64_t* arg, int64_t N,
                           int64_t V, int64_t C, int use_max, int dtype, void* stream);

/* ------------------------------------------------------------------------------------------
 * I5 + P1  fused feature-map gather + atomic pool
 *   replaces image.py:1285 (x[(img, ..., py, px)] NCHW advanced-index gather) followed by
 *   modules.py:497-500 -> pooling.py:63 (BimodalCSRPool over the atomic CSR).
 *   fmap [B,C,H,W] (channels_last=0) or [B,H,W,C] (channels_last=1), dtype
 *   img [Vw] int64 image of each view; pix [P,2] (x,y) int16/int32 (pix_is_i16)
 *   aptr [Vw+1] int64 atomic CSR;  out [Vw,C];  arg [Vw,C] int64 pixel slot (nullable, max/min)
 * ------------------------------------------------------------------------------------------ */
int dva_gather_pool_fwd(const void* fmap, int channels_last, const int64_t* img, const void* pix,
                        int pix_is_i16, const int64_t* aptr, void* out, int64_t* arg,
                        int64_t B, int64_t C, int64_t H, int64_t W, int64_t Vw, int64_t P,
                        int reduce, int dtype, void* stream);
/* grad_fmap must be zero-initialised by the caller; gradients are accumulated with fp32
 * atomics when dtype==DVA_F32 (pixel reuse across views), see DESIGN.md. */
int dva_gather_pool_bwd(const void* grad_out, int channels_last, const int64_t* img,
                        const void* pix, int pix_is_i16, const int64_t* aptr, const int64_t* arg,
                        float* grad_fmap, int64_t B, int64_t C, int64_t H, int64_t W, int64_t Vw,
                        int64_t P, int reduce, int dtype, void* stream);

/* [B,R,S] -> [B,S,R] layout change (dtype-sized elements), e.g. the reference's NCHW-contiguous
 * feature maps (image.py:1884 indexes them as x[b, :, y, x]) to channels-last and map gradients back,
 * so that dva_gather_pool_* / dva_interp_pool_* can run their 16-byte-chunk channels-last kernels. */
int dva_transpose_last2(const void* src, void* dst, int64_t B, int64_t R, int64_t S, int dtype, void* stream);

/* I5b  bilinear variant: the `interpolate=True` branch of get_mapped_features
 *   replaces image.py:1278-1283 -> sparse_interpolation (image.py:105-170, padding 'border')
 *   followed by the same atomic pool.  pix are at the MAPPING resolution (map_w, map_h); every
 *   pixel reads the 4 bilinear corners of the replicate-padded [H,W] map.  The fp32 operation
 *   order is the reference's, so fp32 results (and max / argmax choices) are identical.
 *   A per-pixel interpolation without pooling is aptr = 0..P with reduce = DVA_SUM. */
int dva_interp_pool_fwd(const void* fmap, int channels_last, const int64_t* img, const void* pix,
                        int pix_is_i16, const int64_t* aptr, void* out, int64_t* arg,
                        int64_t B, int64_t C, int64_t H, int64_t W, int64_t map_w, int64_t map_h,
                        int64_t Vw, int64_t P, int reduce, int dtype, void* stream);
int dva_interp_pool_bwd(const void* grad_out, int channels_last, const int64_t* img,
                        const void* pix, int pix_is_i16, const int64_t* aptr, const int64_t* arg,
                        float* grad_fmap, int64_t B, int64_t C, int64_t H, int64_t W,
                        int64_t map_w, int64_t map_h, int64_t Vw, int64_t P, int reduce, int dtype,
                        void* stream);

/* ------------------------------------------------------------------------------------------
 * N1  neighbourhood-based mapping features (density, occlusion)
 *   replaces NeighborhoodBasedMappingFeatures._process,
 *   core/data_transform/multimodal/image.py:483-612 (KeOps argKmin branch :504-514; the FAISS
 *   branch is approximate and not reproduced).
 *   dva_knn_cell_ids : cell[i] = linear cell of point i in a gx x gy x gz grid of `cell_size`
 *                      cubes anchored at (ox,oy,oz) (clamped).  The caller sorts points by cell
 *                      and builds cell_ptr [gx*gy*gz+1] (dva_csr_pointers_from_sorted).
 *   dva_knn_grid     : exact k nearest neighbours (self included), k <= 64, of every point among
 *                      all points; squared distance (dx*dx + dy*dy) + dz*dz in fp32, ties by
 *                      index.  neighbors [n,k] int64 and dist2 [n,k] (nullable) are indexed by
 *                      ORIGINAL point id, ascending (dist2, id).
 *   dva_neighborhood_features : out [V, nk*(density + occlusion)] fp32 = for every k of the
 *                      ascending klist: density of the view's point ((k+1)/(3.1416 d_k^2)/(1/voxel^2),
 *                      NaN -> 1, :527-537), then occlusion of the view ((1 + #neighbours seen by
 *                      the view's image)/(k+1), :563-584).  view_ptr [N+1] / images [V]: the view
 *                      CSR; view_point [V] = point of each view.
 * ------------------------------------------------------------------------------------------ */
int dva_knn_cell_ids(const float* xyz, int64_t* cell, int64_t n, float ox, float oy, float oz,
                     float cell_size, int gx, int gy, int gz, void* stream);
int dva_knn_grid(const float* xyz_sorted, const int64_t* cell_sorted, const int64_t* order,
                 const int64_t* cell_ptr, int64_t n, int k, float ox, float oy, float oz,
                 float cell_size, int gx, int gy, int gz, int64_t* neighbors, float* dist2,
                 void* stream);
int dva_neighborhood_features(const float* xyz, const int64_t* neighbors, int kmax,
                              const int64_t* view_ptr, const int64_t* images,
                              const int64_t* view_point, const int32_t* klist, int nk,
                              double voxel, int density, int occlusion, float* out, int64_t N,
                              int64_t V, void* stream);

/* ------------------------------------------------------------------------------------------
 * P9  dense projection GEMM of an MLP layer (tcgen05 / TMA / TMEM)
 *   replaces the nn.Linear(bias=False) of base_modules.py:42 in every pool MLP.
 *   layout 0: D[M,N] = A[M,K] . B[N,K]^T   (forward,  B = weight [out,in])
 *   layout 1: D[M,N] = A[M,K] . B[K,N]     (backward, dX = dZ . weight)
 *   layout 2: D[N,K] = A[M,N]^T . B[M,K]   (backward, dW = dZ^T . X; stream-K over the M rows)
 *   fp32 row-major operands.  Two kernel families behind the one entry point:
 *     N <= 64 and K <= 64 (any values; every MLP of the map encoders, pooling.py:645-656): "skinny"
 *       kernels -- weights in shared memory, 128-row tiles double-buffered by cp.async, coalesced
 *       16-byte global traffic, 3xTF32 split operands on mma.sync (fp32-grade accuracy, ~1e-6), dW
 *       as per-CTA partials reduced in a fixed order (deterministic);
 *     otherwise the hand-written tcgen05 kernels of csrc/tc_gemm.cu (TMA-fed tcgen05.mma kind::tf32,
 *       TMEM accumulators, 3xTF32 split operands: ~1e-6 of the result's max against fp64; dW as
 *       per-CTA partial tiles reduced in a fixed order): operands 16-byte aligned, N % 4 == 0 and
 *       K % 4 == 0 (else DVA_EUNSUPPORTED; ops.linear zero-pads such widths).
 *   `precision` is accepted for ABI stability (0 or 1) and ignored: every path is fp32-grade.
 *   workspace: dva_linear_gemm_workspace_bytes().
 * ------------------------------------------------------------------------------------------ */
size_t dva_linear_gemm_workspace_bytes(int64_t M, int64_t N, int64_t K, int layout, int precision);
int dva_linear_gemm(const float* A, const float* B, float* D, int64_t M, int64_t N, int64_t K, int layout,
                    int precision, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * P9  Linear with the BatchNorm batch statistics taken in the GEMM epilogue
 *   replaces base_modules.py:42-44 (nn.Linear(bias=False) followed by the statistics half of
 *   FastBatchNorm1d) for the wide layers (E_mod, E_mix, E_main): D[M,n_out] = X[M,k_red] . W[n_out,k_red]^T
 *   by the tcgen05 rows kernel, whose epilogue threads each own one output column and accumulate its
 *   shifted sum / sum of squares while storing; a one-warp-per-column kernel combines the per-CTA
 *   partials in fp64 (fixed order) into mean / invstd [n_out] (biased variance) and updates the running
 *   buffers (momentum, unbiased variance) like nn.BatchNorm1d.  The apply half is dva_bn_act_fwd with
 *   training = 0 on these mean / invstd.  supported(): 32 <= n_out <= 128, n_out % 4 == 0, k_red >= 8,
 *   k_red % 4 == 0 (the shapes dva_linear_gemm serves with the tcgen05 rows kernel); else DVA_EUNSUPPORTED.
 * ------------------------------------------------------------------------------------------ */
int dva_linear_bnstats_supported(int64_t M, int64_t n_out, int64_t k_red);
size_t dva_linear_bnstats_workspace_bytes(int64_t n_out, int64_t k_red);
int dva_linear_bnstats_fwd(const float* X, const float* W, float* D, int64_t M, int64_t n_out, int64_t k_red,
                           float eps, float momentum, float* mean, float* invstd, float* running_mean,
                           float* running_var, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * P9  fused BatchNorm1d (+ LeakyReLU) of an MLP layer
 *   replaces core/common_modules/base_modules.py:38-48 (Linear -> FastBatchNorm1d -> LeakyReLU(0.2))
 *   after the Linear, and FastBatchNorm1d._forward_sparse :139-148: per-column batch statistics
 *   over ALL rows in training (biased variance for normalisation, unbiased for running_var,
 *   momentum update), y = act(gamma * (z - mean) * invstd + beta), act(a) = a > 0 ? a : slope * a
 *   (slope = 1: plain BatchNorm).  z, y [R,C] (dtype); gamma/beta nullable; mean/invstd [C] fp32 are
 *   written in training and READ in eval (host passes running_mean and rsqrt(running_var + eps)).
 *   Backward: dz [R,C] (NULL: statistics pass only); dbeta_dgamma [2,C] fp32 = (sum g ; sum g * zhat) with g = dy * act'.
 *   workspace: dva_bn_workspace_bytes(R, C) bytes (per-CTA partial sums, deterministic).
 * ------------------------------------------------------------------------------------------ */
size_t dva_bn_workspace_bytes(int64_t R, int64_t C);
int dva_bn_act_fwd(const void* z, const float* gamma, const float* beta, float* running_mean,
                   float* running_var, float* mean, float* invstd, void* y, int64_t R, int64_t C,
                   float eps, float momentum, float slope, int training, int dtype, void* workspace,
                   size_t workspace_bytes, void* stream);
int dva_bn_act_bwd(const void* dy, const void* z, const float* gamma, const float* beta,
                   const float* mean, const float* invstd, void* dz, float* dbeta_dgamma, int64_t R,
                   int64_t C, float slope, int training, int dtype, void* workspace,
                   size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * P9 / P5  backward of one narrow MLP layer  a = LeakyReLU(BatchNorm1d(x . W^T))   (training statistics)
 *   replaces the autograd chain of base_modules.py:38-48 for the layers of the map encoders
 *   (DeepSetFeat / MLPSetFeat, pooling.py:645-656, 686: 8 / 32 / 64 -> 32 on one row per view):
 *   pass 1 = the statistics half of dva_bn_act_bwd (dz = NULL there: reduction only), pass 2 = ONE kernel that
 *   forms dz = gamma invstd (g - mean(g) - zhat mean(g zhat)) on chip and emits dX = dz . W and dW = dz^T . x
 *   from the same tile (3xTF32 mma.sync, fp32-grade): 3 reads + 1 write of the rows instead of 5 + 2.
 *   dA, Z [M,N] fp32 (gradient of the layer output, saved pre-BatchNorm linear output); X [M,K] fp32 layer input;
 *   W [N,K]; gamma / beta nullable; mean / invstd [N] of the forward; dX [M,K] nullable (first layer);
 *   dW [N,K]; dbeta_dgamma [2,N] = (sum g ; sum g zhat).  supported(): N <= 32, K <= 64, both % 4 == 0.
 *   Row pointers 16-byte aligned.  Deterministic (per-CTA partials summed in a fixed order).
 * ------------------------------------------------------------------------------------------ */
int dva_mlp_layer_bwd_supported(int64_t M, int64_t N, int64_t K);
size_t dva_mlp_layer_bwd_workspace_bytes(int64_t M, int64_t N, int64_t K);
int dva_mlp_layer_bwd(const float* dA, const float* Z, const float* X, const float* W, const float* gamma,
                      const float* beta, const float* mean, const float* invstd, float* dX, float* dW,
                      float* dbeta_dgamma, int64_t M, int64_t N, int64_t K, float slope, void* workspace,
                      size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Z3  z-buffer visibility from splatting    replaces visibility.py:1073-1195 (CPU/numba oracle)
 *   splat [m,4] int32 (x_a,x_b,y_a,y_b) already clamped, y relative to the un-cropped image;
 *   dist [m] fp32.  Point i wins pixel (x,y) iff dist is the smallest, ties -> lowest i
 *   (strict '<' while iterating ascending, visibility.py:1148-1162) -- realised as one
 *   64-bit atomicMin on (dist_bits<<32 | i).
 *   zbuf [W*Hc] uint64 workspace (Hc = H - crop_top - crop_bottom), initialised by the call.
 *   exact==0: idx_map [W*Hc] int64 (-1 = empty) holds the winning point per pixel.
 *   exact!=0: idx_map re-rasterised with splat centres only: (int(x_proj), int(y_proj)-crop_top),
 *             highest seen index wins a shared centre (visibility.py:1168-1187).
 *   x_proj/y_proj [m] fp64 (numba returns float64, visibility.py:252).
 * ------------------------------------------------------------------------------------------ */
int dva_zbuffer_splat(const int32_t* splat, const float* dist, const double* x_proj,
                      const double* y_proj, unsigned long long* zbuf, int64_t* idx_map,
                      uint8_t* seen, int64_t m, int64_t W, int64_t H, int64_t crop_top,
                      int64_t crop_bottom, int exact, void* stream);

/* Z2  splat boxes                           replaces visibility.py:630-704 (equirectangular),
 *   :761-827 (pinhole).  camera: 0 = s3dis_equirectangular, 1 = pinhole (fx, fy given).
 *   numba evaluates these expressions in float64 (float32 array x Python float), hence the
 *   double parameters.  Output splat [m,4] int32 (16-byte aligned), clamped to the (cropped)
 *   image like the reference; y is relative to the un-cropped image. */
int dva_splat_boxes(const double* x_proj, const double* y_proj, const float* dist,
                    int32_t* splat, int64_t m, int64_t W, int64_t H, int64_t crop_top,
                    int64_t crop_bottom, double voxel, double k_swell, double d_swell, int camera,
                    double fx, double fy, void* stream);

/* Z2  splat boxes from explicit widths        replaces the rounding / clamping tail of
 *   fisheye_splat_cpu (visibility.py:916-951); width [m] fp64 = 2*|proj(xyz) - proj(xyz + dz)|
 *   (visibility.py:903-914) is produced by the host mirror with two dva_project_camera calls. */
int dva_splat_boxes_from_width(const double* x_proj, const double* y_proj, const double* width,
                               int32_t* splat, int64_t m, int64_t W, int64_t H, int64_t crop_top,
                               int64_t crop_bottom, void* stream);

/* Z1  equirectangular camera projection      replaces visibility.py:150-182 + :509-513 + :395-435
 *   xyz [n,3] fp32; img_pose [12] fp32 on device = camera position (3) followed by the 3x3
 *   rotation matrix of pose_to_rotation_matrix (visibility.py:57-90), row-major, computed by the
 *   host mirror.  Outputs dist [n] fp32, x_proj,y_proj [n] fp64, keep [n] uint8 = in
 *   (r_min,r_max) and inside the (cropped) field of view (no image mask). */
int dva_project_equirectangular(const float* xyz, const float* img_pose, float* dist,
                                double* x_proj, double* y_proj, uint8_t* keep, int64_t n,
                                int64_t W, int64_t H, int64_t crop_top, int64_t crop_bottom,
                                float r_min, float r_max, void* stream);

/* Z1  pinhole / fisheye camera projection    replaces visibility.py:219-252 (pinhole_projection_cpu,
 *   cameras 'scannet' and 'kitti360_perspective'), :288-339 (fisheye_projection_cpu,
 *   'kitti360_fisheye') + the range / field-of-view filter of camera_projection_cpu :509-536.
 *   cam [26] fp32 on device = img_xyz(3), A(9 row-major), t0(3), t1(3), intr(8) with
 *   p = A (xyz - t0) + t1  (scannet: A,t1 from inv(extrinsic), t0 = 0; kitti360: A = R^T, t0 = T);
 *   camera 1 = pinhole (intr = fx, fy, cx, cy), 3 = fisheye (intr = xi,k1,k2,gamma1,gamma2,u0,v0). */
int dva_project_camera(const float* xyz, const float* cam, int camera, float* dist, double* x_proj,
                       double* y_proj, uint8_t* keep, int64_t n, int64_t W, int64_t H,
                       int64_t crop_top, int64_t crop_bottom, float r_min, float r_max, void* stream);

/* rows scatter-add: dst[idx[v], :] += src[v, :] for v < V; dst [R, C] fp32 must be zero-initialised by the
 * caller; rows with idx outside [0, R) are skipped.  Backward of `x_mod[row_index]` when row_index repeats
 * rows (modules.py:518 with a caller-supplied index) and of HeuristicBimodalCSRPool's row pick
 * (pooling.py:146-150, "no view" = index V). */
int dva_scatter_add_rows(const void* src, const int64_t* idx, float* dst, int64_t V, int64_t R, int64_t C,
                         int dtype, void* stream);

/* I1 / I4 / I6  native construction of the point -> view -> pixel CSR (csrc/mapping_build.cu)
 *   replaces ImageMapping.from_dense image.py:1728-1795 (lexargsort + unique + cumsum chains) and the
 *   dense expansion / lexargunique / scatter_mean / from_dense sequence of select_points('merge')
 *   image.py:2211-2273.  Items i = 0..n-1: (point_ids[i] in [0, num_points), image_ids[i], pixels[i] = (x, y)
 *   as int16 / int32 / int64 pairs: pix_code 0 / 1 / 2).  Items are bucketed by point (histogram, scan,
 *   scatter) and every point's items ordered by (image, source index) -- or, with dedupe_pixels,
 *   by (image, x, y, source index; 0 <= x, y < 65536) dropping repeated (image, x, y).  Outputs, all
 *   preallocated by the caller with n (resp. n + 1) rows: view_ptr [num_points + 1], images_out [V],
 *   atomic_ptr [V + 1], pixels_out [P, 2] (same integer type), feat_out [V, F] = mean of
 *   feat[feat_row ? feat_row[i] : i] over the view's items with feat_on[i] != 0 (nullable: all), F <= 16;
 *   order_out [P] (nullable) = source item of every kept pixel; counts [3] (device) = V, P, status
 *   (status bit 0: a point id was out of range; such items are skipped).  Deterministic = the result of a
 *   stable lexicographic sort.  Nothing is read back: the caller reads `counts` once to slice the outputs.
 *   dva_view_cat_sorting: ImageData.view_cat_sorting / view_cat_csr_indexing image.py:1549-1588 for S
 *   settings over the same N points in closed form (no argsort): ptrs = device array of S device pointers
 *   to the settings' view pointers [N + 1], bases[s] = views of the settings before s. */
size_t dva_mapping_build_workspace_bytes(int64_t n_items, int64_t num_points);
int dva_mapping_build(const int64_t* point_ids, const int64_t* image_ids, const void* pixels, int pix_code,
                      const float* feat, const int64_t* feat_row, const uint8_t* feat_on, int64_t F,
                      int64_t n_items, int64_t num_points, int dedupe_pixels, int64_t* view_ptr,
                      int64_t* images_out, int64_t* atomic_ptr, void* pixels_out, float* feat_out,
                      int64_t* order_out, int64_t* counts, void* workspace, size_t workspace_bytes, void* stream);
int dva_view_cat_sorting(const int64_t* const* ptrs, const int64_t* bases, int64_t S, int64_t N,
                         int64_t* sorting, int64_t* csr_cat, void* stream);

/* C1  CSR pointers from sorted dense ids     replaces csr.py:158-172 + :197-229
 *   ids [n] int64 sorted ascending, values in [0,num_groups) -> ptr [num_groups+1] int64 with
 *   empty groups inserted (from_dense + insert_empty_groups, image.py:1787-1793). */
int dva_csr_pointers_from_sorted(const int64_t* ids, int64_t* ptr, int64_t n, int64_t num_groups,
                                 void* stream);

/* C1  value index of a group selection       replaces csr.py:235-264 (_index_select_pointers)
 *   ptr_new [k+1] must already hold the exclusive scan of the selected group sizes;
 *   val_idx[p] = ptr[sel[i]] + (p - ptr_new[i]) for p in [ptr_new[i], ptr_new[i+1]). */
int dva_csr_select_values(const int64_t* ptr, const int64_t* sel, const int64_t* ptr_new,
                          int64_t* val_idx, int64_t k, int64_t n_new_items, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DVA_B200_H_ */
