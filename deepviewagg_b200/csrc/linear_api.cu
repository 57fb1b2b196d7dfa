// C ABI of the projection GEMMs of the pool MLPs: dispatch between the skinny mma.sync kernels
// (skinny_gemm.cu: K, N <= 64) and the hand-written tcgen05 kernels (tc_gemm.cu: everything wider).
#include "dva_common.cuh"

extern "C" int dva_skinny_gemm_supported(int64_t M, int64_t N, int64_t K, int layout);
extern "C" size_t dva_skinny_gemm_workspace_bytes(int64_t M, int64_t N, int64_t K, int layout);
extern "C" int dva_skinny_gemm(const float* A, const float* B, float* D, int64_t M, int64_t N, int64_t K,
                               int layout, void* workspace, size_t workspace_bytes, void* stream);
extern "C" size_t dva_tc_rows_workspace_bytes(int64_t n_out, int64_t k_red);
extern "C" int dva_tc_rows_gemm(const float* X, const float* W, float* D, int64_t M, int64_t n_out, int64_t k_red,
                                int64_t ldx, int64_t ldw, int64_t ldo, int transpose_w, float* col_stats,
                                int* stats_ctas, void* workspace, size_t workspace_bytes, void* stream);
extern "C" size_t dva_tc_dw_workspace_bytes(int64_t V, int64_t n_out, int64_t k_in);
extern "C" int dva_tc_dw_gemm(const float* dZ, const float* X, float* D, int64_t V, int64_t n_out, int64_t k_in,
                              int64_t ldz, int64_t ldx, int64_t ldo, void* workspace, size_t workspace_bytes,
                              void* stream);

using namespace dva;

// Which family serves a shape.  The skinny mma.sync kernels take every K, N <= 64; measured on the B200
// (1.28 M rows): 64 -> 64 forward / dX 0.25 / 0.19 ms on the skinny kernels against 0.146 ms on the tcgen05 rows
// kernel, 32-wide layers on a par (0.07 - 0.08 ms) -> rows kernels (layouts 0, 1) go to tcgen05 when both widths
// exceed 32 and are multiples of 4; dW (layout 2) likewise since the tcgen05 dW kernel packs its stages (round 2).
// Round 2: the 32-wide rows GEMMs (N >= 32, K >= 8) go to the tcgen05 kernel too -- on a par as plain GEMMs, but
// the BatchNorm statistics then come out of its epilogue (module step 6.06 -> 5.92 ms at the S3DIS shape).
static bool use_skinny(int64_t M, int64_t N, int64_t K, int layout) {
  if (!dva_skinny_gemm_supported(M, N, K, layout)) return false;
  if (layout == 2) return !(N > 32 && K > 32 && N % 4 == 0 && K % 4 == 0);   // 64 x 64: 2 x 155 us here, tcgen05 dW below that
  return !(N >= 32 && K >= 8 && N % 4 == 0 && K % 4 == 0);
}

static bool gemm_shape_ok(int64_t M, int64_t N, int64_t K) {
  return M >= 1 && N >= 4 && K >= 4 && N % 4 == 0 && K % 4 == 0 && M < (1ll << 40) && N <= 65536 && K <= 65536;
}

extern "C" size_t dva_linear_gemm_workspace_bytes(int64_t M, int64_t N, int64_t K, int layout, int precision) {
  (void)precision;
  // narrow projections (both small dimensions <= 64: every MLP of the map encoders) run on the
  // 3xTF32 mma.sync kernels of skinny_gemm.cu
  if (use_skinny(M, N, K, layout)) return dva_skinny_gemm_workspace_bytes(M, N, K, layout);
  if (!gemm_shape_ok(M, N, K)) return 0;
  size_t w;
  if (layout == 0 || layout == 1) w = dva_tc_rows_workspace_bytes(N, K);   // split weight [n_out = N, reduction = K]
  else w = dva_tc_dw_workspace_bytes(M, N, K);
  return w < 16 ? 16 : w;
}

extern "C" int dva_linear_gemm(const float* A, const float* B, float* D, int64_t M, int64_t N, int64_t K,
                               int layout, int precision, void* workspace, size_t workspace_bytes,
                               void* stream) {
  if (layout < 0 || layout > 2 || (precision != 0 && precision != 1)) return fail(DVA_EINVAL, "linear_gemm: bad layout/precision");
  if (M == 0 && layout != 2) return DVA_OK;
  if (M > 0 && use_skinny(M, N, K, layout))
    return dva_skinny_gemm(A, B, D, M, N, K, layout, workspace, workspace_bytes, stream);
  if (M > 0 && !gemm_shape_ok(M, N, K)) return fail(DVA_EUNSUPPORTED, "linear_gemm: N and K must be multiples of 4 (16-byte TMA rows)");
  if (!A || !B || !D) return fail(DVA_EINVAL, "linear_gemm: null pointer");
  if (!aligned16(A) || !aligned16(B) || !aligned16(D)) return fail(DVA_EALIGN, "linear_gemm: operands must be 16-byte aligned");
  // layout 0: D[M,N] = A[M,K] . B[N,K]^T      -> rows kernel, weight as is
  // layout 1: D[M,N] = A[M,K] . B[K,N]        -> rows kernel, weight read transposed
  // layout 2: D[N,K] = A[M,N]^T . B[M,K]      -> dw kernel (contraction over the M rows)
  if (layout == 0) return dva_tc_rows_gemm(A, B, D, M, N, K, K, K, N, 0, nullptr, nullptr, workspace, workspace_bytes, stream);
  if (layout == 1) return dva_tc_rows_gemm(A, B, D, M, N, K, K, N, N, 1, nullptr, nullptr, workspace, workspace_bytes, stream);
  return dva_tc_dw_gemm(A, B, D, M, N, K, N, K, K, workspace, workspace_bytes, stream);
}
