// Shared between the kernels of the fused view-attention pair:
//   view_attention.cu       streaming forward and backward (row chunks live in registers, one point
//                           per warp at a time; best for long segments and >= 512-byte rows)
//   view_attention_ring.cu  ring forward (rows staged in shared memory by cp.async, several batches
//                           in flight per warp across point boundaries; short segments, rows <= 512 bytes)
//   view_attention_lane.cu  lane-per-view backward (groups of <= 32 views per warp, rows by bulk async
//                           copies; short segments, rows <= 512 bytes)
#pragma once
#include "dva_common.cuh"

namespace dva {

struct VAParams {
  const void* x; const void* idx; int idx64;
  const float* compat; const int64_t* ptr;
  const float* gate_w; const float* gate_b;
  // fwd
  void* out; float* att; float* seg_max; float* seg_den; int32_t* seg_arg;
  // bwd
  const void* gout; const float* s_max; const float* s_den; const int32_t* s_arg;
  void* gx; float* gcompat; float* gate_partial; int scatter;
  int64_t N, V, R;
  int C, G, group_scaling;
  float eps;
};

constexpr int kTileStride = 33;    // att tile is [G][33]: (g,v) -> bank (g+v)%32, conflict-free

// reduce over the lanes that share (lane % G): offsets 16 .. G
__device__ __forceinline__ float group_lane_sum(float v, int G) {
  for (int off = 16; off >= G; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  return v;
}

// row of x of view v: idx[v] (int32 or int64 idx) or v itself; callers check V < 2^31, R < 2^32
__device__ __forceinline__ uint32_t load_row_id(const void* idx, int idx64, int64_t v) {
  if (idx == nullptr) return (uint32_t)v;
  return idx64 ? (uint32_t) reinterpret_cast<const int64_t*>(idx)[v]
               : (uint32_t) reinterpret_cast<const int32_t*>(idx)[v];
}

// *_applicable: shape / alignment conditions of the ring forward and the lane backward; the launchers
// return a DVA_* / cudaError code like every other entry point.
bool va_ring_fwd_applicable(const VAParams& P, int dtype);
int va_ring_fwd(const VAParams& P, int dtype, cudaStream_t st);
bool va_lane_bwd_applicable(const VAParams& P, int dtype);
int va_lane_bwd(const VAParams& P, int dtype, int* grid_out, cudaStream_t st);

}  // namespace dva
