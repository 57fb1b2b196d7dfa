// Shared device/host helpers for libdva_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <atomic>
#include "../../include/dva_b200.h"

namespace dva {

constexpr int kNumSMs = 148;  // B200: 2 dies x 74 SMs; grids are sized in multiples of this

// ---- thread-local error string + launch counter (C ABI: dva_last_error), process-wide launch counter (dva_launch_count)
char* tls_error_buf();
std::atomic<int64_t>& launch_counter();

inline int fail(int code, const char* msg) {
  snprintf(tls_error_buf(), 256, "%s", msg);
  return code;
}

template <typename... A> inline int failf(int code, const char* fmt, A... a) {
  snprintf(tls_error_buf(), 256, fmt, a...);
  return code;
}

inline int check_launch(const char* what) {
  launch_counter().fetch_add(1, std::memory_order_relaxed);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    snprintf(tls_error_buf(), 256, "%s: %s", what, cudaGetErrorString(e));
    return (int)e;
  }
  return DVA_OK;
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// ---- storage-type traits: load/store as fp32
template <typename T> struct Cvt;
template <> struct Cvt<float> {
  static __device__ __forceinline__ float to_f(float v) { return v; }
  static __device__ __forceinline__ float from_f(float v) { return v; }
};
template <> struct Cvt<__nv_bfloat16> {
  static __device__ __forceinline__ float to_f(__nv_bfloat16 v) { return __bfloat162float(v); }
  static __device__ __forceinline__ __nv_bfloat16 from_f(float v) { return __float2bfloat16_rn(v); }
};
template <> struct Cvt<__half> {
  static __device__ __forceinline__ float to_f(__half v) { return __half2float(v); }
  static __device__ __forceinline__ __half from_f(float v) { return __float2half_rn(v); }
};

// 16-byte vector of T: float x4, bf16/half x8
template <typename T> struct Vec16 { static constexpr int N = 16 / sizeof(T); };

template <typename T, int N>
struct alignas(sizeof(T) * N) Pack { T v[N]; };

// streaming 16-byte load/store (rows are touched once: keep them out of L1)
__device__ __forceinline__ uint4 ldg_stream16(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void stg_stream16(void* p, const uint4& v) {
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};"
               :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

template <typename T, int VEC>
__device__ __forceinline__ void unpack16(const uint4& raw, float (&f)[VEC]);
template <> __device__ __forceinline__ void unpack16<float, 4>(const uint4& raw, float (&f)[4]) {
  f[0] = __uint_as_float(raw.x); f[1] = __uint_as_float(raw.y);
  f[2] = __uint_as_float(raw.z); f[3] = __uint_as_float(raw.w);
}
template <> __device__ __forceinline__ void unpack16<__nv_bfloat16, 8>(const uint4& raw, float (&f)[8]) {
  const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {  // bf16 -> fp32 is a 16-bit shift
    f[2 * i] = __uint_as_float(w[i] << 16);
    f[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
  }
}
template <> __device__ __forceinline__ void unpack16<__half, 8>(const uint4& raw, float (&f)[8]) {
  const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    __half2 h = *reinterpret_cast<const __half2*>(&w[i]);
    float2 t = __half22float2(h);
    f[2 * i] = t.x; f[2 * i + 1] = t.y;
  }
}

template <typename T, int VEC>
__device__ __forceinline__ uint4 pack16(const float (&f)[VEC]);
template <> __device__ __forceinline__ uint4 pack16<float, 4>(const float (&f)[4]) {
  return make_uint4(__float_as_uint(f[0]), __float_as_uint(f[1]), __float_as_uint(f[2]),
                    __float_as_uint(f[3]));
}
template <> __device__ __forceinline__ uint4 pack16<__nv_bfloat16, 8>(const float (&f)[8]) {
  uint32_t w[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    __nv_bfloat162 h = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
    w[i] = *reinterpret_cast<uint32_t*>(&h);
  }
  return make_uint4(w[0], w[1], w[2], w[3]);
}
template <> __device__ __forceinline__ uint4 pack16<__half, 8>(const float (&f)[8]) {
  uint32_t w[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    __half2 h = __floats2half2_rn(f[2 * i], f[2 * i + 1]);
    w[i] = *reinterpret_cast<uint32_t*>(&h);
  }
  return make_uint4(w[0], w[1], w[2], w[3]);
}

// ---- async-copy PTX wrappers: cp.async (LDGSTS), mbarriers, bulk copies (UBLKCP)
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
// the destination bytes past src_bytes (0 or 16) are zero-filled
__device__ __forceinline__ void cp_async16_zfill(uint32_t dst, const void* src, int src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
        : "=r"(done) : "r"(bar), "r"(parity) : "memory");
  } while (!done);
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
// orders earlier generic-proxy accesses of shared memory before later async-proxy ones
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- 3xTF32 on mma.sync: x = hi + lo with hi = tf32(x), lo = tf32(x - hi), both rounded to nearest
__device__ __forceinline__ uint32_t to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ void mma_tf32(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// channel -> group of pooling.py:737-755 (group_sizes / expand_group_feat):
// sizes floor(C/G), the first C%G groups one wider.
__host__ __device__ __forceinline__ int group_of_channel(int c, int C, int G) {
  const int base = C / G, rem = C - base * G;
  const int wide = rem * (base + 1);
  return c < wide ? c / (base + 1) : rem + (c - wide) / base;
}

__device__ __forceinline__ int64_t load_idx(const void* idx, bool is64, int64_t v) {
  if (idx == nullptr) return v;
  return is64 ? reinterpret_cast<const int64_t*>(idx)[v]
              : (int64_t) reinterpret_cast<const int32_t*>(idx)[v];
}

}  // namespace dva
