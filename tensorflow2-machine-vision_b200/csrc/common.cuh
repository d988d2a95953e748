// common.cuh — shared host/device plumbing for libb200det.so (error slot, launch checks, warp helpers).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/b200det.h"

// thread-local error message (b200_last_error)
void b200_set_error(const char* fmt, ...);

#define B200_REQUIRE(cond, code, ...)      \
  do {                                     \
    if (!(cond)) {                         \
      b200_set_error(__VA_ARGS__);         \
      return (code);                       \
    }                                      \
  } while (0)

#define B200_CUDA(call)                                                                      \
  do {                                                                                       \
    cudaError_t _e = (call);                                                                 \
    if (_e != cudaSuccess) {                                                                 \
      b200_set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return B200_ERR_CUDA;                                                                  \
    }                                                                                        \
  } while (0)

#define B200_LAUNCH_CHECK()                                                                  \
  do {                                                                                       \
    cudaError_t _e = cudaGetLastError();                                                     \
    if (_e != cudaSuccess) {                                                                 \
      b200_set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, __LINE__); \
      return B200_ERR_CUDA;                                                                  \
    }                                                                                        \
  } while (0)

static inline size_t b200_align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// number of SMs of the current device (cached per thread)
int b200_sm_count();

#ifdef __CUDACC__
#include <cuda_bf16.h>
#include <cuda_fp16.h>

// Head elements in their own type (float, __nv_bfloat16, __half), widened to fp32 on load.  Widening bf16 / fp16 is
// exact, so every decision downstream sees the value that heads.float() would hold.
__device__ __forceinline__ float elem_f32(float x) { return x; }
__device__ __forceinline__ float elem_f32(__nv_bfloat16 x) { return __bfloat162float(x); }
__device__ __forceinline__ float elem_f32(__half x) { return __half2float(x); }
template <typename T>
__device__ __forceinline__ float ldg_f32(const T* p) { return elem_f32(__ldg(p)); }
// four consecutive elements (a box or its head offsets) at a 4-element boundary: one 16-byte load for fp32, one 8-byte
// load for the 2-byte types; STREAM marks data read once (ld.global.cs)
template <bool STREAM>
__device__ __forceinline__ float4 ld4_f32(const float* p) {
  return STREAM ? __ldcs(reinterpret_cast<const float4*>(p)) : __ldg(reinterpret_cast<const float4*>(p));
}
template <bool STREAM, typename H>
__device__ __forceinline__ float4 ld4_f32(const H* p) {
  const uint2 u = STREAM ? __ldcs(reinterpret_cast<const uint2*>(p)) : __ldg(reinterpret_cast<const uint2*>(p));
  const H* h = reinterpret_cast<const H*>(&u);
  return make_float4(elem_f32(h[0]), elem_f32(h[1]), elem_f32(h[2]), elem_f32(h[3]));
}
// Gradient elements in the caller's type (float, __nv_bfloat16, __half): round_elem<TG>(scaled_f32(g, scale)) is
// g * *scale (no multiply when scale is null) rounded once to nearest even, i.e. (g * s).to(dtype) in torch; fp16
// overflow gives +-inf.
__device__ __forceinline__ float scaled_f32(float g, const float* scale) { return scale ? g * __ldg(scale) : g; }
template <typename TG> __device__ __forceinline__ TG round_elem(float v);
template <> __device__ __forceinline__ float round_elem<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 round_elem<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ __half round_elem<__half>(float v) { return __float2half_rn(v); }
template <typename TG> __device__ __forceinline__ uint32_t round_bits16(float v) {
  const TG h = round_elem<TG>(v);
  return (uint32_t)*reinterpret_cast<const unsigned short*>(&h);
}
// four consecutive gradient elements at a 4-element boundary, streaming (st.global.cs): one 16-byte store for fp32, one
// 8-byte store of the four rounded values for the 2-byte types
template <typename TG>
__device__ __forceinline__ void st4(TG* p, float4 v) {
  if constexpr (sizeof(TG) == 4) {
    __stcs(reinterpret_cast<float4*>(p), v);
  } else {
    __stcs(reinterpret_cast<uint2*>(p), make_uint2(round_bits16<TG>(v.x) | (round_bits16<TG>(v.y) << 16),
                                                   round_bits16<TG>(v.z) | (round_bits16<TG>(v.w) << 16)));
  }
}
#endif

// Runs the statements that follow `T` with T bound to the element type of a B200_DTYPE_* code (checked by the caller).
#define B200_DISPATCH_DTYPE(code, T, ...)                                 \
  switch (code) {                                                         \
    case B200_DTYPE_BF16: { using T = __nv_bfloat16; __VA_ARGS__; } break; \
    case B200_DTYPE_F16: { using T = __half; __VA_ARGS__; } break;        \
    default: { using T = float; __VA_ARGS__; } break;                     \
  }
static inline bool b200_dtype_ok(int code) { return code == B200_DTYPE_F32 || code == B200_DTYPE_BF16 || code == B200_DTYPE_F16; }
static inline int b200_dtype_bytes(int code) { return code == B200_DTYPE_F32 ? 4 : 2; }

#ifdef __CUDACC__
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ int warp_sum_i(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// inclusive warp scan
__device__ __forceinline__ int warp_scan_incl(int v) {
  int lane = threadIdx.x & 31;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += t;
  }
  return v;
}
#endif
