// Shared device/host helpers for the crop2seg_b200 kernels (sm_100a only).
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>

#include "../../include/crop2seg_b200.h"

namespace c2s {

// ---------------------------------------------------------------------------------------------
// host-side error plumbing (thread-local, no aborts)
// ---------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
void note_launch(const char* kernel_name);
// C2S_OK when the current device is an sm_100 part, C2S_ERR_NO_DEVICE (with message) otherwise.
int check_device();
// current value of a c2s_option (c2s_set_option); 0 = production behaviour
int option(int which);
// cudaFuncAttributeMaxDynamicSharedMemorySize once per (kernel, device): `done` is a static flag word of the caller
int set_max_dynamic_smem(const void* func, int bytes, std::atomic<unsigned long long>* done);
#define C2S_SMEM_ATTR(kernel, bytes)                                                                \
  do {                                                                                              \
    static std::atomic<unsigned long long> done__{0};                                               \
    const int st__ = ::c2s::set_max_dynamic_smem(reinterpret_cast<const void*>(kernel), static_cast<int>(bytes), &done__); \
    if (st__ != C2S_OK) return st__;                                                                \
  } while (0)

#define C2S_CHECK_ARG(cond, ...)        \
  do {                                  \
    if (!(cond)) {                      \
      ::c2s::set_error(__VA_ARGS__);    \
      return C2S_ERR_BAD_ARGUMENT;      \
    }                                   \
  } while (0)

#define C2S_UNSUPPORTED(...)            \
  do {                                  \
    ::c2s::set_error(__VA_ARGS__);      \
    return C2S_ERR_UNSUPPORTED;         \
  } while (0)

#define C2S_CUDA(call)                                                                  \
  do {                                                                                  \
    cudaError_t err__ = (call);                                                         \
    if (err__ != cudaSuccess) {                                                         \
      ::c2s::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(err__),       \
                       __FILE__, __LINE__);                                             \
      return C2S_ERR_CUDA;                                                              \
    }                                                                                   \
  } while (0)

#define C2S_LAUNCH_CHECK(name)                                                          \
  do {                                                                                  \
    ::c2s::note_launch(name);                                                           \
    cudaError_t err__ = cudaGetLastError();                                             \
    if (err__ != cudaSuccess) {                                                         \
      ::c2s::set_error("launch of %s failed: %s", name, cudaGetErrorString(err__));     \
      return C2S_ERR_CUDA;                                                              \
    }                                                                                   \
  } while (0)

// ---------------------------------------------------------------------------------------------
// element types: 16-byte vectors of V pixels
// ---------------------------------------------------------------------------------------------
template <typename T>
struct Elem;

template <>
struct Elem<float> {
  static constexpr int kVec = 4;  // elements per 16-byte vector
  __device__ static __forceinline__ void unpack(const uint4& v, float (&f)[4]) {
    f[0] = __uint_as_float(v.x);
    f[1] = __uint_as_float(v.y);
    f[2] = __uint_as_float(v.z);
    f[3] = __uint_as_float(v.w);
  }
  __device__ static __forceinline__ uint4 pack(const float (&f)[4]) {
    return make_uint4(__float_as_uint(f[0]), __float_as_uint(f[1]), __float_as_uint(f[2]),
                      __float_as_uint(f[3]));
  }
  __device__ static __forceinline__ float load(const float* p) { return *p; }
  __device__ static __forceinline__ void store(float* p, float v) { *p = v; }
};

template <>
struct Elem<__nv_bfloat16> {
  static constexpr int kVec = 8;
  // bf16 -> fp32 is a 16-bit shift: the low element of a packed pair moves up, the high one is masked.
  __device__ static __forceinline__ void unpack(const uint4& v, float (&f)[8]) {
    f[0] = __uint_as_float(v.x << 16);
    f[1] = __uint_as_float(v.x & 0xffff0000u);
    f[2] = __uint_as_float(v.y << 16);
    f[3] = __uint_as_float(v.y & 0xffff0000u);
    f[4] = __uint_as_float(v.z << 16);
    f[5] = __uint_as_float(v.z & 0xffff0000u);
    f[6] = __uint_as_float(v.w << 16);
    f[7] = __uint_as_float(v.w & 0xffff0000u);
  }
  __device__ static __forceinline__ uint32_t pack2(float lo, float hi) {
    __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&h);
  }
  __device__ static __forceinline__ uint4 pack(const float (&f)[8]) {
    return make_uint4(pack2(f[0], f[1]), pack2(f[2], f[3]), pack2(f[4], f[5]), pack2(f[6], f[7]));
  }
  __device__ static __forceinline__ float load(const __nv_bfloat16* p) { return __bfloat162float(*p); }
  __device__ static __forceinline__ void store(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
};

// Streaming 128-bit load: read-only path, do not allocate in L1 (each input byte is used once).
__device__ __forceinline__ uint4 ld_stream_v4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.L2::128B.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

__device__ __forceinline__ void st_stream_v4(void* p, const uint4& v) {
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y),
               "r"(v.z), "r"(v.w)
               : "memory");
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ATen area_pixel_compute_source_index(scale, dst, align_corners=false) + the i0/i1/lambda split of upsample_bilinear2d
// (nn.Upsample of the attention masks, reference temporal_aggregator.py:17-19).  The aggregator's forward and backward
// must agree on it.
__device__ __forceinline__ void source_index(float scale, int dst, int in_size, int& i0, int& i1, float& l1) {
  float src = scale * (static_cast<float>(dst) + 0.5f) - 0.5f;
  src = src < 0.f ? 0.f : src;
  i0 = static_cast<int>(src);
  i0 = i0 < in_size - 1 ? i0 : in_size - 1;
  i1 = i0 + (i0 < in_size - 1 ? 1 : 0);
  l1 = src - static_cast<float>(i0);
}

inline int ceil_div(long long a, long long b) { return static_cast<int>((a + b - 1) / b); }

}  // namespace c2s
