// common.cuh — shared host/device helpers for libmilb200 (sm_100a only).
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/milb200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libmilb200 is written for sm_100a (B200) only"
#endif

namespace milb200 {

// ---- error plumbing -------------------------------------------------------------------------
void set_error(const char* fmt, ...);
void count_launch(int n = 1);

#define MIL_CHECK_ARG(cond, code, ...)            \
  do {                                            \
    if (!(cond)) {                                \
      ::milb200::set_error(__VA_ARGS__);          \
      return (code);                              \
    }                                             \
  } while (0)

#define MIL_CUDA(call)                                                                   \
  do {                                                                                   \
    cudaError_t e__ = (call);                                                            \
    if (e__ != cudaSuccess) {                                                            \
      ::milb200::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call,                  \
                           cudaGetErrorString(e__));                                     \
      return MILB200_ECUDA;                                                              \
    }                                                                                    \
  } while (0)

#define MIL_LAUNCH_CHECK()                                                               \
  do {                                                                                   \
    ::milb200::count_launch();                                                           \
    cudaError_t e__ = cudaGetLastError();                                                \
    if (e__ != cudaSuccess) {                                                            \
      ::milb200::set_error("%s:%d launch -> %s", __FILE__, __LINE__,                     \
                           cudaGetErrorString(e__));                                     \
      return MILB200_ECUDA;                                                              \
    }                                                                                    \
  } while (0)

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
inline int elem_size(int dtype) { return dtype == MILB200_BF16 ? 2 : 4; }
int sm_count();

// bump allocator over the caller's workspace
struct Workspace {
  char* base;
  size_t size, used;
  Workspace(void* p, size_t n) : base(static_cast<char*>(p)), size(n), used(0) {}
  template <typename T>
  T* take(size_t count) {
    size_t off = align_up(used, 256);
    size_t bytes = count * sizeof(T);
    if (base == nullptr || off + bytes > size) return nullptr;
    used = off + bytes;
    return reinterpret_cast<T*>(base + off);
  }
};
inline size_t ws_need(size_t running, size_t bytes) { return align_up(running, 256) + bytes; }

// ---- device helpers -------------------------------------------------------------------------
#ifdef __CUDACC__
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

// 128-bit streaming load (read-once data: bypass L1 allocation)
__device__ __forceinline__ uint4 ldg_stream(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

__device__ __forceinline__ float bf16lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf16hi(uint32_t u) { return __uint_as_float(u & 0xffff0000u); }
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&h);
}

template <typename T> struct Vec16;  // one 16-byte vector of T, unpacked to fp32
template <> struct Vec16<float> {
  static constexpr int N = 4;
  __device__ static __forceinline__ void unpack(const uint4& v, float* f) {
    f[0] = __uint_as_float(v.x); f[1] = __uint_as_float(v.y);
    f[2] = __uint_as_float(v.z); f[3] = __uint_as_float(v.w);
  }
  __device__ static __forceinline__ uint4 pack(const float* f) {
    return make_uint4(__float_as_uint(f[0]), __float_as_uint(f[1]), __float_as_uint(f[2]),
                      __float_as_uint(f[3]));
  }
};
template <> struct Vec16<__nv_bfloat16> {
  static constexpr int N = 8;
  __device__ static __forceinline__ void unpack(const uint4& v, float* f) {
    f[0] = bf16lo(v.x); f[1] = bf16hi(v.x); f[2] = bf16lo(v.y); f[3] = bf16hi(v.y);
    f[4] = bf16lo(v.z); f[5] = bf16hi(v.z); f[6] = bf16lo(v.w); f[7] = bf16hi(v.w);
  }
  __device__ static __forceinline__ uint4 pack(const float* f) {
    return make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]),
                      pack_bf16(f[6], f[7]));
  }
};

template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) {
  return __bfloat162float(v);
}
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) {
  return __float2bfloat16_rn(v);
}

__device__ __forceinline__ float sigmoid_precise(float x) { return 1.0f / (1.0f + expf(-x)); }
__device__ __forceinline__ float tanh_fast(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float sigmoid_fast(float x) { return fmaf(0.5f, tanh_fast(0.5f * x), 0.5f); }

// Adam's bias correction 1 - beta^step.  Written as -expm1(step * log1p(beta - 1)) (beta - 1 is exact) because
// 1 - powf(beta, step) cancels: at beta = 0.999, step 2 it keeps only 5 correct digits.  Every Adam kernel computes it
// here, on the device, so the eager, graphed and fused updates agree bit for bit.
__device__ __forceinline__ float adam_bias_correction(float beta, int step) {
  return -expm1f(static_cast<float>(step) * log1pf(beta - 1.f));
}

// Philox4x32-10 counter-based generator (dropout masks in core.cu, the feeder's row sampler in resident.cu): a pure
// function of (counter, key), so a mask or a subset is regenerated instead of stored.
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, ctr.x), lo0 = 0xD2511F53u * ctr.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, ctr.z), lo1 = 0xCD9E8D57u * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += 0x9E3779B9u;
    key.y += 0xBB67AE85u;
  }
  return ctr;
}

// index of the bag that owns global row `row`: largest b with offsets[b] <= row
__device__ __forceinline__ int find_bag(const int32_t* __restrict__ offsets, int B, int64_t row) {
  int lo = 0, hi = B;  // invariant: offsets[lo] <= row < offsets[hi]
  while (hi - lo > 1) {
    int mid = (lo + hi) >> 1;
    if (static_cast<int64_t>(__ldg(offsets + mid)) <= row) lo = mid; else hi = mid;
  }
  return lo;
}
#endif  // __CUDACC__

}  // namespace milb200
