// Shared helpers for the damvs_b200 kernels (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include "../../include/damvs.h"

namespace damvs {

// ---- error plumbing (defined in capi.cu) -----------------------------------
int set_error(int code, const char* fmt, ...);
void count_launch();

#define DAMVS_REQUIRE(cond, ...)                                   \
  do {                                                             \
    if (!(cond)) return ::damvs::set_error(DAMVS_ERR_INVALID, __VA_ARGS__); \
  } while (0)

#define DAMVS_CUDA_OK(expr)                                                                   \
  do {                                                                                        \
    cudaError_t e__ = (expr);                                                                 \
    if (e__ != cudaSuccess)                                                                   \
      return ::damvs::set_error(DAMVS_ERR_CUDA, "%s failed: %s", #expr, cudaGetErrorString(e__)); \
  } while (0)

// Check the launch itself (not completion: every entry point is asynchronous).
#define DAMVS_LAUNCH_OK(name)                                                                 \
  do {                                                                                        \
    ::damvs::count_launch();                                                                  \
    cudaError_t e__ = cudaGetLastError();                                                     \
    if (e__ != cudaSuccess)                                                                   \
      return ::damvs::set_error(DAMVS_ERR_CUDA, "launch of %s failed: %s", name, cudaGetErrorString(e__)); \
  } while (0)

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// SM count of the CURRENT device, cached per device ordinal (a process may drive several GPUs, e.g. DataParallel threads).
inline int current_sm_count() {
  static int cache[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0) return 148;
  if (dev < 64 && cache[dev]) return cache[dev];
  int n = 0;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) return 148;
  if (dev < 64) cache[dev] = n;
  return n;
}

// ---- G8 volume addressing ---------------------------------------------------
// element offset of channel 0 of group g at voxel (z,y,x) of batch item b
__host__ __device__ inline size_t g8_offset(int b, int g, int z, int y, int x, int G, int D, int H, int W) {
  return ((((size_t)b * G + g) * D + z) * H + y) * (size_t)W * 8 + (size_t)x * 8;
}

// ---- 8-channel vector load/store in either dtype ----------------------------
struct F8 {
  float v[8];
};

__device__ __forceinline__ F8 load8(const float* p) {
  F8 r;
  float4 a = __ldg(reinterpret_cast<const float4*>(p));
  float4 b = __ldg(reinterpret_cast<const float4*>(p) + 1);
  r.v[0] = a.x; r.v[1] = a.y; r.v[2] = a.z; r.v[3] = a.w;
  r.v[4] = b.x; r.v[5] = b.y; r.v[6] = b.z; r.v[7] = b.w;
  return r;
}

__device__ __forceinline__ F8 load8(const __nv_bfloat16* p) {
  F8 r;
  uint4 u = __ldg(reinterpret_cast<const uint4*>(p));
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    r.v[2 * i] = __uint_as_float(w[i] << 16);
    r.v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
  }
  return r;
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&h);
}

// fp32 pair -> packed fp16x2, round to nearest even, saturating to +-65504 (never inf)
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

__device__ __forceinline__ F8 load8(const __half* p) {
  F8 r;
  uint4 u = __ldg(reinterpret_cast<const uint4*>(p));
  const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 f = __half22float2(h[i]);
    r.v[2 * i] = f.x;
    r.v[2 * i + 1] = f.y;
  }
  return r;
}

// 2-byte element type of a reduced-precision volume and its conversions (F16 = true: IEEE half, false: bfloat16)
template <bool F16> struct HalfT { using type = __nv_bfloat16; };
template <> struct HalfT<true> { using type = __half; };
template <bool F16> __device__ __forceinline__ uint32_t pack_half2(float lo, float hi) { return F16 ? pack_f16x2(lo, hi) : pack_bf16x2(lo, hi); }
// low / high element of a packed pair as fp32
template <bool F16> __device__ __forceinline__ float unpack_lo(uint32_t w) {
  if (F16) return __half2float(__ushort_as_half((unsigned short)(w & 0xffffu)));
  return __uint_as_float(w << 16);
}
template <bool F16> __device__ __forceinline__ float unpack_hi(uint32_t w) {
  if (F16) return __half2float(__ushort_as_half((unsigned short)(w >> 16)));
  return __uint_as_float(w & 0xffff0000u);
}

__device__ __forceinline__ void store8(float* p, const F8& r) {
  reinterpret_cast<float4*>(p)[0] = make_float4(r.v[0], r.v[1], r.v[2], r.v[3]);
  reinterpret_cast<float4*>(p)[1] = make_float4(r.v[4], r.v[5], r.v[6], r.v[7]);
}

__device__ __forceinline__ void store8(__nv_bfloat16* p, const F8& r) {
  uint4 u;
  u.x = pack_bf16x2(r.v[0], r.v[1]);
  u.y = pack_bf16x2(r.v[2], r.v[3]);
  u.z = pack_bf16x2(r.v[4], r.v[5]);
  u.w = pack_bf16x2(r.v[6], r.v[7]);
  *reinterpret_cast<uint4*>(p) = u;
}

__device__ __forceinline__ void store8(__half* p, const F8& r) {
  uint4 u;
  u.x = pack_f16x2(r.v[0], r.v[1]);
  u.y = pack_f16x2(r.v[2], r.v[3]);
  u.z = pack_f16x2(r.v[4], r.v[5]);
  u.w = pack_f16x2(r.v[6], r.v[7]);
  *reinterpret_cast<uint4*>(p) = u;
}

__device__ __forceinline__ void store4(__half* p, float a, float b, float c, float d) {
  uint2 u;
  u.x = pack_f16x2(a, b);
  u.y = pack_f16x2(c, d);
  *reinterpret_cast<uint2*>(p) = u;
}
__device__ __forceinline__ void store4(float* p, float a, float b, float c, float d) {
  *reinterpret_cast<float4*>(p) = make_float4(a, b, c, d);
}
__device__ __forceinline__ void store4(__nv_bfloat16* p, float a, float b, float c, float d) {
  uint2 u;
  u.x = pack_bf16x2(a, b);
  u.y = pack_bf16x2(c, d);
  *reinterpret_cast<uint2*>(p) = u;
}

}  // namespace damvs
