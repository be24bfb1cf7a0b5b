// Shared device/host helpers for libi2it (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <cstdint>
#include <cstdio>
#include <string>
#include <stdexcept>

namespace i2it {

// ---------------------------------------------------------------------------------------------
// host-side error plumbing: everything below the C ABI throws; the ABI layer converts to codes
// ---------------------------------------------------------------------------------------------
struct Error : std::runtime_error {
  using std::runtime_error::runtime_error;
};

#define I2IT_CHECK(cond, msg)                                                                  \
  do {                                                                                         \
    if (!(cond)) throw ::i2it::Error(std::string(__FILE__) + ":" + std::to_string(__LINE__) + \
                                     ": " + (msg));                                            \
  } while (0)

#define I2IT_CUDA(expr)                                                                        \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess)                                                                     \
      throw ::i2it::Error(std::string(__FILE__) + ":" + std::to_string(__LINE__) + ": " #expr \
                          " -> " + cudaGetErrorString(_e));                                    \
  } while (0)

enum DType : int { DT_F16 = 0, DT_BF16 = 1, DT_F32 = 2 };

// ---------------------------------------------------------------------------------------------
// 16-bit element helpers (the path computes in fp16 or bf16 with fp32 accumulation)
// ---------------------------------------------------------------------------------------------
template <typename T> struct Elem;
template <> struct Elem<__half> {
  using V2 = __half2;
  static constexpr int kDType = DT_F16;
  __device__ static __forceinline__ float to_f(__half v) { return __half2float(v); }
  __device__ static __forceinline__ __half from_f(float v) { return __float2half_rn(v); }
  __device__ static __forceinline__ uint32_t pack(float a, float b) {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  }
  __device__ static __forceinline__ float2 unpack(uint32_t u) {
    return __half22float2(*reinterpret_cast<__half2*>(&u));
  }
};
template <> struct Elem<__nv_bfloat16> {
  using V2 = __nv_bfloat162;
  static constexpr int kDType = DT_BF16;
  __device__ static __forceinline__ float to_f(__nv_bfloat16 v) { return __bfloat162float(v); }
  __device__ static __forceinline__ __nv_bfloat16 from_f(float v) { return __float2bfloat16_rn(v); }
  __device__ static __forceinline__ uint32_t pack(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  }
  __device__ static __forceinline__ float2 unpack(uint32_t u) {
    return __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&u));
  }
};

// x * sigmoid(x) with ex2.approx + approximate division (2 MUFU ops; the IEEE division cost ~10 extra instructions/element)
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float silu_f(float x) { return __fdividef(x, 1.0f + ex2_approx(-1.4426950408889634f * x)); }

// erf via Abramowitz-Stegun 7.1.26 (|abs err| < 1.5e-7, far below the 16-bit output rounding): 1 rcp + 1 ex2 + 7 FMA
__device__ __forceinline__ float erf_as(float x) {
  const float ax = fabsf(x);
  const float t = __fdividef(1.0f, fmaf(0.3275911f, ax, 1.0f));
  const float poly = t * (0.254829592f + t * (-0.284496736f + t * (1.421413741f + t * (-1.453152027f + t * 1.061405429f))));
  const float y = 1.0f - poly * ex2_approx(-1.4426950408889634f * ax * ax);
  return copysignf(y, x);
}
__device__ __forceinline__ float gelu_erf_f(float x) { return 0.5f * x * (1.0f + erf_as(x * 0.70710678118654752f)); }

// CLIP's quick_gelu: x * sigmoid(1.702 x)
__device__ __forceinline__ float quick_gelu_f(float x) { return __fdividef(x, 1.0f + ex2_approx(-1.702f * 1.4426950408889634f * x)); }

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

// 16-byte streaming global access (activations are read once per kernel: keep them out of L1)
__device__ __forceinline__ uint4 ld_nc16(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void st16(void* p, const uint4& v) {
  asm volatile("st.global.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

}  // namespace i2it
