// Element types of the data points X (the float32, bfloat16 and float16 paths of class sums, Gram and
// transform). A kernel templated on the element type widens every element to float32 as it is loaded
// (exact: bf16 / fp16 values are float32 values) and then does exactly what it does for float32 points,
// so only the bytes read and how they are staged depend on the type.
#pragma once
#include <cstdint>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

namespace sqfa {

template <typename T>
struct ElemBits;  // float32 value of the raw bits of one element
template <>
struct ElemBits<__nv_bfloat16> {
  static __device__ __forceinline__ float widen(uint32_t u16) { return __uint_as_float(u16 << 16); }
  // the two elements of a 32-bit word (element 0 in the low half)
  static __device__ __forceinline__ float2 widen2(uint32_t w) {
    return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u));
  }
};
template <>
struct ElemBits<__half> {
  static __device__ __forceinline__ float widen(uint32_t u16) { return __half2float(__ushort_as_half((unsigned short)u16)); }
  static __device__ __forceinline__ float2 widen2(uint32_t w) {
    __half2 h;
    *reinterpret_cast<uint32_t*>(&h) = w;
    return __half22float2(h);
  }
};

// four adjacent elements (8 bytes) -> float4
template <typename T>
__device__ __forceinline__ float4 widen4(uint2 v) {
  const float2 a = ElemBits<T>::widen2(v.x), b = ElemBits<T>::widen2(v.y);
  return make_float4(a.x, a.y, b.x, b.y);
}

// one element through the read-only path, widened
template <typename T>
__device__ __forceinline__ float ldg_widen(const T* p) {
  if constexpr (sizeof(T) == 4) {
    return __ldg(reinterpret_cast<const float*>(p));
  } else {
    return ElemBits<T>::widen(__ldg(reinterpret_cast<const unsigned short*>(p)));
  }
}

// four adjacent elements, 4-element aligned (16 bytes for float32, 8 bytes for bf16 / fp16), widened
template <typename T>
__device__ __forceinline__ float4 ldg_widen4(const T* p) {
  if constexpr (sizeof(T) == 4) {
    return __ldg(reinterpret_cast<const float4*>(p));
  } else {
    return widen4<T>(__ldg(reinterpret_cast<const uint2*>(p)));
  }
}

}  // namespace sqfa
