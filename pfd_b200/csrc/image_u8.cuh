// ToPILImage quantisation shared by the control-image pre-processing kernels (canny.cu, hed.cu).
#pragma once
#include <cuda_fp16.h>
#include <stdint.h>

namespace pfd {

// ToPILImage on a float tensor: pic.mul(255).byte() - the product is rounded in the tensor's dtype, then truncated
template <typename T>
__device__ __forceinline__ uint32_t to_u8(T v);
template <>
__device__ __forceinline__ uint32_t to_u8<float>(float v) {
  const float m = v * 255.f;
  return (uint32_t)(unsigned char)(int)m;
}
template <>
__device__ __forceinline__ uint32_t to_u8<__half>(__half v) {
  const float m = __half2float(__hmul(v, __float2half_rn(255.f)));
  return (uint32_t)(unsigned char)(int)m;
}

}  // namespace pfd
