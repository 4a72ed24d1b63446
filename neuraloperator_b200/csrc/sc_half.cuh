// Element conversion of the 16-bit image storage (SC_FLAG_GRID_F16 / SC_FLAG_GRID_BF16): ONE __host__ __device__ pair, used by the
// tensor-core transform kernels (x loads, dx stores), the conversion kernel and the host check sc_hostcheck_convert.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cstdint>

#include "spectral_conv_b200.h"

namespace sc {

template <int G>
__host__ __device__ __forceinline__ float g16_load(uint16_t bits) {
  if constexpr (G == SC_FLAG_GRID_F16) {
    __half_raw r; r.x = bits; return __half2float(__half(r));
  } else {
    __nv_bfloat16_raw r; r.x = bits; return __bfloat162float(__nv_bfloat16(r));
  }
}

template <int G>
__host__ __device__ __forceinline__ uint16_t g16_store(float f) {
  if constexpr (G == SC_FLAG_GRID_F16) return __half_raw(__float2half_rn(f)).x;
  else return __nv_bfloat16_raw(__float2bfloat16_rn(f)).x;
}

// two floats -> one 32-bit word of 16-bit values, the first in the low half
template <int G>
__host__ __device__ __forceinline__ uint32_t g16_pack2(float a, float b) {
  return (uint32_t)g16_store<G>(a) | ((uint32_t)g16_store<G>(b) << 16);
}

}  // namespace sc
