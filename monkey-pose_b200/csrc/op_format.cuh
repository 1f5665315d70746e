// Number format of the 16-bit operands of the hGRU's own tcgen05 convolutions (the gated and H1 operands of the
// 15x15 convs, the 1x1 gate staging tiles, the packed p_r / i_r / o_r weights).  bf16 and fp16 use the same
// instruction (tcgen05.mma kind::f16) at the same rate, with the same 2-byte elements and shared-memory layouts:
// only the A/B format bits of the instruction descriptor and the float -> 16-bit conversions differ, and those live
// here.  The kernels take one of these as a template parameter.  kParts: 16-bit operands stored per value (the split
// GEMM of gemm_tc.cuh also takes the hi + lo pair OpBf16x3).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <cstdint>

namespace hgru {

// bf16: 8 significand bits, fp32's exponent range
struct OpBf16 {
  using T = __nv_bfloat16;
  using T2 = __nv_bfloat162;
  static constexpr uint32_t kIdescFmt = 1;      // sm100::make_idesc format
  static constexpr int kParts = 1;
  __device__ static __forceinline__ T cvt(float v) { return __float2bfloat16(v); }
  __device__ static __forceinline__ float to_float(T v) { return __bfloat162float(v); }
  // (a -> low half, b -> high half: element order in memory)
  __device__ static __forceinline__ T2 cvt2(float a, float b) { return __floats2bfloat162_rn(a, b); }
};

// fp16: 11 significand bits.  Round to nearest with .satfinite: a value beyond +-65504 becomes +-65504, so a
// conversion never creates inf or NaN.  The operands are tanh / sigmoid bounded except the first timestep's gated
// operand G1 . O_0, where an initial state beyond that range is clamped.
struct OpFp16 {
  using T = __half;
  using T2 = __half2;
  static constexpr uint32_t kIdescFmt = 0;
  static constexpr int kParts = 1;
  __device__ static __forceinline__ T cvt(float v) {
    unsigned short u;
    asm("cvt.rn.satfinite.f16.f32 %0, %1;" : "=h"(u) : "f"(v));
    return __ushort_as_half(u);
  }
  __device__ static __forceinline__ float to_float(T v) { return __half2float(v); }
  __device__ static __forceinline__ T2 cvt2(float a, float b) {
    T2 h;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;"      // (first source -> high half)
        : "=r"(*reinterpret_cast<uint32_t*>(&h)) : "f"(b), "f"(a));
    return h;
  }
};

// bf16 hi + lo pairs (hi = bf16(x), lo = bf16(x - hi)): ~16 significand bits from three bf16 products per k-step
// (A_hi*B_hi + A_lo*B_hi + A_hi*B_lo), fp32-class accuracy at a third of the bf16 rate
struct OpBf16x3 : OpBf16 {
  static constexpr int kParts = 2;
};

}  // namespace hgru
