// The operand activation of the fused GroupNorm convolutions K1h (conv_halo.cu) and K1s (conv_halo_swap.cu):
// silu(x*A + B) of two packed bf16 values of the raw stream, with (a, b) = (A/2, B/2) per channel.
#pragma once
#include <stdint.h>

namespace fidm {

// h = x*A/2 + B/2, then silu = h + h*tanh(h): one MUFU op per value.  (tanh.approx.f16x2 was tried: ptxas splits it
// into two MUFU.TANH.F16, so it saves no MUFU issue slots and only costs accuracy.)
__device__ __forceinline__ void silu_pair(uint32_t raw, float a0, float b0, float a1, float b1, float& y0, float& y1) {
  const float h0 = fmaf(__uint_as_float(raw << 16), a0, b0);
  const float h1 = fmaf(__uint_as_float(raw & 0xFFFF0000u), a1, b1);
  float t0, t1;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t0) : "f"(h0));
  asm("tanh.approx.f32 %0, %1;" : "=f"(t1) : "f"(h1));
  y0 = fmaf(h0, t0, h0);
  y1 = fmaf(h1, t1, h1);
}

// -> two packed 16-bit results (fp16 or bf16, channel 0 in the low half)
template <bool OUT_F16>
__device__ __forceinline__ uint32_t act_pair(uint32_t raw, float a0, float b0, float a1, float b1) {
  float y0, y1;
  silu_pair(raw, a0, b0, a1, b1, y0, y1);
  uint32_t o;
  if (OUT_F16) {
    // saturating: |GroupNorm output| <= sqrt(group size) (724 at 256^2), so gamma * (1 + scale) >~ 90 would overflow
    // fp16 (65504) to inf and poison the whole image through the MMA; satfinite clamps at the cost of nothing
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(o) : "f"(y1), "f"(y0));
  } else {
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(o) : "f"(y1), "f"(y0));
  }
  return o;
}

// FP8 operand (tcgen05 kind::f8f6f4, e4m3): -> two packed e4m3 bytes (channel 0 in the low byte).  satfinite: e4m3 has
// no inf, values beyond 448 clamp.
__device__ __forceinline__ uint32_t act_pair_e4m3(uint32_t raw, float a0, float b0, float a1, float b1) {
  float y0, y1;
  silu_pair(raw, a0, b0, a1, b1, y0, y1);
  unsigned short o;
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(o) : "f"(y1), "f"(y0));
  return (uint32_t)o;
}

}  // namespace fidm
