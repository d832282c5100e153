// Leaf pieces of the pixel-row epilogues of K1 (conv_tc.cu) and K1h (conv_halo.cu).  A thread holds one pixel row of a
// 64-channel chunk of the accumulator, `float f[64]`.  Each kernel keeps its own control flow (where operands are
// loaded, barriers, TMEM release, split-K) and calls these for the arithmetic and the staging-tile layout.
#pragma once
#include <cuda_bf16.h>
#include <stdint.h>

#include "sm100_primitives.cuh"

namespace fidm {
namespace epi {

// f[2k] += low bf16 of t's word k, f[2k + 1] += its high bf16
__device__ __forceinline__ void add_bf16x8(float* f, uint4 t) {
  const uint32_t u[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    f[2 * k] += __uint_as_float(u[k] << 16);
    f[2 * k + 1] += __uint_as_float(u[k] & 0xFFFF0000u);
  }
}

// 8 fp32 -> 8 bf16 (round to nearest even), in add_bf16x8's packing
__device__ __forceinline__ uint4 pack_bf16x8(const float* f) {
  uint4 pk;
  __nv_bfloat162 b0 = __floats2bfloat162_rn(f[0], f[1]);
  __nv_bfloat162 b1 = __floats2bfloat162_rn(f[2], f[3]);
  __nv_bfloat162 b2 = __floats2bfloat162_rn(f[4], f[5]);
  __nv_bfloat162 b3 = __floats2bfloat162_rn(f[6], f[7]);
  pk.x = *reinterpret_cast<uint32_t*>(&b0);
  pk.y = *reinterpret_cast<uint32_t*>(&b1);
  pk.z = *reinterpret_cast<uint32_t*>(&b2);
  pk.w = *reinterpret_cast<uint32_t*>(&b3);
  return pk;
}

// f += a 64-channel fp32 row (bias, timestep row): 16-byte aligned
__device__ __forceinline__ void add_f32_row(float (&f)[64], const float* src) {
  const float4* s4 = reinterpret_cast<const float4*>(src);
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    const float4 t = __ldg(s4 + j);
    f[4 * j] += t.x; f[4 * j + 1] += t.y; f[4 * j + 2] += t.z; f[4 * j + 3] += t.w;
  }
}

// f += a 64-channel bf16 row (residual) in global memory: 16-byte aligned
__device__ __forceinline__ void add_bf16_row(float (&f)[64], const __nv_bfloat16* src) {
  const uint4* s = reinterpret_cast<const uint4*>(src);
#pragma unroll
  for (int j = 0; j < 8; ++j) add_bf16x8(f + 8 * j, __ldg(s + j));
}

// f += row `row` of a [128][64] bf16 tile in shared memory with the 128-byte swizzle; row_addr is that row's address
__device__ __forceinline__ void add_bf16_row_smem(float (&f)[64], uint32_t row_addr, int row) {
#pragma unroll
  for (int j = 0; j < 8; ++j) add_bf16x8(f + 8 * j, sm100::ld_shared_u32x4(row_addr + ((j ^ (row & 7)) << 4)));
}

// row `row` of the [128][64] bf16 staging tile (the box of the TMA store, 128-byte swizzle) <- bf16(f); srow is that
// row's address
__device__ __forceinline__ void stage_bf16_row(uint8_t* srow, int row, const float (&f)[64]) {
#pragma unroll
  for (int u = 0; u < 8; ++u) *reinterpret_cast<uint4*>(srow + ((u ^ (row & 7)) << 4)) = pack_bf16x8(f + 8 * u);
}

// Fused GroupNorm statistics: (sum, sum of squares) of channel `col` over rows [64 half, 64 half + 64) of the staged bf16
// tile at shared address `tile`.  With one thread per (col, half), a warp reads 32 consecutive channels of one row
// (conflict-free under the swizzle).
__device__ __forceinline__ float2 staged_col_stats(uint32_t tile, int col, int half) {
  const uint32_t sb0 = tile + (col & 7) * 2;
  const int unit = col >> 3;
  float s1 = 0.0f, s2 = 0.0f;
#pragma unroll 8
  for (int r = half * 64; r < half * 64 + 64; ++r) {
    const float v = __uint_as_float(sm100::ld_shared_u16(sb0 + r * 128 + ((unit ^ (r & 7)) << 4)) << 16);
    s1 += v;
    s2 = fmaf(v, v, s2);
  }
  return make_float2(s1, s2);
}

// The 16-wide head (6 of 16 channels valid): accumulator columns v of output channels c0 .. c0 + 15, + bias + timestep
// row, stored fp32 NCHW at pixel (n, h, w) for the channels below p.cout_valid.
template <class Params>
__device__ __forceinline__ void store_head16(const Params& p, const uint32_t (&v)[16], int c0, int n, int h, int w) {
  const long long hw = (long long)p.H * p.W;
  float* o = p.y_nchw + ((long long)n * p.cout_valid) * hw + (long long)h * p.W + w;
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    const int c = c0 + j;
    if (c < p.cout_valid) {
      float val = __uint_as_float(v[j]);
      if (p.bias) val += __ldg(p.bias + c);
      if (p.row_add) val += __ldg(p.row_add + (long long)n * p.ld_row_add + c);
      o[(long long)c * hw] = val;
    }
  }
}

}  // namespace epi
}  // namespace fidm
