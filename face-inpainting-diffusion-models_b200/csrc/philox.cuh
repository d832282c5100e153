// Counter-based per-image Gaussian noise: Philox4x32-10 (Salmon et al. 2011, "Parallel random numbers: as easy as
// 1, 2, 3") and Box-Muller.  This header is the one place the key/counter layout and the normal transform are
// written; oracle/philox_oracle.py restates them, and the seeded sampler kernels (K4, K6, K7) and fidm_randn_seeded
// all take their values from seeded_normals() below, so every code path gives the same value for the same element.
//
//   key      = (seed & 0xffffffff, seed >> 32)        seed: the image's uint64
//   counter  = (q, draw, tag, 0)                      q = j >> 2, j = c*hw + p: flat NCHW index within the image
//   normals  = Box-Muller on (w0, w1) -> lanes 0, 1 and (w2, w3) -> lanes 2, 3 of group q; element j takes lane j & 3
//   u        = (w + 0.5) * 2^-32 in fp32, never 0:  r = sqrt(-2 log u1) reaches ~6.7 sigma;  theta = 2 pi u2
//
// Every step is an explicit IEEE operation (no FMA contraction, no fast-math intrinsics), so the value of an element
// does not depend on the kernel, the VEC width or the inlining context it is computed in.
#pragma once
#include <stdint.h>

namespace fidm {

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r > 0) {
      k0 += 0x9E3779B9u;
      k1 += 0xBB67AE85u;
    }
    const uint32_t lo0 = 0xD2511F53u * c.x, hi0 = __umulhi(0xD2511F53u, c.x);
    const uint32_t lo1 = 0xCD9E8D57u * c.z, hi1 = __umulhi(0xCD9E8D57u, c.z);
    c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
  }
  return c;
}

// (w + 0.5) * 2^-32: in (0, 1].
__device__ __forceinline__ float philox_uniform(uint32_t w) {
  return __fmul_rn(__fadd_rn(__uint2float_rn(w), 0.5f), 2.3283064365386963e-10f);
}

// Box-Muller on one word pair: (r cos 2 pi u2, r sin 2 pi u2).
__device__ __forceinline__ float2 box_muller(uint32_t w1, uint32_t w2) {
  const float r = sqrtf(__fmul_rn(-2.0f, logf(philox_uniform(w1))));
  float s, c;
  sincospif(__fmul_rn(2.0f, philox_uniform(w2)), &s, &c);
  return make_float2(__fmul_rn(r, c), __fmul_rn(r, s));
}

// The VEC normals of elements j .. j+VEC-1 of one image, draw (tag, draw) under `seed`.  VEC = 4 needs j % 4 == 0
// (one whole group); VEC = 1 computes the word pair of its lane only.
template <int VEC>
__device__ __forceinline__ void seeded_normals(uint64_t seed, long long j, uint32_t tag, uint32_t draw,
                                               float (&n)[VEC]) {
  const uint4 w = philox4x32_10(make_uint4((uint32_t)(j >> 2), draw, tag, 0u), (uint32_t)seed,
                                (uint32_t)(seed >> 32));
  if constexpr (VEC == 4) {
    const float2 a = box_muller(w.x, w.y), b = box_muller(w.z, w.w);
    n[0] = a.x;
    n[1] = a.y;
    n[2] = b.x;
    n[3] = b.y;
  } else {
    const int lane = (int)(j & 3);
    const float2 a = (lane < 2) ? box_muller(w.x, w.y) : box_muller(w.z, w.w);
    n[0] = (lane & 1) ? a.y : a.x;
  }
}

}  // namespace fidm
