// fidm_randn_seeded: a [batch][elems_per_image] buffer of per-image seeded normals (philox.cuh), the values the seeded
// sampler kernels generate for the same draw.  Used for x_T of the seeded loops and as the test oracle's reference.
#include "common.cuh"
#include "philox.cuh"

namespace fidm {

// One thread iteration per group of 4 elements of one image (one Philox block); VEC4: the group is stored with one
// 16-byte store (elems % 4 == 0, 16-byte aligned out).
template <bool VEC4>
__global__ void __launch_bounds__(256) randn_seeded_kernel(float* __restrict__ out, const uint64_t* __restrict__ seeds,
                                                           int batch, long long elems, uint32_t tag, uint32_t draw) {
  const long long groups = (elems + 3) >> 2;
  const long long total = (long long)batch * groups;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int b = (int)(idx / groups);
    const long long j = (idx - (long long)b * groups) << 2;
    float n[4];
    seeded_normals<4>(seeds[b], j, tag, draw, n);
    float* o = out + (long long)b * elems + j;
    if constexpr (VEC4) {
      *reinterpret_cast<float4*>(o) = make_float4(n[0], n[1], n[2], n[3]);
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (j + i < elems) o[i] = n[i];
    }
  }
}

}  // namespace fidm

extern "C" int fidm_randn_seeded(float* out, const uint64_t* seeds, int32_t batch, int64_t elems_per_image,
                                 int32_t tag, int32_t draw, fidm_stream_t stream) {
  using namespace fidm;
  FIDM_REQUIRE(out && seeds, FIDM_E_BADARG, "randn_seeded: out/seeds are required");
  FIDM_REQUIRE(batch > 0 && elems_per_image > 0, FIDM_E_BADARG, "randn_seeded: empty shape");
  FIDM_REQUIRE(elems_per_image <= (4ll << 32), FIDM_E_BADARG, "randn_seeded: more than 2^34 elements per image");
  FIDM_REQUIRE(tag >= FIDM_NOISE_XT && tag <= FIDM_NOISE_UNDO && draw >= 0, FIDM_E_BADARG,
               "randn_seeded: bad tag %d or draw %d", tag, draw);
  const bool vec4 = elems_per_image % 4 == 0 && (uintptr_t)out % 16 == 0;
  const long long total = (long long)batch * ((elems_per_image + 3) >> 2);
  long long blocks = (total + 255) / 256;
  const long long cap = (long long)num_sms() * 16;
  if (blocks > cap) blocks = cap;
  (vec4 ? randn_seeded_kernel<true> : randn_seeded_kernel<false>)<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
      out, seeds, batch, elems_per_image, (uint32_t)tag, (uint32_t)draw);
  FIDM_CHECK_LAUNCH("randn_seeded");
  return 0;
}
