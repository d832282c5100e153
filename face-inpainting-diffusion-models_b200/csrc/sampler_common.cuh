// Pieces shared by the sampler kernels K4 and K8 (sampler_step.cu), K6 (sampler_multistep.cu) and K7
// (sampler_resample.cu).
// The fused-versus-unfused tests and the oracles compare these kernels bit for bit, so each piece exists once.
#pragma once
#include "common.cuh"
#include "philox.cuh"

namespace fidm {

// Grid-stride element `idx` of an NCHW fp32 state [batch, channels, hw], VEC pixels wide: batch b, channel c, pixel
// group pv, the state offset off and the offset moff into a keep mask of 1 or `channels` channels.
struct SamplerElem {
  int b, c, pv;
  long long off, moff;
};

template <int VEC>
__device__ __forceinline__ SamplerElem sampler_elem(long long idx, int channels, int hw, int mask_channels) {
  SamplerElem e;
  const int hw_v = hw / VEC;
  e.pv = (int)(idx % hw_v);
  const int bc = (int)(idx / hw_v);
  e.c = bc % channels;
  e.b = bc / channels;
  e.off = ((long long)e.b * channels + e.c) * hw + (long long)e.pv * VEC;
  const int mc = (mask_channels == 1) ? 0 : e.c;
  e.moff = ((long long)e.b * mask_channels + mc) * hw + (long long)e.pv * VEC;
  return e;
}

// Seeded mode: the VEC normals of element e under its image's seed, draw (tag, draw) -- what fidm_randn_seeded writes
// at the same place of a [batch][channels][hw] buffer.
template <int VEC>
__device__ __forceinline__ void seeded_elem_normals(const fidm_seeded_noise& s, const SamplerElem& e, int hw, int tag,
                                                    int draw, float (&n)[VEC]) {
  seeded_normals<VEC>(s.seeds[e.b], (long long)e.c * hw + (long long)e.pv * VEC, (uint32_t)tag, (uint32_t)draw, n);
}

// Known-region injection (apply_inpainting_injection): m*wg + (1-m)*v, wg = ca*gt + cs*n, one fp32 rounding per
// operation.  Takes values already in registers: the kernels issue every load of an element before any arithmetic.
__device__ __forceinline__ float inject(float v, float m, float g, float n, float ca, float cs) {
  const float wg = __fadd_rn(__fmul_rn(ca, g), __fmul_rn(cs, n));
  return __fadd_rn(__fmul_rn(m, wg), __fmul_rn(__fsub_rn(1.0f, m), v));
}

// Step-boundary fusion: the next evaluation's stem input (channel c of VEC pixels of the NHWC network input, store_stem)
// and its timestep (write_stem: one value for the whole batch).  The roundings are the pack kernel's (layout.cu), so a
// fused loop is bit-identical to pack + evaluate.  Args is any of the sampler arg structs; they share these field names.
template <int VEC, typename Args>
__device__ __forceinline__ void store_stem(const Args& a, const SamplerElem& e, const float (&v)[VEC]) {
  if (a.stem_out) {
    const long long px = (long long)e.b * a.hw + (long long)e.pv * VEC;
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      const long long s = (px + i) * a.stem_ld + e.c;
      if (a.stem_dtype == FIDM_F16)
        reinterpret_cast<__half*>(a.stem_out)[s] = from_f32<__half>(v[i]);
      else if (a.stem_dtype == FIDM_BF16)
        reinterpret_cast<__nv_bfloat16*>(a.stem_out)[s] = from_f32<__nv_bfloat16>(v[i]);
      else
        reinterpret_cast<float*>(a.stem_out)[s] = v[i];
    }
  }
}

template <int VEC, typename Args>
__device__ __forceinline__ void write_stem(const Args& a, long long idx, const SamplerElem& e, const float (&v)[VEC]) {
  store_stem<VEC>(a, e, v);
  if (a.t_out && idx < a.batch) a.t_out[idx] = a.t_out_value;
}

// ---- host side.  `who` prefixes the error text with the entry point's name.
template <typename Args>
inline int check_stem(const Args* a, const char* who) {
  if (a->stem_out)
    FIDM_REQUIRE(a->stem_ld >= a->channels &&
                     (a->stem_dtype == FIDM_F32 || a->stem_dtype == FIDM_BF16 || a->stem_dtype == FIDM_F16),
                 FIDM_E_BADARG, "%s: stem_out needs stem_ld >= channels and a dtype of F32 | BF16 | F16", who);
  return 0;
}

template <typename Args>
inline int check_mask_channels(const Args* a, const char* who) {
  FIDM_REQUIRE(a->mask_channels == 1 || a->mask_channels == a->channels, FIDM_E_BADARG,
               "%s: mask_channels must be 1 or channels", who);
  return 0;
}

// The seeded entries: `s` and its seeds are required, and the injection draw must be a valid one when `inject`.
inline int check_seeded(const fidm_seeded_noise* s, bool inject, const char* who) {
  FIDM_REQUIRE(s != nullptr && s->seeds != nullptr, FIDM_E_BADARG, "%s: seeded noise and its seeds are required", who);
  if (inject)
    FIDM_REQUIRE((s->inject_tag == FIDM_NOISE_INJECT || s->inject_tag == FIDM_NOISE_INJECT_FRESH) && s->inject_draw >= 0,
                 FIDM_E_BADARG, "%s: the injection needs tag INJECT | INJECT_FRESH and a draw >= 0", who);
  return 0;
}

// True when the VEC=4 instantiation may run: hw is a multiple of 4 and every pointer (null or not) is 16-byte aligned.
template <typename... P>
inline bool vec4_ok(int hw, const P*... ptrs) {
  return hw % 4 == 0 && ((uintptr_t)ptrs | ... | (uintptr_t)0) % 16 == 0;
}

// Grid-stride launch over `elems` fp32 elements (`vec4`: 4 per thread and iteration), at most 16 blocks of 256 threads
// per SM.
template <typename Params>
inline int launch_sampler(void (*k4)(Params), void (*k1)(Params), bool vec4, long long elems, const Params& p,
                          fidm_stream_t stream, const char* who) {
  const long long total = elems / (vec4 ? 4 : 1);
  long long blocks = (total + 255) / 256;
  const long long cap = (long long)num_sms() * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  (vec4 ? k4 : k1)<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(p);
  FIDM_CHECK_LAUNCH(who);
  return 0;
}

}  // namespace fidm
