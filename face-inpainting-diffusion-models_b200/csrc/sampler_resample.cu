// K7: RePaint undo-and-inject  [re-noise t-1 -> t_up] -> [known-region injection at t_up] -> [next stem input].
//
// One launch per jump of GaussianDiffusion.repaint_sample_loop, after the DDPM update of K4.  HBM-bound and
// elementwise: with injection it reads x, u, gt, noise (4 x 12 B per pixel) and the mask (4 B), and writes x_next
// (12 B) plus the next evaluation's stem channels.
//
// Rounding contract (as sampler_step.cu): every product and sum is an explicit __fmul_rn / __fadd_rn / __fsub_rn, so
// the compiler may not contract them into FMAs and oracle/repaint_oracle.py can mirror the kernel bit for bit.
#include "common.cuh"

namespace fidm {

struct ResampleParams {
  fidm_resample_args a;
};

template <int VEC>
__global__ void __launch_bounds__(256) resample_undo_kernel(const ResampleParams p) {
  const fidm_resample_args& a = p.a;
  const int hw_v = a.hw / VEC;
  const long long total = (long long)a.batch * a.channels * hw_v;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int pv = (int)(idx % hw_v);
    const int bc = (int)(idx / hw_v);
    const int c = bc % a.channels;
    const int b = bc / a.channels;
    const long long off = ((long long)b * a.channels + c) * a.hw + (long long)pv * VEC;
    const int mc = (a.mask_channels == 1) ? 0 : c;
    const long long moff = ((long long)b * a.mask_channels + mc) * a.hw + (long long)pv * VEC;

    // every load of this element is issued before any arithmetic (one memory round trip)
    float xs[VEC], u[VEC], g[VEC], n[VEC], m[VEC];
    load_vec<float, VEC>(a.x + off, xs);
    load_vec<float, VEC>(a.noise + off, u);
    if (a.inject) {
      load_vec<float, VEC>(a.gt + off, g);
      load_vec<float, VEC>(a.inject_noise + off, n);
      load_vec<float, VEC>(a.keep_mask + moff, m);
    }

    float xn[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      float v = __fadd_rn(__fmul_rn(a.undo_a, xs[i]), __fmul_rn(a.undo_s, u[i]));
      if (a.inject) {  // K4's injection: x = m*wg + (1-m)*x, wg = a*gt + s*n
        const float wg = __fadd_rn(__fmul_rn(a.inject_a, g[i]), __fmul_rn(a.inject_s, n[i]));
        v = __fadd_rn(__fmul_rn(m[i], wg), __fmul_rn(__fsub_rn(1.0f, m[i]), v));
      }
      xn[i] = v;
    }
    store_vec<float, VEC>(a.x_next + off, xn);
    // step-boundary fusion: the next evaluation's stem channels, with the pack kernel's roundings (as K4)
    if (a.stem_out) {
      const long long px = (long long)b * a.hw + (long long)pv * VEC;
#pragma unroll
      for (int i = 0; i < VEC; ++i) {
        const long long e = (px + i) * a.stem_ld + c;
        if (a.stem_dtype == FIDM_F16) reinterpret_cast<__half*>(a.stem_out)[e] = from_f32<__half>(xn[i]);
        else if (a.stem_dtype == FIDM_BF16) reinterpret_cast<__nv_bfloat16*>(a.stem_out)[e] = from_f32<__nv_bfloat16>(xn[i]);
        else reinterpret_cast<float*>(a.stem_out)[e] = xn[i];
      }
    }
    if (a.t_out && idx < a.batch) a.t_out[idx] = a.t_out_value;
  }
}

}  // namespace fidm

extern "C" int fidm_resample_undo(const fidm_resample_args* a, fidm_stream_t stream) {
  using namespace fidm;
  FIDM_REQUIRE(a != nullptr, FIDM_E_BADARG, "resample_undo: null args");
  FIDM_REQUIRE(a->batch > 0 && a->channels > 0 && a->hw > 0, FIDM_E_BADARG, "resample_undo: empty shape");
  FIDM_REQUIRE(a->x && a->noise && a->x_next, FIDM_E_BADARG, "resample_undo: x/noise/x_next are required");
  if (a->inject) {
    FIDM_REQUIRE(a->gt && a->keep_mask && a->inject_noise, FIDM_E_BADARG,
                 "resample_undo: gt/keep_mask/inject_noise required for an injection");
    FIDM_REQUIRE(a->mask_channels == 1 || a->mask_channels == a->channels, FIDM_E_BADARG,
                 "resample_undo: mask_channels must be 1 or channels");
  }
  if (a->stem_out)
    FIDM_REQUIRE(a->stem_ld >= a->channels &&
                     (a->stem_dtype == FIDM_F32 || a->stem_dtype == FIDM_BF16 || a->stem_dtype == FIDM_F16),
                 FIDM_E_BADARG, "resample_undo: stem_out needs stem_ld >= channels and a dtype of F32 | BF16 | F16");
  ResampleParams p;
  p.a = *a;
  const bool vec4 = (a->hw % 4 == 0) && (((uintptr_t)a->x | (uintptr_t)a->noise | (uintptr_t)a->x_next |
                                          (uintptr_t)a->gt | (uintptr_t)a->keep_mask | (uintptr_t)a->inject_noise) %
                                             16 == 0);
  const long long total = (long long)a->batch * a->channels * (a->hw / (vec4 ? 4 : 1));
  long long blocks = (total + 255) / 256;
  const long long cap = (long long)num_sms() * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  if (vec4)
    resample_undo_kernel<4><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(p);
  else
    resample_undo_kernel<1><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(p);
  FIDM_CHECK_LAUNCH("resample_undo");
  return 0;
}
