// K6: DPM-Solver++ multistep step  [x0 prediction at t_k] -> [update to t_{k+1}] -> [known-region injection].
//
// One launch per model evaluation of GaussianDiffusion.dpm_solver_sample_loop.  HBM-bound and elementwise like K4:
// a second-order step with injection reads x, eps, m_{k-1}, gt, noise (5 x 12 B per pixel) and the mask (4 B), and
// writes m_k and x_next (2 x 12 B) plus the next evaluation's stem channels.
//
// Rounding contract (as sampler_step.cu): every product and sum is an explicit __fmul_rn / __fadd_rn / __fsub_rn, so
// the compiler may not contract them into FMAs and oracle/dpm_solver_oracle.py can mirror the kernel bit for bit.
#include "common.cuh"

namespace fidm {

struct MultistepParams {
  fidm_multistep_args a;
};

__device__ __forceinline__ float ms_clamp1(float v) { return fminf(fmaxf(v, -1.0f), 1.0f); }

template <int VEC>
__global__ void __launch_bounds__(256) multistep_step_kernel(const MultistepParams p) {
  const fidm_multistep_args& a = p.a;
  const float* cf = a.coef + (long long)a.step * FIDM_MS_COLS;
  const float c1 = cf[FIDM_MS_X0_C1], c2 = cf[FIDM_MS_X0_C2];
  const float kA = cf[FIDM_MS_A], kB0 = cf[FIDM_MS_B0], kB1 = cf[FIDM_MS_B1];
  const float ca = cf[FIDM_MS_INJ_A], cs = cf[FIDM_MS_INJ_S];
  const bool second = a.m_prev != nullptr;
  const bool upd = a.x_next != nullptr;
  const bool inj = upd && a.inject;
  const int hw_v = a.hw / VEC;
  const long long total = (long long)a.batch * a.channels * hw_v;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int pv = (int)(idx % hw_v);
    const int bc = (int)(idx / hw_v);
    const int c = bc % a.channels;
    const int b = bc / a.channels;
    const long long off = ((long long)b * a.channels + c) * a.hw + (long long)pv * VEC;
    const long long ooff = ((long long)b * a.out_channels + c) * a.hw + (long long)pv * VEC;
    const int mc = (a.mask_channels == 1) ? 0 : c;
    const long long moff = ((long long)b * a.mask_channels + mc) * a.hw + (long long)pv * VEC;

    // every load of this element is issued before any arithmetic (one memory round trip)
    float xs[VEC], mo[VEC], mp[VEC], g[VEC], n[VEC], m[VEC];
    load_vec<float, VEC>(a.x + off, xs);
    load_vec<float, VEC>(a.model_out + ooff, mo);
    if (upd && second) load_vec<float, VEC>(a.m_prev + off, mp);
    if (inj) {
      load_vec<float, VEC>(a.gt + off, g);
      load_vec<float, VEC>(a.inject_noise + off, n);
      load_vec<float, VEC>(a.keep_mask + moff, m);
    }

    float x0[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      float v = (a.mean_type == FIDM_MEAN_START_X) ? mo[i] : __fsub_rn(__fmul_rn(c1, xs[i]), __fmul_rn(c2, mo[i]));
      x0[i] = a.clip_denoised ? ms_clamp1(v) : v;
    }
    store_vec<float, VEC>(a.m_out + off, x0);
    if (!upd) continue;

    float xn[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      float v = __fadd_rn(__fmul_rn(kA, xs[i]), __fmul_rn(kB0, x0[i]));
      if (second) v = __fadd_rn(v, __fmul_rn(kB1, mp[i]));
      if (inj) {  // K4's injection: x = m*wg + (1-m)*x, wg = a*gt + s*n
        const float wg = __fadd_rn(__fmul_rn(ca, g[i]), __fmul_rn(cs, n[i]));
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

extern "C" int fidm_multistep_step(const fidm_multistep_args* a, fidm_stream_t stream) {
  using namespace fidm;
  FIDM_REQUIRE(a != nullptr, FIDM_E_BADARG, "multistep_step: null args");
  FIDM_REQUIRE(a->batch > 0 && a->channels > 0 && a->hw > 0, FIDM_E_BADARG, "multistep_step: empty shape");
  FIDM_REQUIRE(a->mean_type == FIDM_MEAN_EPSILON || a->mean_type == FIDM_MEAN_START_X, FIDM_E_BADARG,
               "multistep_step: mean_type must be EPSILON or START_X");
  FIDM_REQUIRE(a->out_channels == a->channels || a->out_channels == 2 * a->channels, FIDM_E_BADARG,
               "multistep_step: out_channels must be channels or 2*channels");
  FIDM_REQUIRE(a->coef && a->x && a->model_out && a->m_out, FIDM_E_BADARG,
               "multistep_step: coef/x/model_out/m_out are required");
  FIDM_REQUIRE(a->steps > 0 && a->step >= 0 && a->step < a->steps, FIDM_E_BADARG,
               "multistep_step: step %d out of range [0,%d)", a->step, a->steps);
  FIDM_REQUIRE(a->m_prev == nullptr || a->step > 0, FIDM_E_BADARG, "multistep_step: step 0 has no m_prev");
  if (a->inject) {
    FIDM_REQUIRE(a->x_next != nullptr, FIDM_E_BADARG, "multistep_step: an injection needs x_next");
    FIDM_REQUIRE(a->gt && a->keep_mask && a->inject_noise, FIDM_E_BADARG,
                 "multistep_step: gt/keep_mask/inject_noise required for an injection");
    FIDM_REQUIRE(a->mask_channels == 1 || a->mask_channels == a->channels, FIDM_E_BADARG,
                 "multistep_step: mask_channels must be 1 or channels");
  }
  if (a->stem_out)
    FIDM_REQUIRE(a->x_next != nullptr && a->stem_ld >= a->channels &&
                     (a->stem_dtype == FIDM_F32 || a->stem_dtype == FIDM_BF16 || a->stem_dtype == FIDM_F16),
                 FIDM_E_BADARG, "multistep_step: stem_out needs x_next, stem_ld >= channels and a dtype of F32 | BF16 | F16");
  MultistepParams p;
  p.a = *a;
  const bool vec4 = (a->hw % 4 == 0) && (((uintptr_t)a->x | (uintptr_t)a->model_out | (uintptr_t)a->m_prev |
                                          (uintptr_t)a->m_out | (uintptr_t)a->x_next | (uintptr_t)a->gt |
                                          (uintptr_t)a->keep_mask | (uintptr_t)a->inject_noise) % 16 == 0);
  const long long total = (long long)a->batch * a->channels * (a->hw / (vec4 ? 4 : 1));
  long long blocks = (total + 255) / 256;
  const long long cap = (long long)num_sms() * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  if (vec4)
    multistep_step_kernel<4><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(p);
  else
    multistep_step_kernel<1><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(p);
  FIDM_CHECK_LAUNCH("multistep_step");
  return 0;
}
