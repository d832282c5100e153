// K7: RePaint undo-and-inject  [re-noise t-1 -> t_up] -> [known-region injection at t_up] -> [next stem input].
//
// One launch per jump of GaussianDiffusion.repaint_sample_loop, after the DDPM update of K4.  HBM-bound and
// elementwise: with injection it reads x, u, gt, noise (4 x 12 B per pixel) and the mask (4 B), and writes x_next
// (12 B) plus the next evaluation's stem channels.
//
// Rounding contract (as sampler_step.cu): every product and sum is an explicit __fmul_rn / __fadd_rn / __fsub_rn, so
// the compiler may not contract them into FMAs and oracle/repaint_oracle.py can mirror the kernel bit for bit.
#include "sampler_common.cuh"

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
    const SamplerElem e = sampler_elem<VEC>(idx, a.channels, a.hw, a.mask_channels);
    const long long off = e.off;

    // every load of this element is issued before any arithmetic (one memory round trip)
    float xs[VEC], u[VEC], g[VEC], n[VEC], m[VEC];
    load_vec<float, VEC>(a.x + off, xs);
    load_vec<float, VEC>(a.noise + off, u);
    if (a.inject) {
      load_vec<float, VEC>(a.gt + off, g);
      load_vec<float, VEC>(a.inject_noise + off, n);
      load_vec<float, VEC>(a.keep_mask + e.moff, m);
    }

    float xn[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      const float v = __fadd_rn(__fmul_rn(a.undo_a, xs[i]), __fmul_rn(a.undo_s, u[i]));
      xn[i] = a.inject ? inject(v, m[i], g[i], n[i], a.inject_a, a.inject_s) : v;
    }
    store_vec<float, VEC>(a.x_next + off, xn);
    write_stem<VEC>(a, idx, e, xn);
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
    if (int rc = check_mask_channels(a, "resample_undo")) return rc;
  }
  if (int rc = check_stem(a, "resample_undo")) return rc;
  ResampleParams p;
  p.a = *a;
  const bool vec4 = vec4_ok(a->hw, a->x, a->noise, a->x_next, a->gt, a->keep_mask, a->inject_noise);
  return launch_sampler(resample_undo_kernel<4>, resample_undo_kernel<1>, vec4,
                        (long long)a->batch * a->channels * a->hw, p, stream, "resample_undo");
}
