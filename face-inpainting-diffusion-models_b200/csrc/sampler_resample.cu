// K7: RePaint undo-and-inject  [re-noise t-1 -> t_up] -> [known-region injection at t_up] -> [next stem input].
//
// One launch per jump of GaussianDiffusion.repaint_sample_loop, after the DDPM update of K4.  HBM-bound and
// elementwise: with injection it reads x, u, gt, noise (4 x 12 B per pixel) and the mask (4 B), and writes x_next
// (12 B) plus the next evaluation's stem channels.
//
// Rounding contract (as sampler_step.cu): every product and sum is an explicit __fmul_rn / __fadd_rn / __fsub_rn, so
// the compiler may not contract them into FMAs and oracle/repaint_oracle.py can mirror the kernel bit for bit.
//
// SEEDED (fidm_resample_undo_seeded): the undo noise u and the injection noise are generated in registers
// (philox.cuh) instead of read.
#include "sampler_common.cuh"

namespace fidm {

template <bool SEEDED>
struct ResampleParams {
  fidm_resample_args a;
};
template <>
struct ResampleParams<true> {
  fidm_resample_args a;
  fidm_seeded_noise s;
};

template <int VEC, bool SEEDED>
__global__ void __launch_bounds__(256) resample_undo_kernel(const ResampleParams<SEEDED> p) {
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
    if constexpr (SEEDED)
      seeded_elem_normals<VEC>(p.s, e, a.hw, FIDM_NOISE_UNDO, p.s.draw, u);
    else
      load_vec<float, VEC>(a.noise + off, u);
    if (a.inject) {
      load_vec<float, VEC>(a.gt + off, g);
      if constexpr (SEEDED)
        seeded_elem_normals<VEC>(p.s, e, a.hw, p.s.inject_tag, p.s.inject_draw, n);
      else
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

// The unseeded (s == nullptr) and seeded entries; `who` prefixes the error text.
static int resample_undo(const fidm_resample_args* a, const fidm_seeded_noise* s, fidm_stream_t stream,
                         const char* who) {
  FIDM_REQUIRE(a != nullptr, FIDM_E_BADARG, "%s: null args", who);
  FIDM_REQUIRE(a->batch > 0 && a->channels > 0 && a->hw > 0, FIDM_E_BADARG, "%s: empty shape", who);
  FIDM_REQUIRE(a->x && (s || a->noise) && a->x_next, FIDM_E_BADARG, "%s: x/noise/x_next are required", who);
  if (s) {
    if (int rc = check_seeded(s, a->inject != 0, who)) return rc;
    FIDM_REQUIRE(a->noise == nullptr && a->inject_noise == nullptr, FIDM_E_BADARG,
                 "%s: noise/inject_noise must be NULL", who);
    FIDM_REQUIRE(s->draw >= 0, FIDM_E_BADARG, "%s: undo noise draw %d < 0", who, s->draw);
  }
  if (a->inject) {
    FIDM_REQUIRE(a->gt && a->keep_mask && (s || a->inject_noise), FIDM_E_BADARG,
                 "%s: gt/keep_mask/inject_noise required for an injection", who);
    if (int rc = check_mask_channels(a, who)) return rc;
  }
  if (int rc = check_stem(a, who)) return rc;
  const bool vec4 = vec4_ok(a->hw, a->x, a->noise, a->x_next, a->gt, a->keep_mask, a->inject_noise);
  const long long elems = (long long)a->batch * a->channels * a->hw;
  if (s)
    return launch_sampler(resample_undo_kernel<4, true>, resample_undo_kernel<1, true>, vec4, elems,
                          ResampleParams<true>{*a, *s}, stream, who);
  return launch_sampler(resample_undo_kernel<4, false>, resample_undo_kernel<1, false>, vec4, elems,
                        ResampleParams<false>{*a}, stream, who);
}

}  // namespace fidm

extern "C" int fidm_resample_undo(const fidm_resample_args* a, fidm_stream_t stream) {
  return fidm::resample_undo(a, nullptr, stream, "resample_undo");
}

extern "C" int fidm_resample_undo_seeded(const fidm_resample_args* a, const fidm_seeded_noise* s,
                                         fidm_stream_t stream) {
  FIDM_REQUIRE(s != nullptr, FIDM_E_BADARG, "resample_undo_seeded: seeded noise is required");
  return fidm::resample_undo(a, s, stream, "resample_undo_seeded");
}
