// K6: DPM-Solver++ multistep step  [x0 prediction at t_k] -> [update to t_{k+1}] -> [known-region injection].
//
// One launch per model evaluation of GaussianDiffusion.dpm_solver_sample_loop.  HBM-bound and elementwise like K4:
// a second-order step with injection reads x, eps, m_{k-1}, gt, noise (5 x 12 B per pixel) and the mask (4 B), and
// writes m_k and x_next (2 x 12 B) plus the next evaluation's stem channels.
//
// Rounding contract (as sampler_step.cu): every product and sum is an explicit __fmul_rn / __fadd_rn / __fsub_rn, so
// the compiler may not contract them into FMAs and oracle/dpm_solver_oracle.py can mirror the kernel bit for bit.
//
// SEEDED (fidm_multistep_step_seeded): the injection noise is generated in registers (philox.cuh) instead of read.
//
// K9 (fidm_multistep_step_slots, continuous batching) is K6 per slot: the action, the grid point, the seed and the
// draws come per slot from the launch parameters, x_T is generated for an admitted slot, and a slot at its last grid
// point writes its x0 prediction to a separate buffer.  It is a kernel of its own, not a SLOTS instantiation of
// multistep_step_kernel: K6 reads its coefficient row once per launch, before the element loop, and K9 per slot inside
// it, so a shared template would change K6's code.  The x0, update and injection expressions are K6's, operation for
// operation.
#include "sampler_common.cuh"

namespace fidm {

template <bool SEEDED>
struct MultistepParams {
  fidm_multistep_args a;
};
template <>
struct MultistepParams<true> {
  fidm_multistep_args a;
  fidm_seeded_noise s;
};

__device__ __forceinline__ float ms_clamp1(float v) { return fminf(fmaxf(v, -1.0f), 1.0f); }

template <int VEC, bool SEEDED>
__global__ void __launch_bounds__(256) multistep_step_kernel(const MultistepParams<SEEDED> p) {
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
    const SamplerElem e = sampler_elem<VEC>(idx, a.channels, a.hw, a.mask_channels);
    const long long off = e.off;
    const long long ooff = ((long long)e.b * a.out_channels + e.c) * a.hw + (long long)e.pv * VEC;

    // every load of this element is issued before any arithmetic (one memory round trip)
    float xs[VEC], mo[VEC], mp[VEC], g[VEC], n[VEC], m[VEC];
    load_vec<float, VEC>(a.x + off, xs);
    load_vec<float, VEC>(a.model_out + ooff, mo);
    if (upd && second) load_vec<float, VEC>(a.m_prev + off, mp);
    if (inj) {
      load_vec<float, VEC>(a.gt + off, g);
      if constexpr (SEEDED)
        seeded_elem_normals<VEC>(p.s, e, a.hw, p.s.inject_tag, p.s.inject_draw, n);
      else
        load_vec<float, VEC>(a.inject_noise + off, n);
      load_vec<float, VEC>(a.keep_mask + e.moff, m);
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
      xn[i] = inj ? inject(v, m[i], g[i], n[i], ca, cs) : v;
    }
    store_vec<float, VEC>(a.x_next + off, xn);
    write_stem<VEC>(a, idx, e, xn);
  }
}

// The unseeded (s == nullptr) and seeded entries; `who` prefixes the error text.
static int multistep_step(const fidm_multistep_args* a, const fidm_seeded_noise* s, fidm_stream_t stream,
                          const char* who) {
  FIDM_REQUIRE(a != nullptr, FIDM_E_BADARG, "%s: null args", who);
  FIDM_REQUIRE(a->batch > 0 && a->channels > 0 && a->hw > 0, FIDM_E_BADARG, "%s: empty shape", who);
  FIDM_REQUIRE(a->mean_type == FIDM_MEAN_EPSILON || a->mean_type == FIDM_MEAN_START_X, FIDM_E_BADARG,
               "%s: mean_type must be EPSILON or START_X", who);
  FIDM_REQUIRE(a->out_channels == a->channels || a->out_channels == 2 * a->channels, FIDM_E_BADARG,
               "%s: out_channels must be channels or 2*channels", who);
  FIDM_REQUIRE(a->coef && a->x && a->model_out && a->m_out, FIDM_E_BADARG,
               "%s: coef/x/model_out/m_out are required", who);
  FIDM_REQUIRE(a->steps > 0 && a->step >= 0 && a->step < a->steps, FIDM_E_BADARG,
               "%s: step %d out of range [0,%d)", who, a->step, a->steps);
  FIDM_REQUIRE(a->m_prev == nullptr || a->step > 0, FIDM_E_BADARG, "%s: step 0 has no m_prev", who);
  if (s) {
    if (int rc = check_seeded(s, a->inject != 0, who)) return rc;
    FIDM_REQUIRE(a->inject_noise == nullptr, FIDM_E_BADARG, "%s: inject_noise must be NULL", who);
  }
  if (a->inject) {
    FIDM_REQUIRE(a->x_next != nullptr, FIDM_E_BADARG, "%s: an injection needs x_next", who);
    FIDM_REQUIRE(a->gt && a->keep_mask && (s || a->inject_noise), FIDM_E_BADARG,
                 "%s: gt/keep_mask/inject_noise required for an injection", who);
    if (int rc = check_mask_channels(a, who)) return rc;
  }
  FIDM_REQUIRE(a->stem_out == nullptr || a->x_next != nullptr, FIDM_E_BADARG, "%s: stem_out needs x_next", who);
  if (int rc = check_stem(a, who)) return rc;
  const bool vec4 = vec4_ok(a->hw, a->x, a->model_out, a->m_prev, a->m_out, a->x_next, a->gt, a->keep_mask,
                            a->inject_noise);
  const long long elems = (long long)a->batch * a->channels * a->hw;
  if (s)
    return launch_sampler(multistep_step_kernel<4, true>, multistep_step_kernel<1, true>, vec4, elems,
                          MultistepParams<true>{*a, *s}, stream, who);
  return launch_sampler(multistep_step_kernel<4, false>, multistep_step_kernel<1, false>, vec4, elems,
                        MultistepParams<false>{*a}, stream, who);
}

struct MsSlotParams {
  fidm_multistep_args a;
  fidm_ms_slot_args s;
};

template <int VEC>
__global__ void __launch_bounds__(256) multistep_slots_kernel(const MsSlotParams p) {
  const fidm_multistep_args& a = p.a;
  const int hw_v = a.hw / VEC;
  const long long total = (long long)a.batch * a.channels * hw_v;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const SamplerElem e = sampler_elem<VEC>(idx, a.channels, a.hw, a.mask_channels);
    // the slot's action: idle, admit (x_T and the injection at t_0), or the evaluation at grid point k
    const int act = p.s.action[e.b];
    if (act == FIDM_SLOT_IDLE) continue;
    const bool admit = act == FIDM_SLOT_ADMIT;
    const int k = admit ? 0 : act;
    const bool last = !admit && k == a.steps - 1;
    const int next = admit ? 0 : k + 1;             // the grid point of the injection, the state and t_out
    const int draw = last ? -1 : p.s.inject_draw[next];
    const bool inj = draw >= 0;
    // the history is read only where the row is second order: an admitted slot's history is the previous request's
    const bool second = !admit && !last && p.s.order[k] == 2;
    const long long off = e.off;
    const long long ooff = ((long long)e.b * a.out_channels + e.c) * a.hw + (long long)e.pv * VEC;
    const uint64_t seed = p.s.seeds[e.b];
    const long long j = (long long)e.c * a.hw + (long long)e.pv * VEC;

    // every load of this element is issued before any arithmetic (one memory round trip)
    float xs[VEC], mo[VEC], mp[VEC], g[VEC], n[VEC], m[VEC];
    if (admit) {
      seeded_normals<VEC>(seed, j, FIDM_NOISE_XT, 0u, xs);
    } else {
      load_vec<float, VEC>(a.x + off, xs);
      load_vec<float, VEC>(a.model_out + ooff, mo);
    }
    if (second) load_vec<float, VEC>(a.m_prev + off, mp);
    if (inj) {
      load_vec<float, VEC>(a.gt + off, g);
      seeded_normals<VEC>(seed, j, (uint32_t)p.s.inject_tag, (uint32_t)draw, n);
      load_vec<float, VEC>(a.keep_mask + e.moff, m);
    }

    float xn[VEC];
    if (admit) {
#pragma unroll
      for (int i = 0; i < VEC; ++i)
        xn[i] = inj ? inject(xs[i], m[i], g[i], n[i], p.s.admit_inject_a, p.s.admit_inject_s) : xs[i];
    } else {
      const float* cf = a.coef + (long long)k * FIDM_MS_COLS;
      const float c1 = cf[FIDM_MS_X0_C1], c2 = cf[FIDM_MS_X0_C2];
      float x0[VEC];
#pragma unroll
      for (int i = 0; i < VEC; ++i) {
        float v = (a.mean_type == FIDM_MEAN_START_X) ? mo[i] : __fsub_rn(__fmul_rn(c1, xs[i]), __fmul_rn(c2, mo[i]));
        x0[i] = a.clip_denoised ? ms_clamp1(v) : v;
      }
      if (last) {                                   // the request's result: kept apart until the host collects it
        store_vec<float, VEC>(p.s.out + off, x0);
        continue;
      }
      store_vec<float, VEC>(a.m_out + off, x0);
      const float kA = cf[FIDM_MS_A], kB0 = cf[FIDM_MS_B0], kB1 = cf[FIDM_MS_B1];
      const float ca = cf[FIDM_MS_INJ_A], cs = cf[FIDM_MS_INJ_S];
#pragma unroll
      for (int i = 0; i < VEC; ++i) {
        float v = __fadd_rn(__fmul_rn(kA, xs[i]), __fmul_rn(kB0, x0[i]));
        if (second) v = __fadd_rn(v, __fmul_rn(kB1, mp[i]));
        xn[i] = inj ? inject(v, m[i], g[i], n[i], ca, cs) : v;
      }
    }
    store_vec<float, VEC>(a.x_next + off, xn);
    store_stem<VEC>(a, e, xn);
    if (a.t_out && e.c == 0 && e.pv == 0) a.t_out[e.b] = p.s.t_value[next];
  }
}

static int multistep_step_slots(const fidm_multistep_args* a, const fidm_ms_slot_args* s, fidm_stream_t stream) {
  const char* who = "multistep_step_slots";
  FIDM_REQUIRE(a != nullptr && s != nullptr, FIDM_E_BADARG, "%s: null args", who);
  FIDM_REQUIRE(a->batch >= 1 && a->batch <= FIDM_MAX_SLOTS, FIDM_E_BADARG, "%s: %d slots outside [1, %d]", who,
               a->batch, FIDM_MAX_SLOTS);
  FIDM_REQUIRE(a->channels > 0 && a->hw > 0 && a->steps > 0, FIDM_E_BADARG, "%s: empty shape", who);
  FIDM_REQUIRE(a->mean_type == FIDM_MEAN_EPSILON || a->mean_type == FIDM_MEAN_START_X, FIDM_E_BADARG,
               "%s: mean_type must be EPSILON or START_X", who);
  FIDM_REQUIRE(a->out_channels == a->channels || a->out_channels == 2 * a->channels, FIDM_E_BADARG,
               "%s: out_channels must be channels or 2*channels", who);
  FIDM_REQUIRE(a->coef && a->x && a->m_prev && a->m_out && a->x_next && a->gt && a->keep_mask && s->out && s->t_value &&
                   s->inject_draw && s->order,
               FIDM_E_BADARG, "%s: coef/x/m_prev/m_out/x_next/gt/keep_mask/out/t_value/inject_draw/order are required",
               who);
  FIDM_REQUIRE(a->inject_noise == nullptr, FIDM_E_BADARG, "%s: inject_noise must be NULL", who);
  FIDM_REQUIRE(s->inject_tag == FIDM_NOISE_INJECT || s->inject_tag == FIDM_NOISE_INJECT_FRESH, FIDM_E_BADARG,
               "%s: inject_tag must be INJECT | INJECT_FRESH", who);
  if (int rc = check_mask_channels(a, who)) return rc;
  bool any_update = false;
  for (int b = 0; b < a->batch; ++b) {
    const int act = s->action[b];
    FIDM_REQUIRE(act == FIDM_SLOT_IDLE || act == FIDM_SLOT_ADMIT || (act >= 0 && act < a->steps), FIDM_E_BADARG,
                 "%s: slot %d: action %d is not IDLE, ADMIT or a grid point in [0,%d)", who, b, act, a->steps);
    any_update |= act >= 0;
  }
  FIDM_REQUIRE(!any_update || a->model_out != nullptr, FIDM_E_BADARG, "%s: model_out required for an update", who);
  if (int rc = check_stem(a, who)) return rc;
  const bool vec4 = vec4_ok(a->hw, a->x, a->model_out, a->m_prev, a->m_out, a->x_next, a->gt, a->keep_mask, s->out);
  const long long elems = (long long)a->batch * a->channels * a->hw;
  return launch_sampler(multistep_slots_kernel<4>, multistep_slots_kernel<1>, vec4, elems, MsSlotParams{*a, *s}, stream,
                        who);
}

}  // namespace fidm

extern "C" int fidm_multistep_step_slots(const fidm_multistep_args* a, const fidm_ms_slot_args* s,
                                         fidm_stream_t stream) {
  return fidm::multistep_step_slots(a, s, stream);
}

extern "C" int fidm_multistep_step(const fidm_multistep_args* a, fidm_stream_t stream) {
  return fidm::multistep_step(a, nullptr, stream, "multistep_step");
}

extern "C" int fidm_multistep_step_seeded(const fidm_multistep_args* a, const fidm_seeded_noise* s,
                                          fidm_stream_t stream) {
  FIDM_REQUIRE(s != nullptr, FIDM_E_BADARG, "multistep_step_seeded: seeded noise is required");
  return fidm::multistep_step(a, s, stream, "multistep_step_seeded");
}
