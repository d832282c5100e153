// K4: fused reverse-process step  [update at t] -> [known-region injection at t_inject].
//
// One launch replaces the per-step elementwise chain of the reference
// (gaussian_diffusion.py:114-157 inject, :213-298 p_mean_variance tail, :357-388 p_sample,
// :447-485 ddim_sample).  HBM-bound: DDIM eta=0 moves 64 B per pixel (read x, eps, gt, n_inj:
// 4x12 B, mask 4 B; write x 12 B).
//
// Rounding contract: every reference ATen op is one IEEE-754 fp32 rounding, so every product and
// sum below is an explicit __fmul_rn/__fadd_rn/__fsub_rn/__fdiv_rn -- the compiler may not contract
// them into FMAs.  With identical model output and noise the DDIM path is bit-identical to the
// reference; the DDPM path differs only by the ulp of expf.
//
// SEEDED (fidm_sampler_step_seeded): the step noise z and the injection noise are not read but generated in registers
// (philox.cuh), with the values fidm_randn_seeded writes for the same draws: DDIM eta=0 then moves 52 B per pixel.
//
// K8 (fidm_sampler_step_slots, continuous batching) is the same element body with SLOTS set: the action, the timesteps,
// the seed and the draws come per slot from the launch parameters, x_T is generated for an admitted slot, and a slot
// updated at t = 0 writes its sample to a separate buffer.  The update and injection arithmetic is K4's own code.
//
// K10 (fidm_repaint_step_slots, continuous batching of RePaint) is K8 with REPAINT set: the action is the slot's
// evaluation index k, the timesteps and the injection draw come from per-evaluation tables, the step noise is (STEP, k),
// and where a jump follows K7's re-noising (UNDO, k) sits between the update and the injection.  A fused jump
// evaluation therefore computes, operation for operation, the lockstep pair K4 STEP_UPDATE_ONLY -> K7.
#include "sampler_common.cuh"

namespace fidm {

template <bool SEEDED>
struct StepParams {
  fidm_step_args a;
};
template <>
struct StepParams<true> {
  fidm_step_args a;
  fidm_seeded_noise s;
};
struct SlotParams {
  fidm_step_args a;
  fidm_slot_args s;
};
struct RpSlotParams {
  fidm_step_args a;
  fidm_rp_slot_args s;
};
// The parameters of K4 (SLOTS false), K8 (SLOTS and SEEDED true) and K10 (all three true).
template <bool SEEDED, bool SLOTS, bool REPAINT>
struct KernelParams {
  using type = StepParams<SEEDED>;
};
template <>
struct KernelParams<true, true, false> {
  using type = SlotParams;
};
template <>
struct KernelParams<true, true, true> {
  using type = RpSlotParams;
};

__device__ __forceinline__ float clamp1(float v) { return fminf(fmaxf(v, -1.0f), 1.0f); }

template <int VEC, bool SEEDED, bool SLOTS, bool REPAINT = false>
__global__ void __launch_bounds__(256) sampler_step_kernel(const typename KernelParams<SEEDED, SLOTS, REPAINT>::type p) {
  const fidm_step_args& a = p.a;
  const int hw_v = a.hw / VEC;
  const long long total = (long long)a.batch * a.channels * hw_v;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const SamplerElem e = sampler_elem<VEC>(idx, a.channels, a.hw, a.mask_channels);
    const int b = e.b, c = e.c;
    const long long off = e.off;

    // K8: the slot's action -- idle, admit (x_T, injection at T-1), or update at t and injection at t-1 -- and the
    // draw of its injection (< 0: none)
    int act = 0, slot_inj_draw = -1;
    int t_upd = a.t_update, t_inj = a.t_inject;
    if constexpr (SLOTS) {
      act = p.s.action[b];
      if (act == FIDM_SLOT_IDLE) continue;
      if constexpr (REPAINT) {
        // K10: act is the evaluation index k; the walk goes on at next_t[k] (t_up after a jump)
        const bool admit = act == FIDM_SLOT_ADMIT;
        t_upd = admit ? act : p.s.eval_t[act];
        t_inj = admit ? a.num_timesteps - 1 : p.s.next_t[act];
        slot_inj_draw = admit ? p.s.admit_draw : p.s.inject_draw[act];
      } else {
        t_upd = act;
        t_inj = (act == FIDM_SLOT_ADMIT) ? a.num_timesteps - 1 : act - 1;
        if (t_inj >= 0) slot_inj_draw = p.s.inject_draw[t_inj];
      }
    }
    if (!SEEDED && a.t_dev) {
      t_upd = (int)a.t_dev[b];
      t_inj = (a.mode == FIDM_STEP_INJECT_ONLY) ? t_upd : t_upd - 1;
    }

    // Every load of this element is issued up front (one memory round trip instead of two dependent ones), and only
    // what the mode needs is read: the variance channels are skipped when neither the DDPM update nor a caller wants
    // the log-variance (DDIM: 64 B per pixel instead of 76).
    const bool upd = SLOTS ? act != FIDM_SLOT_ADMIT : a.mode != FIDM_STEP_INJECT_ONLY;
    const bool inj = SLOTS ? slot_inj_draw >= 0 : a.mode != FIDM_STEP_UPDATE_ONLY;
    const bool need_var = upd && a.var_type != FIDM_VAR_FIXED && (a.sampler == FIDM_SAMPLER_DDPM || a.logvar_out != nullptr);
    bool has_z;
    if constexpr (REPAINT) has_z = true;                 // DDPM: every update draws its step noise
    else if constexpr (SLOTS) has_z = p.s.step_noise != 0;
    else if constexpr (SEEDED) has_z = p.s.draw >= 0;
    else has_z = a.z != nullptr;
    const bool need_z = upd && has_z;
    const int oc = (a.var_type == FIDM_VAR_FIXED) ? a.channels : 2 * a.channels;
    const long long ooff = ((long long)b * oc + c) * a.hw + (long long)e.pv * VEC;
    float xs[VEC], mo[VEC], vv[VEC], zz[VEC], g[VEC], n[VEC], m[VEC];
    // K8's draws are those of the slot's seed at the element's flat index j within its image
    uint64_t seed = 0;
    long long j = 0;
    if constexpr (SLOTS) {
      seed = p.s.seeds[b];
      j = (long long)c * a.hw + (long long)e.pv * VEC;
    }
    if (!SLOTS || upd) load_vec<float, VEC>(a.x + off, xs);
    else seeded_normals<VEC>(seed, j, FIDM_NOISE_XT, 0u, xs);         // admit: x_T
    if (upd) load_vec<float, VEC>(a.model_out + ooff, mo);
    if (need_var) load_vec<float, VEC>(a.model_out + ooff + (long long)a.channels * a.hw, vv);
    if (need_z) {
      if constexpr (REPAINT)
        seeded_normals<VEC>(seed, j, FIDM_NOISE_STEP, (uint32_t)act, zz);
      else if constexpr (SLOTS)
        seeded_normals<VEC>(seed, j, FIDM_NOISE_STEP, (uint32_t)(a.num_timesteps - 1 - t_upd), zz);
      else if constexpr (SEEDED)
        seeded_elem_normals<VEC>(p.s, e, a.hw, FIDM_NOISE_STEP, p.s.draw, zz);
      else
        load_vec<float, VEC>(a.z + off, zz);
    }
    if (inj) {
      load_vec<float, VEC>(a.gt + off, g);
      if constexpr (SLOTS)
        seeded_normals<VEC>(seed, j, a.cumulative ? FIDM_NOISE_INJECT : FIDM_NOISE_INJECT_FRESH, (uint32_t)slot_inj_draw, n);
      else if constexpr (SEEDED)
        seeded_elem_normals<VEC>(p.s, e, a.hw, p.s.inject_tag, p.s.inject_draw, n);
      else
        load_vec<float, VEC>(a.inject_noise + off, n);
      load_vec<float, VEC>(a.keep_mask + e.moff, m);
    }
    // K10: a jump follows the evaluation where the walk does not go on at t - 1; its undo noise is (UNDO, k)
    [[maybe_unused]] bool jump = false;
    [[maybe_unused]] float uu[VEC];
    if constexpr (REPAINT) {
      jump = upd && t_inj != t_upd - 1;
      if (jump) seeded_normals<VEC>(seed, j, FIDM_NOISE_UNDO, (uint32_t)act, uu);
    }
    float smp[VEC], x0v[VEC];

    if (upd) {
      const float* cf = a.coef + (long long)t_upd * FIDM_COEF_COLS;
      float mv[VEC], lv[VEC];
      const float c1 = cf[FIDM_C_RECIP], c2 = cf[FIDM_C_RECIPM1];
      const float k1 = cf[FIDM_C_POST1], k2 = cf[FIDM_C_POST2];
      const float nz = cf[FIDM_C_NONZERO];
#pragma unroll
      for (int i = 0; i < VEC; ++i) {
        const float x = xs[i];
        // ---- log-variance (gaussian_diffusion.py:241-265)
        float logvar = 0.0f;
        if (!need_var && a.var_type != FIDM_VAR_FIXED) {
          // log-variance not needed (DDIM update, caller does not ask for it)
        } else if (a.var_type == FIDM_VAR_LEARNED_RANGE) {
          const float frac = __fmul_rn(__fadd_rn(vv[i], 1.0f), 0.5f);                 // (v + 1) / 2
          logvar = __fadd_rn(__fmul_rn(frac, cf[FIDM_C_MAX_LOG]),
                             __fmul_rn(__fsub_rn(1.0f, frac), cf[FIDM_C_MIN_LOG]));
        } else if (a.var_type == FIDM_VAR_LEARNED) {
          logvar = vv[i];
        } else {
          logvar = cf[FIDM_C_FIXED_LOGVAR];
        }
        // ---- pred_xstart and posterior mean (:267-286)
        float x0, mean;
        if (a.sampler == FIDM_SAMPLER_DDIM_SCRIPT) {
          // test_inp_ddim_100.py:539-542: pred_x0 = (img - sqrt(1-ab_t) * eps) / sqrt(ab_t)
          x0 = __fdiv_rn(__fsub_rn(x, __fmul_rn(c2, mo[i])), c1);
          if (a.clip_denoised) x0 = clamp1(x0);
          mean = x0;
        } else if (a.mean_type == FIDM_MEAN_EPSILON) {
          x0 = __fsub_rn(__fmul_rn(c1, x), __fmul_rn(c2, mo[i]));
          if (a.clip_denoised) x0 = clamp1(x0);
          mean = __fadd_rn(__fmul_rn(k1, x0), __fmul_rn(k2, x));
        } else if (a.mean_type == FIDM_MEAN_START_X) {
          x0 = a.clip_denoised ? clamp1(mo[i]) : mo[i];
          mean = __fadd_rn(__fmul_rn(k1, x0), __fmul_rn(k2, x));
        } else {  // PREVIOUS_X (:274-278)
          x0 = __fsub_rn(__fmul_rn(cf[FIDM_C_XPREV_A], mo[i]), __fmul_rn(cf[FIDM_C_XPREV_B], x));
          if (a.clip_denoised) x0 = clamp1(x0);
          mean = mo[i];
        }
        x0v[i] = x0;
        mv[i] = mean;
        lv[i] = logvar;
        const float z = need_z ? zz[i] : 0.0f;
        if (a.sampler == FIDM_SAMPLER_DDIM_SCRIPT) {
          // :551-557  img = sqrt(ab_prev) * x0 + sqrt(1 - ab_prev - sigma^2) * eps_raw + sigma * noise
          const float mp = __fadd_rn(__fmul_rn(cf[FIDM_C_DDIM_SQRT_ABP], x0), __fmul_rn(cf[FIDM_C_DDIM_DIR], mo[i]));
          smp[i] = need_z ? __fadd_rn(mp, __fmul_rn(cf[FIDM_C_DDIM_SIGMA], z)) : mp;
        } else if (a.sampler == FIDM_SAMPLER_DDIM) {
          // eps re-derived from the (clamped) x0 (:470, :316-319), then :479-484
          const float e = __fdiv_rn(__fsub_rn(__fmul_rn(c1, x), x0), c2);
          const float mp = __fadd_rn(__fmul_rn(x0, cf[FIDM_C_DDIM_SQRT_ABP]), __fmul_rn(cf[FIDM_C_DDIM_DIR], e));
          smp[i] = need_z ? __fadd_rn(mp, __fmul_rn(__fmul_rn(nz, cf[FIDM_C_DDIM_SIGMA]), z)) : mp;
        } else {
          // :382-387  mean + nonzero * exp(0.5 * logvar) * z
          const float sd = expf(__fmul_rn(0.5f, logvar));
          smp[i] = __fadd_rn(mean, __fmul_rn(__fmul_rn(nz, sd), z));
        }
      }
      if constexpr (!SLOTS) {
        if (a.sample) store_vec<float, VEC>(a.sample + off, smp);
        if (a.pred_xstart) store_vec<float, VEC>(a.pred_xstart + off, x0v);
        if (a.mean_out) store_vec<float, VEC>(a.mean_out + off, mv);
        if (a.logvar_out) store_vec<float, VEC>(a.logvar_out + off, lv);
      }
    } else {
#pragma unroll
      for (int i = 0; i < VEC; ++i) smp[i] = xs[i];
    }
    if constexpr (REPAINT) {
      if (jump) {
        // K7's re-noising from t - 1 to t_up (sampler_resample.cu)
        const float ua = p.s.undo[2 * act], us = p.s.undo[2 * act + 1];
#pragma unroll
        for (int i = 0; i < VEC; ++i) smp[i] = __fadd_rn(__fmul_rn(ua, smp[i]), __fmul_rn(us, uu[i]));
      }
    }

    if (inj) {
      // apply_inpainting_injection (:139-155)
      const float* cf = a.coef + (long long)t_inj * FIDM_COEF_COLS;
      const float ca = a.cumulative ? cf[FIDM_C_SQRT_AB] : cf[FIDM_C_SQRT_AB_F32];
      const float cs = a.cumulative ? cf[FIDM_C_SQRT_1MAB] : cf[FIDM_C_SQRT_1MAB_F32];
#pragma unroll
      for (int i = 0; i < VEC; ++i) smp[i] = inject(smp[i], m[i], g[i], n[i], ca, cs);
    }
    if constexpr (SLOTS) {
      if (upd && t_upd == 0) {                     // the request's result: kept apart until the host collects it
        store_vec<float, VEC>(p.s.out + off, smp);
        continue;
      }
      store_vec<float, VEC>(a.x_next + off, smp);
      store_stem<VEC>(a, e, smp);
      if (a.t_out && c == 0 && e.pv == 0) a.t_out[b] = p.s.t_value[t_inj];
    } else {
      if (a.x_next) store_vec<float, VEC>(a.x_next + off, smp);
      write_stem<VEC>(a, idx, e, smp);
    }
  }
}

// The unseeded (s == nullptr) and seeded entries; `who` prefixes the error text.
static int sampler_step(const fidm_step_args* a, const fidm_seeded_noise* s, fidm_stream_t stream, const char* who) {
  FIDM_REQUIRE(a != nullptr, FIDM_E_BADARG, "%s: null args", who);
  FIDM_REQUIRE(a->batch > 0 && a->channels > 0 && a->hw > 0, FIDM_E_BADARG, "%s: empty shape", who);
  FIDM_REQUIRE(a->mode >= 0 && a->mode <= 2, FIDM_E_BADARG, "%s: bad mode %d", who, a->mode);
  FIDM_REQUIRE(a->coef && a->x, FIDM_E_BADARG, "%s: coef/x are required", who);
  if (int rc = check_mask_channels(a, who)) return rc;
  if (s) {
    if (int rc = check_seeded(s, a->mode != FIDM_STEP_UPDATE_ONLY, who)) return rc;
    FIDM_REQUIRE(a->z == nullptr && a->inject_noise == nullptr && a->t_dev == nullptr, FIDM_E_BADARG,
                 "%s: z/inject_noise/t_dev must be NULL", who);
    FIDM_REQUIRE(s->draw >= -1, FIDM_E_BADARG, "%s: step noise draw %d < -1", who, s->draw);
  }
  if (a->mode != FIDM_STEP_INJECT_ONLY) {
    FIDM_REQUIRE(a->model_out != nullptr, FIDM_E_BADARG, "%s: model_out required for an update", who);
    FIDM_REQUIRE(a->t_dev || (a->t_update >= 0 && a->t_update < a->num_timesteps), FIDM_E_BADARG,
                 "%s: t_update %d out of range [0,%d)", who, a->t_update, a->num_timesteps);
  }
  if (a->mode != FIDM_STEP_UPDATE_ONLY) {
    FIDM_REQUIRE(a->gt && a->keep_mask && (s || a->inject_noise), FIDM_E_BADARG,
                 "%s: gt/keep_mask/inject_noise required for an injection", who);
    FIDM_REQUIRE(a->t_dev || (a->t_inject >= 0 && a->t_inject < a->num_timesteps), FIDM_E_BADARG,
                 "%s: t_inject %d out of range [0,%d)", who, a->t_inject, a->num_timesteps);
  }
  if (int rc = check_stem(a, who)) return rc;
  const bool vec4 = vec4_ok(a->hw, a->x, a->model_out, a->z, a->gt, a->keep_mask, a->inject_noise, a->sample,
                            a->pred_xstart, a->x_next, a->mean_out, a->logvar_out);
  const long long elems = (long long)a->batch * a->channels * a->hw;
  if (s)
    return launch_sampler(sampler_step_kernel<4, true, false>, sampler_step_kernel<1, true, false>, vec4, elems,
                          StepParams<true>{*a, *s}, stream, who);
  return launch_sampler(sampler_step_kernel<4, false, false>, sampler_step_kernel<1, false, false>, vec4, elems,
                        StepParams<false>{*a}, stream, who);
}

static int sampler_step_slots(const fidm_step_args* a, const fidm_slot_args* s, fidm_stream_t stream) {
  const char* who = "sampler_step_slots";
  FIDM_REQUIRE(a != nullptr && s != nullptr, FIDM_E_BADARG, "%s: null args", who);
  FIDM_REQUIRE(a->batch >= 1 && a->batch <= FIDM_MAX_SLOTS, FIDM_E_BADARG, "%s: %d slots outside [1, %d]", who,
               a->batch, FIDM_MAX_SLOTS);
  FIDM_REQUIRE(a->channels > 0 && a->hw > 0 && a->num_timesteps > 0, FIDM_E_BADARG, "%s: empty shape", who);
  FIDM_REQUIRE(a->sampler == FIDM_SAMPLER_DDPM || a->sampler == FIDM_SAMPLER_DDIM, FIDM_E_BADARG,
               "%s: sampler must be DDPM | DDIM", who);
  FIDM_REQUIRE(a->coef && a->x && a->x_next && a->gt && a->keep_mask && s->out && s->t_value && s->inject_draw,
               FIDM_E_BADARG, "%s: coef/x/x_next/gt/keep_mask/out/t_value/inject_draw are required", who);
  FIDM_REQUIRE(a->z == nullptr && a->inject_noise == nullptr && a->t_dev == nullptr, FIDM_E_BADARG,
               "%s: z/inject_noise/t_dev must be NULL", who);
  FIDM_REQUIRE(!a->sample && !a->pred_xstart && !a->mean_out && !a->logvar_out, FIDM_E_BADARG,
               "%s: sample/pred_xstart/mean_out/logvar_out must be NULL", who);
  if (int rc = check_mask_channels(a, who)) return rc;
  bool any_update = false;
  for (int b = 0; b < a->batch; ++b) {
    const int act = s->action[b];
    FIDM_REQUIRE(act == FIDM_SLOT_IDLE || act == FIDM_SLOT_ADMIT || (act >= 0 && act < a->num_timesteps), FIDM_E_BADARG,
                 "%s: slot %d: action %d is not IDLE, ADMIT or a timestep in [0,%d)", who, b, act, a->num_timesteps);
    any_update |= act >= 0;
  }
  FIDM_REQUIRE(!any_update || a->model_out != nullptr, FIDM_E_BADARG, "%s: model_out required for an update", who);
  if (int rc = check_stem(a, who)) return rc;
  const bool vec4 = vec4_ok(a->hw, a->x, a->model_out, a->gt, a->keep_mask, a->x_next, s->out);
  const long long elems = (long long)a->batch * a->channels * a->hw;
  return launch_sampler(sampler_step_kernel<4, true, true>, sampler_step_kernel<1, true, true>, vec4, elems,
                        SlotParams{*a, *s}, stream, who);
}

static int repaint_step_slots(const fidm_step_args* a, const fidm_rp_slot_args* s, fidm_stream_t stream) {
  const char* who = "repaint_step_slots";
  FIDM_REQUIRE(a != nullptr && s != nullptr, FIDM_E_BADARG, "%s: null args", who);
  FIDM_REQUIRE(a->batch >= 1 && a->batch <= FIDM_MAX_SLOTS, FIDM_E_BADARG, "%s: %d slots outside [1, %d]", who,
               a->batch, FIDM_MAX_SLOTS);
  FIDM_REQUIRE(a->channels > 0 && a->hw > 0 && a->num_timesteps > 0 && s->n_evals > 0, FIDM_E_BADARG,
               "%s: empty shape", who);
  FIDM_REQUIRE(a->sampler == FIDM_SAMPLER_DDPM, FIDM_E_BADARG, "%s: sampler must be DDPM", who);
  FIDM_REQUIRE(a->coef && a->x && a->x_next && a->gt && a->keep_mask && s->out && s->t_value && s->eval_t &&
                   s->next_t && s->undo && s->inject_draw,
               FIDM_E_BADARG,
               "%s: coef/x/x_next/gt/keep_mask/out/t_value/eval_t/next_t/undo/inject_draw are required", who);
  FIDM_REQUIRE(a->z == nullptr && a->inject_noise == nullptr && a->t_dev == nullptr, FIDM_E_BADARG,
               "%s: z/inject_noise/t_dev must be NULL", who);
  FIDM_REQUIRE(!a->sample && !a->pred_xstart && !a->mean_out && !a->logvar_out, FIDM_E_BADARG,
               "%s: sample/pred_xstart/mean_out/logvar_out must be NULL", who);
  if (int rc = check_mask_channels(a, who)) return rc;
  bool any_update = false;
  for (int b = 0; b < a->batch; ++b) {
    const int act = s->action[b];
    FIDM_REQUIRE(act == FIDM_SLOT_IDLE || act == FIDM_SLOT_ADMIT || (act >= 0 && act < s->n_evals), FIDM_E_BADARG,
                 "%s: slot %d: action %d is not IDLE, ADMIT or an evaluation in [0,%d)", who, b, act, s->n_evals);
    any_update |= act >= 0;
  }
  FIDM_REQUIRE(!any_update || a->model_out != nullptr, FIDM_E_BADARG, "%s: model_out required for an update", who);
  if (int rc = check_stem(a, who)) return rc;
  const bool vec4 = vec4_ok(a->hw, a->x, a->model_out, a->gt, a->keep_mask, a->x_next, s->out);
  const long long elems = (long long)a->batch * a->channels * a->hw;
  return launch_sampler(sampler_step_kernel<4, true, true, true>, sampler_step_kernel<1, true, true, true>, vec4, elems,
                        RpSlotParams{*a, *s}, stream, who);
}

}  // namespace fidm

extern "C" int fidm_sampler_step_slots(const fidm_step_args* a, const fidm_slot_args* s, fidm_stream_t stream) {
  return fidm::sampler_step_slots(a, s, stream);
}

extern "C" int fidm_repaint_step_slots(const fidm_step_args* a, const fidm_rp_slot_args* s, fidm_stream_t stream) {
  return fidm::repaint_step_slots(a, s, stream);
}

extern "C" int fidm_sampler_step(const fidm_step_args* a, fidm_stream_t stream) {
  return fidm::sampler_step(a, nullptr, stream, "sampler_step");
}

extern "C" int fidm_sampler_step_seeded(const fidm_step_args* a, const fidm_seeded_noise* s, fidm_stream_t stream) {
  FIDM_REQUIRE(s != nullptr, FIDM_E_BADARG, "sampler_step_seeded: seeded noise is required");
  return fidm::sampler_step(a, s, stream, "sampler_step_seeded");
}
