/*
 * fidm_b200.h -- C ABI of the B200-native masked-inpainting sampler kernels (sm_100a).
 *
 * The reference (Sayzal28/Face-Inpainting-Diffusion-Models) is 100 % Python on PyTorch and has no
 * FFI of its own; every FLOP of its sampling path is an ATen library call.  Each entry point below
 * names the reference call site(s) it replaces (paths relative to /root/reference/code).  The
 * library is stateless and re-entrant: the caller owns every buffer (PyTorch allocates, the
 * library never allocates or frees device memory), passes raw device pointers plus an explicit
 * cudaStream_t, and every call is CUDA-graph capturable (no host synchronisation, no host reads
 * of device data).
 *
 * Return value of every int function: 0 = ok, < 0 = bad argument (FIDM_E_*), > 0 = cudaError_t.
 * fidm_last_error_string() describes the last failure on the calling thread.
 *
 * Layout vocabulary: "NHWC" = [N][H][W][C] with an explicit per-pixel stride `ld*` in ELEMENTS
 * (so a tensor may be a channel slice of a wider, zero-copy concat buffer).  "NCHW" = contiguous
 * fp32 as the reference's tensors.  dtype codes: FIDM_F32 / FIDM_BF16.
 */
#ifndef FIDM_B200_H_
#define FIDM_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FIDM_ABI_VERSION 3

#define FIDM_F32  0
#define FIDM_BF16 1
#define FIDM_F16  2   /* normalized conv operands (GroupNorm outputs) and their weights: 11-bit mantissa */
#define FIDM_E4M3 3   /* opt-in FP8 mode: e4m3 weights (per-output-channel scale) x e4m3 normalized operand, fp32 accumulate */

#define FIDM_E_BADARG   (-1)
#define FIDM_E_SHAPE    (-2)   /* shape not supported by this kernel (caller picks another entry) */
#define FIDM_E_ALIGN    (-3)
#define FIDM_E_DRIVER   (-4)   /* cuTensorMapEncode* unavailable / failed */

typedef void* fidm_stream_t;   /* cudaStream_t */

int         fidm_abi_version(void);
const char* fidm_last_error_string(void);
/* 0 if device `dev` is sm_100 (B200); FIDM_E_BADARG otherwise.  No CPU fallback exists. */
int         fidm_device_supported(int dev);

/* ------------------------------------------------------------------------------------------------
 * K4  fused reverse-process step: [update at t] -> [known-region injection at t_inject] .
 * Replaces, per step, the ~40 ATen elementwise kernels, 14 H2D table copies and the .item() sync of
 *   gaussian_diffusion.py:114-157 (apply_inpainting_injection, get_gt_noised, q_sample :172-189),
 *   :213-298 (p_mean_variance arithmetic after the model call), :300-319, :357-388 (p_sample),
 *   :447-485 (ddim_sample).
 * All tensors fp32 NCHW contiguous.  Arithmetic is evaluated with one IEEE rounding per reference
 * ATen op (no FMA contraction), so the DDIM path and the injected known-region pixels are
 * bit-identical to the reference given the same model output and noise.
 * ---------------------------------------------------------------------------------------------- */
#define FIDM_COEF_COLS 20
/* columns of the per-timestep coefficient table (fp32, [T][FIDM_COEF_COLS], built on the host in
 * the reference's own arithmetic: float64 table entry rounded to fp32, gaussian_diffusion.py:12-24) */
enum {
  FIDM_C_SQRT_AB = 0,        /* sqrt_alphas_cumprod[t]                      (:187) */
  FIDM_C_SQRT_1MAB = 1,      /* sqrt_one_minus_alphas_cumprod[t]            (:188) */
  FIDM_C_SQRT_AB_F32 = 2,    /* sqrt_f32(f32(ab[t]))    non-cumulative path (:143-144) */
  FIDM_C_SQRT_1MAB_F32 = 3,  /* sqrt_f32(1 - f32(ab[t]))                    (:145) */
  FIDM_C_RECIP = 4,          /* sqrt_recip_alphas_cumprod[t]                (:303) */
  FIDM_C_RECIPM1 = 5,        /* sqrt_recipm1_alphas_cumprod[t]              (:304) */
  FIDM_C_MAX_LOG = 6,        /* log(betas[t])                               (:247) */
  FIDM_C_MIN_LOG = 7,        /* posterior_log_variance_clipped[t]           (:246) */
  FIDM_C_POST1 = 8,          /* posterior_mean_coef1[t]                     (:199) */
  FIDM_C_POST2 = 9,          /* posterior_mean_coef2[t]                     (:200) */
  FIDM_C_FIXED_LOGVAR = 10,  /* FIXED_LARGE / FIXED_SMALL log-variance      (:254-265) */
  FIDM_C_DDIM_SQRT_ABP = 11, /* sqrt_f32(f32(ab_prev[t]))                   (:480) */
  FIDM_C_DDIM_DIR = 12,      /* sqrt_f32(1 - abp - sigma^2)                 (:481) */
  FIDM_C_DDIM_SIGMA = 13,    /* eta-dependent sigma                         (:474-477) */
  FIDM_C_NONZERO = 14,       /* (t != 0)                                    (:382,:483) */
  FIDM_C_XPREV_A = 15,       /* 1/posterior_mean_coef1[t]                   (:310) */
  FIDM_C_XPREV_B = 16        /* posterior_mean_coef2/posterior_mean_coef1   (:311-313) */
};
enum { FIDM_STEP_INJECT_ONLY = 0, FIDM_STEP_UPDATE_ONLY = 1, FIDM_STEP_UPDATE_INJECT = 2 };
enum { FIDM_SAMPLER_DDPM = 0, FIDM_SAMPLER_DDIM = 1,
       /* the evaluation scripts' strided DDIM update (test_inp_ddim_100.py:539-557): x0 = (x - c5*eps)/c4,
          x <- (c11*x0 + c12*eps) + c13*z with the RAW eps; coefficient rows are indexed by step, not t:
          c4 = sqrt(ab_t), c5 = sqrt(1-ab_t), c0/c1 = injection coefficients at ab_prev (:560-574) */
       FIDM_SAMPLER_DDIM_SCRIPT = 2 };
enum { FIDM_MEAN_PREVIOUS_X = 0, FIDM_MEAN_START_X = 1, FIDM_MEAN_EPSILON = 2 };
enum { FIDM_VAR_LEARNED = 0, FIDM_VAR_FIXED = 1, FIDM_VAR_LEARNED_RANGE = 2 };

typedef struct fidm_step_args {
  int32_t batch, channels, hw;          /* x is [batch][channels][hw] */
  int32_t mode, sampler, mean_type, var_type;
  int32_t clip_denoised;                /* clamp pred_xstart to [-1,1]            (:267-271) */
  int32_t cumulative;                   /* use_cumulative_noise                   (:138-148) */
  int32_t mask_channels;                /* 1 (broadcast, :151-152) or `channels` */
  int32_t num_timesteps;                /* rows of coef */
  int32_t t_update, t_inject;           /* used when t_dev == NULL (whole batch at one timestep) */
  const int64_t* t_dev;                 /* optional [batch] per-sample update timestep; injection then
                                           uses t_dev[b] (INJECT_ONLY) or t_dev[b]-1 (UPDATE_INJECT) */
  const float* coef;                    /* device [num_timesteps][FIDM_COEF_COLS] */
  const float* x;                       /* state fed to the model (UPDATE*) / state to inject into */
  const float* model_out;               /* [batch][channels or 2*channels][hw] */
  const float* z;                       /* step noise; may be NULL when the sigma column is all 0 */
  const float* gt;                      /* [batch][channels][hw] */
  const float* keep_mask;               /* 1 = keep, [batch][mask_channels][hw] */
  const float* inject_noise;            /* n_{t_inject} */
  float* sample;                        /* optional: x_{t-1} before injection ("sample", :485) */
  float* pred_xstart;                   /* optional                                             */
  float* x_next;                        /* optional: state after injection (input of next eval) */
  float* mean_out;                      /* optional: posterior mean      ("mean", :286)          */
  float* logvar_out;                    /* optional: model log-variance  ("log_variance", :251)  */
  /* Step-boundary fusion (the UNet's stem input and timestep are written by THIS kernel, so that no pack / copy
   * launch sits between two evaluations): the state after this call (x_next's value) is also stored as channels
   * [0, channels) of every pixel of the NHWC network input `stem_out` (pixel stride stem_ld elements, dtype
   * stem_dtype = FIDM_F32 | FIDM_BF16 | FIDM_F16; the conditioning channels behind it -- masked image, mask x3:
   * unet.py:199 -- are constant over the loop and are packed once by the caller), and `t_out[0 .. batch)` is set to
   * t_out_value (the timestep the NEXT evaluation sees, already rescaled if rescale_timesteps, :321-324). */
  void* stem_out; int32_t stem_dtype, stem_ld;
  float* t_out; float t_out_value;
} fidm_step_args;
int fidm_sampler_step(const fidm_step_args* a, fidm_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K6  DPM-Solver++ multistep step (Lu et al. 2022, "DPM-Solver++", multistep 2M, data prediction):
 *   m_k    = x0 prediction at t_k:  clamp(c1*x - c2*eps) (EPSILON) | clamp(model_out) (START_X)
 *   x_next = A*x + B0*m_k [+ B1*m_{k-1}]                                    (update t_k -> t_{k+1})
 *   x_next = keep*(ia*gt + is*n) + (1-keep)*x_next                          (optional injection at t_{k+1})
 * The per-step rows are computed on the host in float64 and rounded to fp32 once (dpm_solver.py).  Every product and
 * sum is one IEEE fp32 rounding, in the order written above; the injection and the stem write are K4's expressions.
 * All tensors fp32 NCHW contiguous.
 * ---------------------------------------------------------------------------------------------- */
#define FIDM_MS_COLS 7
/* columns of the per-step table [steps][FIDM_MS_COLS]; row k belongs to the evaluation at t_k */
enum {
  FIDM_MS_X0_C1 = 0,   /* sqrt_recip_alphas_cumprod[t_k]   (as FIDM_C_RECIP) */
  FIDM_MS_X0_C2 = 1,   /* sqrt_recipm1_alphas_cumprod[t_k] (as FIDM_C_RECIPM1) */
  FIDM_MS_A = 2,       /* sigma_{t_{k+1}} / sigma_{t_k} */
  FIDM_MS_B0 = 3,      /* weight of m_k */
  FIDM_MS_B1 = 4,      /* weight of m_{k-1} (second-order rows) */
  FIDM_MS_INJ_A = 5,   /* injection coefficient of gt at t_{k+1} (cumulative: FIDM_C_SQRT_AB, else FIDM_C_SQRT_AB_F32) */
  FIDM_MS_INJ_S = 6    /* injection coefficient of the noise at t_{k+1} */
};
typedef struct fidm_multistep_args {
  int32_t batch, channels, hw;          /* x is [batch][channels][hw] */
  int32_t mean_type;                    /* FIDM_MEAN_EPSILON | FIDM_MEAN_START_X */
  int32_t out_channels;                 /* channels of model_out: channels or 2*channels (learned variance, ignored) */
  int32_t clip_denoised;                /* clamp m_k to [-1,1] */
  int32_t mask_channels;                /* 1 (broadcast) or `channels` */
  int32_t steps, step;                  /* rows of coef, and the row of this call (0 <= step < steps) */
  const float* coef;                    /* device [steps][FIDM_MS_COLS] */
  const float* x;                       /* state at t_k, the model's input */
  const float* model_out;               /* [batch][out_channels][hw] */
  const float* m_prev;                  /* m_{k-1}; NULL selects the first-order update (B1 is not used) */
  float* m_out;                         /* m_k (the next step's history; pred_xstart) */
  float* x_next;                        /* state at t_{k+1}; NULL: no update (the last evaluation, at t = 0) */
  int32_t inject;                       /* 1: injection at t_{k+1} (needs gt, keep_mask, inject_noise, x_next) */
  const float* gt;                      /* [batch][channels][hw] */
  const float* keep_mask;               /* 1 = keep, [batch][mask_channels][hw] */
  const float* inject_noise;            /* n_{t_{k+1}} */
  /* step-boundary fusion, as fidm_step_args: x_next is also stored as channels [0, channels) of the NHWC network
   * input `stem_out` (needs x_next), and t_out[0 .. batch) = t_out_value */
  void* stem_out; int32_t stem_dtype, stem_ld;
  float* t_out; float t_out_value;
} fidm_multistep_args;
int fidm_multistep_step(const fidm_multistep_args* a, fidm_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K7  RePaint undo-and-inject (Lugmayr et al. 2022, "RePaint", Algorithm 1): after the DDPM update of the evaluation
 * at t (K4, STEP_UPDATE_ONLY) the state x at level t-1 is re-noised to level t_up in one draw and the known region is
 * injected for the next evaluation, at t_up:
 *   x'  = undo_a*x + undo_s*u                                undo_a = sqrt(ab[t_up]/ab[t-1]), undo_s = sqrt(1 - ab[t_up]/ab[t-1])
 *   x'' = keep*(inject_a*gt + inject_s*n) + (1-keep)*x'      (optional: injection at t_up, K4's expression)
 * The coefficients are fp32 values the host computes (repaint.py: float64 rounded once; the injection pair is the
 * class table's FIDM_C_SQRT_AB/FIDM_C_SQRT_1MAB columns for cumulative noise, the _F32 columns otherwise).  Every
 * product and sum is one IEEE fp32 rounding, in the order written above.  All tensors fp32 NCHW contiguous.
 * ---------------------------------------------------------------------------------------------- */
typedef struct fidm_resample_args {
  int32_t batch, channels, hw;          /* x is [batch][channels][hw] */
  int32_t mask_channels;                /* 1 (broadcast) or `channels` */
  float undo_a, undo_s;
  const float* x;                       /* state at level t-1 (K4's "sample") */
  const float* noise;                   /* u, the undo noise */
  float* x_next;                        /* state the evaluation at t_up sees */
  int32_t inject;                       /* 1: injection at t_up (needs gt, keep_mask, inject_noise) */
  float inject_a, inject_s;
  const float* gt;                      /* [batch][channels][hw] */
  const float* keep_mask;               /* 1 = keep, [batch][mask_channels][hw] */
  const float* inject_noise;            /* n_{t_up} */
  /* step-boundary fusion, as fidm_step_args: x_next is also stored as channels [0, channels) of the NHWC network
   * input `stem_out`, and t_out[0 .. batch) = t_out_value */
  void* stem_out; int32_t stem_dtype, stem_ld;
  float* t_out; float t_out_value;
} fidm_resample_args;
int fidm_resample_undo(const fidm_resample_args* a, fidm_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Per-image seeded noise.  Every Gaussian value is a function of (the image's uint64 seed, the element's flat NCHW
 * index j within its image, a tag, a draw) only -- Philox4x32-10 keyed by the seed with counter (j >> 2, draw, tag, 0)
 * and Box-Muller, specified in csrc/philox.cuh -- so an image's noise does not depend on its batch, its position in it
 * or the number of GPUs.  The _seeded entries below are the K4 / K6 / K7 entries with their noise tensors generated in
 * registers instead of read: each takes the same arg struct, requires its noise pointers (z, inject_noise, noise) to
 * be NULL, and reads the draws from `s`.  fidm_randn_seeded fills a buffer with the same values.
 * Draws of the sampling loops: x_T (XT, 0); step noise of the k-th evaluation (STEP, k); cumulative injection noise at
 * timestep t (INJECT, t); the i-th fresh injection of a loop (INJECT_FRESH, i); RePaint undo noise after evaluation k
 * (UNDO, k).  K8, K9 and K10 (below) take the same draws per slot; K10 takes (STEP, k) and (UNDO, k) with k the
 * slot's own evaluation index.
 * ---------------------------------------------------------------------------------------------- */
enum { FIDM_NOISE_XT = 0, FIDM_NOISE_STEP = 1, FIDM_NOISE_INJECT = 2, FIDM_NOISE_INJECT_FRESH = 3, FIDM_NOISE_UNDO = 4 };
typedef struct fidm_seeded_noise {
  const uint64_t* seeds;                /* device [batch]: seed of each image */
  int32_t draw;                         /* K4: draw of the step noise (tag STEP; -1: none, as z == NULL);
                                           K7: draw of the undo noise (tag UNDO); K6: unused */
  int32_t inject_tag, inject_draw;      /* the injection noise: FIDM_NOISE_INJECT | FIDM_NOISE_INJECT_FRESH, draw */
} fidm_seeded_noise;
/* K4 with a->z and a->inject_noise NULL; a->t_dev must be NULL (one timestep for the whole batch) */
int fidm_sampler_step_seeded(const fidm_step_args* a, const fidm_seeded_noise* s, fidm_stream_t stream);
/* K6 with a->inject_noise NULL */
int fidm_multistep_step_seeded(const fidm_multistep_args* a, const fidm_seeded_noise* s, fidm_stream_t stream);
/* K7 with a->noise and a->inject_noise NULL */
int fidm_resample_undo_seeded(const fidm_resample_args* a, const fidm_seeded_noise* s, fidm_stream_t stream);
/* out[b][j] = the normal of element j of image b under seeds[b], draw (tag, draw); out is [batch][elems_per_image] */
int fidm_randn_seeded(float* out, const uint64_t* seeds, int32_t batch, int64_t elems_per_image, int32_t tag,
                      int32_t draw, fidm_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K8  per-slot sampler step (continuous batching).  The state [batch][channels][hw] is a fixed set of `batch` SLOTS,
 * each holding its own seeded request at its own timestep; one launch takes, per slot, the action in s->action:
 *   FIDM_SLOT_IDLE   nothing is read or written for the slot (state, stem, t_out, out);
 *   FIDM_SLOT_ADMIT  x_T = draw (XT, 0) under the slot's seed, then the injection at T-1 (unless inject_draw[T-1] < 0),
 *                    written as the state, the stem channels and t_out[b] = t_value[T-1] -- a seeded loop's prologue;
 *   t >= 0           K4's seeded STEP_UPDATE_INJECT / STEP_UPDATE_ONLY at t for the slot: step noise (STEP, T-1-t) when
 *                    s->step_noise, injection at t-1 with draw (INJECT | INJECT_FRESH as a->cumulative,
 *                    inject_draw[t-1]) unless that is < 0; state, stem and t_out[b] = t_value[t-1] are written, and at
 *                    t = 0 the sample goes to out[b] instead (state, stem and t_out are left alone).
 * Every value is bit-identical to what fidm_sampler_step_seeded computes for that image alone (T = a->num_timesteps).
 * Fields of `a` used: the shape (batch = number of slots, at most FIDM_MAX_SLOTS), sampler (DDPM | DDIM), mean_type,
 * var_type, clip_denoised, cumulative, mask_channels, num_timesteps, coef, x, model_out (read for updates), gt,
 * keep_mask, x_next (may equal x: each element is read and written by the same thread), stem_out / stem_dtype /
 * stem_ld and t_out; mode, t_update, t_inject and t_out_value are ignored, and z, inject_noise, t_dev, sample,
 * pred_xstart, mean_out and logvar_out must be NULL.  The per-slot control travels by value in the launch parameters:
 * the host owns the schedule, and no launch reads control state that it or another launch writes.
 * ---------------------------------------------------------------------------------------------- */
#define FIDM_MAX_SLOTS 128
enum { FIDM_SLOT_IDLE = -1, FIDM_SLOT_ADMIT = -2 };
typedef struct fidm_slot_args {
  const float* t_value;                 /* device [num_timesteps]: what the model sees for t (_scale_timesteps) */
  const int32_t* inject_draw;           /* device [num_timesteps]: draw of the injection at t; -1: no injection at t */
  float* out;                           /* [batch][channels][hw]: the sample of a slot updated at t = 0 */
  int32_t step_noise;                   /* 1: updates draw step noise (DDPM, DDIM with eta > 0) */
  int32_t action[FIDM_MAX_SLOTS];       /* per slot: FIDM_SLOT_IDLE | FIDM_SLOT_ADMIT | t (update at t) */
  uint64_t seeds[FIDM_MAX_SLOTS];       /* per slot: the request's seed */
} fidm_slot_args;
int fidm_sampler_step_slots(const fidm_step_args* a, const fidm_slot_args* s, fidm_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K9  per-slot DPM-Solver++ multistep step (continuous batching of dpm_solver_sample_loop): K6 as K8 is K4.  Each slot
 * runs its own seeded request on the grid t_0 = T-1 > ... > t_{steps-1} = 0 of `a->coef` (K6's table); one launch takes,
 * per slot, the action in s->action:
 *   FIDM_SLOT_IDLE   nothing is read or written for the slot (state, history, stem, t_out, out);
 *   FIDM_SLOT_ADMIT  x_T = draw (XT, 0) under the slot's seed, then the injection at t_0 (K4's expression with
 *                    s->admit_inject_a / s->admit_inject_s) unless inject_draw[0] < 0, written as the state, the stem
 *                    channels and t_out[b] = t_value[0] -- the seeded loop's prologue;
 *   k in [0, steps)  K6's row k for the slot: m_k from x and model_out; at k = steps-1 m_k goes to out[b] and nothing
 *                    else is written; otherwise m_k goes to m_out, x' = A*x + B0*m_k [+ B1*m_{k-1}, read from m_prev
 *                    only where order[k] == 2], the injection at t_{k+1} with draw (inject_tag, inject_draw[k+1])
 *                    unless that is < 0, and the state, stem and t_out[b] = t_value[k+1] are written.
 * Every value is bit-identical to what fidm_multistep_step_seeded computes for that image alone (and, for an admission,
 * fidm_randn_seeded followed by fidm_sampler_step_seeded's STEP_INJECT_ONLY at T-1).
 * Fields of `a` used: the shape (batch = number of slots, at most FIDM_MAX_SLOTS), mean_type, out_channels,
 * clip_denoised, mask_channels, steps, coef, x, model_out (read for updates), m_prev, m_out, x_next, gt, keep_mask,
 * stem_out / stem_dtype / stem_ld and t_out; step, inject and t_out_value are ignored and inject_noise must be NULL.
 * x_next may equal x and m_out may equal m_prev (each element is read and written by the same thread).  As for K8 the
 * per-slot control travels by value in the launch parameters.
 * ---------------------------------------------------------------------------------------------- */
typedef struct fidm_ms_slot_args {
  const float* t_value;                 /* device [steps]: what the model sees at grid point k (_scale_timesteps of t_k) */
  const int32_t* inject_draw;           /* device [steps]: draw of the injection at t_k; -1: no injection at t_k */
  const int32_t* order;                 /* device [steps]: 2 where the update out of t_k uses m_{k-1}, else 1 */
  float* out;                           /* [batch][channels][hw]: m_k of a slot at its last grid point */
  int32_t inject_tag;                   /* FIDM_NOISE_INJECT | FIDM_NOISE_INJECT_FRESH */
  float admit_inject_a, admit_inject_s; /* injection coefficients at t_0 = T-1: the K4 table's (FIDM_C_SQRT_AB,
                                           FIDM_C_SQRT_1MAB) for cumulative noise, the _F32 columns otherwise */
  int32_t action[FIDM_MAX_SLOTS];       /* per slot: FIDM_SLOT_IDLE | FIDM_SLOT_ADMIT | k (the grid point evaluated) */
  uint64_t seeds[FIDM_MAX_SLOTS];       /* per slot: the request's seed */
} fidm_ms_slot_args;
int fidm_multistep_step_slots(const fidm_multistep_args* a, const fidm_ms_slot_args* s, fidm_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K10  per-slot RePaint step (continuous batching of repaint_sample_loop): K8 on RePaint's walk.  Every request takes
 * the same n_evals model evaluations (repaint.evaluation_plan); evaluation k is at timestep eval_t[k] and the walk goes
 * on at next_t[k], which is t_up where a jump follows and eval_t[k] - 1 otherwise.  One launch takes, per slot, the
 * action in s->action:
 *   FIDM_SLOT_IDLE   nothing is read or written for the slot (state, stem, t_out, out);
 *   FIDM_SLOT_ADMIT  K8's admission: x_T = draw (XT, 0) under the slot's seed, then the injection at T-1 with draw
 *                    s->admit_draw unless it is < 0, written as the state, the stem channels and t_out[b] = t_value[T-1];
 *   k in [0, n_evals) K4's seeded DDPM update at eval_t[k] with step noise (STEP, k); where a jump follows (next_t[k]
 *                    != eval_t[k] - 1) K7's re-noising x' = undo[k][0]*x + undo[k][1]*u with u = (UNDO, k); then the
 *                    injection at next_t[k] with draw (INJECT | INJECT_FRESH as a->cumulative, inject_draw[k]) unless
 *                    that is < 0 (K4's expression and coefficients); state, stem and t_out[b] = t_value[next_t[k]] are
 *                    written.  At k = n_evals-1 (eval_t = 0, next_t = -1) the sample goes to out[b] instead.
 * Every value is bit-identical to what the seeded lockstep launches compute for that image alone: for a jump
 * evaluation fidm_sampler_step_seeded's STEP_UPDATE_ONLY followed by fidm_resample_undo_seeded, otherwise its
 * STEP_UPDATE_INJECT / STEP_UPDATE_ONLY.  Fields of `a` used: as K8, with sampler DDPM only; as for K8 the per-slot
 * control travels by value in the launch parameters, and x_next may equal x.
 * ---------------------------------------------------------------------------------------------- */
typedef struct fidm_rp_slot_args {
  const float* t_value;                 /* device [num_timesteps]: what the model sees for t (_scale_timesteps) */
  const int32_t* eval_t;                /* device [n_evals]: the timestep evaluation k updates */
  const int32_t* next_t;                /* device [n_evals]: the level of the injection and of evaluation k+1; -1 last.
                                           The kernel takes next_t[k] != eval_t[k] - 1 to mean that a jump follows
                                           (RePaint's t_up is always >= eval_t[k]), so a table without a jump at k
                                           must hold eval_t[k] - 1 there */
  const float* undo;                    /* device [n_evals][2]: (a_u, s_u) in fp32; 0 where no jump follows */
  const int32_t* inject_draw;           /* device [n_evals]: draw of the injection at next_t[k]; -1: none */
  float* out;                           /* [batch][channels][hw]: the sample of a slot at its last evaluation */
  int32_t n_evals;                      /* evaluations per request */
  int32_t admit_draw;                   /* draw of the admission's injection at T-1; -1: none */
  int32_t action[FIDM_MAX_SLOTS];       /* per slot: FIDM_SLOT_IDLE | FIDM_SLOT_ADMIT | k (the evaluation) */
  uint64_t seeds[FIDM_MAX_SLOTS];       /* per slot: the request's seed */
} fidm_rp_slot_args;
int fidm_repaint_step_slots(const fidm_step_args* a, const fidm_rp_slot_args* s, fidm_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Layout converters.  Replace torch.cat([x, masked_image, mask.repeat(1,3,1,1)], 1) of
 * unet.py:199 and the NCHW activations of the reference with one NHWC (bf16|fp32) tensor padded to
 * `c_pad` channels (zeros).  Up to 3 fp32 NCHW sources; a source with repeat>1 is broadcast.
 * ---------------------------------------------------------------------------------------------- */
typedef struct fidm_pack_args {
  int32_t batch, hw, n_src;
  const float* src[4];
  int32_t src_channels[4];              /* channels physically present in src[i] */
  int32_t src_repeat[4];                /* output copies of src[i] (mask: 1 channel x 3) */
  void* dst; int32_t dst_dtype, ld_dst, c_pad;
} fidm_pack_args;
int fidm_pack_nchw_to_nhwc(const fidm_pack_args* a, fidm_stream_t stream);
/* NHWC (bf16|fp32, stride ld) -> NCHW fp32, first `channels` channels. */
int fidm_unpack_nhwc_to_nchw(const void* src, int32_t src_dtype, int32_t ld_src, float* dst,
                             int32_t batch, int32_t hw, int32_t channels, fidm_stream_t stream);

/* I/O adapters (the reference does these on the CPU in its DataLoader / save path):
 *   fidm_prepare_inputs_u8 : data/dataset.py:38-42,130-142 -- image = (u8/255 - 0.5)/0.5, mask = (gray/255 < 0.5)
 *                            (1 = inpaint), masked_image = image*(1-mask), keep = 1-mask; uint8 NHWC -> fp32 NCHW.
 *   fidm_blend_to_u8       : test_inp_ddim_100.py:693-696 + toU8 :33-41 -- ((s*m + gt*(1-m) + 1)*127.5).clamp(0,255)
 *                            -> uint8 NHWC (gt = mask = NULL: no blend). */
int fidm_prepare_inputs_u8(const uint8_t* image_u8_nhwc, const uint8_t* mask_u8, float* image, float* masked_image,
                           float* mask, float* keep_mask, int32_t batch, int32_t hw, fidm_stream_t stream);
int fidm_blend_to_u8(const float* sample, const float* gt, const float* mask, uint8_t* out_u8_nhwc, int32_t batch,
                     int32_t hw, fidm_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K5  timestep path.  timestep_embedding (nn.py:51-61; `freqs` is the host-computed table exactly
 * as the reference computes it on the CPU) and small-batch Linear with optional SiLU on the input
 * (time_embed unet.py:44-48,158 and every ResBlock emb_layers nn.py:167-170,199, concatenated
 * into one weight matrix by the caller).   y[b][o] = bias[o] + sum_k W[o][k] * act(x[b][k]).
 * ---------------------------------------------------------------------------------------------- */
int fidm_timestep_embedding(const float* t, const float* freqs, float* out, int32_t batch,
                            int32_t dim, fidm_stream_t stream);
int fidm_linear_small(const float* x, const void* w, int32_t w_dtype, const float* bias, float* y,
                      int32_t batch, int32_t in_features, int32_t out_features, int32_t silu_input,
                      fidm_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K2  GroupNorm(32) [+ (1+scale),shift] [+ SiLU] [+ 2x avg-pool | 2x nearest-up], NHWC.
 * Replaces nn.GroupNorm(32,C) + nn.SiLU (nn.py:46-48,151-152,173-174; unet.py:149-150; attention
 * norm nn.py:251), the scale/shift modulation nn.py:203-206 and the resampling of up/down
 * ResBlocks nn.py:190-195 (h_upd on the activated tensor and x_upd on the raw tensor).
 * `stats` is a caller-provided workspace of fidm_groupnorm_workspace_bytes(batch, groups) bytes
 * (per-block partial sums, reduced in a fixed order: results are bit-reproducible).  The workspace must
 * be zero-initialised once by the caller; the kernel leaves its completion counters at zero.
 * ---------------------------------------------------------------------------------------------- */
#define FIDM_GN_MAX_BLOCKS 2048
enum { FIDM_RESAMPLE_NONE = 0, FIDM_RESAMPLE_DOWN = 1, FIDM_RESAMPLE_UP = 2 };
typedef struct fidm_gn_args {
  int32_t dtype;                        /* FIDM_BF16 | FIDM_F32: x and y_raw */
  int32_t y_dtype;                      /* dtype of y: = dtype, or FIDM_F16 when dtype is FIDM_BF16 */
  int32_t batch, height, width, channels, groups;
  float eps;
  const void* x; int32_t ld_x;
  const float* gamma; const float* beta;        /* [channels] */
  const float* scale_shift; int32_t ld_ss;      /* optional [batch][ld_ss]: scale at [0,C), shift at [C,2C) */
  int32_t silu;
  int32_t resample;                     /* applied AFTER norm/SiLU (nn.py:192-193) */
  int32_t skip_norm;                    /* 1: plain resample of x (Upsample / Downsample without conv,
                                           nn.py:109,129): no statistics, no affine */
  void* y; int32_t ld_y;                /* activated output (resampled resolution) */
  void* y_raw; int32_t ld_raw;          /* optional: resample(x) without norm (x_upd, nn.py:194) */
  double* stats;                        /* workspace (unused when skip_norm) */
  const float* chansum; int32_t ld_chansum;  /* optional [batch][ld_chansum][2] per-channel (sum, sum of squares)
                                           of x (from fidm_groupnorm_reduce_colsum): replaces the statistics pass */
} fidm_gn_args;
int fidm_groupnorm_silu_nhwc(const fidm_gn_args* a, fidm_stream_t stream);
/* kernels fidm_groupnorm_silu_nhwc launches for these arguments: 1 (statistics from the producer, plain resample, or a
 * small L2-resident tensor handled by the one-pass kernel) or 2 (statistics + apply) */
int fidm_groupnorm_num_launches(const fidm_gn_args* a);
int64_t fidm_groupnorm_workspace_bytes(int32_t batch, int32_t groups);
/* Statistics only (same arguments; y / resample / silu ignored): writes the per-(image, channel) affine coefficients of
 * GroupNorm [* (1+scale) + shift] followed by SiLU, HALVED:  coef[n][c] = (A/2, B/2)  with  A = rstd*gamma*(1+scale),
 * B = (beta - mean*rstd*gamma)*(1+scale) + shift,  so that silu(x*A + B) = h + h*tanh(h), h = x*coef.x + coef.y.
 * Consumed by fidm_conv2d_nhwc_bf16(gn_coef = coef): the normalisation pass itself never runs. */
int fidm_groupnorm_silu_coeff(const fidm_gn_args* a, float* coef, int32_t ld_coef, fidm_stream_t stream);
/* chansum[n][c0 + c] = sum over the `slots` partial rows of image n of colsum[n][slot][c]  (fixed order) */
int fidm_groupnorm_reduce_colsum(const float* colsum, int32_t batch, int32_t slots, int32_t channels,
                                 float* chansum, int32_t ld_chansum, int32_t c0, fidm_stream_t stream);
/* The same fold, and -- when the reduced tensor IS the input of the next GroupNorm (`a`: batch/height/width/channels/
 * groups/eps/gamma/beta/scale_shift of that norm; channels % 32 == 0, channels/groups divides 32) -- the coefficients
 * fidm_groupnorm_silu_coeff would compute from chansum, bit-identical, in the same launch. */
int fidm_groupnorm_reduce_colsum_coeff(const float* colsum, int32_t slots, float* chansum, int32_t ld_chansum, int32_t c0,
                                       const fidm_gn_args* a, float* coef, int32_t ld_coef, fidm_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K1  convolution as implicit GEMM, NHWC activations, KRSC weights ([Cout][kh][kw][Cin]).
 * Replaces every conv_nd(...) call: 3x3 pad 1 (nn.py:102,126,153,176,182; unet.py:55,151),
 * 1x1 skip (nn.py:184) and the Conv1d qkv / proj_out of attention (nn.py:252,254).
 * Epilogue (fused): + bias[c]  (+ row_add[n][c], the additive timestep embedding nn.py:208)
 *                   (+ residual[n,h,w,c], nn.py:212 / :265)  -> bf16|fp32 NHWC, or fp32 NCHW (head).
 * A second (activation, weight) pair may be accumulated into the same output tile: it carries the
 * 1x1 skip_connection of a channel-changing ResBlock (nn.py:184,212) as extra K-slices.
 *
 *   fidm_conv2d_nhwc_bf16  : tcgen05.mma (bf16 x bf16 -> fp32 in TMEM), TMA-staged tiles.
 *                            Requires stride 1, Cin % 64 == 0, Cout % 16 == 0.
 *   fidm_conv2d_nhwc_simt  : FFMA path (fp32 "verification mode", and shapes the tensor-core
 *                            kernel does not take: stride 2, small/odd channel counts).
 * ---------------------------------------------------------------------------------------------- */
typedef struct fidm_conv_args {
  int32_t dtype;                        /* of x and w: FIDM_BF16 | FIDM_F16 (tensor-core entry), FIDM_BF16 |
                                           FIDM_F32 (simt entry).  x2 / w2 / residual / y are bf16 whenever
                                           dtype is a 16-bit type, fp32 otherwise. */
  int32_t batch, height, width;         /* INPUT spatial size */
  int32_t cin, cout, ksize, stride;     /* ksize 1 or 3 (pad = ksize/2); stride 1 or 2 */
  const void* x; int32_t ld_x;
  const void* w;                        /* [cout][ksize][ksize][cin] */
  const void* x2; int32_t ld_x2; int32_t cin2;   /* optional fused 1x1 second source (same H,W as output) */
  const void* w2;                       /* [cout][cin2] */
  const float* bias;                    /* [cout] (already includes the skip bias if x2 is used) */
  const float* row_add; int32_t ld_row_add;     /* optional [batch][ld_row_add], first cout used */
  const void* residual; int32_t ld_res; /* optional NHWC at OUTPUT resolution */
  void* y; int32_t ld_y;
  int32_t y_nchw_f32;                   /* 1: y is fp32 [batch][cout_valid][Ho][Wo] */
  int32_t cout_valid;                   /* channels actually stored (<= cout; head: 6 of 16) */
  float* colsum;                        /* optional (tensor-core entry, NHWC output, images of >= 64 pixels):
                                           per-channel partial (sum, sum of squares) of the stored bf16 output,
                                           [batch][fidm_conv_colsum_slots()][cout][2] fp32 -- the GroupNorm
                                           statistics pass of the consumer, fused into this epilogue */
  void* splitk_ws; int64_t splitk_ws_bytes;  /* optional zero-initialised workspace: lets the tensor-core entry split
                                           the K loop of low-resolution layers over several CTAs (fixed-order fold,
                                           counters are left at zero).  32 MB covers every layer of the UNets here. */
  const float* gn_coef; int32_t ld_gn_coef;  /* optional (tensor-core entry, fidm_conv_gn_fusable() shapes): x is the RAW
                                           bf16 stream and the operand is silu(x*A + B) with per-(image, channel)
                                           coefficients [batch][ld_gn_coef][2] from fidm_groupnorm_silu_coeff -- the
                                           GroupNorm(+scale/shift)+SiLU in front of this conv (nn.py:151-153,173-176,
                                           203-207) is applied while the operand tiles are staged; `dtype` is then the
                                           dtype of w and of the staged operand. */
  int32_t x_half_res;                   /* with gn_coef: x is [batch][height/2][width/2] and the operand is the nearest
                                           2x upsample of silu(x*A + B) -- in_layers of an `up` ResBlock (nn.py:190-195:
                                           GroupNorm, SiLU, Upsample, conv) with no upsampled tensor in memory;
                                           height/width are the OUTPUT size */
  int32_t residual_half_res;            /* with gn_coef: residual is [batch][height/2][width/2] and is read at
                                           (h/2, w/2) -- x_upd of an `up` ResBlock (nn.py:194,212) */
  int32_t halo_copy;                    /* tensor-core entry, 3x3 stride 1, H % 16 == 0, W % 16 == 0, cin % 64 == 0, cout % 128 == 0,
                                           no gn_coef: stage x (already in w's dtype) through the swapped-role halo kernel
                                           (conv_halo_swap.cu) WITHOUT an activation: one halo load per 64-channel slice
                                           instead of one box per tap -- the stem convolution (unet.py:55) */
  const float* w_scale;                 /* dtype FIDM_E4M3 (tensor-core entry, with gn_coef, cin % 128 == 0, cout % 256 == 0):
                                           w holds e4m3 bytes [cout][3][3][cin] and y = acc * w_scale[c] + bias[c] + ...;
                                           the operand is staged as e4m3 (tcgen05 kind::f8f6f4, twice the bf16 rate);
                                           w2 of the fused 1x1 skip stays bf16 and must be pre-divided by w_scale[c] */
} fidm_conv_args;
/* number of partial rows per image the tensor-core conv writes into `colsum` (0: not supported for this size) */
int fidm_conv_colsum_slots(int32_t height, int32_t width);
/* 1 if fidm_conv2d_nhwc_bf16 takes `gn_coef` for this shape (3x3 stride 1, H % 16 == 0, W % 16 == 0, cin % 64 == 0,
 * cout % 128 == 0) AND the layer is large enough to fill the machine's CTA pairs; 0: run the GroupNorm pass. */
int fidm_conv_gn_fusable(int32_t batch, int32_t height, int32_t width, int32_t cin, int32_t cout, int32_t ksize,
                         int32_t stride);
int fidm_conv2d_nhwc_bf16(const fidm_conv_args* a, fidm_stream_t stream);
/* Profiling hook (NULL disables; default).  With a device buffer of 16 x grid uint64, every CTA of the gn_coef kernel
 * records SM cycles: [0..3] MMA issuer (total, waiting for a free accumulator, for a transformed operand copy, for
 * a weight stage), [4..7] transform warps (total, waiting for the halo tile, for a free copy, computing),
 * [8..9] epilogue (total, waiting for an accumulator). */
int fidm_conv_set_profile_buffer(uint64_t* device_buffer);
int fidm_conv2d_nhwc_simt(const fidm_conv_args* a, fidm_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K3  QKV attention over a [batch][tokens][3*C] NHWC qkv buffer (channel order
 * [Q heads | K heads | V heads], head-major inside each third, as nn.py:226-234 views it).
 * softmax_fp32((q*s)^T (k*s)) v with s = head_dim^-1/4, non-causal (nn.py:222-235).
 *   fidm_attention_qkv_nhwc_bf16 : tcgen05 flash-style kernel, head_dim 64 or 128, tokens % 64 == 0.
 *   fidm_attention_qkv_nhwc_simt : fp32 or bf16; tiled FFMA kernel for head_dim 16/32/64/128, a one-warp-per-query
 *                                  kernel for any other head_dim <= 1024 (nn.py:245-249 allows any C / heads).
 * ---------------------------------------------------------------------------------------------- */
typedef struct fidm_attn_args {
  int32_t dtype;
  int32_t batch, tokens, heads, head_dim;
  const void* qkv; int32_t ld_qkv;      /* >= 3*heads*head_dim */
  void* out; int32_t ld_out;            /* [batch][tokens][heads*head_dim] */
} fidm_attn_args;
int fidm_attention_qkv_nhwc_bf16(const fidm_attn_args* a, fidm_stream_t stream);
int fidm_attention_qkv_nhwc_simt(const fidm_attn_args* a, fidm_stream_t stream);

/* Weight repack helper: OIHW fp32 (PyTorch) -> KRSC (bf16|fp32) with Cin/Cout zero padding. */
int fidm_repack_weight_oihw_to_krsc(const float* w, void* dst, int32_t dst_dtype, int32_t cout,
                                    int32_t cin, int32_t ksize, int32_t cout_pad, int32_t cin_pad,
                                    fidm_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* FIDM_B200_H_ */
