"""ctypes binding of the C ABI declared in include/fidm_b200.h.

The shared library is built in-tree by `__graft_entry__.build()` (nvcc, sm_100a).  There is no
CPU or PyTorch fallback: if the library is missing, or a call fails, this module raises.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# FIDM_LIB_PATH: A/B experiments against an older build of the library (symbols it lacks are skipped)
LIB_PATH = os.environ.get("FIDM_LIB_PATH") or os.path.join(_HERE, "libfidm_b200.so")

F32, BF16, F16, E4M3 = 0, 1, 2, 3
COEF_COLS = 20
C_SQRT_AB, C_SQRT_1MAB, C_SQRT_AB_F32, C_SQRT_1MAB_F32 = range(4)
MS_COLS = 7
MS_X0_C1, MS_X0_C2, MS_A, MS_B0, MS_B1, MS_INJ_A, MS_INJ_S = range(7)
STEP_INJECT_ONLY, STEP_UPDATE_ONLY, STEP_UPDATE_INJECT = 0, 1, 2
SAMPLER_DDPM, SAMPLER_DDIM, SAMPLER_DDIM_SCRIPT = 0, 1, 2
MEAN_PREVIOUS_X, MEAN_START_X, MEAN_EPSILON = 0, 1, 2
VAR_LEARNED, VAR_FIXED, VAR_LEARNED_RANGE = 0, 1, 2
RESAMPLE_NONE, RESAMPLE_DOWN, RESAMPLE_UP = 0, 1, 2
NOISE_XT, NOISE_STEP, NOISE_INJECT, NOISE_INJECT_FRESH, NOISE_UNDO = range(5)
MAX_SLOTS = 128
SLOT_IDLE, SLOT_ADMIT = -1, -2

i32, vp, fp, dp = C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p


class StepArgs(C.Structure):
    _fields_ = [("batch", i32), ("channels", i32), ("hw", i32),
                ("mode", i32), ("sampler", i32), ("mean_type", i32), ("var_type", i32),
                ("clip_denoised", i32), ("cumulative", i32), ("mask_channels", i32),
                ("num_timesteps", i32), ("t_update", i32), ("t_inject", i32),
                ("t_dev", vp), ("coef", fp), ("x", fp), ("model_out", fp), ("z", fp), ("gt", fp),
                ("keep_mask", fp), ("inject_noise", fp), ("sample", fp), ("pred_xstart", fp),
                ("x_next", fp), ("mean_out", fp), ("logvar_out", fp),
                ("stem_out", vp), ("stem_dtype", i32), ("stem_ld", i32), ("t_out", fp), ("t_out_value", C.c_float)]


class MultistepArgs(C.Structure):
    _fields_ = [("batch", i32), ("channels", i32), ("hw", i32), ("mean_type", i32), ("out_channels", i32),
                ("clip_denoised", i32), ("mask_channels", i32), ("steps", i32), ("step", i32),
                ("coef", fp), ("x", fp), ("model_out", fp), ("m_prev", fp), ("m_out", fp), ("x_next", fp),
                ("inject", i32), ("gt", fp), ("keep_mask", fp), ("inject_noise", fp),
                ("stem_out", vp), ("stem_dtype", i32), ("stem_ld", i32), ("t_out", fp), ("t_out_value", C.c_float)]


class ResampleArgs(C.Structure):
    _fields_ = [("batch", i32), ("channels", i32), ("hw", i32), ("mask_channels", i32),
                ("undo_a", C.c_float), ("undo_s", C.c_float), ("x", fp), ("noise", fp), ("x_next", fp),
                ("inject", i32), ("inject_a", C.c_float), ("inject_s", C.c_float),
                ("gt", fp), ("keep_mask", fp), ("inject_noise", fp),
                ("stem_out", vp), ("stem_dtype", i32), ("stem_ld", i32), ("t_out", fp), ("t_out_value", C.c_float)]


class SeededNoise(C.Structure):
    _fields_ = [("seeds", vp), ("draw", i32), ("inject_tag", i32), ("inject_draw", i32)]


class SlotArgs(C.Structure):
    _fields_ = [("t_value", fp), ("inject_draw", vp), ("out", fp), ("step_noise", i32),
                ("action", i32 * MAX_SLOTS), ("seeds", C.c_uint64 * MAX_SLOTS)]


class MsSlotArgs(C.Structure):
    _fields_ = [("t_value", fp), ("inject_draw", vp), ("order", vp), ("out", fp), ("inject_tag", i32),
                ("admit_inject_a", C.c_float), ("admit_inject_s", C.c_float),
                ("action", i32 * MAX_SLOTS), ("seeds", C.c_uint64 * MAX_SLOTS)]


class RpSlotArgs(C.Structure):
    _fields_ = [("t_value", fp), ("eval_t", vp), ("next_t", vp), ("undo", fp), ("inject_draw", vp), ("out", fp),
                ("n_evals", i32), ("admit_draw", i32),
                ("action", i32 * MAX_SLOTS), ("seeds", C.c_uint64 * MAX_SLOTS)]


class PackArgs(C.Structure):
    _fields_ = [("batch", i32), ("hw", i32), ("n_src", i32), ("src", fp * 4),
                ("src_channels", i32 * 4), ("src_repeat", i32 * 4),
                ("dst", vp), ("dst_dtype", i32), ("ld_dst", i32), ("c_pad", i32)]


class GnArgs(C.Structure):
    _fields_ = [("dtype", i32), ("y_dtype", i32), ("batch", i32), ("height", i32), ("width", i32), ("channels", i32),
                ("groups", i32), ("eps", C.c_float), ("x", vp), ("ld_x", i32),
                ("gamma", fp), ("beta", fp), ("scale_shift", fp), ("ld_ss", i32),
                ("silu", i32), ("resample", i32), ("skip_norm", i32), ("y", vp), ("ld_y", i32),
                ("y_raw", vp), ("ld_raw", i32), ("stats", dp),
                ("chansum", fp), ("ld_chansum", i32)]


class ConvArgs(C.Structure):
    _fields_ = [("dtype", i32), ("batch", i32), ("height", i32), ("width", i32),
                ("cin", i32), ("cout", i32), ("ksize", i32), ("stride", i32),
                ("x", vp), ("ld_x", i32), ("w", vp),
                ("x2", vp), ("ld_x2", i32), ("cin2", i32), ("w2", vp),
                ("bias", fp), ("row_add", fp), ("ld_row_add", i32),
                ("residual", vp), ("ld_res", i32), ("y", vp), ("ld_y", i32),
                ("y_nchw_f32", i32), ("cout_valid", i32), ("colsum", fp),
                ("splitk_ws", vp), ("splitk_ws_bytes", C.c_int64),
                ("gn_coef", fp), ("ld_gn_coef", i32), ("x_half_res", i32), ("residual_half_res", i32),
                ("halo_copy", i32), ("w_scale", fp)]


class AttnArgs(C.Structure):
    _fields_ = [("dtype", i32), ("batch", i32), ("tokens", i32), ("heads", i32), ("head_dim", i32),
                ("qkv", vp), ("ld_qkv", i32), ("out", vp), ("ld_out", i32)]


# every symbol include/fidm_b200.h declares: name -> (restype, argtypes)
_P = C.POINTER
SYMBOLS = {
    "fidm_abi_version": (C.c_int, []),
    "fidm_last_error_string": (C.c_char_p, []),
    "fidm_device_supported": (C.c_int, [C.c_int]),
    "fidm_sampler_step": (C.c_int, [_P(StepArgs), vp]),
    "fidm_multistep_step": (C.c_int, [_P(MultistepArgs), vp]),
    "fidm_resample_undo": (C.c_int, [_P(ResampleArgs), vp]),
    "fidm_sampler_step_seeded": (C.c_int, [_P(StepArgs), _P(SeededNoise), vp]),
    "fidm_multistep_step_seeded": (C.c_int, [_P(MultistepArgs), _P(SeededNoise), vp]),
    "fidm_resample_undo_seeded": (C.c_int, [_P(ResampleArgs), _P(SeededNoise), vp]),
    "fidm_randn_seeded": (C.c_int, [fp, vp, i32, C.c_int64, i32, i32, vp]),
    "fidm_sampler_step_slots": (C.c_int, [_P(StepArgs), _P(SlotArgs), vp]),
    "fidm_multistep_step_slots": (C.c_int, [_P(MultistepArgs), _P(MsSlotArgs), vp]),
    "fidm_repaint_step_slots": (C.c_int, [_P(StepArgs), _P(RpSlotArgs), vp]),
    "fidm_pack_nchw_to_nhwc": (C.c_int, [_P(PackArgs), vp]),
    "fidm_unpack_nhwc_to_nchw": (C.c_int, [vp, i32, i32, fp, i32, i32, i32, vp]),
    "fidm_prepare_inputs_u8": (C.c_int, [vp, vp, fp, fp, fp, fp, i32, i32, vp]),
    "fidm_blend_to_u8": (C.c_int, [fp, fp, fp, vp, i32, i32, vp]),
    "fidm_timestep_embedding": (C.c_int, [fp, fp, fp, i32, i32, vp]),
    "fidm_linear_small": (C.c_int, [fp, vp, i32, fp, fp, i32, i32, i32, i32, vp]),
    "fidm_groupnorm_silu_nhwc": (C.c_int, [_P(GnArgs), vp]),
    "fidm_groupnorm_num_launches": (C.c_int, [_P(GnArgs)]),
    "fidm_groupnorm_workspace_bytes": (C.c_int64, [i32, i32]),
    "fidm_groupnorm_reduce_colsum": (C.c_int, [fp, i32, i32, i32, fp, i32, i32, vp]),
    "fidm_groupnorm_silu_coeff": (C.c_int, [_P(GnArgs), fp, i32, vp]),
    "fidm_groupnorm_reduce_colsum_coeff": (C.c_int, [fp, i32, fp, i32, i32, _P(GnArgs), fp, i32, vp]),
    "fidm_conv_colsum_slots": (C.c_int, [i32, i32]),
    "fidm_conv_gn_fusable": (C.c_int, [i32, i32, i32, i32, i32, i32, i32]),
    "fidm_conv2d_nhwc_bf16": (C.c_int, [_P(ConvArgs), vp]),
    "fidm_conv_set_profile_buffer": (C.c_int, [vp]),
    "fidm_conv2d_nhwc_simt": (C.c_int, [_P(ConvArgs), vp]),
    "fidm_attention_qkv_nhwc_bf16": (C.c_int, [_P(AttnArgs), vp]),
    "fidm_attention_qkv_nhwc_simt": (C.c_int, [_P(AttnArgs), vp]),
    "fidm_repack_weight_oihw_to_krsc": (C.c_int, [fp, vp, i32, i32, i32, i32, i32, i32, vp]),
}

_lib = None


class FidmError(RuntimeError):
    pass


class ArgumentError(FidmError, ValueError):
    """An argument the library refuses (negative status): a FidmError, and a ValueError like any bad argument."""


def lib():
    """The loaded shared library; raises if it has not been built (no fallback path exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FidmError(
                f"{LIB_PATH} is missing: build the sm_100a extension first "
                "(`python -c 'import __graft_entry__ as g; g.build()'`). There is no CPU fallback.")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            if os.environ.get("FIDM_LIB_PATH") and not hasattr(handle, name):
                continue
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = res, args
        if handle.fidm_abi_version() != 3:
            raise FidmError("libfidm_b200.so ABI version mismatch; rebuild")
        _lib = handle
    return _lib


def check(rc, what=""):
    if rc == 0:
        return
    msg = lib().fidm_last_error_string().decode(errors="replace")
    if rc < 0:
        raise ArgumentError(f"fidm {what}: {msg} (code {rc})")
    raise FidmError(f"fidm {what}: CUDA error {rc}: {msg}")


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t, byte_offset=0):
    return None if t is None else C.c_void_p(t.data_ptr() + byte_offset)


def dtype_code(dt):
    if dt == torch.bfloat16:
        return BF16
    if dt == torch.float32:
        return F32
    if dt == torch.float16:
        return F16
    if dt in (torch.float8_e4m3fn, torch.uint8):
        return E4M3
    raise ValueError(f"unsupported dtype {dt}")


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise FidmError("fidm_b200 runs on sm_100a GPUs only; got a CPU tensor (no CPU fallback exists)")
