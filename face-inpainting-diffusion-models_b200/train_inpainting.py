"""Model + diffusion factory and the sampling helper of the reference's `train_inpainting.py`
(`:199-262` and `:265-310`).  The training loop utilities of that file (`train_epoch`, `validate`,
checkpoint writers, schedulers) are outside the sampling path and are not provided.
"""
import torch

from .unet import DiffusionInpaintingModel, UNetModel
from .utils.schedules import create_gaussian_diffusion

# the architecture the reference hard-codes (train_inpainting.py:208-224)
FFHQ_UNET_KWARGS = dict(in_channels=3, model_channels=128, out_channels=6, num_res_blocks=1,
                        attention_resolutions=(16,), channel_mult=(1, 1, 2, 2, 4, 4), conv_resample=True,
                        dims=2, use_checkpoint=False, use_fp16=False, num_heads=4, num_head_channels=64,
                        use_scale_shift_norm=True, resblock_updown=True)


def unwrap_state_dict(checkpoint, keys=("state_dict", "model")):
    """Checkpoint container sniffing (train_inpainting.py:230-238; the evaluation scripts use
    keys=("model_state_dict", "state_dict"), test_inp_ddim_100.py:337-349)."""
    if isinstance(checkpoint, dict):
        for k in keys:
            if k in checkpoint:
                return checkpoint[k]
    return checkpoint


def fold_lora(state_dict, alpha_over_r=None):
    """Optional loader helper: fold `<name>.lora_A.weight` / `<name>.lora_B.weight` pairs into
    `<name>.weight` (W += (alpha/r) * B @ A) and drop them.  The reference has no LoRA code; a
    "LoRA-merged" checkpoint is simply one whose qkv / proj_out weights already contain the update
    (SURVEY.md fact 2), which needs no special handling."""
    out = dict(state_dict)
    for k in list(state_dict):
        if k.endswith(".lora_A.weight"):
            base = k[: -len(".lora_A.weight")]
            A, Bm = state_dict[k], state_dict[base + ".lora_B.weight"]
            scale = alpha_over_r if alpha_over_r is not None else 1.0
            w = out[base + ".weight"]
            out[base + ".weight"] = (w.reshape(w.shape[0], -1) + scale * (Bm.reshape(Bm.shape[0], -1) @
                                                                      A.reshape(A.shape[0], -1))).reshape(w.shape)
            del out[k], out[base + ".lora_B.weight"]
    return out


def create_model_and_diffusion(checkpoint_path, device, img_size=256):
    """Same contract as the reference (train_inpainting.py:199-262): returns
    (DiffusionInpaintingModel, GaussianDiffusion, {'missing_keys', 'unexpected_keys'}).
    `checkpoint_path=None` skips the load (random init), which the benchmarks use."""
    base_model = UNetModel(image_size=img_size, **FFHQ_UNET_KWARGS)
    missing, unexpected = [], []
    if checkpoint_path is not None:
        print(f"Loading checkpoint from {checkpoint_path}")
        ckpt = torch.load(checkpoint_path, map_location="cpu", weights_only=False)
        res = base_model.load_state_dict(unwrap_state_dict(ckpt), strict=False)
        missing, unexpected = list(res.missing_keys), list(res.unexpected_keys)
        print(f"Missing keys: {len(missing)}, Unexpected keys: {len(unexpected)}")
    model = DiffusionInpaintingModel(base_model, in_channels=9).to(device)
    diffusion = create_gaussian_diffusion(steps=1000, learn_sigma=True, noise_schedule="quadratic",
                                          use_kl=False, predict_xstart=False, rescale_timesteps=False)
    return model, diffusion, {"missing_keys": missing, "unexpected_keys": unexpected}


def conditioning(gt, gt_keep_mask):
    """(masked_image, mask) the UNet is fed for the known image gt and its keep mask (test_inp_ddim_100.py:373-385)."""
    return gt * gt_keep_mask + torch.zeros_like(gt) * (1 - gt_keep_mask), 1 - gt_keep_mask


class InpaintingModelFn:
    """The `model_fn` closure every working call site of the reference wraps the model in
    (test_inp_ddim_100.py:373-385): swallows `gt` / `gt_keep_mask`, feeds the UNet
    masked_image = gt * keep and mask = 1 - keep.  The two conditioning tensors are computed once
    instead of once per step."""

    def __init__(self, model):
        self.model = model
        self._key = None
        self._cond = None

    def parameters(self):
        return self.model.parameters()

    def eval(self):
        self.model.eval()
        return self

    def train(self, mode=True):
        self.model.train(mode)
        return self

    def _conditioning(self, gt, gt_keep_mask):
        # the cache holds references, so identity (not an address that could be recycled) is compared
        k = self._key
        if k is None or k[0] is not gt or k[1] is not gt_keep_mask or k[2:] != (gt._version, gt_keep_mask._version):
            self._cond = conditioning(gt, gt_keep_mask)
            self._key = (gt, gt_keep_mask, gt._version, gt_keep_mask._version)
        return self._cond

    def __call__(self, x, t, gt=None, gt_keep_mask=None, masked_image=None, mask=None, **kwargs):
        if masked_image is None or mask is None:
            if gt is None or gt_keep_mask is None:
                raise ValueError("Ground truth and mask required for inpainting")
            masked_image, mask = self._conditioning(gt, gt_keep_mask)
        return self.model(x, t, masked_image=masked_image, mask=mask)

    def fused_plan(self, shape, x, t_first, model_kwargs):
        """Step-boundary fusion hook of GaussianDiffusion's loops: pack the loop-invariant conditioning channels
        (masked image, mask x3: unet.py:199) together with the initial state `x` and timestep into the engine plan's
        network input ONCE and return the plan; from then on the sampler step kernel writes the three state channels
        and the timestep itself and `plan.run()` is the whole model call.  None: the caller uses __call__ per step."""
        mk = model_kwargs or {}
        gt, keep = mk.get("gt"), mk.get("gt_keep_mask")
        masked_image, mask = mk.get("masked_image"), mk.get("mask")
        inner = self.model
        if getattr(inner, "fused_plan", None) is None or len(shape) != 4:       # not this package's DiffusionInpaintingModel
            return None
        if masked_image is None or mask is None:
            if gt is None or keep is None:
                return None
            masked_image, mask = self._conditioning(gt, keep)
        if not (x.is_cuda and x.dtype == torch.float32 and tuple(x.shape) == tuple(shape)):
            return None
        return inner.fused_plan(x, t_first, masked_image, mask)

    def slot_plan(self, batch, channels, height, width):
        """Continuous-batching hook (continuous.py): the engine plan of `batch` slots, whose state channels and
        timesteps the sampler step kernel writes, or None: the caller uses __call__ per iteration."""
        inner = self.model
        if getattr(inner, "slot_plan", None) is None:
            return None
        return inner.slot_plan(batch, channels, height, width)

    def load_slot(self, plan, slot, gt, gt_keep_mask):
        """Pack the conditioning channels of one request (gt [1, C, H, W], keep [1, 1 or C, H, W]) into slot `slot` of
        a plan from slot_plan."""
        masked_image, mask = conditioning(gt, gt_keep_mask)
        self.model.load_slot(plan, slot, masked_image, mask)


def sample_with_advanced_inpainting(model, diffusion, masked_images, masks, device, num_steps=50, use_ddim=True,
                                    eta=0.0, injection_schedule="all", use_cumulative_noise=True):
    """Helper of train_inpainting.py:265-310: masks are 1 = inpaint; gt is re-derived from the masked
    image exactly as the reference does (`masked / (1 - mask + 1e-8)`, clamped)."""
    model.eval()
    gt = torch.clamp(masked_images / (1 - masks + 1e-8), -1, 1)
    keep = 1 - masks
    with torch.no_grad():
        return diffusion.sample_with_advanced_inpainting(
            model=model if isinstance(model, InpaintingModelFn) else InpaintingModelFn(model),
            shape=masked_images.shape, gt=gt, gt_keep_mask=keep, use_ddim=use_ddim, eta=eta, progress=False,
            device=device, injection_schedule=injection_schedule, use_cumulative_noise=use_cumulative_noise)
