"""`UNetModel` and `DiffusionInpaintingModel` with the reference's constructor and call surface
(`unet.py:17-21`, `:154`, `:179`, `:197`) and its exact `state_dict` layout, executed on a B200 by
the fused engine (`engine.Plan`).  There is no per-module PyTorch forward and no CPU fallback.
"""
import os

import torch
import torch.nn as nn

from . import _lib as L
from . import nn as layers
from .arch import unet_topology
from .engine import STEM_CIN_PAD, Plan, Weights


class UNetModel(nn.Module):
    """The full UNet with attention and timestep embedding (reference ctor: unet.py:17-21)."""

    def __init__(self, image_size, in_channels, model_channels, out_channels, num_res_blocks,
                 attention_resolutions, dropout=0, channel_mult=(1, 2, 4, 8), conv_resample=True,
                 dims=2, num_classes=None, use_checkpoint=False, use_fp16=False, num_heads=1,
                 num_head_channels=-1, num_heads_upsample=-1, use_scale_shift_norm=False,
                 resblock_updown=False, use_new_attention_order=False):
        super().__init__()
        if num_heads_upsample == -1:
            num_heads_upsample = num_heads
        self.topology = unet_topology(
            image_size, in_channels, model_channels, out_channels, num_res_blocks, attention_resolutions,
            dropout=dropout, channel_mult=tuple(channel_mult), conv_resample=conv_resample, dims=dims,
            num_classes=num_classes, use_checkpoint=use_checkpoint, use_fp16=use_fp16, num_heads=num_heads,
            num_head_channels=num_head_channels, num_heads_upsample=num_heads_upsample,
            use_scale_shift_norm=use_scale_shift_norm, resblock_updown=resblock_updown,
            use_new_attention_order=use_new_attention_order)
        topo = self.topology
        # attributes the reference exposes (unet.py:27-40)
        self.image_size, self.in_channels, self.model_channels = image_size, in_channels, model_channels
        self.out_channels, self.num_res_blocks = out_channels, num_res_blocks
        self.attention_resolutions, self.dropout, self.channel_mult = attention_resolutions, dropout, channel_mult
        self.conv_resample, self.num_classes, self.use_checkpoint = conv_resample, num_classes, use_checkpoint
        self.dtype = torch.float16 if use_fp16 else torch.float32
        self.num_heads, self.num_head_channels = num_heads, num_head_channels
        self.num_heads_upsample = num_heads_upsample

        ted = topo.time_embed_dim
        self.time_embed = nn.Sequential(nn.Linear(model_channels, ted), nn.SiLU(), nn.Linear(ted, ted))
        ssn = topo.cfg["use_scale_shift_norm"]

        def build(layer):
            if layer.kind == "stem":
                return nn.Conv2d(layer.cin, layer.cout, 3, padding=1)
            if layer.kind == "res":
                return layers.ResBlock(layer, ted, ssn, dropout)
            if layer.kind == "attn":
                return layers.AttentionBlock(layer)
            if layer.kind == "down":
                return layers.Downsample(layer)
            if layer.kind == "up":
                return layers.Upsample(layer)
            raise NotImplementedError(layer.kind)

        def seq(blk):
            return layers.TimestepEmbedSequential(*[build(l) for l in blk.layers])

        self.input_blocks = nn.ModuleList([seq(b) for b in topo.input_blocks])
        self.middle_block = seq(topo.middle)
        self.output_blocks = nn.ModuleList([seq(b) for b in topo.output_blocks])
        self.out = nn.Sequential(nn.GroupNorm(32, topo.head_ch), nn.SiLU(),
                                 layers._zero_(nn.Conv2d(topo.head_ch, out_channels, 3, padding=1)))
        self.eval()

        # ---- engine state (not part of the state_dict)
        self.precision = os.environ.get("FIDM_PRECISION", "bf16")
        self.use_cuda_graph = os.environ.get("FIDM_CUDA_GRAPH", "1") != "0"
        self._weights = None
        self._plans = {}
        # checkpoints may be loaded through a wrapper (DiffusionInpaintingModel.load_state_dict)
        self.register_load_state_dict_post_hook(lambda module, incompatible: module.invalidate())

    # ------------------------------------------------------------------ engine management
    def set_precision(self, precision):
        """"bf16" (tcgen05 tensor cores), "fp32" (FFMA verification mode) or the opt-in "fp8" (bf16 engine with the large
        GroupNorm-fused 3x3 convolutions on e4m3 operands, engine.py)."""
        if precision not in ("bf16", "fp32", "fp8"):
            raise ValueError(precision)
        if precision != self.precision:
            self.precision = precision
            self.invalidate()
        return self

    def invalidate(self):
        """Drop repacked weights and plans (call after mutating parameters in place)."""
        self._weights = None
        self._plans = {}

    def _apply(self, fn, *a, **k):
        out = super()._apply(fn, *a, **k)
        self.invalidate()
        return out

    def _stem_in_channels(self):
        return self.input_blocks[0][0].weight.shape[1]

    def plan_for(self, batch, height, width):
        dev = self.out[2].weight.device
        if dev.type != "cuda":
            raise L.FidmError("fidm_b200 models run on sm_100a GPUs only: move the model to CUDA "
                              "(there is no CPU fallback)")
        if self._weights is None:
            topo = self.topology
            cin = self._stem_in_channels()
            if cin != topo.cfg["in_channels"]:       # stem swapped by DiffusionInpaintingModel
                cfg = dict(topo.cfg)
                for k in ("image_size", "in_channels", "model_channels", "out_channels", "num_res_blocks",
                          "attention_resolutions"):
                    cfg.pop(k)
                topo = unet_topology(self.image_size, cin, self.model_channels, self.out_channels,
                                     self.num_res_blocks, self.attention_resolutions, **cfg)
                self.topology = topo
            if cin > STEM_CIN_PAD:
                raise NotImplementedError(f"in_channels {cin} > {STEM_CIN_PAD}")
            with torch.no_grad():
                self._weights = Weights(topo, self.state_dict(), dev, self.precision)
        key = (batch, height, width)
        if key not in self._plans:
            self._plans[key] = Plan(self._weights, batch, height, width, use_graph=self.use_cuda_graph)
        return self._plans[key]

    def _evaluate(self, sources, timesteps, batch, height, width, clone=True):
        """sources: [(fp32 NCHW tensor, channels, repeat)] concatenated along channels."""
        plan = self.plan_for(batch, height, width)
        srcs = []
        for t, c, r in sources:
            L.require_cuda(t)
            srcs.append((t.detach().to(torch.float32).contiguous(), c, r))
        ts = timesteps.detach().to(device=srcs[0][0].device, dtype=torch.float32)
        plan.load_inputs(srcs, ts)
        out = plan.run()
        return out.clone() if clone else out

    def forward(self, x, timesteps, y=None):
        """x: [N, in_channels, H, W] fp32 CUDA; timesteps: [N].  Returns [N, out_channels, H, W] fp32."""
        assert (y is not None) == (self.num_classes is not None)
        n, c, h, w = x.shape
        assert c == self._stem_in_channels()
        return self._evaluate([(x, c, 1)], timesteps, n, h, w)


class DiffusionInpaintingModel(nn.Module):
    """9-channel inpainting wrapper (reference: unet.py:176-200)."""

    def __init__(self, base_model, in_channels=9):
        super().__init__()
        self.base_model = base_model
        old = base_model.input_blocks[0][0]
        new = nn.Conv2d(in_channels, old.out_channels, old.kernel_size, old.stride, old.padding)
        with torch.no_grad():
            if old.weight.shape[1] <= in_channels:
                # RGB filters are kept, the masked-image / mask channels start at zero (unet.py:190-195)
                new.weight.zero_()
                new.weight[:, :old.weight.shape[1]] = old.weight
        new.to(old.weight.device)
        base_model.input_blocks[0] = layers.TimestepEmbedSequential(new)
        base_model.invalidate()
        self.eval()

    def fused_plan(self, x, t_value, masked_image, mask):
        """Pack [x | masked_image | mask x3] and a uniform timestep into the plan's network input and return the plan
        (see train_inpainting.InpaintingModelFn.fused_plan).  The caller owns the plan's inputs until its loop ends."""
        n, c, h, w = x.shape
        if c + masked_image.shape[1] + 3 > 16:
            return None
        base = self.base_model
        plan = base.plan_for(n, h, w)
        rep = 3 if mask.shape[1] == 1 else 1
        srcs = [(t.detach().to(torch.float32).contiguous(), t.shape[1], r)
                for t, r in ((x, 1), (masked_image, 1), (mask, rep))]
        plan.load_inputs(srcs, torch.full((n,), float(t_value), device=x.device, dtype=torch.float32))
        return plan

    def slot_plan(self, batch, channels, height, width):
        """The engine plan of `batch` slots for continuous batching (continuous.py), or None when the network input
        [x | masked_image | mask x3] does not fit the 16-channel stem pack.  The plan is the one the loops of this
        batch size use: the caller owns its inputs while it has work."""
        if 2 * channels + 3 > 16:
            return None
        return self.base_model.plan_for(batch, height, width)

    def load_slot(self, plan, slot, masked_image, mask):
        """Pack one image's conditioning channels (masked image, mask x3: unet.py:199) into image `slot` of the plan's
        network input, behind the state channels that the sampler step kernel writes."""
        c = masked_image.shape[1]
        rep = 3 if mask.shape[1] == 1 else 1
        plan.load_slot(slot, [(t.detach().to(torch.float32).contiguous(), t.shape[1], r)
                              for t, r in ((masked_image, 1), (mask, rep))], c)

    def forward(self, x, t, masked_image, mask):
        """cat([x, masked_image, mask x3]) -> base UNet (unet.py:197-200); the concat is fused into the
        NCHW->NHWC pack kernel."""
        n, c, h, w = x.shape
        rep = 3 if mask.shape[1] == 1 else 1
        return self.base_model._evaluate([(x, c, 1), (masked_image, masked_image.shape[1], 1),
                                          (mask, mask.shape[1], rep)], t, n, h, w)
