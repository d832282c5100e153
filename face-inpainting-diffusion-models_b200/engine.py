"""Execution plan of one UNet evaluation on a B200.

The reference evaluates the UNet as ~700 eager ATen launches on NCHW fp32 tensors
(`unet.py:154-173`).  Here the topology (`arch.py`) is compiled once per (batch, H, W) into a flat
list of C-ABI kernel calls on NHWC activations:

  * weights are repacked once: OIHW fp32 -> KRSC 16-bit (stem Cin 9 -> 64, head Cout 6 -> 16);
  * `torch.cat([h, hs.pop()], 1)` (`unet.py:170`) never runs: every producer of `h` / `hs[i]` writes
    straight into its channel slice of a pre-planned concat buffer (pixel stride `ld`);
  * GroupNorm+SiLU(+scale/shift)(+2x resample) is one K2 call, conv+bias+emb+residual(+1x1 skip)
    one K1 call, attention one K3 call, the whole timestep path three K5 calls;
  * the list is captured into a CUDA graph after one eager warm-up, so an evaluation is a single
    graph launch (no Python, no per-kernel launch latency).

precision "bf16": tcgen05 tensor-core kernels, fp32 accumulate / statistics / softmax; the residual stream,
                  qkv and attention tensors are bf16, the normalized conv operands (GroupNorm outputs) and
                  the weights they multiply are fp16 (same tensor rate, 8x smaller rounding error).
precision "fp32": FFMA verification mode (north star: eps within rel-L2 1e-5 of the reference).
precision "fp8":  opt-in (SURVEY 8-f row 4): as "bf16", except that the large 3x3 convolutions behind a GroupNorm
                  (cin % 128 == 0, cout % 256 == 0, >= FP8_MIN_PIXELS output pixels -- the 256->256 / 512->256 layers that
                  hold over half of ADM256's FLOPs) multiply an e4m3 operand with e4m3 weights (per-output-channel scale)
                  on tcgen05 kind::f8f6f4 at twice the bf16 rate.  Outside the north star's eps bar; reported with its own
                  PSNR next to bf16.
"""
import ctypes as C
import math
import os

import torch

from . import _lib as L
from .arch import Topology


class Ref:
    """A [B,H,W,channels] NHWC view: channel slice [c0, c0+channels) of `storage` [B,H,W,ld]."""

    __slots__ = ("storage", "c0", "channels", "H", "W")

    def __init__(self, storage, c0, channels, H, W):
        self.storage, self.c0, self.channels, self.H, self.W = storage, c0, channels, H, W

    @property
    def ld(self):
        return self.storage.shape[-1]

    @property
    def ptr(self):
        return C.c_void_p(self.storage.data_ptr() + self.c0 * self.storage.element_size())


class _Pool:
    """Plan-time scratch allocator: buffers live as long as the plan, and are recycled between
    layers because execution is strictly sequential on one stream."""

    def __init__(self, device, dtype):
        self.device, self.dtype = device, dtype
        self.free = {}
        self.all = []

    def get(self, B, H, W, Cn, dtype=None):
        dtype = dtype or self.dtype
        key = (B, H, W, Cn, dtype)
        lst = self.free.setdefault(key, [])
        if lst:
            return lst.pop()
        t = torch.empty(B, H, W, Cn, device=self.device, dtype=dtype)
        self.all.append(t)
        return t

    def put(self, t):
        self.free.setdefault(tuple(t.shape) + (t.dtype,), []).append(t)

    def nbytes(self):
        return sum(t.numel() * t.element_size() for t in self.all)


STEM_CIN_PAD = 64
HEAD_COUT_PAD = 16


def tc_eligible(cin, cout, stride=1, head=False):
    """Shapes the tcgen05 conv kernel takes (fidm_conv2d_nhwc_bf16): stride 1, or the stride-2 3x3 of
    Downsample(use_conv=True) (nn.py:126) through TMA element strides."""
    return stride in (1, 2) and cin % 64 == 0 and (cout % 64 == 0 or (head and cout == 16 and stride == 1))


class Weights:
    """Device-resident, kernel-ready parameters (built once per model / device / precision)."""

    def __init__(self, topo: Topology, sd, device, precision):
        self.topo, self.device, self.precision = topo, device, precision
        self.fp8 = precision == "fp8"
        precision = "bf16" if self.fp8 else precision          # everything but the selected layers is the bf16 engine
        self.tc = precision == "bf16"                           # tensor-core kernels (vs the FFMA verification mode)
        self.conv8 = {}     # name -> (e4m3 krsc weight as uint8, fp32 per-output-channel scale)
        self.skip8 = {}     # out_layers name -> bf16 1x1 skip weight pre-divided by that scale
        self.dtype = torch.bfloat16 if precision == "bf16" else torch.float32
        self.code = L.dtype_code(self.dtype)
        self.conv = {}      # name -> (krsc weight, bias fp32, cin_pad, cout_pad, ksize)
        # In "bf16" mode the *normalized* conv operands (GroupNorm outputs, the packed network input) and
        # the weights they meet are stored as fp16: same tcgen05 rate, 11-bit instead of 8-bit mantissa,
        # and their range is bounded by the normalisation.  The unnormalized residual stream, the qkv /
        # attention tensors and everything they are multiplied with stay bf16.
        self.norm_dtype = torch.float16 if precision == "bf16" else torch.float32
        if self.tc and os.environ.get("FIDM_NORM_DTYPE", "fp16") == "bf16":
            self.norm_dtype = torch.bfloat16          # A/B switch: pure-bf16 operands
        self.vec = {}       # name -> fp32 vector (GroupNorm gamma/beta)
        lib = L.lib()

        def f32(name):
            return sd[name].detach().to(device=device, dtype=torch.float32).contiguous()

        def conv(name, cin_pad=None, cout_pad=None, extra_bias=None, normalized=False, stride=1, head=False):
            w = f32(name + ".weight")
            if w.dim() == 3:                      # Conv1d k=1 (nn.py:252,254)
                w = w.unsqueeze(-1)
            cout, cin, ks, _ = w.shape
            cin_pad, cout_pad = cin_pad or cin, cout_pad or cout
            wdt = self.dtype
            if normalized and self.tc and tc_eligible(cin_pad, cout_pad, stride, head):
                wdt = self.norm_dtype
            dst = torch.empty(cout_pad, ks, ks, cin_pad, device=device, dtype=wdt)
            L.check(lib.fidm_repack_weight_oihw_to_krsc(L.ptr(w), L.ptr(dst), L.dtype_code(wdt), cout, cin, ks,
                                                        cout_pad, cin_pad, L.stream()), "repack " + name)
            b = torch.zeros(cout_pad, device=device, dtype=torch.float32)
            b[:cout] = f32(name + ".bias")
            if extra_bias is not None:
                b[:cout] += extra_bias
            self.conv[name] = (dst, b, cin_pad, cout_pad, ks)
            if self.fp8 and normalized and ks == 3 and stride == 1 and cin_pad % 128 == 0 and cout_pad % 256 == 0:
                # e4m3 copy: w = q * scale[c], scale[c] = max|w[c]| / 448 (the largest finite e4m3)
                wk = torch.empty(cout_pad, ks, ks, cin_pad, device=device, dtype=torch.float32)
                L.check(lib.fidm_repack_weight_oihw_to_krsc(L.ptr(w), L.ptr(wk), L.F32, cout, cin, ks, cout_pad, cin_pad,
                                                            L.stream()), "repack fp8 " + name)
                amax = wk.abs().amax(dim=(1, 2, 3)).clamp_min(1e-12)
                scale = (amax / 448.0).contiguous()
                q = (wk / scale[:, None, None, None]).clamp(-448.0, 448.0).to(torch.float8_e4m3fn)
                self.conv8[name] = (q.view(torch.uint8).contiguous(), scale)

        def norm(name):
            self.vec[name + ".weight"] = f32(name + ".weight")
            self.vec[name + ".bias"] = f32(name + ".bias")

        emb_w, emb_b, self.emb_off = [], [], {}
        off = 0
        from .arch import all_layers
        for layer in all_layers(topo):
            n = layer.name
            if layer.kind == "stem":
                conv(n, cin_pad=STEM_CIN_PAD, normalized=True)
            elif layer.kind == "res":
                norm(n + ".in_layers.0")
                conv(n + ".in_layers.2", normalized=True)
                norm(n + ".out_layers.0")
                if layer.skip == "identity":
                    conv(n + ".out_layers.3", normalized=True)
                else:
                    conv(n + ".skip_connection")
                    # the 1x1 skip rides the out_layers conv as extra K slices (Plan._conv, x2): that launch takes the
                    # tensor-core kernel -- and fp16 normalized operands -- only if the skip source qualifies too
                    # (the same predicate _conv applies); otherwise it is the SIMT kernel on bf16 operands
                    conv(n + ".out_layers.3", extra_bias=f32(n + ".skip_connection.bias"),
                         normalized=layer.skip != "conv1x1" or layer.cin % 64 == 0)
                    if (n + ".out_layers.3") in self.conv8:
                        # the 1x1 skip shares the accumulator that is later multiplied by the e4m3 scale: pre-divide it
                        w2 = self.conv[n + ".skip_connection"][0].float() / self.conv8[n + ".out_layers.3"][1][:, None, None, None]
                        self.skip8[n + ".out_layers.3"] = w2.to(torch.bfloat16).contiguous()
                w = f32(n + ".emb_layers.1.weight")
                emb_w.append(w)
                emb_b.append(f32(n + ".emb_layers.1.bias"))
                self.emb_off[n] = off
                off += w.shape[0]
            elif layer.kind == "attn":
                norm(n + ".norm")
                conv(n + ".qkv", normalized=True)
                conv(n + ".proj_out")
            elif layer.kind == "down" and layer.use_conv:
                conv(n + ".op", stride=2)
            elif layer.kind == "up" and layer.use_conv:
                conv(n + ".conv")
        norm("out.0")
        conv("out.2", cout_pad=HEAD_COUT_PAD, normalized=True, head=True)
        self.emb_total = off
        self.emb_w = torch.cat(emb_w, 0).contiguous()
        self.emb_b = torch.cat(emb_b, 0).contiguous()
        self.te0_w, self.te0_b = f32("time_embed.0.weight"), f32("time_embed.0.bias")
        self.te2_w, self.te2_b = f32("time_embed.2.weight"), f32("time_embed.2.bias")
        mc = topo.cfg["model_channels"]
        half = mc // 2
        # computed on the CPU exactly as the reference does (nn.py:54-56), then uploaded
        self.freqs = torch.exp(-math.log(10000) * torch.arange(start=0, end=half, dtype=torch.float32) / half
                               ).to(device)
        torch.cuda.synchronize(device)


class Plan:
    """Flat kernel schedule + buffers for one (batch, H, W)."""

    def __init__(self, weights: Weights, B, H, W, use_graph=True, out=None):
        self.w, self.B, self.H, self.W = weights, B, H, W
        topo = weights.topo
        dev, dt = weights.device, weights.dtype
        self.ops = []
        self.n_fp8 = 0           # convolutions of this plan that run on the e4m3 path (precision "fp8")
        self.pool = _Pool(dev, dt)
        self.keep = []
        # fused GroupNorm statistics: per-storage [B, ld, 2] channel sums written by the producing convs
        self.fuse_stats = os.environ.get("FIDM_FUSE_GN_STATS", "1") != "0" and weights.tc
        # GroupNorm + SiLU applied in the consumer conv's operand path (K1h) where fidm_conv_gn_fusable() says so
        self.fuse_gn = os.environ.get("FIDM_FUSE_GN_APPLY", "1") != "0"
        self.fuse_up = os.environ.get("FIDM_FUSE_UPSAMPLE", "1") != "0"
        self.fuse_reduce_coeff = os.environ.get("FIDM_FUSE_REDUCE_COEFF", "1") != "0"
        self.chansum = {}        # id(storage) -> fp32 [B, ld, 2]
        self.coverage = {}       # id(storage) -> [(c0, channels)]
        self.colsum_scratch = {}  # numel -> fp32 scratch for the per-tile partial rows
        self.splitk_ws = torch.zeros(32 << 20, device=dev, dtype=torch.uint8)   # zero-initialised, kernels re-arm it
        cfg = topo.cfg
        mc, ted = cfg["model_channels"], topo.time_embed_dim
        self.ssn = cfg["use_scale_shift_norm"]
        lib = L.lib()
        self.lib = lib

        # ---- static inputs / outputs
        self.x_in = torch.zeros(B, H, W, STEM_CIN_PAD, device=dev, dtype=weights.conv["input_blocks.0.0"][0].dtype)
        self.t_in = torch.zeros(B, device=dev, dtype=torch.float32)
        self.out = out if out is not None else torch.empty(B, topo.out_channels, H, W, device=dev,
                                                           dtype=torch.float32)
        assert self.out.is_contiguous() and self.out.shape[0] == B
        self.stats = torch.zeros(lib.fidm_groupnorm_workspace_bytes(B, 32) // 8, device=dev, dtype=torch.float64)

        # ---- K5: timestep path
        self.temb = torch.empty(B, mc, device=dev, dtype=torch.float32)
        self.e1 = torch.empty(B, ted, device=dev, dtype=torch.float32)
        self.emb = torch.empty(B, ted, device=dev, dtype=torch.float32)
        self.emb_all = torch.empty(B, weights.emb_total, device=dev, dtype=torch.float32)
        w = weights
        self._op(lib.fidm_timestep_embedding, L.ptr(self.t_in), L.ptr(w.freqs), L.ptr(self.temb), B, mc)
        self._op(lib.fidm_linear_small, L.ptr(self.temb), L.ptr(w.te0_w), L.F32, L.ptr(w.te0_b), L.ptr(self.e1),
                 B, mc, ted, 0)
        self._op(lib.fidm_linear_small, L.ptr(self.e1), L.ptr(w.te2_w), L.F32, L.ptr(w.te2_b), L.ptr(self.emb),
                 B, ted, ted, 1)
        self._op(lib.fidm_linear_small, L.ptr(self.emb), L.ptr(w.emb_w), L.F32, L.ptr(w.emb_b), L.ptr(self.emb_all),
                 B, ted, w.emb_total, 1)
        self._last_reduce = None             # (op index, storage id, c0, channels, colsum ptr, slots, chansum) of the last fold
        self.n_time_ops = len(self.ops)      # K5 depends only on t: a parallel branch of the graph (see launch_all)
        self.first_emb_use = None            # index of the first op that reads emb_all

        # ---- concat buffers of the output path (unet.py:170): cat_j = [h | hs.pop()]
        n_in = len(topo.input_blocks)
        assert n_in == len(topo.output_blocks)
        res = [(H // b.ds, W // b.ds) for b in topo.input_blocks]
        self.cats = []
        for j, blk in enumerate(topo.output_blocks):
            i = n_in - 1 - j
            hh, ww = res[i]
            self.cats.append(torch.empty(B, hh, ww, blk.cin, device=dev, dtype=dt))

        def in_dst(i):
            j = n_in - 1 - i
            blk = topo.output_blocks[j]
            hh, ww = res[i]
            return Ref(self.cats[j], blk.cin - blk.skip_ch, blk.skip_ch, hh, ww)

        def h_dst(j):
            blk = topo.output_blocks[j]
            hh, ww = res[n_in - 1 - j]
            return Ref(self.cats[j], 0, blk.cin - blk.skip_ch, hh, ww)

        # ---- walk the topology
        x = Ref(self.x_in, 0, STEM_CIN_PAD, H, W)
        for i, blk in enumerate(topo.input_blocks):
            x = self._block(blk, x, in_dst(i))
        x = self._block(topo.middle, x, h_dst(0))
        for j, blk in enumerate(topo.output_blocks):
            full = Ref(self.cats[j], 0, blk.cin, x.H, x.W)
            if j + 1 < len(topo.output_blocks):
                dst = h_dst(j + 1)
            else:
                dst = self._new(self.H, self.W, blk.cout)
            x = self._block(blk, full, dst)
        # ---- head: out = conv3x3(SiLU(GN(h)))  (unet.py:148-152,173)
        if self._fusable("out.2", x.H, x.W):
            coef = self._gn_coeff(x, "out.0")
            self._conv("out.2", x, None, nchw_out=self.out, cout_valid=topo.out_channels, gn_coef=coef)
        else:
            a = self._new(x.H, x.W, x.channels, self._wdtype("out.2"))
            self._gn(x, a, "out.0", silu=True)
            self._conv("out.2", a, None, nchw_out=self.out, cout_valid=topo.out_channels)

        self.graph = None
        self.use_graph = use_graph
        self._warm = False

    # ------------------------------------------------------------------ op builders
    def _op(self, fn, *args):
        self.ops.append((fn, args))

    def _uses_emb(self):
        """The op about to be appended reads the timestep table (join point of the K5 branch)."""
        if self.first_emb_use is None:
            self.first_emb_use = len(self.ops)

    def _new(self, H, W, Cn, dtype=None):
        t = self.pool.get(self.B, H, W, Cn, dtype)
        self.coverage.pop(id(t), None)           # new contents: previously fused statistics are stale
        return Ref(t, 0, Cn, H, W)

    def _covered(self, x):
        """True if fused channel sums exist for every channel of the view `x`."""
        rng = sorted(self.coverage.get(id(x.storage), []))
        pos = x.c0
        for c0, n in rng:
            if c0 <= pos < c0 + n:
                pos = c0 + n
        return pos >= x.c0 + x.channels

    def _wdtype(self, name):
        """dtype of the weights of conv `name` == dtype its (normalized) input operand must have."""
        return self.w.conv[name][0].dtype

    def _release(self, ref):
        self.pool.put(ref.storage)

    def _gn(self, x, y, name, silu, scale_shift=None, resample=L.RESAMPLE_NONE, y_raw=None, skip_norm=False):
        w = self.w
        a = L.GnArgs()
        a.dtype, a.y_dtype = L.dtype_code(x.storage.dtype), L.dtype_code(y.storage.dtype)
        a.batch, a.height, a.width, a.channels, a.groups = self.B, x.H, x.W, x.channels, 32
        a.eps = 1e-5
        a.x, a.ld_x = x.ptr, x.ld
        if not skip_norm:
            a.gamma, a.beta = L.ptr(w.vec[name + ".weight"]), L.ptr(w.vec[name + ".bias"])
        if scale_shift is not None:
            off = scale_shift
            a.scale_shift = L.ptr(self.emb_all, off * 4)
            a.ld_ss = self.emb_all.shape[1]
            self._uses_emb()
        a.silu, a.resample, a.skip_norm = int(silu), resample, int(skip_norm)
        a.y, a.ld_y = y.ptr, y.ld
        if y_raw is not None:
            a.y_raw, a.ld_raw = y_raw.ptr, y_raw.ld
        a.stats = L.ptr(self.stats)
        if not skip_norm and self._covered(x):
            cs = self.chansum[id(x.storage)]
            a.chansum, a.ld_chansum = L.ptr(cs, x.c0 * 8), cs.shape[1]
        self.keep.append(a)
        self._op(self.lib.fidm_groupnorm_silu_nhwc, C.byref(a))

    def _fusable(self, name, H, W):
        """True if conv `name` at HxW can apply its GroupNorm+SiLU input in the operand path (K1h)."""
        if not (self.fuse_gn and self.w.tc):
            return False
        wt, _, cin_pad, cout_pad, ks = self.w.conv[name]
        return bool(self.lib.fidm_conv_gn_fusable(self.B, H, W, cin_pad, cout_pad, ks, 1))

    def _gn_coeff(self, x, name, scale_shift=None):
        """Statistics of x -> halved affine coefficients [B, C, 2] for a conv with a fused GroupNorm+SiLU operand."""
        w = self.w
        coef = torch.empty(self.B, x.channels, 2, device=w.device, dtype=torch.float32)
        a = L.GnArgs()
        a.dtype = a.y_dtype = L.dtype_code(x.storage.dtype)
        a.batch, a.height, a.width, a.channels, a.groups = self.B, x.H, x.W, x.channels, 32
        a.eps = 1e-5
        a.x, a.ld_x = x.ptr, x.ld
        a.gamma, a.beta = L.ptr(w.vec[name + ".weight"]), L.ptr(w.vec[name + ".bias"])
        if scale_shift is not None:
            a.scale_shift = L.ptr(self.emb_all, scale_shift * 4)
            a.ld_ss = self.emb_all.shape[1]
            self._uses_emb()
        a.silu = 1
        a.stats = L.ptr(self.stats)
        if self._covered(x):
            cs = self.chansum[id(x.storage)]
            a.chansum, a.ld_chansum = L.ptr(cs, x.c0 * 8), cs.shape[1]
        self.keep.append((a, coef))
        lr = self._last_reduce
        cpg = x.channels // 32
        if (lr is not None and lr[0] == len(self.ops) - 1 and lr[1:4] == (id(x.storage), x.c0, x.channels) and
                x.channels % 32 == 0 and cpg <= 32 and 32 % cpg == 0 and self.fuse_reduce_coeff):
            # x was produced by the conv just before and its statistics were folded by the previous op: redo that
            # fold together with the coefficients (one launch instead of two, identical results)
            self.ops.pop()
            _, _, c0, ch, colsum, slots, cs = lr
            self._op(self.lib.fidm_groupnorm_reduce_colsum_coeff, colsum, slots, L.ptr(cs), cs.shape[1], c0, C.byref(a),
                     L.ptr(coef), x.channels)
            self._last_reduce = None
        else:
            self._op(self.lib.fidm_groupnorm_silu_coeff, C.byref(a), L.ptr(coef), x.channels)
        return coef

    def _conv(self, name, x, y, residual=None, row_add=None, x2=None, name2=None, stride=1, nchw_out=None,
              cout_valid=None, stats=True, gn_coef=None, x_half=False, residual_half=False, halo_copy=False):
        w = self.w
        wt, bias, cin_pad, cout_pad, ks = w.conv[name]
        assert x.channels == cin_pad, (name, x.channels, cin_pad)
        a = L.ConvArgs()
        if gn_coef is None:
            assert x.storage.dtype == wt.dtype, (name, x.storage.dtype, wt.dtype)
        else:       # raw bf16 stream in; the kernel stages silu(x*A + B) in the weights' dtype
            assert x.storage.dtype == torch.bfloat16 and wt.dtype in (torch.float16, torch.bfloat16)
            a.gn_coef, a.ld_gn_coef = L.ptr(gn_coef), gn_coef.shape[1]
        # x_half (K1h only): x is the half-resolution raw stream of an `up` ResBlock; the conv runs at 2H x 2W
        Ho, Wo = (2 * x.H, 2 * x.W) if x_half else (x.H, x.W)
        assert not (x_half or residual_half) or gn_coef is not None
        a.x_half_res, a.residual_half_res = int(x_half), int(residual_half)
        a.dtype, a.batch, a.height, a.width = L.dtype_code(wt.dtype), self.B, Ho, Wo
        a.cin, a.cout, a.ksize, a.stride = cin_pad, cout_pad, ks, stride
        a.x, a.ld_x, a.w = x.ptr, x.ld, L.ptr(wt)
        # stem: one halo load per slice through the swapped-role kernel instead of one TMA box per tap, where the layer
        # fills the machine (one 16 x 16 pixel box x 128 output channels per SM)
        if (halo_copy and w.tc and ks == 3 and stride == 1 and Ho % 16 == 0 and Wo % 16 == 0 and cout_pad % 128 == 0 and
                self.B * (Ho // 16) * (Wo // 16) * (cout_pad // 128) * 100 >= 148 * 75 and
                os.environ.get("FIDM_STEM_HALO", "1") != "0"):
            a.halo_copy = 1
        use_fp8 = (gn_coef is not None and name in w.conv8 and not x_half and Ho * Wo >= self.FP8_MIN_PIXELS and
                   (x2 is None or name in w.skip8))
        if use_fp8:          # e4m3 operand x e4m3 weights (kind::f8f6f4), per-output-channel scale in the epilogue
            w8, scale = w.conv8[name]
            a.dtype, a.w, a.w_scale = L.E4M3, L.ptr(w8), L.ptr(scale)
            self.n_fp8 += 1
        if x2 is not None:
            w2 = w.skip8[name] if use_fp8 else w.conv[name2][0]
            a.x2, a.ld_x2, a.cin2, a.w2 = x2.ptr, x2.ld, x2.channels, L.ptr(w2)
        a.bias = L.ptr(bias)
        if row_add is not None:
            a.row_add = L.ptr(self.emb_all, row_add * 4)
            a.ld_row_add = self.emb_all.shape[1]
            self._uses_emb()
        if residual is not None:
            a.residual, a.ld_res = residual.ptr, residual.ld
        if nchw_out is not None:
            a.y, a.ld_y, a.y_nchw_f32 = L.ptr(nchw_out), 0, 1
        else:
            a.y, a.ld_y = y.ptr, y.ld
        a.cout_valid = cout_valid or cout_pad
        a.splitk_ws, a.splitk_ws_bytes = L.ptr(self.splitk_ws), self.splitk_ws.numel()
        self.keep.append(a)
        tc_ok = (w.tc and tc_eligible(cin_pad, cout_pad, stride, nchw_out is not None) and
                 (x2 is None or x2.channels % 64 == 0) and (stride == 1 or (ks == 3 and Ho % 2 == 0 and Wo % 2 == 0)))
        assert tc_ok or (wt.dtype != torch.float16 and gn_coef is None)
        fn = self.lib.fidm_conv2d_nhwc_bf16 if tc_ok else self.lib.fidm_conv2d_nhwc_simt
        # Fusing the consumer GroupNorm's statistics into this epilogue pays off where the separate statistics
        # pass is HBM-bound (large tensors) and the epilogue is off the critical path (long K loop); measured
        # on B200: 128^2 and larger, K >= 1152.  Small tensors keep the (L2-resident) statistics kernel.
        k_total = ks * ks * cin_pad + (x2.channels if x2 is not None else 0)
        if name == "input_blocks.0.0" and os.environ.get("FIDM_STEM_STATS", "1") != "0":
            k_total = 1152      # the stem output feeds TWO GroupNorms (first ResBlock, last skip concat): fuse its statistics
        Hy, Wy = Ho // stride, Wo // stride                      # output resolution (Ho, Wo are the INPUT's for stride 2)
        slots = self.lib.fidm_conv_colsum_slots(Hy, Wy) if (
            tc_ok and nchw_out is None and stats and self.fuse_stats and cout_pad % 64 == 0 and
            Hy * Wy >= self.FUSE_MIN_PIXELS and k_total >= 1152) else 0
        if slots > 0:
            n = self.B * slots * cout_pad * 2
            if n not in self.colsum_scratch:
                self.colsum_scratch[n] = torch.empty(n, device=w.device, dtype=torch.float32)
            a.colsum = L.ptr(self.colsum_scratch[n])
        self._op(fn, C.byref(a))
        if slots > 0:
            sid = id(y.storage)
            if sid not in self.chansum:
                self.chansum[sid] = torch.zeros(self.B, y.ld, 2, device=w.device, dtype=torch.float32)
            cs = self.chansum[sid]
            self._op(self.lib.fidm_groupnorm_reduce_colsum, a.colsum, self.B, slots, cout_pad, L.ptr(cs), y.ld, y.c0)
            self._last_reduce = (len(self.ops) - 1, sid, y.c0, cout_pad, a.colsum, slots, cs)
            self.coverage.setdefault(sid, []).append((y.c0, cout_pad))
        elif y is not None:
            # a producer without fused statistics invalidates whatever was recorded for these channels
            self.coverage[id(y.storage)] = [r for r in self.coverage.get(id(y.storage), [])
                                            if r[0] + r[1] <= y.c0 or r[0] >= y.c0 + cout_pad]

    def _attention(self, qkv, out, heads, head_dim):
        w = self.w
        a = L.AttnArgs()
        a.dtype, a.batch, a.tokens, a.heads, a.head_dim = w.code, self.B, qkv.H * qkv.W, heads, head_dim
        a.qkv, a.ld_qkv, a.out, a.ld_out = qkv.ptr, qkv.ld, out.ptr, out.ld
        self.keep.append(a)
        tc_ok = (w.tc and head_dim in (64, 128) and a.tokens % 64 == 0 and
                 hasattr(self.lib, "fidm_attention_qkv_nhwc_bf16") and Plan.TC_ATTENTION)
        fn = self.lib.fidm_attention_qkv_nhwc_bf16 if tc_ok else self.lib.fidm_attention_qkv_nhwc_simt
        self._op(fn, C.byref(a))

    TC_ATTENTION = True
    FUSE_MIN_PIXELS = int(os.environ.get("FIDM_FUSE_MIN_PIXELS", 128 * 128))
    FP8_MIN_PIXELS = int(os.environ.get("FIDM_FP8_MIN_PIXELS", 128 * 128))

    # ------------------------------------------------------------------ layers
    def _block(self, blk, x, dst):
        layers = blk.layers
        for k, layer in enumerate(layers):
            last = k == len(layers) - 1
            if layer.kind == "stem":
                y = dst
                self._conv(layer.name, x, y, halo_copy=True)
            elif layer.kind == "res":
                y = self._res(layer, x, dst if last else None)
            elif layer.kind == "attn":
                y = self._attn(layer, x, dst if last else None)
            elif layer.kind == "down":
                y = self._down(layer, x, dst if last else None)
            elif layer.kind == "up":
                y = self._up(layer, x, dst if last else None)
            else:
                raise NotImplementedError(layer.kind)
            if k > 0:
                self._release(x)          # intermediate of this block
            x = y
        return x

    def _res(self, layer, x, dst):
        """ResBlock._forward (nn.py:189-212)."""
        n, w = layer.name, self.w
        H, W = x.H, x.W
        if layer.up:
            H, W, mode = 2 * H, 2 * W, L.RESAMPLE_UP
        elif layer.down:
            H, W, mode = H // 2, W // 2, L.RESAMPLE_DOWN
        else:
            mode = L.RESAMPLE_NONE
        off = w.emb_off[n]
        xr = None
        h = None
        fuse_up = (mode == L.RESAMPLE_UP and layer.skip == "identity" and self.fuse_up and
                   self._fusable(n + ".in_layers.2", H, W) and self._fusable(n + ".out_layers.3", H, W))
        if mode == L.RESAMPLE_NONE and self._fusable(n + ".in_layers.2", H, W):
            # GroupNorm + SiLU of x applied inside the conv (K1h): no normalized tensor, no apply pass
            coef = self._gn_coeff(x, n + ".in_layers.0")
            h = self._new(H, W, layer.cout)
            self._conv(n + ".in_layers.2", x, h, row_add=None if self.ssn else off, gn_coef=coef)
        elif fuse_up:
            # `up` ResBlock: GroupNorm + SiLU + nearest 2x upsample of the half-resolution x inside the conv, and
            # x_upd (nn.py:194) read at (h/2, w/2) by the second conv's epilogue: no upsampled tensor exists
            coef = self._gn_coeff(x, n + ".in_layers.0")
            h = self._new(H, W, layer.cout)
            self._conv(n + ".in_layers.2", x, h, row_add=None if self.ssn else off, gn_coef=coef, x_half=True)
            y = dst if dst is not None else self._new(H, W, layer.cout)
            coef = self._gn_coeff(h, n + ".out_layers.0", scale_shift=off if self.ssn else None)
            self._conv(n + ".out_layers.3", h, y, gn_coef=coef, residual=x, residual_half=True)
            self._release(h)
            return y
        else:
            a1 = self._new(H, W, layer.cin, self._wdtype(n + ".in_layers.2"))
            xr = self._new(H, W, layer.cin) if mode != L.RESAMPLE_NONE else None
            self._gn(x, a1, n + ".in_layers.0", silu=True, resample=mode, y_raw=xr)
            h = self._new(H, W, layer.cout)
            self._conv(n + ".in_layers.2", a1, h, row_add=None if self.ssn else off)
            self._release(a1)
        y = dst if dst is not None else self._new(H, W, layer.cout)
        xs = xr if xr is not None else x
        skip = dict(residual=xs) if layer.skip == "identity" else dict(x2=xs, name2=n + ".skip_connection")
        if self._fusable(n + ".out_layers.3", H, W) and (layer.skip == "identity" or layer.cin % 64 == 0):
            coef = self._gn_coeff(h, n + ".out_layers.0", scale_shift=off if self.ssn else None)
            self._conv(n + ".out_layers.3", h, y, gn_coef=coef, **skip)
        else:
            a2 = self._new(H, W, layer.cout, self._wdtype(n + ".out_layers.3"))
            self._gn(h, a2, n + ".out_layers.0", silu=True, scale_shift=off if self.ssn else None)
            self._conv(n + ".out_layers.3", a2, y, **skip)
            self._release(a2)
        self._release(h)
        if xr is not None:
            self._release(xr)
        return y

    def _attn(self, layer, x, dst):
        """AttentionBlock._forward (nn.py:259-265)."""
        n, Cn = layer.name, layer.channels
        a = self._new(x.H, x.W, Cn, self._wdtype(n + ".qkv"))
        self._gn(x, a, n + ".norm", silu=False)
        qkv = self._new(x.H, x.W, 3 * Cn)
        self._conv(n + ".qkv", a, qkv, stats=False)
        self._release(a)
        o = self._new(x.H, x.W, Cn)
        self._attention(qkv, o, layer.heads, Cn // layer.heads)
        self._release(qkv)
        y = dst if dst is not None else self._new(x.H, x.W, Cn)
        self._conv(n + ".proj_out", o, y, residual=x)
        self._release(o)
        return y

    def _down(self, layer, x, dst):
        """Downsample (nn.py:115-133): conv3x3 stride 2, or 2x average pooling."""
        H, W = x.H // 2, x.W // 2
        y = dst if dst is not None else self._new(H, W, layer.channels)
        if layer.use_conv:
            self._conv(layer.name + ".op", x, y, stride=2)
        else:
            self._gn(x, y, None, silu=False, resample=L.RESAMPLE_DOWN, skip_norm=True)
        return y

    def _up(self, layer, x, dst):
        """Upsample (nn.py:92-112): nearest 2x, then optional conv3x3."""
        H, W = 2 * x.H, 2 * x.W
        if layer.use_conv:
            u = self._new(H, W, layer.channels)
            self._gn(x, u, None, silu=False, resample=L.RESAMPLE_UP, skip_norm=True)
            y = dst if dst is not None else self._new(H, W, layer.channels)
            self._conv(layer.name + ".conv", u, y)
            self._release(u)
        else:
            y = dst if dst is not None else self._new(H, W, layer.channels)
            self._gn(x, y, None, silu=False, resample=L.RESAMPLE_UP, skip_norm=True)
        return y

    # ------------------------------------------------------------------ execution
    def load_inputs(self, sources, timesteps, batch_offset=0):
        """Pack the fp32 NCHW `sources` [(tensor, channels, repeat)] (rows batch_offset .. +B) into the
        NHWC network input and copy the timesteps."""
        a = L.PackArgs()
        hw = self.H * self.W
        a.batch, a.hw, a.n_src = self.B, hw, len(sources)
        total_c = 0
        for i, (t, c, r) in enumerate(sources):
            a.src[i] = t.data_ptr() + batch_offset * c * hw * 4
            a.src_channels[i], a.src_repeat[i] = c, r
            total_c += c * r
        a.dst, a.dst_dtype = self.x_in.data_ptr(), L.dtype_code(self.x_in.dtype)
        # only the first 16 channels are rewritten per call; x_in was zero-filled at allocation
        a.ld_dst, a.c_pad = STEM_CIN_PAD, (16 if total_c <= 16 else STEM_CIN_PAD)
        L.check(self.lib.fidm_pack_nchw_to_nhwc(a, L.stream()), "pack")
        self.t_in.copy_(timesteps[batch_offset:batch_offset + self.B], non_blocking=True)

    def load_slot(self, slot, sources, c0):
        """Pack the fp32 NCHW `sources` [(tensor [1, channels, H, W], channels, repeat)] of ONE image into image `slot`
        of the network input, from channel c0 on: the pack kernel with a destination offset.  The other images, the
        channels outside the sources and the timesteps are left alone (continuous batching admits one request per slot
        while the sampler step kernel writes the state channels)."""
        a = L.PackArgs()
        hw = self.H * self.W
        a.batch, a.hw, a.n_src = 1, hw, len(sources)
        total_c = 0
        for i, (t, c, r) in enumerate(sources):
            assert t.is_contiguous() and t.dtype == torch.float32 and t.numel() == c * hw, (tuple(t.shape), c)
            a.src[i] = t.data_ptr()
            a.src_channels[i], a.src_repeat[i] = c, r
            total_c += c * r
        assert 0 <= slot < self.B and c0 + total_c <= 16, (slot, c0, total_c)
        a.dst = self.x_in.data_ptr() + (slot * hw * STEM_CIN_PAD + c0) * self.x_in.element_size()
        a.dst_dtype, a.ld_dst, a.c_pad = L.dtype_code(self.x_in.dtype), STEM_CIN_PAD, total_c
        L.check(self.lib.fidm_pack_nchw_to_nhwc(a, L.stream()), "pack")

    def _launch(self, ops):
        st = L.stream()
        for fn, args in ops:
            rc = fn(*args, st)
            if rc != 0:
                L.check(rc, fn.__name__)

    def launch_all(self, fork_time_path=False):
        """Launch the schedule on the current stream.  fork_time_path (used under graph capture): the timestep path
        (K5: embedding + three small Linears, 300 MB of weights) depends only on t, so it runs on a side stream next
        to the stem convolution and the first statistics pass and joins before its first consumer."""
        k, j = self.n_time_ops, self.first_emb_use
        if not fork_time_path or j is None or j <= k:
            return self._launch(self.ops)
        main = torch.cuda.current_stream()
        side = self._side_stream
        side.wait_stream(main)
        with torch.cuda.stream(side):
            self._launch(self.ops[:k])
        self._launch(self.ops[k:j])
        main.wait_stream(side)
        self._launch(self.ops[j:])

    def run(self):
        """Evaluate the UNet on self.x_in / self.t_in into self.out."""
        if not self.use_graph:
            self.launch_all()
            return self.out
        if self.graph is None:
            if not self._warm:
                self.launch_all()                     # sets func attributes, resolves driver entry points
                torch.cuda.current_stream().synchronize()
                self._warm = True
            g = torch.cuda.CUDAGraph()
            self._side_stream = torch.cuda.Stream()
            with torch.cuda.graph(g):
                self.launch_all(fork_time_path=os.environ.get("FIDM_FORK_TIME_PATH", "1") != "0")
            self.graph = g
        self.graph.replay()
        return self.out

    def n_launches(self):
        """Kernel launches per evaluation (groupnorm = stats + apply)."""
        n = 0
        for fn, args in self.ops:
            if fn is self.lib.fidm_groupnorm_silu_nhwc:
                n += self.lib.fidm_groupnorm_num_launches(args[0])
            elif fn is self.lib.fidm_groupnorm_silu_coeff:
                n += 1
            else:
                n += 1
        return n


class PlanGroup:
    """Two (or more) half-batch plans captured as PARALLEL branches of one CUDA graph.

    The UNet alternates tensor-pipe-bound kernels (K1 conv, K3 attention) with HBM-bound ones (K2
    GroupNorm).  Samples are independent, so the batch is split into micro-batches whose kernel chains run
    on separate streams: while one micro-batch is in a convolution the other's GroupNorm blocks co-reside
    on the same SMs (the conv CTAs use 192 threads and no more than one CTA per SM) and use the idle HBM
    bandwidth.  Results are identical to the single-plan execution (every kernel is per-sample)."""

    def __init__(self, weights: Weights, B, H, W, parts=2, use_graph=True):
        assert B % parts == 0
        self.B, self.H, self.W, self.w = B, H, W, weights
        b = B // parts
        self.out = torch.empty(B, weights.topo.out_channels, H, W, device=weights.device, dtype=torch.float32)
        self.parts = [Plan(weights, b, H, W, use_graph=False, out=self.out[i * b:(i + 1) * b]) for i in range(parts)]
        self.use_graph = use_graph
        self.graph = None
        self.pool = self                         # bench.py reads plan.pool.nbytes()

    def nbytes(self):
        return sum(p.pool.nbytes() for p in self.parts)

    def n_launches(self):
        return sum(p.n_launches() for p in self.parts)

    def load_inputs(self, sources, timesteps):
        for i, p in enumerate(self.parts):
            p.load_inputs(sources, timesteps, batch_offset=i * p.B)

    def run(self):
        if not self.use_graph:
            for p in self.parts:
                p.launch_all()
            return self.out
        if self.graph is None:
            for p in self.parts:                  # eager warm-up: func attributes, driver entry points
                p.launch_all()
            torch.cuda.current_stream().synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                main = torch.cuda.current_stream()
                fork = torch.cuda.Event()
                fork.record(main)
                joins = []
                for p in self.parts[1:]:
                    side = torch.cuda.Stream()
                    side.wait_event(fork)
                    with torch.cuda.stream(side):
                        p.launch_all()
                        ev = torch.cuda.Event()
                        ev.record(side)
                    joins.append(ev)
                self.parts[0].launch_all()
                for ev in joins:
                    main.wait_event(ev)
            self.graph = g
        self.graph.replay()
        return self.out
