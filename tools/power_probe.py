"""Sustained (seconds-long) behaviour of the hot kernels under the 1 kW cap: time per launch, power, SM clock."""
import math
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pynvml
import torch

import fidm_b200 as F
from fidm_b200 import ops

pynvml.nvmlInit()
h = pynvml.nvmlDeviceGetHandleByIndex(0)


class Sampler:
    def __init__(self):
        self.p, self.c, self.stop = [], [], threading.Event()
        self.th = threading.Thread(target=self.run, daemon=True)

    def run(self):
        while not self.stop.is_set():
            self.p.append(pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0)
            self.c.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
            time.sleep(0.02)

    def __enter__(self):
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.th.join()


def sustained(name, fn, seconds=3.0, work=None, unit=""):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    n = 0
    with Sampler() as s:
        t0 = time.time()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        while time.time() - t0 < seconds:
            for _ in range(20):
                fn()
            n += 20
            torch.cuda.synchronize()
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    half = len(s.p) // 2
    pw = sum(s.p[half:]) / max(1, len(s.p) - half)
    ck = sum(s.c[half:]) / max(1, len(s.c) - half)
    rate = f"{work / ms / 1e9:.1f} {unit}" if work else ""
    print(f"{name:42s} {ms * 1e3:9.1f} us/launch  {rate:>16s}  power {pw:6.0f} W  sm {ck:6.0f} MHz", flush=True)


dev = "cuda:0"
B, H, W, Cc = 8, 256, 256, 256
x16 = torch.randn(B, H, W, Cc, device=dev).half()
xb = torch.randn(B, H, W, Cc, device=dev).bfloat16()
w16 = ops.repack_weight(torch.randn(Cc, Cc, 3, 3, device=dev) / math.sqrt(Cc * 9), torch.float16)
wb = ops.repack_weight(torch.randn(Cc, Cc, 3, 3, device=dev) / math.sqrt(Cc * 9), torch.bfloat16)
bias = torch.zeros(Cc, device=dev)
y = torch.empty(B, H, W, Cc, device=dev, dtype=torch.bfloat16)
yh = torch.empty(B, H, W, Cc, device=dev, dtype=torch.float16)
gamma = torch.ones(Cc, device=dev)
beta = torch.zeros(Cc, device=dev)
flops = 2.0 * B * H * W * Cc * Cc * 9
nbytes = B * H * W * Cc * 2
sustained("conv 3x3 256->256 @256^2 fp16 operands", lambda: ops.conv2d(x16, w16, bias, out=y, impl="tc"), work=flops, unit="TFLOP/s")
sustained("conv 3x3 256->256 @256^2 bf16 operands", lambda: ops.conv2d(xb, wb, bias, out=y, impl="tc"), work=flops, unit="TFLOP/s")
a = torch.randn(8192, 8192, device=dev).bfloat16()
b = torch.randn(8192, 8192, device=dev).bfloat16()
sustained("torch.matmul bf16 8192^3 (cuBLAS)", lambda: torch.matmul(a, b), work=2.0 * 8192 ** 3, unit="TFLOP/s")
sustained("groupnorm+silu apply+stats (bf16->fp16)", lambda: ops.groupnorm_silu(xb, gamma, beta, out=yh), work=3 * nbytes, unit="GB/s x1e-3")
sustained("copy_ bf16 268 MB", lambda: y.copy_(xb), work=2 * nbytes, unit="GB/s x1e-3")
cfg = F.CONFIGS["ADM256"]
from fidm_b200.utils.synth import synth_batch, synth_state_dict
m = F.DiffusionInpaintingModel(F.UNetModel(**dict(cfg, in_channels=3)))
m.load_state_dict(synth_state_dict(cfg, seed=0), strict=True)
m.to(dev)
data = synth_batch(B, 256, seed=1, device=dev)
xin = torch.randn(B, 3, 256, 256, device=dev)
tt = torch.full((B,), 50, device=dev)
sustained("ADM256 UNet eval batch 8", lambda: m(xin, tt, masked_image=data["masked_image"], mask=data["mask"]), seconds=5.0,
          work=2241.48e9 * B, unit="TFLOP/s")
