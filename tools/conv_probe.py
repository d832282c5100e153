"""Sustained TFLOP/s of conv shapes (tensor-core kernel) under the power cap."""
import math, os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
import fidm_b200 as F
from fidm_b200 import ops
dev = "cuda:0"

def run(name, B, H, W, Cin, Cout, ks, dtype=torch.bfloat16, seconds=2.0):
    x = torch.randn(B, H, W, Cin, device=dev).to(dtype)
    w = ops.repack_weight(torch.randn(Cout, Cin, ks, ks, device=dev) / math.sqrt(Cin * ks * ks), dtype)
    b = torch.zeros(Cout, device=dev)
    y = torch.empty(B, H, W, Cout, device=dev, dtype=torch.bfloat16)
    for _ in range(3):
        ops.conv2d(x, w, b, out=y, impl="tc")
    torch.cuda.synchronize()
    n = 0
    t0 = time.time()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    while time.time() - t0 < seconds:
        for _ in range(20):
            ops.conv2d(x, w, b, out=y, impl="tc")
        n += 20
        torch.cuda.synchronize()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    fl = 2.0 * B * H * W * Cin * Cout * ks * ks
    print(f"{name:46s} {ms*1e3:9.1f} us  {fl/ms/1e9:8.1f} TFLOP/s", flush=True)

def run_halo(name, B, H, W, Cin, Cout, seconds=2.0):
    """the same layer with GroupNorm+SiLU applied in the operand path (K1h): raw bf16 in, no separate norm pass"""
    x = torch.randn(B, H, W, Cin, device=dev).bfloat16()
    w = ops.repack_weight(torch.randn(Cout, Cin, 3, 3, device=dev) / math.sqrt(Cin * 9), torch.float16)
    b = torch.zeros(Cout, device=dev)
    y = torch.empty(B, H, W, Cout, device=dev, dtype=torch.bfloat16)
    coef = ops.groupnorm_silu_coeff(x, torch.ones(Cin, device=dev), torch.zeros(Cin, device=dev))
    for _ in range(3):
        ops.conv2d(x, w, b, out=y, impl="tc", gn_coef=coef)
    torch.cuda.synchronize()
    n = 0
    t0 = time.time()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    while time.time() - t0 < seconds:
        for _ in range(20):
            ops.conv2d(x, w, b, out=y, impl="tc", gn_coef=coef)
        n += 20
        torch.cuda.synchronize()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    fl = 2.0 * B * H * W * Cin * Cout * 9
    print(f"{name:46s} {ms*1e3:9.1f} us  {fl/ms/1e9:8.1f} TFLOP/s", flush=True)


if "--halo" in sys.argv:
    secs = 0.5 if "--quick" in sys.argv else 2.0
    run("3x3 256->256 @256^2 B8 fp16 (K1, normalized in)", 8, 256, 256, 256, 256, 3, torch.float16, secs)
    run_halo("3x3 256->256 @256^2 B8 (K1h, GN fused)", 8, 256, 256, 256, 256, secs)
    run_halo("3x3 512->256 @256^2 B8 (K1h, GN fused)", 8, 256, 256, 512, 256, secs)
    run_halo("3x3 256->256 @128^2 B8 (K1h, GN fused)", 8, 128, 128, 256, 256, secs)
    run_halo("3x3 512->512 @128^2 B8 (K1h, GN fused)", 8, 128, 128, 512, 512, secs)
    run_halo("3x3 512->512 @64^2 B8 (K1h, GN fused)", 8, 64, 64, 512, 512, secs)
    run_halo("3x3 128->128 @256^2 B8 (K1h, GN fused)", 8, 256, 256, 128, 128, secs)
    sys.exit(0)

run("3x3 256->256 @256^2 B8 (K=2304)", 8, 256, 256, 256, 256, 3)
run("1x1 2304->256 @256^2 B8 (pure GEMM, K=2304)", 8, 256, 256, 2304, 256, 1)
run("3x3 512->256 @256^2 B8 (K=4608)", 8, 256, 256, 512, 256, 3)
run("3x3 512->512 @128^2 B8", 8, 128, 128, 512, 512, 3)
run("3x3 512->512 @64^2 B8", 8, 64, 64, 512, 512, 3)
run("3x3 1024->1024 @16^2 B8", 8, 16, 16, 1024, 1024, 3)
run("3x3 1024->1024 @8^2 B8", 8, 8, 8, 1024, 1024, 3)
