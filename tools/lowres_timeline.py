"""Timeline of ONE launch of the K1 kernel (conv_tc) on a low-resolution layer: %globaltimer stamps written by the
kernel when a probe buffer is set (fidm_conv_set_profile_buffer), per CTA, first work unit only.  Answers where the
~8 us of a low-resolution launch go (prologue, first operand round trip, K loop, split-K fold, store)."""
import math
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch

import fidm_b200 as F  # noqa: F401
from fidm_b200 import _lib as L
from fidm_b200 import ops

dev = "cuda:0"
# stamps 7 / 8: partial tile written to the workspace / past the cluster barrier (cluster split-K) or arrival counted
# (FIDM_CONV_SPLIT_CLUSTER=0); 9 / 10 only exist on the workspace-fold and unsplit paths
NAMES = ["entry", "setup done", "first TMA issued", "last TMA issued", "first stage full", "last MMA issued",
         "accumulator ready", "partial parked", "barrier passed", "fold loaded", "TMA store issued", "epilogue done",
         "exit"]


def timeline(B, H, Cin, Cout, ks=3):
    x = torch.randn(B, H, H, Cin, device=dev).half()
    w = ops.repack_weight(torch.randn(Cout, Cin, ks, ks, device=dev) / math.sqrt(Cin * ks * ks), torch.float16)
    b = torch.zeros(Cout, device=dev)
    y = torch.empty(B, H, H, Cout, device=dev, dtype=torch.bfloat16)
    flush = torch.empty(256 << 20, device=dev, dtype=torch.uint8)
    for _ in range(3):
        ops.conv2d(x, w, b, out=y, impl="tc")
    prof = torch.zeros(32 * 148, device=dev, dtype=torch.int64)
    rows = []
    for cold in (False, True):
        if cold:
            flush.zero_()
        torch.cuda.synchronize()
        prof.zero_()
        L.lib().fidm_conv_set_profile_buffer(L.ptr(prof))
        ops.conv2d(x, w, b, out=y, impl="tc")
        torch.cuda.synchronize()
        L.lib().fidm_conv_set_profile_buffer(None)
        pr = prof.view(148, 32).cpu()
        geo = int(pr[0, 14])
        grid, bn, S = geo >> 32, (geo >> 8) & 0xFFFF, geo & 0xFF
        pr = pr[:grid]
        t0 = int(pr[:, 0].min())
        fin = pr[:, 13] == 1 if S > 1 else torch.ones(grid, dtype=torch.bool)
        print(f"conv{ks}x{ks} {Cin}->{Cout} @{H}^2 B{B}  grid {grid}  N tile {bn}  split {S}  "
              f"{'weights cold (L2 flushed)' if cold else 'weights warm in L2'}")
        for i, nm in enumerate(NAMES):
            col = pr[:, i]
            sel = col[(col > 0) & (fin if i in (9, 10) else torch.ones(grid, dtype=torch.bool))]
            if sel.numel() == 0:
                continue
            rel = (sel - t0).double() / 1e3
            print(f"   {nm:20s} min {rel.min():6.2f}  median {rel.median():6.2f}  max {rel.max():6.2f} us   (n={sel.numel()})")
        for i, nm in ((16, "producer: start"), (17, "producer: indices")):
            col = pr[:, i]
            rel = (col[col > 0] - t0).double() / 1e3
            if rel.numel():
                print(f"   {nm:24s} min {rel.min():6.2f}  median {rel.median():6.2f}  max {rel.max():6.2f} us")
        rows.append((pr[:, 12].max() - t0).item() / 1e3)
    return rows


SHAPES = [(8, 512, 512, 3), (16, 512, 512, 3), (8, 1024, 1024, 3), (16, 1024, 1024, 3), (32, 512, 512, 3),
          (32, 512, 1536, 1)]
if len(sys.argv) > 1:
    SHAPES = SHAPES[:int(sys.argv[1])]
for B in (1, 8):
    for H, ci, co, ks in SHAPES:
        timeline(B, H, ci, co, ks)
