"""Time the fused q|k|v projection + attention kernel against the two kernels it replaces (vit3d_linear_fwd, then
vit3d_attn_fwd_padded / vit3d_attn_fwd), BF16 mode, with CUDA events.  Every timed call reads its own yn from a rotation
of input copies whose total exceeds the 126 MB L2, so the inputs come from HBM as they do in the model."""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import vit3d_b200  # noqa: F401  (registers the package path)
from vit3d_b200._lib import ACT_NONE, PREC, call, ptr, stream

ap = argparse.ArgumentParser()
ap.add_argument("--batches", default="256,1024")
ap.add_argument("--heads", type=int, default=8)
ap.add_argument("--iters", type=int, default=50)
a = ap.parse_args()
dev = "cuda:0"
S, H = 65, 256
D = H // a.heads
print(torch.cuda.get_device_name(0))
w32 = torch.randn(3 * H, H, device=dev) / 16
w = w32.to(torch.bfloat16)
b = torch.randn(3 * H, device=dev) * 0.1
for B in [int(x) for x in a.batches.split(",")]:
    n_in = max(2, -(-160 * 2**20 // (B * S * H * 2)))
    yns = [torch.randn(B, S, H, device=dev).to(torch.bfloat16) for _ in range(n_in)]
    qkv = torch.empty(B, S, 3 * H, device=dev, dtype=torch.bfloat16)
    ctx = torch.empty(B, S, H, device=dev, dtype=torch.bfloat16)
    for vis in (1, 0):
        probs = torch.empty(B, a.heads, S, 72, device=dev) if vis else None

        def two(yn):
            call("vit3d_linear_fwd", ptr(yn), H, 0, ptr(w32), ptr(w), ptr(b), None, ptr(qkv), 0, None, ACT_NONE, B * S,
                 3 * H, H, PREC["bf16"], stream())
            if vis:
                call("vit3d_attn_fwd_padded", ptr(qkv), ptr(ctx), ptr(probs), 72, B, S, a.heads, D, stream())
            else:
                call("vit3d_attn_fwd", ptr(qkv), ptr(ctx), None, B, S, a.heads, D, PREC["bf16"], stream())

        def one(yn):
            call("vit3d_qkv_attn_fwd", ptr(yn), ptr(w), ptr(b), ptr(ctx), ptr(probs), 72, B, S, a.heads, D, stream())

        res = {}
        for name, fn in (("two-kernel", two), ("fused", one), ("two-kernel ", two), ("fused ", one)):
            for i in range(3):
                fn(yns[i % n_in])
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(a.iters):
                fn(yns[i % n_in])
            e1.record()
            torch.cuda.synchronize()
            res.setdefault(name.strip(), []).append(e0.elapsed_time(e1) / a.iters * 1e3)
        byts = B * S * H * 2 * 2 + (B * a.heads * S * 72 * 4 if vis else 0)     # yn in, ctx (+ probabilities) out
        f = min(res["fused"])
        print(f"B={B} heads={a.heads} vis={vis}: two-kernel {min(res['two-kernel']):.1f} us, fused {f:.1f} us "
              f"({byts / f / 1e3:.0f} GB/s of the {byts / 1e6:.1f} MB the fused kernel must move)")
