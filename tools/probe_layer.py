"""Per-kernel timing of one encoder layer's operators at bench shapes (CUDA events, kernel alone, inputs far
larger than nothing-fits-in-L2 not required: each launch streams 100+ MB), sweeping the run-time tuning
switches (vit3d_set_tuning) so variants are compared in ONE process on ONE GPU.

    python tools/probe_layer.py [--batch 1024] [--d 2048] [--heads 8] [--iters 20]
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import vit3d_b200  # noqa: F401
from vit3d_b200._lib import PREC, call, lib, ptr, stream

ap = argparse.ArgumentParser()
ap.add_argument("--batch", type=int, default=1024)
ap.add_argument("--d", type=int, default=2048)
ap.add_argument("--heads", type=int, default=8)
ap.add_argument("--iters", type=int, default=20)
ap.add_argument("--json", default="")
a = ap.parse_args()
dev = "cuda:0"
L = lib()
B, S, H, d = a.batch, 65, 256, a.d
M = B * S
bf = torch.bfloat16
HBM = 6464.9e9


def timeit(fn, iters=a.iters):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e3      # us


def linear(x, w, wl, b, res, y, pre, act, N, K):
    yf = y.dtype == torch.float32
    call("vit3d_linear_fwd", ptr(x), K, 0, ptr(w), ptr(wl), ptr(b), ptr(res), ptr(y), int(yf), ptr(pre), act, M, N, K,
         PREC["bf16"], stream())


results = {}


def report(name, us, flops, bytes_):
    results[name] = {"us": round(us, 2), "tflops": round(flops / us / 1e6, 1), "hbm_gbs": round(bytes_ / us / 1e3, 1),
                     "hbm_frac": round(bytes_ / (us * 1e-6) / HBM, 3)}
    print(f"{name:44s} {us:8.1f} us  {flops / us / 1e6:7.1f} TFLOP/s  {bytes_ / us / 1e3:7.1f} GB/s ({bytes_ / (us * 1e-6) / HBM:.0%} HBM)")


xn = (torch.randn(M, H, device=dev) * 0.8).to(bf)
x32 = torch.randn(M, H, device=dev)
gamma = torch.ones(H, device=dev)
beta = torch.zeros(H, device=dev)


def mk(N, K):
    w = torch.randn(N, K, device=dev) / K ** 0.5
    return w, w.to(bf), torch.randn(N, device=dev) * 0.01


w_qkv, wl_qkv, b_qkv = mk(3 * H, H)
w_o, wl_o, b_o = mk(H, H)
w1, wl1, b1 = mk(d, H)
w2, wl2, b2 = mk(H, d)
qkv = torch.empty(M, 3 * H, device=dev, dtype=bf)
ctx = torch.empty(M, H, device=dev, dtype=bf)
probs = torch.empty(B, a.heads, S, S, device=dev)
h = torch.empty(M, d, device=dev, dtype=bf)
pre = torch.empty(M, d, device=dev, dtype=bf)
y32 = torch.empty(M, H, device=dev)
yn = torch.empty(M, H, device=dev, dtype=bf)
mean = torch.empty(M, device=dev)
rstd = torch.empty(M, device=dev)

def gemm_suite():
    report("qkv GEMM", timeit(lambda: linear(xn, w_qkv, wl_qkv, b_qkv, None, qkv, None, 0, 3 * H, H)),
           2.0 * M * 3 * H * H, M * H * 2 + M * 3 * H * 2)
    report("fc1 GEMM + GELU", timeit(lambda: linear(xn, w1, wl1, b1, None, h, None, 1, d, H)),
           2.0 * M * d * H, M * H * 2 + M * d * 2)
    report("fc1 GEMM + GELU + pre (training)", timeit(lambda: linear(xn, w1, wl1, b1, None, h, pre, 1, d, H)),
           2.0 * M * d * H, M * H * 2 + 2 * M * d * 2)
    report("fc1 GEMM + bias, no act", timeit(lambda: linear(xn, w1, wl1, b1, None, h, None, 0, d, H)),
           2.0 * M * d * H, M * H * 2 + M * d * 2)
    report("out-proj GEMM + residual", timeit(lambda: linear(ctx, w_o, wl_o, b_o, x32, y32, None, 0, H, H)),
           2.0 * M * H * H, M * H * 2 + 2 * M * H * 4)
    report("fc2 GEMM + residual", timeit(lambda: linear(h, w2, wl2, b2, x32, y32, None, 0, H, d)),
           2.0 * M * d * H, M * d * 2 + 2 * M * H * 4)
    if L.vit3d_linear_ln_supported(M, H, H):
        report("out-proj GEMM + residual + LN (fused)",
               timeit(lambda: call("vit3d_linear_ln_fwd", ptr(ctx), ptr(wl_o), ptr(b_o), ptr(x32), ptr(y32), ptr(gamma),
                                   ptr(beta), 1e-6, ptr(yn), None, None, M, H, H, stream())),
               2.0 * M * H * H, M * H * 2 + 2 * M * H * 4 + M * H * 2)
        report("fc2 GEMM + residual + LN (fused)",
               timeit(lambda: call("vit3d_linear_ln_fwd", ptr(h), ptr(wl2), ptr(b2), ptr(x32), ptr(y32), ptr(gamma),
                                   ptr(beta), 1e-6, ptr(yn), None, None, M, H, d, stream())),
               2.0 * M * d * H, M * d * 2 + 2 * M * H * 4 + M * H * 2)


# tuning keys (include/vit3d.h): 1 attention threads, 5 fused-MLP weight multicast
gemm_suite()
w2h = w2.to(torch.float16)
for pair in (0, 1):
    L.vit3d_set_tuning(5, pair)
    tag = f"[multicast pair={pair}]"
    report(f"fused MLP (fc1+GELU+fc2+res) {tag}",
           timeit(lambda: call("vit3d_mlp_fwd", ptr(xn), ptr(wl1), ptr(b1), ptr(w2h), ptr(b2), ptr(x32), ptr(y32), M, H, d,
                               stream())), 4.0 * M * d * H, M * H * 2 + 2 * M * H * 4)
    report(f"fused MLP + LN {tag}",
           timeit(lambda: call("vit3d_mlp_ln_fwd", ptr(xn), ptr(wl1), ptr(b1), ptr(w2h), ptr(b2), ptr(x32), ptr(y32),
                               ptr(gamma), ptr(beta), 1e-6, ptr(yn), M, H, d, stream())),
           4.0 * M * d * H, M * H * 2 + 2 * M * H * 4 + M * H * 2)
L.vit3d_set_tuning(5, 0)
vol = torch.randn(B, 1, 128, 128, 5, device=dev)
wp = torch.randn(H, 1, 16, 16, 5, device=dev) * 0.02
bp = torch.randn(H, device=dev) * 0.01
cls = torch.randn(1, 1, H, device=dev) * 0.02
pos = torch.randn(1, 65, H, device=dev) * 0.02
tok = torch.empty(B, 65, H, device=dev)
report("patch embedding (TF32, TMA im2col)",
       timeit(lambda: call("vit3d_patch_embed_fwd", ptr(vol), ptr(wp), ptr(bp), ptr(cls), ptr(pos), ptr(tok), B, 128, 128, 5,
                           16, 16, 5, H, PREC["bf16"], None, 0, stream())),
       2.0 * B * 64 * 1280 * H, B * 327680 + B * 65 * H * 4)
report("fused MLP + final LN (fp32 out only)",
       timeit(lambda: call("vit3d_mlp_lnf_fwd", ptr(xn), ptr(wl1), ptr(b1), ptr(w2h), ptr(b2), ptr(x32), ptr(gamma), ptr(beta),
                           1e-6, ptr(y32), M, H, d, stream())), 4.0 * M * d * H, M * H * 2 + 2 * M * H * 4)
report("LayerNorm fp32 -> bf16",
       timeit(lambda: call("vit3d_ln_fwd", ptr(x32), ptr(gamma), ptr(beta), ptr(yn), 1, ptr(mean), ptr(rstd), M, H, 1e-6,
                           stream())), 8.0 * M * H, M * H * 4 + M * H * 2)
qkv.copy_((torch.randn(M, 3 * H, device=dev) * 0.5).to(bf))
D = H // a.heads
for thr in (512, 640):
    L.vit3d_set_tuning(1, thr)
    for vis in (1, 0):
        report(f"attention fwd vis={vis} [threads={thr}]",
               timeit(lambda: call("vit3d_attn_fwd", ptr(qkv), ptr(ctx), ptr(probs) if vis else None, B, S, a.heads, D,
                                   PREC["bf16"], stream())),
               4.0 * B * S * S * H, M * 4 * H * 2 + (B * a.heads * S * S * 4 if vis else 0))
L.vit3d_set_tuning(1, 0)
if a.json:
    json.dump(results, open(a.json, "w"), indent=1)
