"""Times the data gradient of the patch embedding (d tokens / d x, written into the volume) at the reference geometry
(128 x 128 x 5 volumes, 16 x 16 x 5 patches, hidden 256), CUDA events over 20 calls after 5 warm-up calls, on rotating
dtokens / dx buffers whose total exceeds the 126 MB L2:

  tcgen05    vit3d_patch_embed_dgrad in BF16 mode: one TF32 tcgen05 kernel that stores straight into dx
  composed   the alternative built from existing pieces: tensor-core vit3d_linear_fwd (bf16 dY x bf16 transposed filter
             bank -> fp32 dpatches), then the inverse-im2col scatter.  The bf16 compaction of dY is NOT timed (in the
             composition's favour); the scatter's time is that of its kernel in the fp32 path (torch.profiler, separate run;
             the scatter is an ordinary launch, so its span does not include a PDL wait for its predecessor)
  fp32       vit3d_patch_embed_dgrad in FP32 mode (patch-row compaction + FMA GEMM + scatter)

Achieved bandwidth counts the bytes the product needs: dx written (B*X*Y*Z*4) + the patch rows of dtokens read
(B*P*H*4).  The card's name and power limit are printed with the numbers.

    python tools/probe_patch_dgrad.py [--batches 256 1024]
"""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from vit3d_b200 import functional as F  # noqa: E402
from vit3d_b200._lib import PREC, call, lib, ptr, stream  # noqa: E402

X, Y, Z, PATCH, H = 128, 128, 5, (16, 16, 5), 256
L2_BYTES = 126 << 20


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # pragma: no cover
        pl = f"unknown ({e})"
    return f"{name}, power limit / max SM clock: {pl}"


def timed(fn, n_sets, reps=20, warm=5):
    for i in range(warm):
        fn(i % n_sets)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(reps):
        fn(i % n_sets)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3      # us per call


def kernel_us(fn, name_part, n_sets, reps=10):
    """Mean device time of the kernels whose name contains name_part, from torch.profiler."""
    for i in range(3):
        fn(i % n_sets)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for i in range(reps):
            fn(i % n_sets)
        torch.cuda.synchronize()
    rows = [r for r in prof.key_averages() if name_part in r.key and r.count > 0]
    if not rows:
        raise RuntimeError(f"no kernel named *{name_part}* in the profile")
    # per-launch mean of each matching kernel (a kernel may be listed more than once per launch)
    return sum(r.self_device_time_total / r.count for r in rows)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[256, 1024])
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    print(card())
    p0, p1, p2 = PATCH
    P = (X // p0) * (Y // p1) * (Z // p2)
    Kp = p0 * p1 * p2
    w = torch.randn(H, 1, *PATCH, device=dev) * 0.05
    w_t = F.lp_weight(w, "tf32_t")
    w_t_bf16 = F.lp_weight(w.reshape(H, Kp), "bf16_t")       # [Kp, H] bf16
    for B in args.batches:
        per_set = B * (P + 1) * H * 4 + B * X * Y * Z * 4
        n_sets = max(2, -(-2 * L2_BYTES // per_set))
        dtoks = [torch.randn(B, P + 1, H, device=dev) for _ in range(n_sets)]
        dxs = [torch.empty(B, 1, X, Y, Z, device=dev) for _ in range(n_sets)]
        dys = [torch.randn(B * P, H, device=dev).to(torch.bfloat16) for _ in range(n_sets)]
        dps = [torch.empty(B * P, Kp, device=dev) for _ in range(n_sets)]
        wsb = lib().vit3d_patch_embed_ws_bytes(B, X, Y, Z, p0, p1, p2, H, PREC["bf16"])
        ws = torch.empty(wsb, device=dev, dtype=torch.uint8)
        nbytes = B * X * Y * Z * 4 + B * P * H * 4

        def dgrad(prec):
            def fn(i):
                call("vit3d_patch_embed_dgrad", ptr(dtoks[i]), ptr(w), ptr(w_t if prec != "fp32" else None), ptr(dxs[i]),
                     B, X, Y, Z, p0, p1, p2, H, PREC[prec], ptr(ws), wsb, stream())
            return fn

        def linear(i):
            call("vit3d_linear_fwd", ptr(dys[i]), H, 0, ptr(w_t_bf16), ptr(w_t_bf16), None, None, ptr(dps[i]), 1, None, 0,
                 B * P, Kp, H, PREC["bf16"], stream())

        # correctness of what is timed: the tcgen05 result against the exact fp32 path
        dgrad("fp32")(0)
        ref = dxs[0].clone()
        dgrad("bf16")(0)
        rel = float((dxs[0] - ref).norm() / ref.norm())

        us_tc = timed(dgrad("bf16"), n_sets)
        us_lin = timed(linear, n_sets)
        us_fp32 = timed(dgrad("fp32"), n_sets)
        us_scatter = kernel_us(dgrad("fp32"), "patch_scatter", n_sets)
        floor = nbytes / 7.7e12 * 1e6
        print(f"B={B:5d}  bytes {nbytes / 1e6:7.1f} MB  ({n_sets} rotating sets, {n_sets * per_set / 1e6:.0f} MB)  "
              f"HBM floor at 7.7 TB/s: {floor:6.1f} us   tcgen05 vs fp32 rel. L2 {rel:.1e}")
        print(f"  tcgen05 dgrad      {us_tc:8.1f} us  {nbytes / us_tc / 1e3:6.0f} GB/s")
        print(f"  composed           {us_lin + us_scatter:8.1f} us  {nbytes / (us_lin + us_scatter) / 1e3:6.0f} GB/s   "
              f"(linear_fwd {us_lin:.1f} us + scatter {us_scatter:.1f} us)")
        print(f"  fp32 generic path  {us_fp32:8.1f} us  {nbytes / us_fp32 / 1e3:6.0f} GB/s")
        del dtoks, dxs, dys, dps, ws
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
