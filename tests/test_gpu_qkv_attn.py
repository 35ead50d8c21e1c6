"""The fused q|k|v projection + attention kernel (vit3d_qkv_attn_fwd, BF16 inference) against the two-kernel path it
replaces - vit3d_linear_fwd into a packed qkv matrix, then vit3d_attn_fwd / vit3d_attn_fwd_padded - and against fp64."""
import math

import pytest
import torch

import vit3d_b200
from oracle import vit3d_oracle as O
from vit3d_b200._lib import ACT_NONE, PREC, call, lib, ptr, stream
from vit3d_b200.graphs import GraphedInference
from vit3d_b200.models.modeling import VisionTransformer

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
S, H = 65, 256


def two_kernel(yn, w32, w, b, heads, vis):
    B = yn.shape[0]
    qkv = torch.empty(B, S, 3 * H, device=DEV, dtype=torch.bfloat16)
    call("vit3d_linear_fwd", ptr(yn), H, 0, ptr(w32), ptr(w), ptr(b), None, ptr(qkv), 0, None, ACT_NONE, B * S, 3 * H, H,
         PREC["bf16"], stream())
    ctx = torch.full((B, S, H), float("nan"), device=DEV, dtype=torch.bfloat16)
    if vis:
        probs = torch.full((B, heads, S, 72), float("nan"), device=DEV)
        call("vit3d_attn_fwd_padded", ptr(qkv), ptr(ctx), ptr(probs), 72, B, S, heads, H // heads, stream())
    else:
        probs = None
        call("vit3d_attn_fwd", ptr(qkv), ptr(ctx), None, B, S, heads, H // heads, PREC["bf16"], stream())
    return qkv, ctx, probs


def fused(yn, w, b, heads, vis):
    B = yn.shape[0]
    ctx = torch.full((B, S, H), float("nan"), device=DEV, dtype=torch.bfloat16)
    probs = torch.full((B, heads, S, 72), float("nan"), device=DEV) if vis else None
    call("vit3d_qkv_attn_fwd", ptr(yn), ptr(w), ptr(b), ptr(ctx), ptr(probs), 72, B, S, heads, H // heads, stream())
    return ctx, probs


@pytest.mark.parametrize("heads", [8, 16])
@pytest.mark.parametrize("B", [1, 2, 3, 64, 257, 1024])
@pytest.mark.parametrize("vis", [True, False])
def test_qkv_attn_equals_two_kernel_path(heads, B, vis):
    assert lib().vit3d_qkv_attn_supported(S, heads, H // heads) == 1
    g = torch.Generator().manual_seed(B * 7 + heads)
    yn = torch.randn(B, S, H, generator=g).to(DEV, torch.bfloat16)
    w32 = (torch.randn(3 * H, H, generator=g) / 16).to(DEV)
    w = w32.to(torch.bfloat16)
    b = (torch.randn(3 * H, generator=g) * 0.1).to(DEV)
    qkv, ctx0, probs0 = two_kernel(yn, w32, w, b, heads, vis)
    ctx1, probs1 = fused(yn, w, b, heads, vis)
    torch.cuda.synchronize()
    assert torch.equal(ctx0, ctx1)
    if vis:
        assert torch.equal(probs0[..., :S], probs1[..., :S])
        assert bool((probs1[..., S:] == 0).all())

    # fp64 attention over the fp64 projection of the same bf16 inputs: ctx within bf16 rounding, probabilities within
    # the rounding of q and k to bf16
    D = H // heads
    q, k, v = ((yn.double() @ w.double().t() + b.double())[..., i * H:(i + 1) * H].view(B, S, heads, D).permute(0, 2, 1, 3)
               for i in range(3))
    p = torch.softmax(q @ k.transpose(-1, -2) / math.sqrt(D), dim=-1)
    ref = (p @ v).permute(0, 2, 1, 3).reshape(B, S, H)
    assert (ctx1.double() - ref).abs().max().item() < 3e-2 * max(1.0, ref.abs().max().item())
    if vis:
        assert (probs1[..., :S].double() - p).abs().max().item() < 2e-2


def test_qkv_attn_support():
    """Head groups are 32 q|k|v columns wide: head dimensions 16 and 32; 64 (4 heads) keeps the two kernels."""
    assert [lib().vit3d_qkv_attn_supported(S, k, H // k) for k in (4, 8, 16)] == [0, 1, 1]
    assert lib().vit3d_qkv_attn_supported(64, 8, 32) == 0


def _conf5_launches(train):
    cfg = vit3d_b200.north_star_config(5)
    m = VisionTransformer(cfg, 128, zero_head=True, num_classes=1, vis=True, precision="bf16").to(DEV)
    x = O.synth_volumes(2, seed=3).to(DEV)
    if train:
        m.train()
        n0 = lib().vit3d_launch_count()
        logits, _, _ = m(x)
        n = lib().vit3d_launch_count() - n0
        return n, None
    m.eval()
    g = GraphedInference(m)
    logits, weights, _ = g(x)
    with torch.no_grad():
        eager = m(x)
    assert all(torch.equal(a, b) for a, b in zip(weights, eager[1]))
    assert len(weights) == 6 and weights[0].shape == (2, 8, S, S)
    return g.launches_per_replay, weights


def test_conf5_inference_launches():
    """conf 5 in BF16 mode: one kernel per layer for q|k|v and attention (22 launches per replayed step, 28 before);
    the training forward keeps the projection and the attention core as separate kernels (its backward needs qkv)."""
    n, _ = _conf5_launches(train=False)
    assert n == 22, n
    n_train, _ = _conf5_launches(train=True)
    assert n_train > 28, n_train
