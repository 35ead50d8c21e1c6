"""Gradient with respect to the input volume (d loss / d x through the patch embedding, the Conv3d data gradient):
the C entry vit3d_patch_embed_dgrad against fp64, and x.grad of the per-operator path, the fused BF16 training step,
a frozen-parameter saliency pass and the ensemble against autograd over the oracle in fp64.

Tolerances (relative L2 norm): the kernel 1e-5 in fp32 mode, 2e-3 in TF32 / BF16 mode (TF32 operands); the models
use the parameter-gradient tolerances of the low-precision parity tests (fp32 2e-3, TF32 0.02, BF16 0.08)."""
import functools

import pytest
import torch

import vit3d_b200
from oracle import vit3d_oracle as O
from tests.helpers import case_setup, load_golden, unpack_masks
from vit3d_b200 import _lib, functional as F, fused_train
from vit3d_b200._lib import PREC, call, ptr, stream
from vit3d_b200.models.modeling import TransformerEnsemble, VisionTransformer

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
H_KERNEL = 256


def relerr(got, want):
    want = want.double()
    return float((got.detach().double().cpu() - want).norm() / want.norm())


def launches():
    return _lib.lib().vit3d_launch_count()


@functools.lru_cache(maxsize=2)
def kernel_case(shape, patch, B):
    """Seeded dtokens / filter bank and the fp64 data gradient: (dtok[:, 1:] @ W) scattered by the inverse of
    oracle.patch_gather (its autograd backward: a pure permutation, 0 where no patch covers a voxel)."""
    X, Y, Z = shape
    gen = torch.Generator().manual_seed(1000 * B + X + patch[0])
    P = (X // patch[0]) * (Y // patch[1]) * (Z // patch[2])
    dtok = torch.randn(B, P + 1, H_KERNEL, generator=gen)
    w = torch.randn(H_KERNEL, 1, *patch, generator=gen) * 0.05
    xx = torch.zeros(B, 1, X, Y, Z, dtype=torch.float64, requires_grad=True)
    dp = dtok[:, 1:].double() @ w.double().reshape(H_KERNEL, -1)
    O.patch_gather(xx, patch).backward(dp)
    return dtok, w, xx.grad


GEOMETRIES = [
    ((128, 128, 5), (16, 16, 5)),     # the reference geometry: tensor-core path in BF16 / TF32 mode
    ((128, 128, 5), (8, 8, 5)),       # P = 256 (shipped_p8): generic path
    ((130, 130, 5), (16, 16, 5)),     # uncovered remainder (Conv3d drops 2 rows and 2 columns): generic path
]


@pytest.mark.parametrize("prec", ["fp32", "tf32", "bf16"])
@pytest.mark.parametrize("B", [1, 2, 3, 64, 257, 1024])
@pytest.mark.parametrize("geom", GEOMETRIES, ids=["p16", "p8", "remainder"])
def test_patch_embed_dgrad_kernel_vs_fp64(geom, B, prec):
    (X, Y, Z), patch = geom
    p0, p1, p2 = patch
    dtok, w, want = kernel_case((X, Y, Z), patch, B)
    dtok_d, w_d = dtok.to(DEV), w.to(DEV)
    pid = PREC[prec]
    wsb = _lib.lib().vit3d_patch_embed_ws_bytes(B, X, Y, Z, p0, p1, p2, H_KERNEL, pid)
    ws = torch.empty(wsb, device=DEV, dtype=torch.uint8)
    w_t = F.lp_weight(w_d, "tf32_t") if prec != "fp32" else None
    assert w_t is None or w_t.shape == (p0 * p1 * p2, H_KERNEL)
    dx = torch.full((B, 1, X, Y, Z), float("nan"), device=DEV)      # every voxel must be written
    n0 = launches()
    call("vit3d_patch_embed_dgrad", ptr(dtok_d), ptr(w_d), ptr(w_t), ptr(dx), B, X, Y, Z, p0, p1, p2, H_KERNEL, pid,
         ptr(ws), wsb, stream())
    n = launches() - n0
    got = dx.cpu()
    assert torch.isfinite(got).all()
    tol = 1e-5 if prec == "fp32" else 2e-3
    assert relerr(got, want) <= tol, (prec, B, relerr(got, want))
    if X % p0 or Y % p1:
        assert (got[:, :, X - X % p0:] == 0).all() and (got[:, :, :, Y - Y % p1:] == 0).all()
    # path coverage: one tcgen05 launch in BF16 mode, TF32 rounding + tcgen05 in TF32 mode; the exact fp32 path is
    # patch-row compaction + FMA GEMM + inverse im2col
    tc = prec != "fp32" and patch == (16, 16, 5) and X == 128
    assert n == ({"bf16": 1, "tf32": 2}[prec] if tc else 3), (prec, patch, n)


def test_patch_embed_dgrad_empty_batch_and_bad_arguments():
    w = torch.randn(H_KERNEL, 1, 16, 16, 5, device=DEV)
    wsb = _lib.lib().vit3d_patch_embed_ws_bytes(0, 128, 128, 5, 16, 16, 5, H_KERNEL, PREC["bf16"])
    ws = torch.empty(wsb, device=DEV, dtype=torch.uint8)
    dx = torch.empty(0, 1, 128, 128, 5, device=DEV)
    dtok = torch.empty(0, 65, H_KERNEL, device=DEV)
    w_t = F.lp_weight(w, "tf32_t")
    n0 = launches()
    call("vit3d_patch_embed_dgrad", ptr(dtok), ptr(w), ptr(w_t), ptr(dx), 0, 128, 128, 5, 16, 16, 5, H_KERNEL, PREC["bf16"],
         ptr(ws), wsb, stream())
    assert launches() == n0
    with pytest.raises(vit3d_b200.Vit3dError):
        call("vit3d_patch_embed_dgrad", ptr(dtok), ptr(w), None, ptr(dx), 1, 128, 128, 5, 16, 16, 5, H_KERNEL,
             PREC["fp32"], ptr(ws), 16, stream())


# ----------------------------------------------------------------------------- models
def build(name, prec):
    cfg, sd, x, y, w = case_setup(name)
    m = VisionTransformer(cfg, 128, zero_head=True, num_classes=1, precision=prec)
    m.load_state_dict(sd)
    return cfg, sd, m.to(DEV), x, y, w


@pytest.mark.parametrize("name,prec,tol", [("tiny", "fp32", 2e-3), ("conf5", "fp32", 2e-3), ("shipped_p8", "fp32", 2e-3),
                                           ("tiny", "tf32", 0.02), ("conf5", "tf32", 0.02),
                                           ("tiny", "bf16", 0.08), ("conf5", "bf16", 0.08)])
def test_model_input_grad_per_operator_path(name, prec, tol):
    cfg, sd, m, x, y, w = build(name, prec)
    m.eval()
    F._STATE["fused_train"] = False
    try:
        m(x.to(DEV), y.to(DEV), w).backward()          # warm-up: weight shadows are built once
        if prec != "fp32":
            F.lp_weight(m.transformer.embeddings.patch_embeddings.weight, "tf32_t")
        m.zero_grad(set_to_none=True)
        n0 = launches()
        m(x.to(DEV), y.to(DEV), w).backward()
        n_plain = launches() - n0
        ref = {k: p.grad.clone() for k, p in m.named_parameters()}
        m.zero_grad(set_to_none=True)
        xg = x.to(DEV).requires_grad_()
        n0 = launches()
        m(xg, y.to(DEV), w).backward()
        n_dx = launches() - n0
    finally:
        F._STATE["fused_train"] = True
    _, _, dxo = O.vit_loss_and_grads(sd, cfg, x, y, w, dtype=torch.float64)
    assert xg.grad is not None and xg.grad.shape == x.shape and xg.grad.dtype == torch.float32
    assert relerr(xg.grad, dxo) <= tol, (name, prec, relerr(xg.grad, dxo))
    tc = prec != "fp32" and cfg.hidden_size == 256 and cfg.patches["size"][0] == 16
    assert n_dx - n_plain == ({"bf16": 1, "tf32": 2}[prec] if tc else 3), (n_plain, n_dx)
    # the parameter gradients take the same kernels on the same inputs whether or not x needs a gradient (their
    # split-K reductions use fp32 atomics, so two runs agree to rounding, not necessarily bit for bit; the key.bias
    # gradients are 0 in exact arithmetic, hence the floor relative to the largest gradient)
    gscale = max(float(v.norm()) for v in ref.values())
    for k, p in m.named_parameters():
        a, b = p.grad, ref[k]
        err = float((a - b).norm())
        assert err <= 1e-5 * float(b.norm()) + 1e-6 * gscale, (k, err, float(b.norm()))


def test_fused_training_step_input_grad_eval_mode():
    cfg, sd, m, x, y, w = build("conf5", "bf16")
    m.eval()
    xd = x.to(DEV)
    assert fused_train.supported(m, xd)
    m(xd, y.to(DEV), w).backward()                  # warm-up: weight shadows are built once
    F.lp_weight(m.transformer.embeddings.patch_embeddings.weight, "tf32_t")
    n0 = launches()
    m(xd, y.to(DEV), w).backward()
    n_plain = launches() - n0
    xg = xd.clone().requires_grad_()
    n0 = launches()
    loss = m(xg, y.to(DEV), w)
    assert type(loss.grad_fn).__name__.startswith("VitTrainFn")
    loss.backward()
    assert launches() - n0 == n_plain + 1           # the tcgen05 data-gradient kernel
    _, _, dxo = O.vit_loss_and_grads(sd, cfg, x, y, w, dtype=torch.float64)
    assert relerr(xg.grad, dxo) <= 0.08, relerr(xg.grad, dxo)


def test_fused_training_step_input_grad_with_reference_dropout_masks():
    g = load_golden("conf5")
    cfg, sd, m, x, y, w = build("conf5", "bf16")
    masks = unpack_masks(g)
    sites = {0: masks["emb"].reshape(-1)}
    for i in range(cfg.transformer["num_layers"]):
        sites[1 + 2 * i] = masks[("fc1", i)].reshape(-1)
        sites[2 + 2 * i] = masks[("fc2", i)].reshape(-1)
    m.train()
    xg = x.to(DEV).requires_grad_()
    assert fused_train.supported(m, xg)
    with F.mask_injection(sites):
        loss = m(xg, y.to(DEV), w)
        assert type(loss.grad_fn).__name__.startswith("VitTrainFn")
        loss.backward()
    _, _, dxo = O.vit_loss_and_grads(sd, cfg, x, y, w, masks=masks, dtype=torch.float64)
    assert relerr(xg.grad, dxo) <= 0.08, relerr(xg.grad, dxo)


@pytest.mark.parametrize("prec,tol", [("fp32", 2e-3), ("tf32", 0.02), ("bf16", 0.08)])
def test_frozen_parameter_saliency(prec, tol):
    cfg, sd, m, x, _, _ = build("conf5", prec)
    m.eval()
    for p in m.parameters():
        p.requires_grad_(False)
    xg = x.to(DEV).requires_grad_()
    m(xg)[0].sum().backward()
    assert all(p.grad is None for p in m.parameters())
    p64 = O.to_dtype(sd, torch.float64)
    xx = x.double().requires_grad_()
    O.vit_forward(p64, cfg, xx)[0].sum().backward()
    assert relerr(xg.grad, xx.grad) <= tol, relerr(xg.grad, xx.grad)


@pytest.mark.parametrize("prec,tol", [("fp32", 2e-3), ("bf16", 0.08)])
def test_ensemble_input_grad(prec, tol):
    cfgs = [vit3d_b200.north_star_config(c) for c in (5, 9, 11)]
    members_sd = [O.init_state_dict(c, seed=42 + j) for j, c in enumerate(cfgs)]
    sd = O.ensemble_state_dict(members_sd, seed=7)
    members = [VisionTransformer(c, 128, zero_head=True, num_classes=1, precision=prec) for c in cfgs]
    ens = TransformerEnsemble(*members, in_features=1)
    ens.load_state_dict(sd)
    ens.to(DEV).eval()
    x = O.synth_volumes(3, seed=42, kind="img")
    xg = x.to(DEV).requires_grad_()
    ens(xg).sum().backward()
    xx = x.double().requires_grad_()
    O.ensemble_forward(O.to_dtype(sd, torch.float64), cfgs, xx).sum().backward()
    assert relerr(xg.grad, xx.grad) <= tol, relerr(xg.grad, xx.grad)
