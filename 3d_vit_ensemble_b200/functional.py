"""torch.autograd.Function wrappers over the C ABI (one Function per operator of the path).

PyTorch is used for device memory, streams and autograd bookkeeping only; every
arithmetic operation is a kernel of libvit3d_sm100.so.  Reference line numbers cite
evapachetti/3d_vit_ensemble `models/modeling.py`.
"""
from __future__ import annotations

import os
import weakref
from typing import Optional

import torch

from . import _lib
from ._lib import ACT_GELU, ACT_NONE, PREC, call, ptr, stream

_STATE = {"precision": os.environ.get("VIT3D_PRECISION", "bf16"), "step": 0, "mask_override": None}


def set_precision(p: str) -> None:
    """'fp32' (exact FMA path), 'tf32' or 'bf16' (tcgen05 paths); default for new models."""
    if p not in PREC:
        raise ValueError(f"unknown precision {p!r}; choose from {list(PREC)}")
    _STATE["precision"] = p


def get_precision() -> str:
    return _STATE["precision"]


def act_dtype(prec: str) -> torch.dtype:
    return torch.bfloat16 if prec == "bf16" else torch.float32


def next_dropout_step() -> int:
    _STATE["step"] += 1
    return _STATE["step"]


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise _lib.Vit3dError("vit3d operators run on CUDA tensors only (no CPU fallback); "
                                  "move the model and its inputs to a cuda device")


def _c(t):
    return t if t.is_contiguous() else t.contiguous()


def enable_direct_grads(on: bool = True) -> None:
    """When on, backward kernels accumulate a parameter's gradient straight into its existing `.grad`
    (e.g. a view of optim.FlatArena's flat buffer) and hand autograd `None` for it - no zero-filled
    temporary and no extra add per parameter.  Turned on by the fused optimizers / GradReducer; leave it
    off if you call torch.autograd.grad() for parameter gradients."""
    _STATE["direct_grads"] = bool(on)


def _grad_target(p):
    """The tensor a parameter gradient can be accumulated into in place, or None."""
    if not _STATE.get("direct_grads") or not isinstance(p, torch.nn.Parameter):
        return None
    g = p.grad
    if g is None or g.dtype != torch.float32 or g.device != p.device or not g.is_contiguous() or g.shape != p.shape:
        return None
    return g


def _grad_done(p):
    hook = _STATE.get("grad_hook")
    if hook is not None:
        hook(p)


# bf16 shadow copies of fp32 master weights (parameters only), refreshed when the parameter
# changes (optimizer step / load_state_dict bump _version, .to() changes data_ptr).  Keyed by the
# parameter object itself so that a freed-and-reallocated address can never alias a stale copy.
_LP_CACHE = {}   # id(param) -> (weakref(param), version, data_ptr, bf16 copy, epoch)


def invalidate_weight_shadows() -> None:
    """Call after weights were modified by a kernel torch does not know about (fused optimizers)."""
    _STATE["epoch"] = _STATE.get("epoch", 0) + 1


def lp_weight(w: torch.Tensor, prec: str = "bf16") -> torch.Tensor:
    """bf16 copy (BF16 mode) or TF32-rounded fp32 copy (TF32 mode) of an fp32 weight; "bf16_t" / "tf32_t": the same,
    transposed to [K, N] (K = product of the trailing dimensions)."""
    cacheable = isinstance(w, torch.nn.Parameter)
    if cacheable:
        ent = _LP_CACHE.get((id(w), prec))
        if (ent is not None and ent[0]() is w and ent[1] == w._version and ent[2] == w.data_ptr()
                and ent[4] == _STATE.get("epoch", 0)):
            return ent[3]
    if prec == "bf16":
        out = torch.empty(w.shape, dtype=torch.bfloat16, device=w.device)
        call("vit3d_cast_f32_to_bf16", ptr(w.detach()), ptr(out), w.numel(), stream())
    elif prec == "f16":             # fp16 shadow (fc2 weight of the fused MLP)
        out = torch.empty(w.shape, dtype=torch.float16, device=w.device)
        call("vit3d_cast_f32_to_f16", ptr(w.detach()), ptr(out), w.numel(), stream())
    elif prec == "bf16_t":          # transposed bf16 shadow [K,N] of a [N,K] weight: dgrad operand
        out = torch.empty(w.shape[1], w.shape[0], dtype=torch.bfloat16, device=w.device)
        call("vit3d_transpose_f32_to_bf16", ptr(w.detach()), ptr(out), w.shape[0], w.shape[1], stream())
    elif prec == "tf32_t":          # transposed TF32 shadow [K,N] of an [N,...] weight: patch-embedding dgrad operand
        out = lp_weight(w, "tf32").reshape(w.shape[0], -1).t().contiguous()
    else:
        out = torch.empty(w.shape, dtype=torch.float32, device=w.device)
        call("vit3d_round_tf32", ptr(w.detach()), ptr(out), w.numel(), stream())
    if cacheable:
        key = (id(w), prec)
        _LP_CACHE[key] = (weakref.ref(w, lambda _r, key=key: _LP_CACHE.pop(key, None)), w._version, w.data_ptr(), out,
                          _STATE.get("epoch", 0))
    return out


# ----------------------------------------------------------------------------- a1
class PatchEmbedFn(torch.autograd.Function):
    """Conv3d(kernel=stride=patch) + flatten/transpose + cls concat + position add
    (Embeddings.forward, modeling.py:162-173) as one gather-GEMM."""

    @staticmethod
    def forward(ctx, x, w, bias, cls, pos, prec):
        _need_cuda(x, w, bias, cls, pos)
        ctx.x_dtype = x.dtype
        x = _c(x.float())
        B, Cc, X, Y, Z = x.shape
        if Cc != 1:
            raise _lib.Vit3dError("patch embedding expects a single input channel")
        H = w.shape[0]
        p0, p1, p2 = w.shape[2:]
        P = (X // p0) * (Y // p1) * (Z // p2)
        if pos.shape[1] != P + 1:
            raise _lib.Vit3dError(f"position_embeddings has {pos.shape[1]} rows, input gives {P + 1} tokens")
        tokens = torch.empty(B, P + 1, H, device=x.device, dtype=torch.float32)
        pid = PREC[prec]
        wsb = _lib.lib().vit3d_patch_embed_ws_bytes(B, X, Y, Z, p0, p1, p2, H, pid)
        ws = torch.empty(wsb, device=x.device, dtype=torch.uint8)
        # BF16 and TF32 modes run the embedding on the tensor cores in TF32: give it round-to-nearest weights
        # (TF32 mode also rounds the volume first; fp32 mode uses the exact fp32 embedding, see vit3d_patch_embed_fwd)
        w_use = lp_weight(w, "tf32") if (prec in ("bf16", "tf32") and w.is_contiguous()) else _c(w)
        call("vit3d_patch_embed_fwd", ptr(x), ptr(w_use), ptr(_c(bias)), ptr(_c(cls)), ptr(_c(pos)), ptr(tokens),
             B, X, Y, Z, p0, p1, p2, H, pid, ptr(ws), wsb, stream())
        ctx.save_for_backward(x)
        ctx.meta = (w.shape, cls.shape, pos.shape, prec)
        ctx.params = (w, bias, cls, pos)
        return tokens

    @staticmethod
    def backward(ctx, dtok):
        (x,) = ctx.saved_tensors
        wshape, cshape, pshape, prec = ctx.meta
        B, _, X, Y, Z = x.shape
        H, _, p0, p1, p2 = wshape
        dev = x.device
        pid = PREC[prec]
        wsb = _lib.lib().vit3d_patch_embed_ws_bytes(B, X, Y, Z, p0, p1, p2, H, pid)
        ws = torch.empty(wsb, device=dev, dtype=torch.uint8)
        dtok = _c(dtok.float())
        grads = [None] * 6
        if any(ctx.needs_input_grad[1:5]):
            targets = [_grad_target(p) for p in ctx.params]
            direct = all(t is not None for t in targets)
            if direct:
                dw, db, dcls, dpos = targets
            else:
                dw = torch.zeros(wshape, device=dev)
                db = torch.zeros(H, device=dev)
                dcls = torch.zeros(cshape, device=dev)
                dpos = torch.zeros(pshape, device=dev)
            call("vit3d_patch_embed_bwd", ptr(x), ptr(dtok), ptr(dw), ptr(db), ptr(dcls), ptr(dpos),
                 B, X, Y, Z, p0, p1, p2, H, pid, ptr(ws), wsb, stream())
            if direct:
                for p in ctx.params:
                    _grad_done(p)
            else:
                grads[1:5] = dw, db, dcls, dpos
        if ctx.needs_input_grad[0]:
            # d tokens / d x (Conv3d data gradient): BF16 and TF32 modes hand the tensor-core kernel the transposed
            # TF32-rounded filter bank, fp32 mode takes the exact path from the master weight
            w = ctx.params[0]
            w_t = lp_weight(w, "tf32_t") if (prec in ("bf16", "tf32") and w.is_contiguous()) else None
            dx = torch.empty(x.shape, device=dev, dtype=torch.float32)
            call("vit3d_patch_embed_dgrad", ptr(dtok), ptr(_c(w.detach())), ptr(w_t), ptr(dx), B, X, Y, Z, p0, p1, p2, H,
                 pid, ptr(ws), wsb, stream())
            grads[0] = dx.to(ctx.x_dtype)
        return tuple(grads)


def u8_volumes_to_f32(x_u8: torch.Tensor, mean: float) -> torch.Tensor:
    """N2: uint8 volumes (as stored on disk, create_dataset.py:46-59) -> fp32 minus the training mean
    (tools.py:18-26), on the device; 4x less host->device traffic than shipping fp32 volumes."""
    _need_cuda(x_u8)
    x_u8 = _c(x_u8)
    y = torch.empty(x_u8.shape, device=x_u8.device, dtype=torch.float32)
    call("vit3d_u8_to_f32", ptr(x_u8), ptr(y), x_u8.numel(), float(mean), stream())
    return y


def patch_gather(x: torch.Tensor, patch) -> torch.Tensor:
    """Bit-exact im2col permutation used by the embedding (for tests / inspection)."""
    _need_cuda(x)
    x = _c(x.float())
    B, _, X, Y, Z = x.shape
    p0, p1, p2 = patch
    P = (X // p0) * (Y // p1) * (Z // p2)
    out = torch.empty(B, P, p0 * p1 * p2, device=x.device)
    call("vit3d_patch_gather", ptr(x), ptr(out), B, X, Y, Z, p0, p1, p2, stream())
    return out


# ----------------------------------------------------------------------------- LayerNorm
class LayerNormFn(torch.autograd.Function):
    """nn.LayerNorm(H, eps) forward/backward (modeling.py:189,194,253)."""

    @staticmethod
    def forward(ctx, x, gamma, beta, eps, out_mode):
        """out_mode: 0 fp32, 1 bf16, 2 fp32 rounded to TF32 (operand of a TF32 GEMM)."""
        _need_cuda(x, gamma, beta)
        x = _c(x.float())
        H = x.shape[-1]
        M = x.numel() // H
        out_mode = int(out_mode)
        od = torch.bfloat16 if out_mode == 1 else torch.float32
        y = torch.empty(x.shape, device=x.device, dtype=od)
        mean = torch.empty(M, device=x.device)
        rstd = torch.empty(M, device=x.device)
        call("vit3d_ln_fwd", ptr(x), ptr(_c(gamma)), ptr(_c(beta)), ptr(y), out_mode, ptr(mean),
             ptr(rstd), M, H, float(eps), stream())
        ctx.save_for_backward(x, gamma, mean, rstd)
        ctx.params = (gamma, beta)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, gamma, mean, rstd = ctx.saved_tensors
        H = x.shape[-1]
        M = x.numel() // H
        dy = _c(dy.float())
        dx = torch.empty_like(x)
        tg, tb = _grad_target(ctx.params[0]), _grad_target(ctx.params[1])
        direct = tg is not None and tb is not None
        dg = tg if direct else torch.zeros_like(gamma)
        db = tb if direct else torch.zeros_like(gamma)
        call("vit3d_ln_bwd", ptr(dy), ptr(x), ptr(mean), ptr(rstd), ptr(_c(gamma)), None, ptr(dx), ptr(dg), ptr(db),
             M, H, stream())
        if direct:
            _grad_done(ctx.params[0])
            _grad_done(ctx.params[1])
            return dx, None, None, None, None
        return dx, dg, db, None, None


# ----------------------------------------------------------------------------- Linear
class LinearFn(torch.autograd.Function):
    """y = act(x W^T + b) (+ residual): nn.Linear at modeling.py:63-67,105-106,277 with the GELU
    (modeling.py:120) and the residual add (modeling.py:191,196) folded into the epilogue."""

    @staticmethod
    def forward(ctx, x, w, b, residual, act, prec, out_f32, drop=None):
        """drop = (p, seed, site, step): Dropout applied to the activation output (modeling.py:121); its
        backward is folded into the GELU backward kernel."""
        _need_cuda(x, w, b, residual)
        N, K = w.shape
        lead = x.shape[:-1]
        ad = act_dtype(prec)
        if x.dtype not in (torch.float32, torch.bfloat16) or (x.dtype == torch.bfloat16 and prec != "bf16"):
            x = x.float()
        if x.dim() == 2 and x.stride(1) == 1 and x.stride(0) >= K:
            x2, ldx = x, x.stride(0)           # strided rows (the head reads token 0 of each volume)
        else:
            x2, ldx = _c(x).reshape(-1, K), K
        M = x2.shape[0]
        yd = torch.float32 if (residual is not None or out_f32) else ad
        y = torch.empty(M, N, device=x.device, dtype=yd)
        # the pre-activation is only needed by the GELU backward: inference (no_grad) does not write it
        pre = torch.empty(M, N, device=x.device, dtype=yd) if (act == ACT_GELU and any(ctx.needs_input_grad)) else None
        shadow = prec in ("bf16", "tf32")
        w_obj = w
        w_lp = lp_weight(w, prec) if (shadow and w.is_contiguous()) else None
        w = _c(w)
        if shadow and w_lp is None:
            w_lp = lp_weight(w, prec)
        res = None if residual is None else _c(residual.float()).reshape(M, N)
        call("vit3d_linear_fwd", ptr(x2), ldx, int(x2.dtype == torch.float32), ptr(w), ptr(w_lp),
             ptr(None if b is None else _c(b)), ptr(res), ptr(y), int(yd == torch.float32), ptr(pre), act, M, N, K,
             PREC[prec], stream())
        ctx.drop = None
        if drop is not None:
            p_, seed_, site_, step_ = drop
            call("vit3d_dropout", ptr(y), None, ptr(y), y.numel(), int(yd == torch.float32), float(p_), seed_, site_,
                 step_, ptr(_STATE.get("step_dev")), stream())
            ctx.drop = drop
        ctx.save_for_backward(x2, w, w_lp, pre)
        ctx.w_obj = w_obj if (prec == "bf16" and w_obj.is_contiguous() and w_obj.dim() == 2) else None
        ctx.params = (w_obj, b)
        ctx.meta = (ldx, act, prec, b is not None, residual is not None, x.shape, x.dtype)
        return y.reshape(*lead, N)

    @staticmethod
    def backward(ctx, dy):
        x2, w, w_lp, pre = ctx.saved_tensors
        ldx, act, prec, has_b, has_res, xshape, xdtype = ctx.meta
        N, K = w.shape
        M = x2.shape[0]
        dy2 = _c(dy).reshape(M, N)
        d_res = dy2.reshape(*xshape[:-1], N) if has_res else None
        if act == ACT_GELU:
            if dy2.dtype != pre.dtype:
                dy2 = dy2.to(pre.dtype)
            dh = torch.empty_like(pre)
            pid = PREC["fp32"] if pre.dtype == torch.float32 else PREC["bf16"]
            if ctx.drop is not None:
                p_, seed_, site_, step_ = ctx.drop
                fused = (pre.dtype == torch.bfloat16 and dh.numel() % 8 == 0 and dy2.data_ptr() % 16 == 0
                         and pre.data_ptr() % 16 == 0 and dh.data_ptr() % 16 == 0)
                if fused:       # dropout' and gelu' in one pass over the [M, mlp_dim] gradient
                    call("vit3d_gelu_dropout_bwd", ptr(dy2), ptr(pre), ptr(dh), dh.numel(), pid, float(p_), seed_,
                         site_, step_, ptr(_STATE.get("step_dev")), stream())
                else:
                    tmp = torch.empty_like(dy2)
                    call("vit3d_dropout", ptr(dy2), None, ptr(tmp), dy2.numel(), int(dy2.dtype == torch.float32),
                         float(p_), seed_, site_, step_, ptr(_STATE.get("step_dev")), stream())
                    call("vit3d_gelu_bwd", ptr(tmp), ptr(pre), ptr(dh), dh.numel(), pid, stream())
            else:
                # gelu'(pre) * dy
                call("vit3d_gelu_bwd", ptr(dy2), ptr(pre), ptr(dh), dh.numel(), pid, stream())
            dy2 = dh
        need_dx = ctx.needs_input_grad[0]
        dx = torch.empty(M, K, device=dy.device, dtype=x2.dtype) if need_dx else None
        tw = _grad_target(ctx.params[0]) if ctx.needs_input_grad[1] else None
        tb = _grad_target(ctx.params[1]) if (has_b and ctx.needs_input_grad[2]) else None
        dw = tw if tw is not None else (torch.zeros_like(w) if ctx.needs_input_grad[1] else None)
        db = tb if tb is not None else (torch.zeros(N, device=dy.device) if (has_b and ctx.needs_input_grad[2]) else None)
        w_t = None
        if prec == "bf16":
            # tensor-core backward wants bf16 operands: the residual-stream gradient arrives fp32
            if dy2.dtype == torch.float32 and x2.dtype == torch.bfloat16:
                dyb = torch.empty(M, N, device=dy.device, dtype=torch.bfloat16)
                call("vit3d_cast_f32_to_bf16", ptr(dy2), ptr(dyb), dy2.numel(), stream())
                dy2 = dyb
            if need_dx and dy2.dtype == torch.bfloat16:
                w_t = lp_weight(ctx.w_obj if ctx.w_obj is not None else w, "bf16_t")
        call("vit3d_linear_bwd", ptr(dy2), int(dy2.dtype == torch.float32), ptr(x2), ldx,
             int(x2.dtype == torch.float32), ptr(w), ptr(w_t), ptr(dx), K, int(x2.dtype == torch.float32), ptr(dw),
             ptr(db), M, N, K, PREC[prec], stream())
        if dx is not None:
            dx = dx.reshape(xshape).to(xdtype)
        if tw is not None:
            _grad_done(ctx.params[0])
            dw = None
        if tb is not None:
            _grad_done(ctx.params[1])
            db = None
        return dx, dw, db, d_res, None, None, None, None


def mlp_fused_supported(M: int, H: int, d: int) -> bool:
    return bool(_lib.lib().vit3d_mlp_supported(M, H, d))


def mlp_fused(xn, w1, b1, w2, b2, residual):
    """Inference-only fused fc1 -> GELU -> fc2 (+ residual): the [M, d] intermediate never reaches HBM.
    xn: bf16 LayerNorm output (..., H); residual fp32 (..., H); returns fp32 (..., H).  No autograd."""
    _need_cuda(xn, w1, b1, w2, b2, residual)
    H = xn.shape[-1]
    d = w1.shape[0]
    x2 = _c(xn).reshape(-1, H)
    if x2.dtype != torch.bfloat16:
        x2 = x2.to(torch.bfloat16)
    M = x2.shape[0]
    res = _c(residual.float()).reshape(M, H)
    out = torch.empty(M, H, device=xn.device, dtype=torch.float32)
    call("vit3d_mlp_fwd", ptr(x2), ptr(lp_weight(w1, "bf16")), ptr(_c(b1)), ptr(lp_weight(w2, "f16")), ptr(_c(b2)),
         ptr(res), ptr(out), M, H, d, stream())
    return out.reshape(residual.shape)


def mlp_fused_ln(xn, w1, b1, w2, b2, residual, ln_weight, ln_bias, eps):
    """Inference-only fused `y = residual + fc2(GELU(fc1(xn)))` and `yn = LayerNorm(y)` (the next Block's
    attention_norm) in one kernel.  Returns (y fp32, yn bf16).  No autograd."""
    _need_cuda(xn, w1, b1, w2, b2, residual, ln_weight, ln_bias)
    H = xn.shape[-1]
    d = w1.shape[0]
    x2 = _c(xn).reshape(-1, H)
    if x2.dtype != torch.bfloat16:
        x2 = x2.to(torch.bfloat16)
    M = x2.shape[0]
    res = _c(residual.float()).reshape(M, H)
    out = torch.empty(M, H, device=xn.device, dtype=torch.float32)
    yn = torch.empty(M, H, device=xn.device, dtype=torch.bfloat16)
    call("vit3d_mlp_ln_fwd", ptr(x2), ptr(lp_weight(w1, "bf16")), ptr(_c(b1)), ptr(lp_weight(w2, "f16")), ptr(_c(b2)),
         ptr(res), ptr(out), ptr(_c(ln_weight)), ptr(_c(ln_bias)), float(eps), ptr(yn), M, H, d, stream())
    return out.reshape(residual.shape), yn.reshape(residual.shape)


def mlp_fused_final_ln(xn, w1, b1, w2, b2, residual, ln_weight, ln_bias, eps):
    """Inference-only: the last Block's MLP with the encoder's final LayerNorm folded in (modeling.py:196, :253).
    Returns `LayerNorm(residual + fc2(GELU(fc1(xn))))` as fp32; the un-normalised sum is never written."""
    _need_cuda(xn, w1, b1, w2, b2, residual, ln_weight, ln_bias)
    H = xn.shape[-1]
    d = w1.shape[0]
    x2 = _c(xn).reshape(-1, H)
    if x2.dtype != torch.bfloat16:
        x2 = x2.to(torch.bfloat16)
    M = x2.shape[0]
    res = _c(residual.float()).reshape(M, H)
    out = torch.empty(M, H, device=xn.device, dtype=torch.float32)
    call("vit3d_mlp_lnf_fwd", ptr(x2), ptr(lp_weight(w1, "bf16")), ptr(_c(b1)), ptr(lp_weight(w2, "f16")), ptr(_c(b2)),
         ptr(res), ptr(_c(ln_weight)), ptr(_c(ln_bias)), float(eps), ptr(out), M, H, d, stream())
    return out.reshape(residual.shape)


def mlp_fused_ln_supported(M: int, H: int, d: int) -> bool:
    return bool(_lib.lib().vit3d_mlp_ln_supported(M, H, d))


def linear(x, w, b=None, residual=None, act=ACT_NONE, prec=None, out_f32=False, drop=None):
    return LinearFn.apply(x, w, b, residual, act, prec or get_precision(), out_f32, drop)


def linear_ln_supported(x, w, prec) -> bool:
    """Can `linear_ln` run?  (inference only: BF16 mode, bf16 input, 256 output features)"""
    if prec != "bf16" or torch.is_grad_enabled() or not x.is_cuda or x.dtype != torch.bfloat16:
        return False
    N, K = w.shape
    return bool(_lib.lib().vit3d_linear_ln_supported(x.numel() // K, N, K))


def linear_ln(x, w, b, residual, ln_weight, ln_bias, eps):
    """Inference-only fused `y = x W^T + b + residual; yn = LayerNorm(y)` (modeling.py:190-194: the residual
    add followed by the next LayerNorm): one tcgen05 GEMM whose epilogue owns whole rows.  x bf16 (..., K),
    residual fp32 (..., N).  Returns (y fp32, yn bf16).  No autograd."""
    _need_cuda(x, w, b, residual, ln_weight, ln_bias)
    N, K = w.shape
    x2 = _c(x).reshape(-1, K)
    M = x2.shape[0]
    res = _c(residual.float()).reshape(M, N)
    y = torch.empty(M, N, device=x.device, dtype=torch.float32)
    yn = torch.empty(M, N, device=x.device, dtype=torch.bfloat16)
    call("vit3d_linear_ln_fwd", ptr(x2), ptr(lp_weight(w, "bf16")), ptr(None if b is None else _c(b)), ptr(res), ptr(y),
         ptr(_c(ln_weight)), ptr(_c(ln_bias)), float(eps), ptr(yn), None, None, M, N, K, stream())
    return y.reshape(residual.shape), yn.reshape(residual.shape)


# packed q|k|v weight of an Attention module for inference: built once per weight version instead of a
# torch.cat + bf16 cast on every forward (training keeps the cat: autograd splits the gradient through it)
_QKV_CACHE = {}   # id(query.weight) -> (weakref, versions, ptrs, epoch, packed fp32 weight, packed bias, lp shadow)


def packed_qkv(attn, prec: str):
    ws = (attn.query.weight, attn.key.weight, attn.value.weight)
    bs = (attn.query.bias, attn.key.bias, attn.value.bias)
    sig = (tuple(t._version for t in ws + bs), tuple(t.data_ptr() for t in ws + bs), _STATE.get("epoch", 0), prec)
    key = id(ws[0])
    ent = _QKV_CACHE.get(key)
    if ent is not None and ent[0]() is ws[0] and ent[1] == sig:
        return ent[2], ent[3], ent[4]
    with torch.no_grad():
        w = torch.cat([t.detach() for t in ws], dim=0).contiguous()
        b = torch.cat([t.detach() for t in bs], dim=0).contiguous()
    w_lp = lp_weight(w, prec) if prec in ("bf16", "tf32") else None
    _QKV_CACHE[key] = (weakref.ref(ws[0], lambda _r, key=key: _QKV_CACHE.pop(key, None)), sig, w, b, w_lp)
    return w, b, w_lp


def linear_packed(x, w, b, w_lp, prec):
    """Inference-only Linear with a caller-supplied low-precision weight shadow (no autograd)."""
    _need_cuda(x, w, b)
    N, K = w.shape
    lead = x.shape[:-1]
    ad = act_dtype(prec)
    if x.dtype != ad:
        x = x.to(ad)
    x2 = _c(x).reshape(-1, K)
    M = x2.shape[0]
    y = torch.empty(M, N, device=x.device, dtype=ad)
    call("vit3d_linear_fwd", ptr(x2), K, int(ad == torch.float32), ptr(w), ptr(w_lp), ptr(b), None, ptr(y),
         int(ad == torch.float32), None, ACT_NONE, M, N, K, PREC[prec], stream())
    return y.reshape(*lead, N)


# ----------------------------------------------------------------------------- attention core
class AttnCoreFn(torch.autograd.Function):
    """softmax(q k^T / sqrt(D)) v per (volume, head) (modeling.py:83-96) on the packed qkv matrix."""

    @staticmethod
    def forward(ctx, qkv, heads, vis, prec):
        _need_cuda(qkv)
        B, S, A3 = qkv.shape
        A = A3 // 3
        D = A // heads
        ad = act_dtype(prec)
        qkv = _c(qkv.to(ad))
        out = torch.empty(B, S, A, device=qkv.device, dtype=ad)
        probs = None
        if vis and prec == "bf16" and _lib.lib().vit3d_attn_padded_supported(S, heads, D):
            # rows padded to 72 floats (9 whole 32-byte sectors): sector-aligned stores; callers get the [..., :S] view -
            # the shape and values of the reference's attention_probs (modeling.py:89-90), not contiguous
            ld = 72
            store = torch.empty(B, heads, S, ld, device=qkv.device)
            call("vit3d_attn_fwd_padded", ptr(qkv), ptr(out), ptr(store), ld, B, S, heads, D, stream())
            probs = store[..., :S]
        else:
            probs = torch.empty(B, heads, S, S, device=qkv.device) if vis else None
            call("vit3d_attn_fwd", ptr(qkv), ptr(out), ptr(probs), B, S, heads, D, PREC[prec], stream())
        ctx.save_for_backward(qkv)
        ctx.meta = (heads, D, prec)
        if probs is None:
            return out, None
        ctx.mark_non_differentiable(probs)
        return out, probs

    @staticmethod
    def backward(ctx, dctx, _dprobs):
        (qkv,) = ctx.saved_tensors
        heads, D, prec = ctx.meta
        B, S, _ = qkv.shape
        dctx = _c(dctx.to(qkv.dtype))
        dqkv = torch.empty_like(qkv)
        call("vit3d_attn_bwd", ptr(dctx), ptr(qkv), ptr(dqkv), B, S, heads, D, PREC[prec], stream())
        return dqkv, None, None, None


# ----------------------------------------------------------------------------- dropout
class DropoutFn(torch.autograd.Function):
    """Inverted dropout with a counter-based mask (modeling.py:121,123,174), optionally fused with the
    residual add that follows it (modeling.py:196)."""

    @staticmethod
    def forward(ctx, x, residual, p, seed, site, step, mask):
        _need_cuda(x, residual)
        x = _c(x)
        if residual is not None:
            residual = _c(residual.to(x.dtype))
        y = torch.empty_like(x)
        f32 = int(x.dtype == torch.float32)
        if mask is not None:
            mask = _c(mask.to(device=x.device, dtype=torch.uint8))
            if mask.numel() != x.numel():
                raise _lib.Vit3dError("dropout mask has the wrong number of elements")
            call("vit3d_dropout_masked", ptr(x), ptr(mask), ptr(residual), ptr(y), x.numel(), f32, float(p), stream())
        else:
            call("vit3d_dropout", ptr(x), ptr(residual), ptr(y), x.numel(), f32, float(p), seed, site, step,
                 ptr(_STATE.get("step_dev")), stream())
        ctx.meta = (p, seed, site, step, mask, residual is not None)
        return y

    @staticmethod
    def backward(ctx, dy):
        p, seed, site, step, mask, has_res = ctx.meta
        dy = _c(dy)
        dx = torch.empty_like(dy)
        f32 = int(dy.dtype == torch.float32)
        if mask is not None:
            call("vit3d_dropout_masked", ptr(dy), ptr(mask), None, ptr(dx), dy.numel(), f32, float(p), stream())
        else:
            call("vit3d_dropout", ptr(dy), None, ptr(dx), dy.numel(), f32, float(p), seed, site, step,
                 ptr(_STATE.get("step_dev")), stream())
        return dx, (dy if has_res else None), None, None, None, None, None


def dropout(x, p: float, training: bool, site: int, step: int, mask=None, residual=None):
    if not training or p <= 0.0:
        assert residual is None
        return x
    if mask is None and _STATE["mask_override"] is not None:
        mask = _STATE["mask_override"].get(site)
    seed = torch.initial_seed() & 0xFFFFFFFFFFFFFFFF
    return DropoutFn.apply(x, residual, p, seed, site, step, mask)


def dropout_mask(n: int, p: float, site: int, step: int, device) -> torch.Tensor:
    """The keep-mask DropoutFn draws for (current torch seed, site, step): for parity tests."""
    m = torch.empty(n, device=device, dtype=torch.uint8)
    call("vit3d_dropout_mask", ptr(m), n, float(p), torch.initial_seed() & 0xFFFFFFFFFFFFFFFF, site, step, stream())
    return m


class mask_injection:
    """Context manager: replay explicit dropout keep-masks {site: mask} (parity with the reference's RNG
    stream is impossible, SURVEY.md §7; its masks are injected instead)."""

    def __init__(self, masks):
        self.masks = masks

    def __enter__(self):
        _STATE["mask_override"] = self.masks

    def __exit__(self, *a):
        _STATE["mask_override"] = None


# ----------------------------------------------------------------------------- loss
class BceLogitsFn(torch.autograd.Function):
    """BCEWithLogitsLoss(pos_weight)(logits.view(-1,1), labels.view(-1,1)) mean (modeling.py:283-286)."""

    @staticmethod
    def forward(ctx, logits, labels, pos_weight):
        _need_cuda(logits, labels)
        z = _c(logits.float()).reshape(-1)
        y = _c(labels.to(device=z.device, dtype=torch.float32)).reshape(-1)
        if y.numel() != z.numel():
            raise _lib.Vit3dError("BCE: logits and labels differ in size")
        loss = torch.empty((), device=z.device)
        pw_dev = None
        if isinstance(pos_weight, torch.Tensor) and pos_weight.is_cuda:
            # device-resident class weight (CUDA-graph replays): read by the kernel, no host sync
            pw_dev = pos_weight.reshape(1).float()
            pw = 1.0
        else:
            pw = -1.0 if pos_weight is None else float(pos_weight)
        call("vit3d_bce_logits_fwd", ptr(z), ptr(y), pw, ptr(pw_dev), ptr(loss), z.numel(), stream())
        ctx.save_for_backward(z, y, pw_dev)
        ctx.meta = (pw, logits.shape)
        return loss

    @staticmethod
    def backward(ctx, dloss):
        z, y, pw_dev = ctx.saved_tensors
        pw, shape = ctx.meta
        dz = torch.empty_like(z)
        dl = _c(dloss.float())
        call("vit3d_bce_logits_bwd", ptr(z), ptr(y), pw, ptr(pw_dev), ptr(dl), ptr(dz), z.numel(), stream())
        return dz.reshape(shape), None, None


# ----------------------------------------------------------------------------- meta classifier
class MetaFn(torch.autograd.Function):
    """sigmoid(Linear(cat(member logits))) (TransformerEnsemble.forward, modeling.py:355-356)."""

    @staticmethod
    def forward(ctx, feats, w, b):
        _need_cuda(feats, w, b)
        feats = _c(feats.float())
        B, F = feats.shape
        Cn = w.shape[0]
        if w.shape[1] != F:
            raise _lib.Vit3dError(f"meta-classifier expects {w.shape[1]} features, members give {F} "
                                  "(use in_features == num_classes of the members)")
        out = torch.empty(B, Cn, device=feats.device)
        call("vit3d_meta_fwd", ptr(feats), ptr(_c(w)), ptr(_c(b)), ptr(out), B, F, Cn, stream())
        ctx.save_for_backward(feats, w, out)
        return out

    @staticmethod
    def backward(ctx, dout):
        feats, w, out = ctx.saved_tensors
        B, F = feats.shape
        Cn = w.shape[0]
        df = torch.empty_like(feats)
        dw = torch.zeros_like(w)
        db = torch.zeros(Cn, device=w.device)
        call("vit3d_meta_bwd", ptr(_c(dout.float())), ptr(out), ptr(feats), ptr(_c(w)), ptr(df), ptr(dw), ptr(db),
             B, F, Cn, stream())
        return df, dw, db
