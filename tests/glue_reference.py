"""Float64 references of the small kernels that sit between the GEMMs (LayerNorm, classification head, BCE loss,
patch-embedding parameter gradients, meta-classifier, GELU), written in closed form.

tests/test_train_glue_reference_cpu.py pins each of them against torch.autograd in float64;
tests/test_gpu_train_glue.py compares the CUDA kernels with them.  Every function takes the operands exactly as the
kernel sees them (already rounded to fp32 or bf16 by the caller) and computes in float64."""
import math

import torch

from oracle import vit3d_oracle as O

f64 = torch.float64


def bf16_round(t):
    """t rounded to bfloat16 (round to nearest even), returned as float64."""
    return t.to(torch.float32).to(torch.bfloat16).to(f64)


def unpack_bits(bits, n):
    """Keep mask from packed bits: bit e of byte k is element 8k + e (the layout of vit3d_dropout_bits)."""
    b = bits.reshape(-1).to(torch.int64)
    return ((b.unsqueeze(-1) >> torch.arange(8)) & 1).reshape(-1)[:n].to(torch.bool)


def pack_bits(keep):
    """Inverse of unpack_bits (numel a multiple of 8) -> uint8 tensor."""
    k = keep.reshape(-1, 8).to(torch.int64)
    return (k << torch.arange(8)).sum(-1).to(torch.uint8)


# --------------------------------------------------------------------------- LayerNorm
def layer_norm(x, gamma, beta, eps):
    """Row LayerNorm (biased variance): (y, mean, rstd), all float64."""
    x = x.to(f64)
    mu = x.mean(-1)
    var = ((x - mu[:, None]) ** 2).mean(-1)
    rstd = 1.0 / torch.sqrt(var + eps)
    y = (x - mu[:, None]) * rstd[:, None] * gamma.to(f64) + beta.to(f64)
    return y, mu, rstd


def layer_norm_bwd(dy, x, mean, rstd, gamma, dres=None, keep=None, scale=1.0):
    """LayerNorm backward at the GIVEN statistics, with what vit3d_ln256_bwd fuses around it:
        o  = dres + rstd (g dy - mean_h(g dy) - xhat mean_h(g dy xhat)),   ob = o keep scale
        dgamma = sum_m dy xhat,  dbeta = sum_m dy,  dbias = sum_m ob
    Also returns `mag`, a per-element bound on the magnitude of the terms that make up o (the scale its fp32
    rounding error is measured against)."""
    dy, x, g = dy.to(f64), x.to(f64), gamma.to(f64)
    mean, rstd = mean.to(f64)[:, None], rstd.to(f64)[:, None]
    xh = (x - mean) * rstd
    gd = g * dy
    s1 = gd.mean(-1, keepdim=True)
    s2 = (gd * xh).mean(-1, keepdim=True)
    o = rstd * (gd - s1 - xh * s2)
    mag = rstd * (gd.abs() + s1.abs() + (xh * s2).abs())
    if dres is not None:
        o = o + dres.to(f64)
        mag = mag + dres.to(f64).abs()
    ob = o if keep is None else o * keep.to(f64) * scale
    return dict(o=o, ob=ob, mag=mag, xhat=xh, dgamma=(dy * xh).sum(0), dbeta=dy.sum(0), dbias=ob.sum(0))


# --------------------------------------------------------------------------- classification head (num_classes 1)
def head_fwd(enc, w, b, S):
    """logits[b] = enc[b*S, :] . w + bias  over the cls rows of the [B*S, H] token matrix."""
    cls = enc.to(f64).reshape(-1, S, enc.shape[-1])[:, 0]
    return cls @ w.to(f64).reshape(-1) + b.to(f64).reshape(())


def head_bwd(dlogit, enc, w, S):
    """(dencoded [B*S, H], dw [H], db []) of head_fwd."""
    H = enc.shape[-1]
    dl = dlogit.to(f64).reshape(-1)
    B = dl.numel()
    cls = enc.to(f64).reshape(B, S, H)[:, 0]
    denc = torch.zeros(B, S, H, dtype=f64)
    denc[:, 0] = dl[:, None] * w.to(f64).reshape(1, H)
    return denc.reshape(B * S, H), dl @ cls, dl.sum()


# --------------------------------------------------------------------------- BCE with logits (mean)
def bce(z, y, pos_weight=None, dloss=1.0):
    """(loss, dz) of BCEWithLogitsLoss(pos_weight) with mean reduction, dz scaled by dloss."""
    z, y = z.to(f64), y.to(f64)
    w = 1.0 if pos_weight is None else float(pos_weight)
    n = z.numel()
    logsig = lambda t: torch.clamp(t, max=0) - torch.log1p(torch.exp(-t.abs()))      # noqa: E731
    loss = -(w * y * logsig(z) + (1.0 - y) * logsig(-z)).sum() / n
    s = torch.sigmoid(z)
    dz = ((1.0 - y) * s - w * y * (1.0 - s)) * dloss / n
    return loss, dz


# --------------------------------------------------------------------------- patch embedding, parameter gradients
def embed_param_grads(x, dtok, patch, bf16_operands=False):
    """Gradients of tokens = cat(cls, patches @ w^T + bias) + pos with respect to w [H, Kp], bias, cls, pos.
    bf16_operands: the patches and the patch rows of dtok enter dw / dbias rounded to bf16 (BF16 mode); dcls and
    dpos always come from the fp32 dtok.  Returns the gradients and, under key + "_abs", the sums of the absolute
    values of their terms."""
    B, S, H = dtok.shape
    pt = O.patch_gather(x.to(f64), patch).reshape(B * (S - 1), -1)
    dY = dtok[:, 1:].reshape(-1, H).to(f64)
    if bf16_operands:
        pt, dY = bf16_round(pt), bf16_round(dY)
    d = dtok.to(f64)
    return dict(dw=dY.t() @ pt, dw_abs=dY.abs().t() @ pt.abs(), dbias=dY.sum(0), dbias_abs=dY.abs().sum(0),
                dcls=d[:, 0].sum(0), dcls_abs=d[:, 0].abs().sum(0), dpos=d.sum(0), dpos_abs=d.abs().sum(0))


# --------------------------------------------------------------------------- meta-classifier
def meta_fwd(f, w, b):
    """out[B, C] = sigmoid(f[B, F] @ w[C, F]^T + b)."""
    return torch.sigmoid(f.to(f64) @ w.to(f64).t() + b.to(f64))


def meta_bwd(dout, out, f, w):
    """(dfeats, dw, db) of meta_fwd at the GIVEN output `out` (dz = dout * out * (1 - out))."""
    dz = dout.to(f64) * out.to(f64) * (1.0 - out.to(f64))
    return dz @ w.to(f64), dz.t() @ f.to(f64), dz.sum(0)


# --------------------------------------------------------------------------- GELU (exact erf)
def gelu(x):
    x = x.to(f64)
    return 0.5 * x * (1.0 + torch.erf(x / math.sqrt(2.0)))


def gelu_grad(x):
    x = x.to(f64)
    return 0.5 * (1.0 + torch.erf(x / math.sqrt(2.0))) + x * torch.exp(-0.5 * x * x) / math.sqrt(2.0 * math.pi)


# coefficients of the fitted tanh-form GELU that the BF16 path differentiates (gelu_grad_fast, csrc/common.cuh):
# y = 0.5 x (1 + tanh(u)),  u = x (C0 + C1 x^2 + C2 x^4),  x^2 clamped at 100
GELU_FIT = (0.797458471, 0.0370503451, -3.58732362e-4)


def gelu_grad_fit(x):
    """gelu_grad_fast in float64 (exact tanh): the derivative of the fitted form."""
    c0, c1, c2 = GELU_FIT
    x = x.to(f64)
    x2 = torch.clamp(x * x, max=100.0)
    t = torch.tanh(x * (c0 + x2 * (c1 + x2 * c2)))
    du = c0 + x2 * (3.0 * c1 + x2 * 5.0 * c2)
    return 0.5 * (1.0 + t) + 0.5 * x * (1.0 - t * t) * du
