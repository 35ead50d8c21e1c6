"""The float64 references of tests/glue_reference.py against torch.autograd in float64 on small shapes, so that the
kernel tests in tests/test_gpu_train_glue.py compare with references that are themselves right.  No GPU needed."""
import math

import pytest
import torch
import torch.nn.functional as TF

from tests import glue_reference as R

f64 = torch.float64
TOL = dict(rtol=1e-12, atol=1e-12)


def gen(seed):
    return torch.Generator().manual_seed(seed)


def test_bit_packing_round_trip_and_layout():
    g = gen(1)
    keep = torch.rand(3 * 256, generator=g) < 0.9
    bits = R.pack_bits(keep)
    assert bits.dtype == torch.uint8 and bits.numel() == 3 * 32
    assert torch.equal(R.unpack_bits(bits, keep.numel()), keep)
    # bit e of byte k is element 8k + e
    one = torch.zeros(16, dtype=torch.bool)
    one[8 + 3] = True
    assert R.pack_bits(one).tolist() == [0, 8]


def test_bf16_round_is_round_to_nearest_even():
    x = torch.tensor([1.0, 1.0 + 2.0 ** -8, 1.0 + 3 * 2.0 ** -8, 1.0 + 2.0 ** -9, -1.0 - 2.0 ** -8], dtype=f64)
    assert R.bf16_round(x).tolist() == [1.0, 1.0, 1.0 + 2.0 ** -6, 1.0, -1.0]


@pytest.mark.parametrize("M,H", [(1, 8), (5, 256), (3, 257)])
def test_layer_norm_matches_torch(M, H):
    g = gen(M * H)
    x = torch.randn(M, H, generator=g, dtype=f64) * 3 + 2
    x[0] += 1000.0
    gamma, beta = torch.randn(H, generator=g, dtype=f64), torch.randn(H, generator=g, dtype=f64)
    y, mu, rstd = R.layer_norm(x, gamma, beta, 1e-6)
    torch.testing.assert_close(y, TF.layer_norm(x, (H,), gamma, beta, 1e-6), rtol=1e-10, atol=1e-10)
    torch.testing.assert_close(mu, x.mean(-1), **TOL)
    torch.testing.assert_close(rstd, 1 / torch.sqrt(x.var(-1, unbiased=False) + 1e-6), rtol=1e-10, atol=0)


@pytest.mark.parametrize("with_dres,with_keep", [(False, False), (True, False), (False, True), (True, True)])
def test_layer_norm_bwd_matches_autograd(with_dres, with_keep):
    M, H, scale = 6, 256, 1 / 0.9
    g = gen(7 + 2 * with_dres + with_keep)
    x = torch.randn(M, H, generator=g, dtype=f64)
    x[1] += 1000.0
    gamma, beta = torch.randn(H, generator=g, dtype=f64), torch.randn(H, generator=g, dtype=f64)
    dy = torch.randn(M, H, generator=g, dtype=f64)
    dres = torch.randn(M, H, generator=g, dtype=f64) if with_dres else None
    keep = (torch.rand(M, H, generator=g) < 0.9) if with_keep else None
    _, mu, rstd = R.layer_norm(x, gamma, beta, 1e-6)
    ref = R.layer_norm_bwd(dy, x, mu, rstd, gamma, dres, keep, scale)

    xa, ga, ba = (t.clone().requires_grad_() for t in (x, gamma, beta))
    TF.layer_norm(xa, (H,), ga, ba, 1e-6).backward(dy)
    o = xa.grad + (dres if with_dres else 0)
    torch.testing.assert_close(ref["o"], o, rtol=1e-9, atol=1e-9)
    ob = o * keep * scale if with_keep else o
    torch.testing.assert_close(ref["ob"], ob, rtol=1e-9, atol=1e-9)
    torch.testing.assert_close(ref["dgamma"], ga.grad, rtol=1e-9, atol=1e-9)
    torch.testing.assert_close(ref["dbeta"], ba.grad, **TOL)
    torch.testing.assert_close(ref["dbias"], ob.sum(0), rtol=1e-9, atol=1e-9)
    assert (ref["mag"] >= ref["o"].abs() * (1 - 1e-12)).all()


@pytest.mark.parametrize("B,S", [(1, 5), (3, 65)])
def test_head_matches_autograd(B, S):
    H = 256
    g = gen(B * S)
    enc = torch.randn(B * S, H, generator=g, dtype=f64)
    w, b = torch.randn(1, H, generator=g, dtype=f64), torch.randn(1, generator=g, dtype=f64)
    dl = torch.randn(B, generator=g, dtype=f64)
    ea, wa, ba = (t.clone().requires_grad_() for t in (enc, w, b))
    logits = TF.linear(ea.reshape(B, S, H)[:, 0], wa, ba).reshape(-1)
    torch.testing.assert_close(R.head_fwd(enc, w, b, S), logits.detach(), **TOL)
    logits.backward(dl)
    denc, dw, db = R.head_bwd(dl, enc, w, S)
    torch.testing.assert_close(denc, ea.grad, **TOL)
    torch.testing.assert_close(dw, wa.grad.reshape(-1), **TOL)
    torch.testing.assert_close(db, ba.grad.reshape(()), **TOL)


@pytest.mark.parametrize("pw", [None, 0.5, 3.0])
@pytest.mark.parametrize("soft", [False, True])
def test_bce_matches_torch(pw, soft):
    g = gen(11)
    n = 9
    z = torch.randn(n, generator=g, dtype=f64) * 4
    z[:5] = torch.tensor([0.0, 20.0, -20.0, 90.0, -90.0], dtype=f64)
    y = torch.rand(n, generator=g, dtype=f64) if soft else (torch.rand(n, generator=g) < 0.5).to(f64)
    dloss = 0.37
    za = z.clone().requires_grad_()
    pwt = None if pw is None else torch.tensor([pw], dtype=f64)
    loss = TF.binary_cross_entropy_with_logits(za.view(-1, 1), y.view(-1, 1), pos_weight=pwt)
    (loss * dloss).backward()
    lr, dz = R.bce(z, y, pw, dloss)
    torch.testing.assert_close(lr, loss.detach(), **TOL)
    torch.testing.assert_close(dz, za.grad, **TOL)


@pytest.mark.parametrize("size,patch", [((32, 32, 5), (16, 16, 5)), ((34, 36, 5), (8, 8, 5))])
def test_embed_param_grads_match_conv3d(size, patch):
    """Against a plain nn.Conv3d embedding (Embeddings.forward, modeling.py:162-173), including the voxels Conv3d
    drops."""
    B, H = 3, 16
    g = gen(sum(size) + patch[0])
    x = torch.randn(B, 1, *size, generator=g, dtype=f64)
    conv = torch.nn.Conv3d(1, H, kernel_size=patch, stride=patch).double()
    P = math.prod(s // p for s, p in zip(size, patch))
    cls = torch.randn(1, 1, H, generator=g, dtype=f64, requires_grad=True)
    pos = torch.randn(1, P + 1, H, generator=g, dtype=f64, requires_grad=True)
    t = conv(x).flatten(2).transpose(-1, -2)
    t = torch.cat((cls.expand(B, -1, -1), t), dim=1) + pos
    dtok = torch.randn(t.shape, generator=g, dtype=f64)
    t.backward(dtok)
    ref = R.embed_param_grads(x, dtok, patch)
    torch.testing.assert_close(ref["dw"], conv.weight.grad.reshape(H, -1), **TOL)
    torch.testing.assert_close(ref["dbias"], conv.bias.grad, **TOL)
    torch.testing.assert_close(ref["dcls"], cls.grad.reshape(H), **TOL)
    torch.testing.assert_close(ref["dpos"], pos.grad.reshape(P + 1, H), **TOL)
    for k in ("dw", "dbias", "dcls", "dpos"):
        assert (ref[k + "_abs"] >= ref[k].abs() * (1 - 1e-12)).all()
    rb = R.embed_param_grads(x, dtok, patch, bf16_operands=True)
    pt = R.bf16_round(R.O.patch_gather(x, patch).reshape(B * P, -1))
    dY = R.bf16_round(dtok[:, 1:].reshape(-1, H))
    torch.testing.assert_close(rb["dw"], dY.t() @ pt, **TOL)
    torch.testing.assert_close(rb["dcls"], ref["dcls"], rtol=0, atol=0)


@pytest.mark.parametrize("B,F,C", [(1, 3, 1), (4, 5, 2)])
def test_meta_matches_autograd(B, F, C):
    g = gen(B * F * C)
    f = torch.randn(B, F, generator=g, dtype=f64)
    w, b = torch.randn(C, F, generator=g, dtype=f64), torch.randn(C, generator=g, dtype=f64)
    dout = torch.randn(B, C, generator=g, dtype=f64)
    fa, wa, ba = (t.clone().requires_grad_() for t in (f, w, b))
    out = torch.sigmoid(TF.linear(fa, wa, ba))
    torch.testing.assert_close(R.meta_fwd(f, w, b), out.detach(), **TOL)
    out.backward(dout)
    df, dw, db = R.meta_bwd(dout, out.detach(), f, w)
    torch.testing.assert_close(df, fa.grad, **TOL)
    torch.testing.assert_close(dw, wa.grad, **TOL)
    torch.testing.assert_close(db, ba.grad, **TOL)


def test_gelu_and_its_derivative_match_torch():
    x = torch.linspace(-12, 12, 4001, dtype=f64)
    xa = x.clone().requires_grad_()
    y = TF.gelu(xa)
    torch.testing.assert_close(R.gelu(x), y.detach(), **TOL)
    y.sum().backward()
    torch.testing.assert_close(R.gelu_grad(x), xa.grad, **TOL)


def test_fitted_gelu_derivative_error_bound():
    """The BF16 backward differentiates a fitted tanh form of GELU.  Its distance from the exact erf derivative over
    [-12, 12] (1.214e-4) is part of the 1e-3 the kernel test budgets for, next to tanh.approx's ~2^-11."""
    x = torch.linspace(-12, 12, 240001, dtype=f64)
    err = (R.gelu_grad_fit(x) - R.gelu_grad(x)).abs().max().item()
    assert err <= 1.25e-4, err
