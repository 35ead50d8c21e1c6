"""The kernels between the GEMMs of the training step, one by one against float64: LayerNorm-256 forward / backward
(vit3d_ln256_fwd / _bwd), the classification head (vit3d_linear_fwd with N = 1, vit3d_head_bwd), BCE-with-logits,
the patch-embedding parameter gradients, the per-operator LayerNorm (vit3d_ln_fwd / _bwd), the meta-classifier and the
element-wise kernels (GELU, dropout, uint8 input).  The references are tests/glue_reference.py (pinned against
autograd by tests/test_train_glue_reference_cpu.py); they take the operands rounded as the kernel documents (bf16
patches and dY in BF16 mode, the fp32 mean / rstd handed to a backward) and nothing else, so that what is left is
indexing and reduction error.

Shapes are chosen where these kernels change behaviour: LayerNorm-256 backward runs 2 * sm_count blocks of 8 warps,
so M = 16 * sm_count + 1 makes one warp take a second row; the head gradient reduces 64 volumes per block (B = 63, 64,
65); the embedding gradients split the batch over grid.y above 32 volumes; the loss is one block of 256 threads
(n = 255, 256, 257); dropout, uint8 conversion and the GELU backward have vector bodies and scalar tails.

Every fully written output starts as NaN and must come back finite; every accumulated output (+=) starts from a
random non-zero value of the order of the sum it receives, and `got - start` is compared.  Tolerances:
  - fp32 results of short reductions (<= 256 terms): |err| <= 1e-5 x the scale of the row / element (the sum of the
    magnitudes of the terms), about 100 fp32 ulps.
  - column sums over M rows (dgamma, dbeta, dbias, dw, db, dcls, dpos): |err| <= 1e-5 x sum_m |term| per column,
    robust to cancellation and far below a lost row or block.
  - LayerNorm forward outputs: |y - ref| <= 4e-6 |gamma| (1 + |mean| rstd) + 1 fp32 ulp; the mean by
    4e-6 (1 / rstd + |mean|), rstd by 4e-6 rstd (1 + |mean| rstd).  The fp32 mean carries an error that grows with
    |mean| / sigma: an emulation of the kernel's summation order gave an xhat error of 3.9e-7 at mean 0 and 7.6e-5 at
    mean 1000, sigma 1 (a one-pass variance: 0.25).  So a row at 1000 + N(0, 1) passes the two-pass kernel and fails
    a one-pass rewrite.
  - bf16 outputs: one bf16 ulp of the float64 value on top of the fp32 tolerance of the value before rounding;
    TF32-rounded outputs (vit3d_ln_fwd y_bf16 = 2): low 13 mantissa bits zero and one TF32 ulp (2^-10 relative).
  - exactly 0 where the operation gives 0 (dropped elements, the non-cls rows of d(encoded)); bit-exact where the
    operation is exact (uint8 -> fp32, the dropped LayerNorm input, dropout against its fp32 formula).
  - BCE gradient: absolute, 2e-6 (w + 1) |dloss| / n: 1 - sigmoid(z) cancels in fp32 for large |z|, as in torch.
  - GELU: forward 5e-7 |x| + the output's ulp (erff is within 2 ulp; 1 + erf cancels for negative x).  Backward in
    fp32 and on the exact bf16 path (unaligned or n % 8 != 0): 1e-5 |da|.  The aligned bf16 path differentiates the
    fitted tanh form with tanh.approx: the fit is within 1.22e-4 of the erf derivative on [-12, 12]
    (test_fitted_gelu_derivative_error_bound) and tanh.approx adds about 2^-11, so 1e-3 |da| + one bf16 ulp.  Both
    are absolute: gelu' crosses 0 near h = -0.75.
  - dropout: y = x * float32(1 / (1 - p)) + residual under the mask vit3d_dropout_mask exports, bit for bit, either
    as a rounded product plus the residual or as one fused multiply-add (ptxas may contract them).  Today's kernels
    give the unfused form on every path (vector body, scalar tail, vit3d_dropout_masked).  bf16 output is the bf16
    rounding of that value."""
import ctypes
import functools

import pytest
import torch

import vit3d_b200
from tests import glue_reference as R
from tests.test_gpu_input_grad import GEOMETRIES
from vit3d_b200 import _lib
from vit3d_b200._lib import PREC, call, ptr, stream

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
f32, bf16, f64 = torch.float32, torch.bfloat16, torch.float64
H = 256
EPS = 1e-6
EPS32 = float(torch.tensor(EPS, dtype=f32))
P_DROP = 0.1
# the library computes 1 / (1 - p) in fp32 on the host
DROP_SCALE = float(torch.tensor(1.0, dtype=f32) / (torch.tensor(1.0, dtype=f32) - torch.tensor(P_DROP, dtype=f32)))
SEED, SITE = 0x1234ABCD5678, 5
SM_ROWS = "16sm+1"


@functools.lru_cache(maxsize=1)
def sm_count():
    sms, cc = ctypes.c_int(), ctypes.c_int()
    call("vit3d_device_info", ctypes.byref(sms), ctypes.byref(cc))
    return sms.value


def rows(M):
    return 16 * sm_count() + 1 if M == SM_ROWS else M


def launches():
    return _lib.lib().vit3d_launch_count()


def cpu_gen(seed):
    return torch.Generator().manual_seed(seed)


def gpu_gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def nan(shape, dtype=f32):
    return torch.full(shape if isinstance(shape, tuple) else (shape,), float("nan"), device=DEV, dtype=dtype)


def ulp(ref, mant):
    """Spacing of a float with `mant` stored mantissa bits at |ref| (23 fp32, 10 TF32, 7 bf16)."""
    a = ref.abs().clamp(min=2.0 ** -126)
    return torch.exp2(torch.floor(torch.log2(a)) - mant)


def check(got, ref, tol, what):
    """|got - ref| <= tol element-wise (NaN fails)."""
    got = got.detach().to("cpu", f64)
    ref = ref.to(f64)
    err = (got - ref).abs()
    tol = torch.as_tensor(tol, dtype=f64).expand(err.shape)
    bad = ~(err <= tol)
    if bool(bad.any()):
        i = tuple(int(k) for k in bad.nonzero()[0])
        worst = float(torch.where(bad & (err == err), err / tol, torch.zeros_like(err)).max())
        pytest.fail(f"{what}: {int(bad.sum())} of {bad.numel()} out of tolerance; first at {i}: got {float(got[i])!r} "
                    f"want {float(ref[i])!r} tol {float(tol[i]):.3g}; worst err/tol {worst:.3g}")


def check_colsum(got, start, ref, ref_abs, what):
    check(got.detach().to("cpu", f64) - start.to("cpu", f64), ref, 1e-5 * ref_abs, what)


def acc_start(ref_abs, g):
    """Start value of an accumulated output: random sign and magnitude U(0.5, 1) x the sum of |terms| the element
    receives.  Adding a sum into a start value rounds at the start's ulp, so a start of the order of the sum keeps that
    rounding (about one fp32 ulp of the result) inside the column-sum tolerance."""
    a = ref_abs.to(f64).clamp(min=1e-20)
    u = torch.rand(a.shape, generator=g, dtype=f64) * 0.5 + 0.5
    sign = torch.where(torch.rand(a.shape, generator=g) < 0.5, -1.0, 1.0).to(f64)
    return (sign * u * a).to(f32)


def ln_stat_tols(mu, rstd):
    """Bounds of the LayerNorm statistics (module docstring)."""
    k = 1.0 + mu.abs() * rstd
    return 4e-6 * (1.0 / rstd + mu.abs()), 4e-6 * rstd * k, k


# ============================================================================ LayerNorm 256
@functools.lru_cache(maxsize=1)
def ln256_case(M):
    """x [M, 256] with an offset row (1000 + N(0, 1)) first and a constant row last, gamma, beta, keep bits, dy, dres."""
    g = cpu_gen(M)
    x = torch.randn(M, H, generator=g)
    x[0] += 1000.0
    if M > 1:
        x[M - 1] = 0.5
    gamma, beta = torch.randn(H, generator=g), torch.randn(H, generator=g)
    keep = torch.rand(M, H, generator=g) >= P_DROP
    dy, dres = torch.randn(M, H, generator=g), torch.randn(M, H, generator=g)
    return x, gamma, beta, keep, R.pack_bits(keep), dy, dres


@pytest.mark.parametrize("M", [1, 7, 130, SM_ROWS, 66560])
def test_ln256_fwd_vs_fp64(M):
    M = rows(M)
    x, gamma, beta, keep, bits, _, _ = ln256_case(M)
    xd = torch.where(keep, x * torch.tensor(DROP_SCALE, dtype=f32), torch.zeros((), dtype=f32))
    refs = {}
    for drop, xin in ((False, x), (True, xd)):
        y, mu, rstd = R.layer_norm(xin, gamma, beta, EPS32)
        tm, tr, k = ln_stat_tols(mu, rstd)
        refs[drop] = (y, mu, rstd, tm, tr, 4e-6 * gamma.abs().to(f64) * k[:, None] + ulp(y, 23))
    xg, gg, bg, bitsg = x.to(DEV), gamma.to(DEV), beta.to(DEV), bits.to(DEV)
    # (bf16 output, fp32 output, statistics, keep bits, x_dropped)
    for y_b, y_f, stats, drop, want_xd in ((1, 0, 1, 1, 1), (0, 1, 0, 0, 0), (1, 1, 1, 0, 0), (1, 1, 0, 1, 0)):
        what = f"M={M} bf16={y_b} f32={y_f} stats={stats} bits={drop} x_dropped={want_xd}"
        yb = nan((M, H), bf16) if y_b else None
        yf = nan((M, H)) if y_f else None
        mean, rstd = (nan(M), nan(M)) if stats else (None, None)
        xdg = nan((M, H)) if want_xd else None
        call("vit3d_ln256_fwd", ptr(xg), ptr(bitsg) if drop else None, DROP_SCALE, ptr(xdg), ptr(gg), ptr(bg), ptr(yb),
             ptr(yf), ptr(mean), ptr(rstd), M, EPS, stream())
        y, mu, rs, tm, tr, ty = refs[bool(drop)]
        if want_xd:
            assert torch.equal(xdg.cpu(), xd), what
        if y_f:
            check(yf, y, ty, "y_f32 " + what)
        if y_b:
            check(yb, y, ty + ulp(y, 7), "y_bf16 " + what)
        if stats:
            check(mean, mu, tm, "mean " + what)
            check(rstd, rs, tr, "rstd " + what)


# (dres, bits, mask_f32, outputs, dbias, dgamma / dbeta, dx aliases dres): the fused step's four calls first
LN256_BWD_FLAGS = [
    (0, 1, 0, "both", 1, 1, 0),      # encoder_norm, under the last fc2 Dropout
    (1, 0, 0, "both", 1, 1, 0),      # ffn_norm
    (1, 1, 0, "both", 1, 1, 0),      # attention_norm of Block i > 0, under Block i-1's fc2 Dropout
    (1, 1, 1, "dx", 0, 1, 0),        # attention_norm of Block 0, under the embedding Dropout
    (0, 0, 0, "dxb", 0, 0, 0),
    (1, 1, 1, "both", 1, 0, 1),
    (0, 0, 1, "dx", 1, 1, 0),
    (1, 0, 0, "dx", 0, 1, 1),
]


@pytest.mark.parametrize("M", [1, 7, 130, SM_ROWS, 66560])
def test_ln256_bwd_vs_fp64(M):
    M = rows(M)
    x, gamma, _, keep, bits, dy, dres = ln256_case(M)
    _, mu64, rs64 = R.layer_norm(x, gamma, gamma, EPS32)
    mean, rstd = mu64.to(f32), rs64.to(f32)               # the kernel's operands; the reference uses them as they are
    core = R.layer_norm_bwd(dy, x, mean, rstd, gamma)
    dres64, keep64 = dres.to(f64), keep.to(f64) * DROP_SCALE
    dgamma_abs, dbeta_abs = (dy.to(f64) * core["xhat"]).abs().sum(0), dy.to(f64).abs().sum(0)
    dyg, xg, mg, rg, gg, bitsg = (t.to(DEV) for t in (dy, x, mean, rstd, gamma, bits))
    dresg = dres.to(DEV)
    g = cpu_gen(M + 1)
    for has_dres, drop, mask_f32, outs, has_dbias, has_dgb, alias in LN256_BWD_FLAGS:
        what = f"M={M} dres={has_dres} bits={drop} mask_f32={mask_f32} out={outs} dbias={has_dbias} dgb={has_dgb} alias={alias}"
        o = core["o"] + dres64 if has_dres else core["o"]
        mag = core["mag"] + dres64.abs() if has_dres else core["mag"]
        ob = o * keep64 if drop else o
        rowtol = 1e-5 * mag.amax(1, keepdim=True) * (DROP_SCALE if drop else 1.0)
        dx = dxb = None
        if outs in ("dx", "both"):
            dx = dresg.clone() if alias else nan((M, H))
        if outs in ("dxb", "both"):
            dxb = nan((M, H), bf16)
        dres_arg = (dx if alias else dresg) if has_dres else None
        dbias_abs = (mag * keep64 if drop else mag).sum(0)
        starts = {k: acc_start(a, g) for k, a in (("dgamma", dgamma_abs), ("dbeta", dbeta_abs), ("dbias", dbias_abs))}
        acc = {k: v.to(DEV) for k, v in starts.items()}
        call("vit3d_ln256_bwd", ptr(dyg), ptr(xg), ptr(mg), ptr(rg), ptr(gg), ptr(dres_arg), ptr(bitsg) if drop else None,
             DROP_SCALE, mask_f32, ptr(dx), ptr(dxb), ptr(acc["dgamma"]) if has_dgb else None,
             ptr(acc["dbeta"]) if has_dgb else None, ptr(acc["dbias"]) if has_dbias else None, M, stream())
        if dx is not None:
            check(dx, ob if mask_f32 else o, rowtol, "dx " + what)
        if dxb is not None:
            check(dxb, ob, rowtol + ulp(ob, 7), "dx_bf16 " + what)
        if drop:
            dropped = ~keep
            if dxb is not None:
                assert (dxb.cpu()[dropped] == 0).all(), what
            if dx is not None and mask_f32:
                assert (dx.cpu()[dropped] == 0).all(), what
        for k, used, ref, ref_abs in (("dgamma", has_dgb, core["dgamma"], dgamma_abs), ("dbeta", has_dgb, core["dbeta"], dbeta_abs),
                                      ("dbias", has_dbias, ob.sum(0), dbias_abs)):
            if used:
                check_colsum(acc[k], starts[k], ref, ref_abs, f"{k} " + what)
            else:
                assert torch.equal(acc[k].cpu(), starts[k]), f"{k} written although not requested: " + what


def test_ln256_fwd_then_bwd_vs_autograd():
    """The fused step's pairing: vit3d_ln256_fwd's own statistics feed vit3d_ln256_bwd; against autograd over fp64
    F.layer_norm."""
    M = 130
    g = cpu_gen(77)
    x = torch.randn(M, H, generator=g) * 2 + 0.5
    gamma, beta, dy = torch.randn(H, generator=g), torch.randn(H, generator=g), torch.randn(M, H, generator=g)
    xg, gg, bg, dyg = x.to(DEV), gamma.to(DEV), beta.to(DEV), dy.to(DEV)
    y, mean, rstd = nan((M, H)), nan(M), nan(M)
    call("vit3d_ln256_fwd", ptr(xg), None, 1.0, None, ptr(gg), ptr(bg), None, ptr(y), ptr(mean), ptr(rstd), M, EPS, stream())
    dx = nan((M, H))
    dgamma, dbeta = torch.zeros(H, device=DEV), torch.zeros(H, device=DEV)
    call("vit3d_ln256_bwd", ptr(dyg), ptr(xg), ptr(mean), ptr(rstd), ptr(gg), None, None, 1.0, 0, ptr(dx), None, ptr(dgamma),
         ptr(dbeta), None, M, stream())
    xa, ga, ba = (t.to(f64).requires_grad_() for t in (x, gamma, beta))
    ya = torch.nn.functional.layer_norm(xa, (H,), ga, ba, EPS32)
    ya.backward(dy.to(f64))
    _, mu, rs = R.layer_norm(x, gamma, beta, EPS32)
    k = ln_stat_tols(mu, rs)[2]
    ref = R.layer_norm_bwd(dy, x, mu, rs, gamma)
    check(y, ya.detach(), 4e-6 * gamma.abs().to(f64) * k[:, None] + ulp(ya.detach(), 23), "y")
    check(dx, xa.grad, 1e-5 * ref["mag"].amax(1, keepdim=True), "dx")
    check(dgamma, ga.grad, 1e-5 * (dy.to(f64) * ref["xhat"]).abs().sum(0), "dgamma")
    check(dbeta, ba.grad, 1e-5 * dy.to(f64).abs().sum(0), "dbeta")


# ============================================================================ classification head
@pytest.mark.parametrize("S", [65, 257])
@pytest.mark.parametrize("B", [1, 2, 63, 64, 65, 257, 1024])
def test_head_fwd_and_bwd_vs_fp64(B, S):
    gg = gpu_gen(B * 1000 + S)
    enc = torch.randn(B * S, H, generator=gg, device=DEV)
    cls = enc.view(B, S, H)[:, 0].cpu()
    g = cpu_gen(B + S)
    w, b = torch.randn(1, H, generator=g), torch.randn(1, generator=g)
    dl = torch.randn(B, generator=g)
    wg, bg, dlg = w.to(DEV), b.to(DEV), dl.to(DEV)
    # forward: logits = enc[b*S] . w + bias (vit3d_linear_fwd: fp32, N = 1, strided rows -> rowdot_kernel)
    logits = nan((B, 1))
    n0 = launches()
    call("vit3d_linear_fwd", ptr(enc), S * H, 1, ptr(wg), None, ptr(bg), None, ptr(logits), 1, None, 0, B, 1, H,
         PREC["fp32"], stream())
    assert launches() - n0 == 1
    terms = (cls.to(f64) * w.to(f64)).abs().sum(1) + b.abs().to(f64)
    check(logits.view(-1), R.head_fwd(cls, w, b, 1), 1e-5 * terms, f"logits B={B} S={S}")     # S = 1: cls rows only
    # backward
    denc = nan((B * S, H))
    dw_abs, db_abs = dl.to(f64).abs() @ cls.to(f64).abs(), dl.to(f64).abs().sum().reshape(1)
    dw0, db0 = acc_start(dw_abs, g), acc_start(db_abs, g)
    dw, db = dw0.to(DEV), db0.to(DEV)
    call("vit3d_head_bwd", ptr(dlg), ptr(enc), ptr(wg), ptr(denc), ptr(dw), ptr(db), B, S, H, stream())
    d3 = denc.view(B, S, H)
    assert bool((d3[:, 1:] == 0).all()), f"non-cls rows of dencoded not exactly 0 (B={B} S={S})"
    dcls_ref, dw_ref, db_ref = R.head_bwd(dl, cls, w, 1)
    check(d3[:, 0], dcls_ref, ulp(dcls_ref, 23), f"dencoded cls rows B={B} S={S}")      # one fp32 product each
    check_colsum(dw, dw0, dw_ref, dw_abs, f"dw B={B} S={S}")
    check_colsum(db, db0, db_ref.reshape(1), db_abs, f"db B={B} S={S}")


def test_head_bwd_rejects_other_hidden_sizes():
    enc = torch.zeros(65, 128, device=DEV)
    w, dl = torch.zeros(128, device=DEV), torch.zeros(1, device=DEV)
    dw, db, denc = torch.zeros(128, device=DEV), torch.zeros(1, device=DEV), torch.zeros(65, 128, device=DEV)
    n0 = launches()
    assert _lib.lib().vit3d_head_bwd(ptr(dl), ptr(enc), ptr(w), ptr(denc), ptr(dw), ptr(db), 1, 65, 128, stream()) == -2
    with pytest.raises(vit3d_b200.Vit3dError):
        call("vit3d_head_bwd", ptr(dl), ptr(enc), ptr(w), ptr(denc), ptr(dw), ptr(db), 1, 65, 128, stream())
    assert launches() == n0


# ============================================================================ BCE with logits
def bce_case(n, soft, seed):
    g = cpu_gen(seed)
    z = torch.randn(n, generator=g) * 4
    special = torch.tensor([0.0, 20.0, -20.0, 90.0, -90.0])
    z[:min(n, 5)] = special[:min(n, 5)]
    y = torch.rand(n, generator=g) if soft else (torch.rand(n, generator=g) < 0.5).to(f32)
    return z, y


# (host pos_weight, device pos_weight or None, the weight in effect or None)
PW_MODES = {"none": (-1.0, None, None), "host": (2.5, None, 2.5), "device": (7.0, 0.75, 0.75),
            "device_negative": (3.0, -1.0, None)}


def run_bce(z, y, mode, dloss):
    n = z.numel()
    pw_host, pw_dev, w = PW_MODES[mode]
    zg, yg = z.to(DEV), y.to(DEV)
    pwg = None if pw_dev is None else torch.tensor([pw_dev], device=DEV)
    dlg = None if dloss is None else torch.tensor([dloss], device=DEV)
    loss, dz = nan(1), nan(n)
    call("vit3d_bce_logits_fwd", ptr(zg), ptr(yg), pw_host, ptr(pwg), ptr(loss), n, stream())
    call("vit3d_bce_logits_bwd", ptr(zg), ptr(yg), pw_host, ptr(pwg), ptr(dlg), ptr(dz), n, stream())
    what = f"n={n} pos_weight={mode} dloss={dloss}"
    lref, dref = R.bce(z, y, w, 1.0 if dloss is None else dloss)
    ww = 1.0 if w is None else w
    z64, y64 = z.to(f64), y.to(f64)
    lsig = torch.nn.functional.logsigmoid
    scale = ((ww * y64 * lsig(z64)).abs() + ((1 - y64) * lsig(-z64)).abs()).sum() / n
    check(loss.view(()), lref, 1e-5 * scale, "loss " + what)
    check(dz, dref, 2e-6 * (ww + 1) * abs(1.0 if dloss is None else dloss) / n, "dlogits " + what)


@pytest.mark.parametrize("mode", list(PW_MODES))
@pytest.mark.parametrize("n", [1, 2, 7, 255, 256, 257, 1000, 1024])
def test_bce_logits_vs_fp64(n, mode):
    z, y = bce_case(n, False, n)
    for dloss in (None, 0.37):
        run_bce(z, y, mode, dloss)


def test_bce_logits_soft_labels_vs_fp64():
    z, y = bce_case(257, True, 5)
    run_bce(z, y, "device", 0.37)


# ============================================================================ patch embedding: parameter gradients
@functools.lru_cache(maxsize=2)
def embed_ref(geom, B, bf16_operands):
    (X, Y, Z), patch = geom
    x, dtok = embed_inputs(geom, B)
    return R.embed_param_grads(x.cpu(), dtok.cpu(), patch, bf16_operands)


@functools.lru_cache(maxsize=1)
def embed_inputs(geom, B):
    (X, Y, Z), patch = geom
    P = (X // patch[0]) * (Y // patch[1]) * (Z // patch[2])
    g = gpu_gen(B * 7 + X + patch[0])
    return torch.randn(B, 1, X, Y, Z, generator=g, device=DEV), torch.randn(B, P + 1, H, generator=g, device=DEV)


EMBED_CASES = [(gi, B) for gi in range(3) for B in (1, 3, 33, 257)] + [(0, 1024)]


@pytest.mark.parametrize("gi,B", EMBED_CASES, ids=[f"{['p16', 'p8', 'remainder'][gi]}-B{B}" for gi, B in EMBED_CASES])
def test_patch_embed_param_grads_vs_fp64(gi, B):
    geom = GEOMETRIES[gi]
    (X, Y, Z), (p0, p1, p2) = geom
    Kp = p0 * p1 * p2
    x, dtok = embed_inputs(geom, B)
    S = dtok.shape[1]
    g = cpu_gen(B + gi)
    for prec in ("fp32", "tf32", "bf16"):
        what = f"{prec} geometry={geom} B={B}"
        pid = PREC[prec]
        # BF16 mode takes the tensor-core weight gradient when it serves the [H, Kp] product over B*P rows
        # (tc_wgrad_supported: at least 64 rows, H and Kp multiples of 64): every case here
        tc = prec == "bf16" and B * (S - 1) >= 64 and H % 64 == 0 and Kp % 64 == 0
        ref = embed_ref(geom, B, tc)
        wsb = _lib.lib().vit3d_patch_embed_ws_bytes(B, X, Y, Z, p0, p1, p2, H, pid)
        ws = torch.empty(wsb, device=DEV, dtype=torch.uint8)
        starts = {k: acc_start(ref[k + "_abs"], g) for k in ("dw", "dbias", "dcls", "dpos")}
        acc = {k: v.to(DEV) for k, v in starts.items()}
        n0 = launches()
        call("vit3d_patch_embed_bwd", ptr(x), ptr(dtok), ptr(acc["dw"]), ptr(acc["dbias"]), ptr(acc["dcls"]), ptr(acc["dpos"]),
             B, X, Y, Z, p0, p1, p2, H, pid, ptr(ws), wsb, stream())
        # im2col, patch-row compaction, the dw GEMM, the dbias column sums, dcls / dpos: five launches on either path
        assert launches() - n0 == 5, what
        for k in ("dw", "dbias", "dcls", "dpos"):
            check_colsum(acc[k], starts[k], ref[k], ref[k + "_abs"], f"{k} {what}")
        if tc:
            # the tensor-core weight gradient took bf16 operands: its dw is far closer to the bf16-operand reference than
            # the fp32-operand one is (the launch counts of the two paths are equal, so this is what pins the path)
            got = acc["dw"].cpu().to(f64) - starts["dw"].to(f64)
            gap = float((embed_ref(geom, B, False)["dw"] - ref["dw"]).norm())
            assert float((got - ref["dw"]).norm()) < 0.1 * gap, what


# ============================================================================ per-operator LayerNorm (any H)
def ln_case(M, Hn):
    g = cpu_gen(M * 10000 + Hn)
    x = torch.randn(M, Hn, generator=g)
    x[0] += 1000.0
    return (x, torch.randn(Hn, generator=g), torch.randn(Hn, generator=g), torch.randn(M, Hn, generator=g),
            torch.randn(M, Hn, generator=g))


@pytest.mark.parametrize("M", [1, 9, 4097])
@pytest.mark.parametrize("Hn", [8, 16, 32, 64, 255, 256, 257, 768, 8192])
def test_ln_fwd_bwd_any_width_vs_fp64(Hn, M):
    x, gamma, beta, dy, dres = ln_case(M, Hn)
    y, mu, rs = R.layer_norm(x, gamma, beta, EPS32)
    tm, tr, k = ln_stat_tols(mu, rs)
    ty = 4e-6 * gamma.abs().to(f64) * k[:, None] + ulp(y, 23)
    xg, gg, bg = x.to(DEV), gamma.to(DEV), beta.to(DEV)
    for mode in (0, 1, 2):
        what = f"H={Hn} M={M} y_bf16={mode}"
        out = nan((M, Hn), bf16 if mode == 1 else f32)
        mean, rstd = nan(M), nan(M)
        call("vit3d_ln_fwd", ptr(xg), ptr(gg), ptr(bg), ptr(out), mode, ptr(mean), ptr(rstd), M, Hn, EPS, stream())
        check(mean, mu, tm, "mean " + what)
        check(rstd, rs, tr, "rstd " + what)
        if mode == 0:
            check(out, y, ty, "y " + what)
        elif mode == 1:
            check(out, y, ty + ulp(y, 7), "y " + what)
        else:
            assert bool(((out.view(torch.int32) & 0x1FFF) == 0).all()), "TF32 low mantissa bits " + what
            check(out, y, ty + ulp(y, 10), "y " + what)
    mean, rstd = mu.to(f32), rs.to(f32)
    core = R.layer_norm_bwd(dy, x, mean, rstd, gamma)
    dgamma_abs, dbeta_abs = (dy.to(f64) * core["xhat"]).abs().sum(0), dy.to(f64).abs().sum(0)
    dyg, mg, rg, dresg = dy.to(DEV), mean.to(DEV), rstd.to(DEV), dres.to(DEV)
    g = cpu_gen(M + Hn)
    for has_dres in (False, True):
        what = f"H={Hn} M={M} dres={has_dres}"
        o = core["o"] + dres.to(f64) if has_dres else core["o"]
        mag = core["mag"] + dres.to(f64).abs() if has_dres else core["mag"]
        dx = nan((M, Hn))
        dg0, db0 = acc_start(dgamma_abs, g), acc_start(dbeta_abs, g)
        dgamma, dbeta = dg0.to(DEV), db0.to(DEV)
        call("vit3d_ln_bwd", ptr(dyg), ptr(xg), ptr(mg), ptr(rg), ptr(gg), ptr(dresg) if has_dres else None, ptr(dx),
             ptr(dgamma), ptr(dbeta), M, Hn, stream())
        check(dx, o, 1e-5 * mag.amax(1, keepdim=True), "dx " + what)
        check_colsum(dgamma, dg0, core["dgamma"], dgamma_abs, "dgamma " + what)
        check_colsum(dbeta, db0, core["dbeta"], dbeta_abs, "dbeta " + what)


# ============================================================================ meta-classifier
@pytest.mark.parametrize("C", [1, 2])
@pytest.mark.parametrize("Fn", [3, 5])
@pytest.mark.parametrize("B", [1, 3, 300])
def test_meta_fwd_bwd_vs_fp64(B, Fn, C):
    g = cpu_gen(B * 100 + Fn * 10 + C)
    f = torch.randn(B, Fn, generator=g)
    w, b = torch.randn(C, Fn, generator=g) * 0.5, torch.randn(C, generator=g) * 0.5
    dout = torch.randn(B, C, generator=g)
    fg, wg, bg, doutg = f.to(DEV), w.to(DEV), b.to(DEV), dout.to(DEV)
    what = f"B={B} F={Fn} C={C}"
    out = nan((B, C))
    call("vit3d_meta_fwd", ptr(fg), ptr(wg), ptr(bg), ptr(out), B, Fn, C, stream())
    ref = R.meta_fwd(f, w, b)
    terms = f.to(f64).abs() @ w.to(f64).abs().t() + b.to(f64).abs()
    check(out, ref, 1e-5 * ref * (1 + terms), "out " + what)
    o = out.cpu()                                  # the backward's operand: the reference uses it as it is
    df_ref, dw_ref, db_ref = R.meta_bwd(dout, o, f, w)
    dz_abs = (dout.to(f64) * o.to(f64) * (1 - o.to(f64))).abs()
    dw_abs, db_abs = dz_abs.t() @ f.to(f64).abs(), dz_abs.sum(0)
    dfeats = nan((B, Fn))
    dw0, db0 = acc_start(dw_abs, g), acc_start(db_abs, g)
    dw, db = dw0.to(DEV), db0.to(DEV)
    call("vit3d_meta_bwd", ptr(doutg), ptr(out), ptr(fg), ptr(wg), ptr(dfeats), ptr(dw), ptr(db), B, Fn, C, stream())
    check(dfeats, df_ref, 1e-5 * (dz_abs @ w.to(f64).abs()), "dfeats " + what)
    check_colsum(dw, dw0, dw_ref, dw_abs, "dw " + what)
    check_colsum(db, db0, db_ref, db_abs, "db " + what)


# ============================================================================ element-wise
def gelu_inputs(n, seed):
    g = cpu_gen(seed)
    h = torch.randn(n, generator=g) * 3
    special = torch.tensor([0.0, 1e-3, -1e-3, -0.75, 5.0, -5.0, 10.0, -10.0, 20.0, -20.0])
    h[:min(n, special.numel())] = special[:min(n, special.numel())]
    return h, torch.randn(n, generator=g)


@pytest.mark.parametrize("dtype", [f32, bf16])
def test_gelu_fwd_vs_fp64(dtype):
    n = 2 ** 20 + 3
    h, _ = gelu_inputs(n, 1)
    h = h.to(dtype)
    hg, a = h.to(DEV), nan(n, dtype)
    call("vit3d_gelu_fwd", ptr(hg), ptr(a), n, PREC["fp32" if dtype == f32 else "bf16"], stream())
    ref = R.gelu(h)
    tol = 5e-7 * h.to(f64).abs() + ulp(ref, 23 if dtype == f32 else 7)
    check(a, ref, tol, f"gelu {dtype}")


def mask_of(n, step):
    m = torch.empty(n, dtype=torch.uint8, device=DEV)
    call("vit3d_dropout_mask", ptr(m), n, P_DROP, SEED, SITE, step, stream())
    return m.cpu().to(torch.bool)


@pytest.mark.parametrize("case", ["f32-8", "f32-9", "f32-1M", "f32-1M+3", "bf16-8", "bf16-9", "bf16-1M", "bf16-1M+3",
                                  "bf16-offset"])
def test_gelu_bwd_vs_fp64(case):
    dt, size = case.split("-")
    dtype = f32 if dt == "f32" else bf16
    n = {"8": 8, "9": 9, "1M": 2 ** 20, "1M+3": 2 ** 20 + 3, "offset": 2 ** 20}[size]
    off = 1 if size == "offset" else 0            # one bf16 element: the buffers sit 2 bytes past a 16-byte boundary
    h, da = gelu_inputs(n, n)
    h, da = h.to(dtype), da.to(dtype)
    hg, dag = torch.empty(n + off, device=DEV, dtype=dtype), torch.empty(n + off, device=DEV, dtype=dtype)
    hg[off:], dag[off:] = h.to(DEV), da.to(DEV)
    dh = nan(n + off, dtype)
    call("vit3d_gelu_bwd", ptr(dag[off:]), ptr(hg[off:]), ptr(dh[off:]), n, PREC["fp32" if dt == "f32" else "bf16"], stream())
    ref = da.to(f64) * R.gelu_grad(h)
    fast = dtype == bf16 and n % 8 == 0 and not off
    tol = (1e-3 if fast else 1e-5) * da.to(f64).abs() + (ulp(ref, 7) if dtype == bf16 else 0)
    check(dh[off:], ref, tol, f"gelu_bwd {case}")


@pytest.mark.parametrize("n", [8, 2 ** 20])
@pytest.mark.parametrize("use_step_dev", [False, True])
def test_gelu_dropout_bwd_vs_fp64(n, use_step_dev):
    h, da = gelu_inputs(n, n + 1)
    h, da = h.to(bf16), da.to(bf16)
    step, step_dev = (3, torch.tensor([4], device=DEV, dtype=torch.int32)) if use_step_dev else (7, None)
    dag, hg, dh = da.to(DEV), h.to(DEV), nan(n, bf16)
    call("vit3d_gelu_dropout_bwd", ptr(dag), ptr(hg), ptr(dh), n, PREC["bf16"], P_DROP, SEED, SITE, step, ptr(step_dev),
         stream())
    keep = mask_of(n, 7)
    got = dh.cpu()
    assert bool((got[~keep] == 0).all()), "dropped elements not exactly 0"
    ref = da.to(f64) * DROP_SCALE * R.gelu_grad(h)
    check(got[keep], ref[keep], (1e-3 * DROP_SCALE * da.to(f64).abs() + ulp(ref, 7))[keep], f"gelu_dropout_bwd n={n}")


def dropout_candidates(x, res, keep, dtype):
    """The fp32 values y = keep ? x * scale : 0 (+ residual) may take: product rounded then added, or one fused
    multiply-add; bf16 output rounds each."""
    sc = torch.tensor(DROP_SCALE, dtype=f32)
    xf = x.to(f32)
    prod = torch.where(keep, xf * sc, torch.zeros((), dtype=f32))
    if res is None:
        c = [prod]
    else:
        fused = torch.where(keep, xf.to(f64) * DROP_SCALE + res.to(f64), res.to(f64)).to(f32)
        c = [prod + res.to(f32), fused]
    return [v.to(dtype) for v in c]


def check_dropout(got, cands, what):
    got = got.cpu()
    ok = torch.zeros(got.shape, dtype=torch.bool)
    for c in cands:
        ok |= got == c
    assert bool(ok.all()), f"{what}: {int((~ok).sum())} elements match neither the fused nor the unfused formula"


@pytest.mark.parametrize("use_step_dev", [False, True])
@pytest.mark.parametrize("tail", [0, 1, 2, 3])
@pytest.mark.parametrize("with_res", [False, True])
@pytest.mark.parametrize("dtype", [f32, bf16])
def test_dropout_vs_exported_mask(dtype, with_res, tail, use_step_dev):
    n = 16384 + tail
    g = cpu_gen(n + 2 * with_res)
    x = torch.randn(n, generator=g).to(dtype)
    res = torch.randn(n, generator=g).to(dtype) if with_res else None
    step, step_dev = (3, torch.tensor([4], device=DEV, dtype=torch.int32)) if use_step_dev else (7, None)
    xg, resg, y = x.to(DEV), None if res is None else res.to(DEV), nan(n, dtype)
    call("vit3d_dropout", ptr(xg), ptr(resg), ptr(y), n, int(dtype == f32), P_DROP, SEED, SITE, step, ptr(step_dev), stream())
    keep = mask_of(n, 7)
    assert 0.05 < 1 - keep.float().mean() < 0.15
    check_dropout(y, dropout_candidates(x, res, keep, dtype), f"dropout {dtype} n={n} residual={with_res}")


@pytest.mark.parametrize("with_res", [False, True])
@pytest.mark.parametrize("dtype", [f32, bf16])
def test_dropout_masked_vs_formula(dtype, with_res):
    n = 16384 + 3
    g = cpu_gen(n + with_res)
    x = torch.randn(n, generator=g).to(dtype)
    res = torch.randn(n, generator=g).to(dtype) if with_res else None
    keep = torch.rand(n, generator=g) >= P_DROP
    xg, kg, resg, y = x.to(DEV), keep.to(torch.uint8).to(DEV), None if res is None else res.to(DEV), nan(n, dtype)
    call("vit3d_dropout_masked", ptr(xg), ptr(kg), ptr(resg), ptr(y), n, int(dtype == f32), P_DROP, stream())
    check_dropout(y, dropout_candidates(x, res, keep, dtype), f"dropout_masked {dtype} residual={with_res}")


@pytest.mark.parametrize("n", [1, 15, 16, 17, 81920 * 3 + 5])
def test_u8_to_f32_bit_exact(n):
    g = cpu_gen(n)
    x = torch.randint(0, 256, (n,), generator=g, dtype=torch.uint8)
    mean = torch.tensor(41.7, dtype=f32)
    xg, y = x.to(DEV), nan(n)
    call("vit3d_u8_to_f32", ptr(xg), ptr(y), n, float(mean), stream())
    assert torch.equal(y.cpu(), x.to(f32) - mean)
