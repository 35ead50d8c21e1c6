"""Fused BF16 training step of a VisionTransformer (SURVEY.md §8 a8): `loss = model(x, y, w); loss.backward()`
(train_baseline_cv.py:171-176) as ONE explicit kernel sequence instead of one autograd node per operator.

What the per-operator path (functional.py) pays and this one does not:
  * residual-gradient adds, dtype copies, zero fills and torch.cat run as framework kernels  -> none here: the
    LayerNorm backward kernel adds the skip gradient, emits the bf16 operand of the next GEMMs and the bias
    gradient's column sums in the same pass (vit3d_ln256_bwd);
  * separate Dropout / GELU' / column-sum passes over the [M, mlp_dim] tensors -> keep masks are bit arrays made
    by one launch per step (vit3d_dropout_bits) and applied inside the GEMM epilogues; the fc1 epilogue saves
    gelu'(pre) x mask instead of pre, and dgrad(fc2) -> x that factor -> dgrad(fc1) + fc1-bias column sums are ONE
    kernel (vit3d_mlp_bwd): the [M, mlp_dim] gradient is written once, for the weight-gradient GEMMs;
  * bf16 / transposed-bf16 weight shadows re-derived by ~80 cast / transpose launches after every optimizer
    step -> one launch over a device job table (vit3d_refresh_shadows), into persistent buffers;
  * q, k, v as one packed projection without torch.cat: packed shadows, and the packed weight gradient lands in
    the three parameters' gradients directly (vit3d_wgrad with row segments).

Per encoder Block: 5 launches forward (+1 mask launch on a side stream), 10 backward; one launch per step sums the
weight-gradient partial tiles.  Reference line numbers: models/modeling.py.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional

import numpy as np
import torch

from . import _lib
from . import functional as F
from ._lib import PREC, call, ptr, stream

_BF16 = PREC["bf16"]
_JOB_DTYPE = np.dtype([("src", "<u8"), ("dst", "<u8"), ("rows", "<i4"), ("cols", "<i4"), ("ld", "<i4"), ("kind", "<i4"),
                       ("tile0", "<i4"), ("tiles_c", "<i4")])
K_BF16, K_BF16_T, K_F16, K_TF32, K_F32 = 0, 1, 2, 3, 4


class _WgradJob(C.Structure):
    """include/vit3d.h: record of vit3d_wgrad_reduce (VIT3D_WGRAD_JOB_BYTES = 64)."""
    _fields_ = [("ws", C.c_void_p), ("dst", C.c_void_p * 3), ("seg_rows", C.c_int), ("rows", C.c_int), ("cols", C.c_int),
                ("bn", C.c_int), ("splits", C.c_int), ("tiles_n", C.c_int), ("block0", C.c_int), ("pad", C.c_int)]


class _Wgrads:
    """The weight-gradient GEMMs of one backward pass.  Default: split-K work items accumulate into the gradients with
    fp32 vector atomics.  `functional._STATE["wgrad_partial"] = True`: every work item stores its partial tile into one
    workspace (plain stores) and ONE reduce launch at the end adds them to the gradients - built on the estimate
    that the atomics of 148 partial tiles cost ~20 us per GEMM; MEASURED slower (conf 18, batch 256: 4.52 ms per step
    against 4.28 ms): the 1.2 GB of extra HBM traffic costs more than the atomics, which the L2 absorbs."""

    def __init__(self, M, shapes, dev):
        self.M = M
        self.partial = F._STATE.get("wgrad_partial", False) and all(N % 128 == 0 for N, _ in shapes)
        self.jobs = (_WgradJob * max(1, len(shapes)))()
        self.n = 0
        self.off = 0
        self.ws = None
        if self.partial:
            L = _lib.lib()
            total = sum(L.vit3d_wgrad_ws_bytes(M, N, K) for N, K in shapes)
            self.ws = torch.empty(total // 4, device=dev, dtype=torch.float32)

    def __call__(self, dy, x, dsts, seg_rows, N, K, st):
        if not self.partial:
            d = list(dsts) + [None] * (3 - len(dsts))
            call("vit3d_wgrad", ptr(dy), ptr(x), d[0], d[1], d[2], seg_rows, self.M, N, K, st)
            return
        bn, sp = C.c_int(0), C.c_int(0)
        wp = self.ws.data_ptr() + self.off
        call("vit3d_wgrad_partial", ptr(dy), ptr(x), wp, self.M, N, K, C.byref(bn), C.byref(sp), st)
        j = self.jobs[self.n]
        j.ws = wp
        for i in range(3):
            j.dst[i] = dsts[i] if i < len(dsts) else None
        j.seg_rows, j.rows, j.cols, j.bn, j.splits, j.tiles_n = seg_rows, N, K, bn.value, sp.value, K // bn.value
        self.n += 1
        self.off += _lib.lib().vit3d_wgrad_ws_bytes(self.M, N, K)

    def finish(self, st):
        if self.partial and self.n:
            call("vit3d_wgrad_reduce", C.cast(self.jobs, C.c_void_p), self.n, st)


def supported(model, x) -> bool:
    """Can the fused step serve this call?  BF16 mode, hidden 256, 65 tokens, CUDA, num_classes 1."""
    if getattr(model, "precision", None) != "bf16" or not x.is_cuda or model.num_classes != 1:
        return False
    if F._STATE.get("fused_train", True) is False:
        return False
    emb = model.transformer.embeddings
    if x.dim() != 5 or x.shape[1] != 1:
        return False
    w = emb.patch_embeddings.weight
    S = emb.position_embeddings.shape[1]
    blk = model.transformer.encoder.layer[0]
    d = blk.ffn.fc1.weight.shape[0]
    if blk.attn.attn_dropout.p > 0.0:
        return False
    B = x.shape[0]
    if not _lib.lib().vit3d_train_supported(B, S, w.shape[0], blk.attn.num_attention_heads, d):
        return False
    # the tensor-core patch embedding must serve the geometry as well (whole volumes per 128-row tile)
    return (x.shape[2] // w.shape[2]) * (x.shape[3] // w.shape[3]) + 1 == S and w.shape[4] == x.shape[4]


class TrainPlan:
    """Persistent low-precision weight shadows of one model + the device job table that rewrites all of them
    in one launch.  Buffers never move, so CUDA graphs that read them stay valid across optimizer steps."""

    def __init__(self, model):
        self.model = model
        enc = model.transformer.encoder
        emb = model.transformer.embeddings
        self.L = len(enc.layer)
        self.H = emb.patch_embeddings.weight.shape[0]
        self.d = enc.layer[0].ffn.fc1.weight.shape[0]
        dev = emb.patch_embeddings.weight.device
        self.device = dev
        H, d, L = self.H, self.d, self.L
        per_layer_bf16 = 2 * 3 * H * H + 2 * H * H + 4 * H * d
        self.lp = torch.empty(L * per_layer_bf16, device=dev, dtype=torch.bfloat16)
        kp = emb.patch_embeddings.weight[0].numel()
        self.f32 = torch.empty(L * 3 * H + H * kp, device=dev, dtype=torch.float32)
        jobs = []
        self.layers: List[Dict[str, torch.Tensor]] = []
        off = 0
        foff = 0

        def take(n, shape):
            nonlocal off
            t = self.lp[off:off + n].view(*shape)
            off += n
            return t

        def job(src, dst_ptr, rows, cols, ld, kind):
            jobs.append((src, dst_ptr, rows, cols, ld, kind))

        self._params = []
        for blk in enc.layer:
            a, f = blk.attn, blk.ffn
            sh = {"wqkv": take(3 * H * H, (3 * H, H)), "wqkv_t": take(3 * H * H, (H, 3 * H)),
                  "wo": take(H * H, (H, H)), "wo_t": take(H * H, (H, H)),
                  "w1": take(H * d, (d, H)), "w1_t": take(H * d, (H, d)),
                  "w2": take(H * d, (H, d)), "w2_t": take(H * d, (d, H))}
            sh["bqkv"] = self.f32[foff:foff + 3 * H]
            foff += 3 * H
            for j, lin in enumerate((a.query, a.key, a.value)):
                job(lin.weight, sh["wqkv"].data_ptr() + j * H * H * 2, H, H, H, K_BF16)
                job(lin.weight, sh["wqkv_t"].data_ptr() + j * H * 2, H, H, 3 * H, K_BF16_T)
                job(lin.bias, sh["bqkv"].data_ptr() + j * H * 4, 1, H, H, K_F32)
            job(a.out.weight, sh["wo"].data_ptr(), H, H, H, K_BF16)
            job(a.out.weight, sh["wo_t"].data_ptr(), H, H, H, K_BF16_T)
            job(f.fc1.weight, sh["w1"].data_ptr(), d, H, H, K_BF16)
            job(f.fc1.weight, sh["w1_t"].data_ptr(), d, H, d, K_BF16_T)
            job(f.fc2.weight, sh["w2"].data_ptr(), H, d, d, K_BF16)
            job(f.fc2.weight, sh["w2_t"].data_ptr(), H, d, H, K_BF16_T)
            self.layers.append(sh)
        self.w_patch = self.f32[foff:foff + H * kp].view(H, kp)
        job(emb.patch_embeddings.weight, self.w_patch.data_ptr(), H, kp, kp, K_TF32)
        self._job_src = [j[0] for j in jobs]
        self._job_rest = [j[1:] for j in jobs]
        self.jobs_dev = None
        self._sig = None
        self._build_table()

    def _build_table(self):
        arr = np.zeros(len(self._job_src), dtype=_JOB_DTYPE)
        t0 = 0
        for i, (src, (dst, rows, cols, ld, kind)) in enumerate(zip(self._job_src, self._job_rest)):
            if not src.is_contiguous() or src.dtype != torch.float32:
                raise _lib.Vit3dError("fused training needs contiguous fp32 parameters")
            tiles_c = (cols + _lib.SHADOW_TILE - 1) // _lib.SHADOW_TILE
            arr[i] = (src.data_ptr(), dst, rows, cols, ld, kind, t0, tiles_c)
            t0 += tiles_c * ((rows + _lib.SHADOW_TILE - 1) // _lib.SHADOW_TILE)
        self.total_tiles = t0
        self.njobs = len(arr)
        host = torch.from_numpy(arr.view(np.uint8).copy())
        self.jobs_dev = host.to(self.device)
        self._ptrs = tuple(s.data_ptr() for s in self._job_src)

    def side_stream(self):
        if getattr(self, "_side", None) is None:
            self._side = torch.cuda.Stream(device=self.device)
        return self._side

    def signature(self):
        return (tuple(s._version for s in self._job_src), F._STATE.get("epoch", 0))

    def refresh(self, step_dev=None, force=False):
        """Rewrites the shadows when a weight changed since the last refresh (optimizer step, load_state_dict,
        .to()).  step_dev: device counter the kernel increments (CUDA-graph replays)."""
        ptrs = tuple(s.data_ptr() for s in self._job_src)
        if ptrs != self._ptrs:          # parameters were re-homed (FlatArena, .to()): new source addresses
            self._build_table()
            self._sig = None
        sig = self.signature()
        if not force and sig == self._sig and step_dev is None:
            return
        call("vit3d_refresh_shadows", ptr(self.jobs_dev), self.njobs, self.total_tiles, ptr(step_dev), stream())
        self._sig = sig


def plan_of(model) -> TrainPlan:
    p = getattr(model, "_train_plan", None)
    if p is None or p.device != model.head.weight.device:
        p = TrainPlan(model)
        object.__setattr__(model, "_train_plan", p)
    return p


def _pack_mask_bits(mask: torch.Tensor, dev) -> torch.Tensor:
    """keep mask (bool / uint8, any shape) -> little-endian bit array (uint8), element e = byte e//8, bit e%8."""
    m = mask.to(device=dev).reshape(-1).to(torch.uint8)
    assert m.numel() % 32 == 0
    wts = (2 ** torch.arange(8, device=dev, dtype=torch.int32))
    return (m.view(-1, 8).to(torch.int32) * wts).sum(dim=1).to(torch.uint8)


class _Grads:
    """Where each parameter's gradient accumulates: its existing `.grad` (flat arena) when direct accumulation
    is on, else a zeroed temporary handed back to autograd."""

    def __init__(self, params):
        self.targets = {}
        self.temps = {}
        for p in params:
            t = F._grad_target(p) if p.requires_grad else None
            if t is None:
                t = torch.zeros_like(p, memory_format=torch.contiguous_format)
                self.temps[id(p)] = t
            self.targets[id(p)] = t

    def __call__(self, p):
        return ptr(self.targets[id(p)])

    def result(self, params):
        return tuple(self.temps.get(id(p)) for p in params)


def forward(model, x, labels, pos_weight, step: Optional[int] = None):
    """Training-mode (or eval-mode) forward that keeps what backward needs.  Returns (loss, saved)."""
    plan = plan_of(model)
    step_dev = F._STATE.get("step_dev")
    plan.refresh()
    tr = model.transformer
    emb, enc = tr.embeddings, tr.encoder
    dev = x.device
    x = F._c(x.float())
    B = x.shape[0]
    H, d, L = plan.H, plan.d, plan.L
    S = emb.position_embeddings.shape[1]
    M = B * S
    heads = enc.layer[0].attn.num_attention_heads
    D = H // heads
    p = float(emb.dropout.p)
    training = model.training and p > 0.0
    st = stream()
    bf, f32 = torch.bfloat16, torch.float32

    # ---- dropout keep bits of every site of this step: one launch (or injected masks in parity tests)
    bits0 = None
    bits1 = [None] * L
    bits2 = [None] * L
    bits_ready = []          # per Block: event after which its two masks exist (side stream)
    scale = 1.0
    if training:
        scale = 1.0 / (1.0 - p)
        nel = [M * H] + [n for _ in range(L) for n in (M * d, M * H)]
        sites = list(range(1 + 2 * L))
        offs = np.concatenate([[0], np.cumsum(nel)]) // 8
        allbits = torch.empty(int(offs[-1]), device=dev, dtype=torch.uint8)
        override = F._STATE["mask_override"]
        if override is not None:
            for s_, (o0, o1) in enumerate(zip(offs[:-1], offs[1:])):
                if s_ not in override:
                    raise _lib.Vit3dError(f"mask injection: no mask for dropout site {s_}")
                allbits[int(o0):int(o1)] = _pack_mask_bits(override[s_], dev)
        else:
            if step is None:
                step = F.next_dropout_step()
            seed = torch.initial_seed() & 0xFFFFFFFFFFFFFFFF
            # the embedding mask is needed at once; the masks of Block l (2 sites, M*(d+H) decisions: ALU-bound Philox,
            # 30 registers, no shared memory) are drawn on a SIDE stream, one launch per Block, and co-reside with the
            # forward's GEMM CTAs (one per SM, half of the issue slots idle) - the main stream waits for Block l's
            # event just before fc1 of Block l.  Inside a CUDA graph these become a parallel branch.
            call("vit3d_dropout_bits", ptr(allbits), 1, (C.c_uint * 1)(0), (C.c_longlong * 1)(nel[0]), p, seed, step,
                 ptr(step_dev), st)
            main = torch.cuda.current_stream(dev)
            side = plan.side_stream()
            side.wait_stream(main)
            allbits.record_stream(side)
            with torch.cuda.stream(side):
                sst = stream()
                for l in range(L):
                    base = allbits[int(offs[1 + 2 * l]):]
                    call("vit3d_dropout_bits", ptr(base), 2, (C.c_uint * 2)(1 + 2 * l, 2 + 2 * l),
                         (C.c_longlong * 2)(nel[1 + 2 * l], nel[2 + 2 * l]), p, seed, step, ptr(step_dev), sst)
                    ev = torch.cuda.Event()
                    ev.record(side)
                    bits_ready.append(ev)
        seg = [allbits[int(o0):int(o1)] for o0, o1 in zip(offs[:-1], offs[1:])]
        bits0 = seg[0]
        bits1 = seg[1::2]
        bits2 = seg[2::2]

    # ---- a1: patch embedding (+cls, +pos), then Dropout + the first attention_norm in one pass
    w = emb.patch_embeddings.weight
    _, _, X, Y, Z = x.shape
    p0, p1, p2 = w.shape[2:]
    tok = torch.empty(B, S, H, device=dev, dtype=f32)
    wsb = _lib.lib().vit3d_patch_embed_ws_bytes(B, X, Y, Z, p0, p1, p2, H, _BF16)
    ws = torch.empty(wsb, device=dev, dtype=torch.uint8)      # only touched when the TMA-gather GEMM cannot serve the geometry
    call("vit3d_patch_embed_fwd", ptr(x), ptr(plan.w_patch), ptr(emb.patch_embeddings.bias), ptr(emb.cls_token),
         ptr(emb.position_embeddings), ptr(tok), B, X, Y, Z, p0, p1, p2, H, _BF16, ptr(ws), wsb, st)
    l0 = enc.layer[0]
    x0 = torch.empty(M, H, device=dev, dtype=f32) if training else tok.view(M, H)
    xn = torch.empty(M, H, device=dev, dtype=bf)
    mean = torch.empty(M, device=dev, dtype=f32)
    rstd = torch.empty(M, device=dev, dtype=f32)
    call("vit3d_ln256_fwd", ptr(tok), ptr(bits0), scale, ptr(x0) if training else None, ptr(l0.attention_norm.weight),
         ptr(l0.attention_norm.bias), ptr(xn), None, ptr(mean), ptr(rstd), M, float(l0.attention_norm.eps), st)

    saved_layers = []
    for i, blk in enumerate(enc.layer):
        sh = plan.layers[i]
        a, f = blk.attn, blk.ffn
        qkv = torch.empty(M, 3 * H, device=dev, dtype=bf)
        call("vit3d_linear_fwd", ptr(xn), H, 0, ptr(sh["wqkv"]), ptr(sh["wqkv"]), ptr(sh["bqkv"]), None, ptr(qkv), 0, None, 0,
             M, 3 * H, H, _BF16, st)
        ctx = torch.empty(M, H, device=dev, dtype=bf)
        call("vit3d_attn_fwd", ptr(qkv), ptr(ctx), None, B, S, heads, D, _BF16, st)
        x1 = torch.empty(M, H, device=dev, dtype=f32)
        xn2 = torch.empty(M, H, device=dev, dtype=bf)
        mean2 = torch.empty(M, device=dev, dtype=f32)
        rstd2 = torch.empty(M, device=dev, dtype=f32)
        call("vit3d_linear_res_train_fwd", ptr(ctx), ptr(sh["wo"]), ptr(a.out.bias), ptr(x0), ptr(x1), None, 1.0,
             ptr(blk.ffn_norm.weight), ptr(blk.ffn_norm.bias), float(blk.ffn_norm.eps), ptr(xn2), ptr(mean2), ptr(rstd2),
             M, H, H, st)
        if bits_ready:
            torch.cuda.current_stream(dev).wait_event(bits_ready[i])
        dact = torch.empty(M, d, device=dev, dtype=bf)       # gelu'(pre) * keep / (1-p): all the backward needs of fc1's output
        act = torch.empty(M, d, device=dev, dtype=bf)
        call("vit3d_fc1_train_fwd", ptr(xn2), ptr(sh["w1"]), ptr(f.fc1.bias), ptr(dact), ptr(act), ptr(bits1[i]), scale,
             M, d, H, st)
        x2 = torch.empty(M, H, device=dev, dtype=f32)
        rec = dict(x0=x0, xn1=xn, mean1=mean, rstd1=rstd, qkv=qkv, ctx=ctx, x1=x1, xn2=xn2, mean2=mean2, rstd2=rstd2,
                   dact=dact, act=act)
        if i + 1 < L:
            nl = enc.layer[i + 1].attention_norm
            xn = torch.empty(M, H, device=dev, dtype=bf)
            mean = torch.empty(M, device=dev, dtype=f32)
            rstd = torch.empty(M, device=dev, dtype=f32)
            call("vit3d_linear_res_train_fwd", ptr(act), ptr(sh["w2"]), ptr(f.fc2.bias), ptr(x1), ptr(x2), ptr(bits2[i]),
                 scale, ptr(nl.weight), ptr(nl.bias), float(nl.eps), ptr(xn), ptr(mean), ptr(rstd), M, H, d, st)
        else:
            call("vit3d_linear_res_train_fwd", ptr(act), ptr(sh["w2"]), ptr(f.fc2.bias), ptr(x1), ptr(x2), ptr(bits2[i]),
                 scale, None, None, 0.0, None, None, None, M, H, d, st)
        saved_layers.append(rec)
        x0 = x2

    # ---- encoder_norm (modeling.py:253), head on the cls rows (:281), BCE-with-logits (:283-286)
    en = enc.encoder_norm
    encd = torch.empty(M, H, device=dev, dtype=f32)
    mean_f = torch.empty(M, device=dev, dtype=f32)
    rstd_f = torch.empty(M, device=dev, dtype=f32)
    call("vit3d_ln256_fwd", ptr(x0), None, 1.0, None, ptr(en.weight), ptr(en.bias), None, ptr(encd), ptr(mean_f), ptr(rstd_f),
         M, float(en.eps), st)
    logits = torch.empty(B, 1, device=dev, dtype=f32)
    call("vit3d_linear_fwd", ptr(encd), S * H, 1, ptr(model.head.weight), None, ptr(model.head.bias), None, ptr(logits), 1,
         None, 0, B, 1, H, PREC["fp32"], st)
    y = F._c(labels.to(device=dev, dtype=f32)).reshape(-1)
    if y.numel() != B:
        raise _lib.Vit3dError("BCE: logits and labels differ in size")
    loss = torch.empty((), device=dev, dtype=f32)
    pw_dev = None
    if isinstance(pos_weight, torch.Tensor) and pos_weight.is_cuda:
        pw_dev, pw = pos_weight.reshape(1).float(), 1.0
    else:
        pw = -1.0 if pos_weight is None else float(pos_weight)
    call("vit3d_bce_logits_fwd", ptr(logits), ptr(y), pw, ptr(pw_dev), ptr(loss), B, st)
    saved = dict(x=x, layers=saved_layers, x_last=x0, mean_f=mean_f, rstd_f=rstd_f, enc=encd, logits=logits, y=y, pw=pw,
                 pw_dev=pw_dev, bits0=bits0, bits1=bits1, bits2=bits2, scale=scale, B=B, S=S, M=M, heads=heads, D=D,
                 training=training)
    return loss, saved


def backward(model, saved, dloss: Optional[torch.Tensor] = None):
    """Gradients of every parameter from `saved` (see forward).  Accumulates into the parameters' `.grad`
    (flat arena) where possible; returns the tuple autograd expects (None where accumulated in place), in
    `model.parameters()` order."""
    gen = backward_steps(model, saved, dloss, ())
    while True:
        try:
            next(gen)
        except StopIteration as e:
            return e.value


def backward_steps(model, saved, dloss: Optional[torch.Tensor] = None, cuts=()):
    """`backward` as a generator: yields the Block index i after the backward of Block i when i is in `cuts` - every
    gradient of the head, encoder_norm and Blocks >= i is complete at that point (data-parallel steps all-reduce that
    part of the flat arena while the rest of the backward runs, graphs.GraphedTrainStep).  The generator's return value
    is `backward`'s."""
    plan = plan_of(model)
    tr = model.transformer
    emb, enc = tr.embeddings, tr.encoder
    params = list(model.parameters())
    G = _Grads(params)
    B, S, M, heads, D = saved["B"], saved["S"], saved["M"], saved["heads"], saved["D"]
    H, d, L = plan.H, plan.d, plan.L
    scale = saved["scale"]
    bits0, bits1, bits2 = saved["bits0"], saved["bits1"], saved["bits2"]
    dev = saved["x"].device
    st = stream()
    bf, f32 = torch.bfloat16, torch.float32

    dlog = torch.empty(B, device=dev, dtype=f32)
    dl = None if dloss is None else F._c(dloss.float())
    call("vit3d_bce_logits_bwd", ptr(saved["logits"]), ptr(saved["y"]), saved["pw"], ptr(saved["pw_dev"]), ptr(dl), ptr(dlog),
         B, st)
    denc = torch.empty(M, H, device=dev, dtype=f32)
    call("vit3d_head_bwd", ptr(dlog), ptr(saved["enc"]), ptr(model.head.weight), ptr(denc), G(model.head.weight),
         G(model.head.bias), B, S, H, st)
    F._grad_done(model.head.weight)
    F._grad_done(model.head.bias)
    en = enc.encoder_norm
    g = torch.empty(M, H, device=dev, dtype=f32)         # dL/d(block output), fp32
    g1 = torch.empty(M, H, device=dev, dtype=f32)
    gb = torch.empty(M, H, device=dev, dtype=bf)          # its bf16 (dropout-masked) copy: GEMM operand
    g1b = torch.empty(M, H, device=dev, dtype=bf)
    dwide = torch.empty(M, d, device=dev, dtype=bf)       # da, overwritten in place by dh
    dctx = torch.empty(M, H, device=dev, dtype=bf)
    dqkv = torch.empty(M, 3 * H, device=dev, dtype=bf)
    dxn = denc                                            # fp32 [M,H] scratch for the dgrad outputs
    fused_mlp = F._STATE.get("fused_mlp_bwd", True) and bool(_lib.lib().vit3d_mlp_bwd_supported(M, H, d))
    wg = _Wgrads(M, [s_ for _ in range(L) for s_ in ((H, d), (d, H), (H, H), (3 * H, H))], dev)
    last = enc.layer[L - 1]
    call("vit3d_ln256_bwd", ptr(denc), ptr(saved["x_last"]), ptr(saved["mean_f"]), ptr(saved["rstd_f"]), ptr(en.weight), None,
         ptr(bits2[L - 1]), scale, 0, ptr(g), ptr(gb), G(en.weight), G(en.bias), G(last.ffn.fc2.bias), M, st)
    F._grad_done(en.weight)
    F._grad_done(en.bias)
    for i in range(L - 1, -1, -1):
        blk = enc.layer[i]
        a, f = blk.attn, blk.ffn
        sh = plan.layers[i]
        r = saved["layers"][i]
        # ---- Mlp backward (modeling.py:118-124): fc2, Dropout + GELU, fc1
        wg(gb, r["act"], [G(f.fc2.weight)], 0, H, d, st)
        if fused_mlp:
            # dgrad(fc2) -> GELU' x mask -> dgrad(fc1) in one kernel: `da` stays on chip, dh is written once
            call("vit3d_mlp_bwd", ptr(gb), ptr(sh["w2_t"]), ptr(sh["w1_t"]), ptr(r["dact"]), ptr(dwide), ptr(dxn),
                 G(f.fc1.bias), M, H, d, st)
            wg(dwide, r["xn2"], [G(f.fc1.weight)], 0, d, H, st)
        else:
            call("vit3d_linear_fwd", ptr(gb), H, 0, ptr(sh["w2_t"]), ptr(sh["w2_t"]), None, None, ptr(dwide), 0, None, 0, M, d,
                 H, _BF16, st)
            call("vit3d_mul_colsum_bwd", ptr(dwide), ptr(r["dact"]), ptr(dwide), G(f.fc1.bias), M, d, st)
            wg(dwide, r["xn2"], [G(f.fc1.weight)], 0, d, H, st)
            call("vit3d_linear_fwd", ptr(dwide), d, 0, ptr(sh["w1_t"]), ptr(sh["w1_t"]), None, None, ptr(dxn), 1, None, 0, M, H,
                 d, _BF16, st)
        # ---- ffn_norm backward + skip gradient; bf16 copy and column sums for the out-projection
        call("vit3d_ln256_bwd", ptr(dxn), ptr(r["x1"]), ptr(r["mean2"]), ptr(r["rstd2"]), ptr(blk.ffn_norm.weight), ptr(g),
             None, 1.0, 0, ptr(g1), ptr(g1b), G(blk.ffn_norm.weight), G(blk.ffn_norm.bias), G(a.out.bias), M, st)
        # ---- Attention backward (modeling.py:78-99)
        wg(g1b, r["ctx"], [G(a.out.weight)], 0, H, H, st)
        call("vit3d_linear_fwd", ptr(g1b), H, 0, ptr(sh["wo_t"]), ptr(sh["wo_t"]), None, None, ptr(dctx), 0, None, 0, M, H, H,
             _BF16, st)
        call("vit3d_attn_bwd_bias", ptr(dctx), ptr(r["qkv"]), ptr(dqkv), G(a.query.bias), G(a.key.bias), G(a.value.bias),
             B, S, heads, D, st)
        wg(dqkv, r["xn1"], [G(a.query.weight), G(a.key.weight), G(a.value.weight)], H, 3 * H, H, st)
        call("vit3d_linear_fwd", ptr(dqkv), 3 * H, 0, ptr(sh["wqkv_t"]), ptr(sh["wqkv_t"]), None, None, ptr(dxn), 1, None, 0,
             M, H, 3 * H, _BF16, st)
        # ---- attention_norm backward + skip gradient; below it: the previous Block's fc2 Dropout, or the embedding Dropout
        an = blk.attention_norm
        if i > 0:
            prev = enc.layer[i - 1]
            call("vit3d_ln256_bwd", ptr(dxn), ptr(r["x0"]), ptr(r["mean1"]), ptr(r["rstd1"]), ptr(an.weight), ptr(g1),
                 ptr(bits2[i - 1]), scale, 0, ptr(g), ptr(gb), G(an.weight), G(an.bias), G(prev.ffn.fc2.bias), M, st)
        else:
            call("vit3d_ln256_bwd", ptr(dxn), ptr(r["x0"]), ptr(r["mean1"]), ptr(r["rstd1"]), ptr(an.weight), ptr(g1),
                 ptr(bits0), scale, 1, ptr(g), None, G(an.weight), G(an.bias), None, M, st)
        if not wg.partial:
            for p_ in blk.parameters():
                F._grad_done(p_)
            if i in cuts and i > 0:
                yield i
    wg.finish(st)                      # one launch: partial tiles of all 4 L weight-gradient GEMMs -> the gradients
    if wg.partial:
        for blk in reversed(list(enc.layer)):
            for p_ in blk.parameters():
                F._grad_done(p_)
    # ---- Embeddings backward (modeling.py:162-174): g = dL/d(tokens) with the embedding Dropout already undone
    x = saved["x"]
    w = emb.patch_embeddings.weight
    _, _, X, Y, Z = x.shape
    p0, p1, p2 = w.shape[2:]
    wsb = _lib.lib().vit3d_patch_embed_ws_bytes(B, X, Y, Z, p0, p1, p2, H, _BF16)
    ws = torch.empty(wsb, device=dev, dtype=torch.uint8)
    call("vit3d_patch_embed_bwd", ptr(x), ptr(g), G(w), G(emb.patch_embeddings.bias), G(emb.cls_token),
         G(emb.position_embeddings), B, X, Y, Z, p0, p1, p2, H, _BF16, ptr(ws), wsb, st)
    if saved.get("need_dx"):       # the input volume's gradient (autograd callers whose x requires grad)
        dx = torch.empty(x.shape, device=dev, dtype=f32)
        call("vit3d_patch_embed_dgrad", ptr(g), ptr(w), ptr(F.lp_weight(w, "tf32_t")), ptr(dx), B, X, Y, Z, p0, p1, p2, H,
             _BF16, ptr(ws), wsb, st)
        saved["dx"] = dx
    for p_ in emb.parameters():
        F._grad_done(p_)
    return G.result(params)


class VitTrainFn(torch.autograd.Function):
    """loss = BCEWithLogits(head(encoder(embeddings(x)))[:,0]) with the whole backward as one node."""

    @staticmethod
    def forward(ctx, model, x, labels, pos_weight, *params):
        loss, saved = forward(model, x, labels, pos_weight)
        saved["need_dx"] = ctx.needs_input_grad[1]
        ctx.model = model
        ctx.saved = saved
        ctx.x_dtype = x.dtype
        return loss

    @staticmethod
    def backward(ctx, dloss):
        grads = backward(ctx.model, ctx.saved, dloss)
        dx = ctx.saved.get("dx")
        ctx.saved = None
        return (None, None if dx is None else dx.to(ctx.x_dtype), None, None) + tuple(grads)


def loss(model, x, labels, pos_weight):
    """Autograd entry: `model(x, labels, weights)` in BF16 mode routes here when `supported`."""
    return VitTrainFn.apply(model, x, labels, pos_weight, *model.parameters())


def loss_and_grads_steps(model, x, labels, pos_weight, cuts):
    """`loss_and_grads` as a generator over the segments `backward_steps(cuts=...)` defines: yields the (static) loss
    tensor after the forward + first backward segment and after every further segment but the last; returns it."""
    with torch.no_grad():
        lo, saved = forward(model, x, labels, pos_weight)
        gen = backward_steps(model, saved, None, cuts)
        while True:
            try:
                next(gen)
            except StopIteration as e:
                grads = e.value
                break
            yield lo
    if any(g is not None for g in grads):
        raise _lib.Vit3dError("loss_and_grads needs every parameter's .grad to be an fp32 buffer it can accumulate into "
                              "(build an optim.FusedSGD / FusedAdam over model.parameters() first)")
    return lo


def loss_and_grads(model, x, labels, pos_weight):
    """Forward + backward without autograd (CUDA-graph capture of a training step: no framework kernels at all).
    Gradients accumulate into the parameters' `.grad` buffers, which must exist (fused optimizers' flat arena)."""
    with torch.no_grad():
        lo, saved = forward(model, x, labels, pos_weight)
        grads = backward(model, saved, None)
    if any(g is not None for g in grads):
        raise _lib.Vit3dError("loss_and_grads needs every parameter's .grad to be an fp32 buffer it can accumulate into "
                              "(build an optim.FusedSGD / FusedAdam over model.parameters() first)")
    return lo
