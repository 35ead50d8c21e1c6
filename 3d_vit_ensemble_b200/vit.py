"""Drop-in `models.modeling` surface of evapachetti/3d_vit_ensemble on B200 kernels.

Same class names, constructor and ``forward`` signatures, parameter creation order (so the
same torch seed yields the same initial weights) and ``state_dict`` keys as the reference
``models/modeling.py``; the arithmetic runs in libvit3d_sm100.so.  The scripts' call pattern
is unchanged::

    from models.modeling import VisionTransformer, TransformerEnsemble
    model = VisionTransformer(config, 128, zero_head=True, num_classes=1).to("cuda")
    loss = model(x, y, weights); loss.backward()          # train_baseline_cv.py:171-176
    logits, attn, enc = model(x)                          # train_baseline_cv.py:79-80
    probs = TransformerEnsemble(m5, m9, m11, in_features=1)(x)

There is no CPU path: calling a module with CPU tensors raises.
"""
from __future__ import annotations

import copy
import math

import torch
import torch.nn as nn
from torch.nn import Conv3d, Dropout, LayerNorm, Linear

from . import functional as F
from . import fused_train
from ._lib import ACT_GELU, ACT_NONE, Vit3dError

Z_SIZE = 5  # slices per volume (modeling.py:134)


def _triple(size):
    if isinstance(size, (tuple, list)):
        if len(size) == 3:
            return tuple(int(s) for s in size)
        if len(size) == 2:
            return (int(size[0]), int(size[1]), Z_SIZE)
    return (int(size), int(size), Z_SIZE)


class Attention(nn.Module):
    """modeling.py:55-99.  q/k/v run as one packed [3A, H] GEMM."""

    def __init__(self, config, vis):
        super().__init__()
        self.vis = vis
        self.num_attention_heads = config.transformer["num_heads"]
        self.attention_head_size = int(config.hidden_size / self.num_attention_heads)
        self.all_head_size = self.num_attention_heads * self.attention_head_size
        self.query = Linear(config.hidden_size, self.all_head_size)
        self.key = Linear(config.hidden_size, self.all_head_size)
        self.value = Linear(config.hidden_size, self.all_head_size)
        self.out = Linear(config.hidden_size, config.hidden_size)
        self.attn_dropout = Dropout(config.transformer["attention_dropout_rate"])
        self.proj_dropout = Dropout(config.transformer["attention_dropout_rate"])
        self.precision = F.get_precision()
        self._site = 0

    def forward(self, hidden_states, residual=None, next_ln=None):
        """next_ln (inference): the LayerNorm that consumes `residual + out`; when the fused kernel applies it
        the call returns (out, weights, LN(out)) - otherwise the third item is None."""
        prec = self.precision
        if torch.is_grad_enabled() or not hidden_states.is_cuda:
            w = torch.cat((self.query.weight, self.key.weight, self.value.weight), dim=0)
            b = torch.cat((self.query.bias, self.key.bias, self.value.bias), dim=0)
            qkv = F.linear(hidden_states, w, b, prec=prec)
            ctx, weights = F.AttnCoreFn.apply(qkv, self.num_attention_heads, bool(self.vis), prec)
        elif prec == "bf16" and F.qkv_attn_supported(hidden_states, self.num_attention_heads):
            # one kernel: the q|k|v matrix stays on chip
            _, b, w_lp = F.packed_qkv(self, prec)
            ctx, weights = F.qkv_attn(hidden_states, w_lp, b, self.num_attention_heads, bool(self.vis))
        else:
            qkv = F.linear_packed(hidden_states, *F.packed_qkv(self, prec), prec)
            ctx, weights = F.AttnCoreFn.apply(qkv, self.num_attention_heads, bool(self.vis), prec)
        p = self.attn_dropout.p
        if p > 0.0 and self.training:
            raise Vit3dError("attention_dropout_rate > 0 is not implemented (the reference config fixes it at 0.0, "
                             "tools.py:93)")
        if next_ln is not None and residual is not None and F.linear_ln_supported(ctx, self.out.weight, prec):
            out, normed = F.linear_ln(ctx, self.out.weight, self.out.bias, residual, next_ln.weight, next_ln.bias,
                                      next_ln.eps)
            return out, weights, normed
        out = F.linear(ctx, self.out.weight, self.out.bias, residual=residual, prec=prec, out_f32=True)
        if next_ln is not None:
            return out, weights, None
        return out, weights


class Mlp(nn.Module):
    """modeling.py:102-124: fc1 -> exact GELU -> Dropout -> fc2 -> Dropout."""

    def __init__(self, config):
        super().__init__()
        self.fc1 = Linear(config.hidden_size, config.transformer["mlp_dim"])
        self.fc2 = Linear(config.transformer["mlp_dim"], config.hidden_size)
        self.dropout = Dropout(config.transformer["dropout_rate"])
        self._init_weights()
        self.precision = F.get_precision()
        self._site = 1

    def _init_weights(self):
        nn.init.xavier_uniform_(self.fc1.weight)
        nn.init.xavier_uniform_(self.fc2.weight)
        nn.init.normal_(self.fc1.bias, std=1e-6)
        nn.init.normal_(self.fc2.bias, std=1e-6)

    def forward(self, x, residual=None, step=None, next_ln=None, final=False):
        """next_ln (inference): LayerNorm applied to the block output inside the fc2 kernel; the call then
        returns (out, LN(out) or None).  final=True (last Block, next_ln = encoder_norm): the fused kernel
        writes ONLY the fp32 LayerNorm output and the call returns (None, LN(out)); if the fused kernel
        cannot run it returns (out, None) like the other fallbacks."""
        if next_ln is not None:
            prec = self.precision
            infer = (not (self.training and self.dropout.p > 0.0) and residual is not None
                     and not torch.is_grad_enabled())
            can_fuse = (infer and prec == "bf16" and self.fc1.weight.is_contiguous()
                        and self.fc2.weight.is_contiguous()
                        and F.mlp_fused_ln_supported(x.numel() // x.shape[-1], x.shape[-1], self.fc1.weight.shape[0]))
            if final:
                if can_fuse:
                    return None, F.mlp_fused_final_ln(x, self.fc1.weight, self.fc1.bias, self.fc2.weight, self.fc2.bias,
                                                      residual, next_ln.weight, next_ln.bias, next_ln.eps)
                return self.forward(x, residual=residual, step=step), None
            if can_fuse:
                # one kernel: fc1 -> GELU -> fc2 -> + residual -> next LayerNorm
                return F.mlp_fused_ln(x, self.fc1.weight, self.fc1.bias, self.fc2.weight, self.fc2.bias, residual,
                                      next_ln.weight, next_ln.bias, next_ln.eps)
            if infer:
                h = F.linear(x, self.fc1.weight, self.fc1.bias, act=ACT_GELU, prec=prec)
                if F.linear_ln_supported(h, self.fc2.weight, prec):
                    return F.linear_ln(h, self.fc2.weight, self.fc2.bias, residual, next_ln.weight, next_ln.bias,
                                       next_ln.eps)
                return F.linear(h, self.fc2.weight, self.fc2.bias, residual=residual, prec=prec, out_f32=True), None
            return self.forward(x, residual=residual, step=step), None
        prec = self.precision
        p = self.dropout.p
        train = self.training and p > 0.0
        if train and step is None:
            step = F.next_dropout_step()
        if (not train and prec == "bf16" and residual is not None and not torch.is_grad_enabled()
                and x.is_cuda and self.fc1.weight.is_contiguous() and self.fc2.weight.is_contiguous()
                and F.mlp_fused_supported(x.numel() // x.shape[-1], x.shape[-1], self.fc1.weight.shape[0])):
            # inference: one kernel, the (M, mlp_dim) intermediate stays in TMEM / shared memory
            return F.mlp_fused(x, self.fc1.weight, self.fc1.bias, self.fc2.weight, self.fc2.bias, residual)
        if train and F._STATE["mask_override"] is None:
            # Dropout after the GELU rides along with fc1: applied in place on its output, undone inside the
            # GELU backward kernel (no separate pass over the (M, mlp_dim) gradient)
            seed = torch.initial_seed() & 0xFFFFFFFFFFFFFFFF
            h = F.linear(x, self.fc1.weight, self.fc1.bias, act=ACT_GELU, prec=prec, drop=(p, seed, self._site, step))
        else:
            h = F.linear(x, self.fc1.weight, self.fc1.bias, act=ACT_GELU, prec=prec)
            h = F.dropout(h, p, train, self._site, step)
        if train:
            # Dropout follows fc2 and precedes the residual add (modeling.py:123, :196)
            y = F.linear(h, self.fc2.weight, self.fc2.bias, prec=prec, out_f32=True)
            return F.dropout(y, p, True, self._site + 1, step, residual=residual)
        return F.linear(h, self.fc2.weight, self.fc2.bias, residual=residual, prec=prec, out_f32=True)


class Embeddings(nn.Module):
    """modeling.py:127-175 (non-hybrid): patch Conv3d + cls token + position embeddings + Dropout."""

    def __init__(self, config, img_size, in_channels=1):
        super().__init__()
        self.hybrid = None
        self.z_size = Z_SIZE
        img_size = (img_size, img_size, self.z_size)
        if config.patches.get("grid") is not None:
            raise NotImplementedError("the ResNetV2 hybrid stem is unreachable from the reference's configs "
                                      "(tools.py:87) and is out of scope")
        patch_size = _triple(config.patches["size"])
        n_patches = (img_size[0] // patch_size[0]) * (img_size[1] // patch_size[1]) * (img_size[2] // patch_size[2])
        self.hybrid = False
        self.patch_embeddings = Conv3d(in_channels=in_channels, out_channels=config.hidden_size,
                                       kernel_size=patch_size, stride=patch_size)
        self.position_embeddings = nn.Parameter(torch.zeros(1, n_patches + 1, config.hidden_size))
        self.cls_token = nn.Parameter(torch.zeros(1, 1, config.hidden_size))
        self.dropout = Dropout(config.transformer["dropout_rate"])
        self.precision = F.get_precision()

    def forward(self, x, step=None):
        tok = F.PatchEmbedFn.apply(x, self.patch_embeddings.weight, self.patch_embeddings.bias, self.cls_token,
                                   self.position_embeddings, self.precision)
        p = self.dropout.p
        if self.training and p > 0.0:
            if step is None:
                step = F.next_dropout_step()
            tok = F.dropout(tok, p, True, 0, step)
        return tok


class Block(nn.Module):
    """modeling.py:178-197: x + Attn(LN(x)); x + Mlp(LN(x)), both LayerNorm eps=1e-6."""

    def __init__(self, config, vis):
        super().__init__()
        self.hidden_size = config.hidden_size
        self.attention_norm = LayerNorm(config.hidden_size, eps=1e-6)
        self.ffn_norm = LayerNorm(config.hidden_size, eps=1e-6)
        self.ffn = Mlp(config)
        self.attn = Attention(config, vis)
        self.precision = F.get_precision()

    def forward(self, x, step=None, normed=None, next_ln=None, final=False):
        """The reference signature is forward(x).  `normed` / `next_ln` are the inference fast path of
        Encoder.forward: `normed` = attention_norm(x) already produced by the previous block's fc2 kernel,
        `next_ln` = the LayerNorm that will consume this block's output (the next block's attention_norm);
        with next_ln the call returns (x, weights, next_ln(x) or None).  final=True: this is the last Block and
        next_ln the encoder_norm - when the fused kernel runs, x comes back as None (only next_ln(x), fp32, exists)."""
        prec = self.precision
        x = x.float()
        h = x
        lp = {"bf16": 1, "tf32": 2}.get(prec, 0)     # LayerNorm output feeds a GEMM: bf16 / TF32-rounded / fp32
        fuse = prec == "bf16" and not torch.is_grad_enabled() and x.is_cuda
        xn = normed
        if xn is None:
            xn = F.LayerNormFn.apply(x, self.attention_norm.weight, self.attention_norm.bias, self.attention_norm.eps, lp)
        if fuse:
            x, weights, xn = self.attn(xn, residual=h, next_ln=self.ffn_norm)
        else:
            x, weights = self.attn(xn, residual=h)
            xn = None
        h = x
        if xn is None:
            xn = F.LayerNormFn.apply(x, self.ffn_norm.weight, self.ffn_norm.bias, self.ffn_norm.eps, lp)
        if next_ln is not None and fuse:
            x, xn_next = self.ffn(xn, residual=h, step=step, next_ln=next_ln, final=final)
            return x, weights, xn_next
        x = self.ffn(xn, residual=h, step=step)
        if next_ln is not None:
            return x, weights, None
        return x, weights


class Encoder(nn.Module):
    """modeling.py:237-254."""

    def __init__(self, config, vis):
        super().__init__()
        self.vis = vis
        self.layer = nn.ModuleList()
        self.encoder_norm = LayerNorm(config.hidden_size, eps=1e-6)
        for _ in range(config.transformer["num_layers"]):
            layer = Block(config, vis)
            self.layer.append(copy.deepcopy(layer))
        for i, blk in enumerate(self.layer):       # dropout sites: 0 = embeddings, then 2 per block
            blk.ffn._site = 1 + 2 * i
        self.precision = F.get_precision()

    def forward(self, hidden_states, step=None):
        attn_weights = []
        if self.training and step is None:
            step = F.next_dropout_step()
        # inference in BF16 mode: each block's fc2 kernel also applies the NEXT block's attention_norm
        chain = (self.precision == "bf16" and not torch.is_grad_enabled() and hidden_states.is_cuda)
        normed = None
        n_layers = len(self.layer)
        for i, layer_block in enumerate(self.layer):
            if chain and i + 1 < n_layers:
                hidden_states, weights, normed = layer_block(hidden_states, step=step, normed=normed,
                                                             next_ln=self.layer[i + 1].attention_norm)
            elif chain:
                # last Block: encoder_norm rides in its MLP kernel, which then writes only `encoded`
                hidden_states, weights, encoded = layer_block(hidden_states, step=step, normed=normed,
                                                              next_ln=self.encoder_norm, final=True)
                if self.vis:
                    attn_weights.append(weights)
                if encoded is not None:
                    return encoded, attn_weights
                break
            else:
                hidden_states, weights = layer_block(hidden_states, step=step, normed=normed)
                normed = None
            if self.vis:
                attn_weights.append(weights)
        encoded = F.LayerNormFn.apply(hidden_states, self.encoder_norm.weight, self.encoder_norm.bias,
                                      self.encoder_norm.eps, 0)
        return encoded, attn_weights


class Transformer(nn.Module):
    """modeling.py:257-266."""

    def __init__(self, config, img_size, vis):
        super().__init__()
        self.embeddings = Embeddings(config, img_size=img_size)
        self.encoder = Encoder(config, vis)

    def forward(self, input_ids, step=None):
        if self.training and step is None:
            step = F.next_dropout_step()
        embedding_output = self.embeddings(input_ids, step=step)
        encoded, attn_weights = self.encoder(embedding_output, step=step)
        return encoded, attn_weights


class VisionTransformer(nn.Module):
    """modeling.py:269-288.  ``precision`` ('fp32' | 'tf32' | 'bf16') is the only addition."""

    def __init__(self, config, img_size=224, num_classes=21843, zero_head=False, vis=True, precision=None):
        super().__init__()
        self.num_classes = num_classes
        self.zero_head = zero_head
        self.classifier = config.classifier
        self.config = config
        self.img_size = img_size
        self.transformer = Transformer(config, img_size, vis)
        self.head = Linear(config.hidden_size, num_classes)
        self.input_mean = 0.0      # N2: subtracted from uint8 volumes on the device (tools.normalize's mean)
        self.set_precision(precision or F.get_precision())

    def set_precision(self, precision: str):
        if precision not in ("fp32", "tf32", "bf16"):
            raise ValueError(precision)
        for m in self.modules():
            if hasattr(m, "precision"):
                m.precision = precision
        self.precision = precision
        return self

    def forward(self, x, labels=None, weights=None):
        F._need_cuda(x)
        if x.dtype == torch.uint8:          # N2: raw 8-bit volumes; (u8 - mean) happens on the device
            x = F.u8_volumes_to_f32(x, self.input_mean)
        if labels is not None and fused_train.supported(self, x):
            # BF16 mode, hidden 256: forward + loss with ONE autograd node whose backward is the fused kernel
            # sequence of fused_train.py (the per-operator Functions below stay the generic path)
            return fused_train.loss(self, x, labels, weights)
        x, attn_weights = self.transformer(x)
        logits = F.linear(x[:, 0], self.head.weight, self.head.bias, prec="fp32", out_f32=True)
        if labels is not None:
            if self.num_classes != 1:
                raise Vit3dError("the BCE loss path needs num_classes == 1 (as in the reference scripts)")
            return F.BceLogitsFn.apply(logits.view(-1, self.num_classes), labels.view(-1).unsqueeze(dim=1), weights)
        return logits, attn_weights, x

    def load_from(self, weights):
        raise NotImplementedError("importing JAX .npz checkpoints (modeling.py:291-344) is never called by the "
                                  "reference scripts and is out of scope; use load_state_dict")


class TransformerEnsemble(nn.Module):
    """modeling.py:347-356: member logits -> cat -> Linear -> sigmoid."""

    def __init__(self, *transformers, in_features=3, n_classes=1):
        super().__init__()
        self.transformers = nn.ModuleList(transformers)
        self.classifier = nn.Linear(len(transformers) * in_features, n_classes)

    def forward(self, x):
        if x.dtype == torch.uint8:          # N2: convert once for all members (they share input_mean of member 0)
            x = F.u8_volumes_to_f32(x, self.transformers[0].input_mean)
        outputs = [transformer(x)[0] for transformer in self.transformers]
        concatenated_output = torch.cat(outputs, dim=1)
        return F.MetaFn.apply(concatenated_output, self.classifier.weight, self.classifier.bias)
