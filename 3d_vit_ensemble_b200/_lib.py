"""ctypes binding of libvit3d_sm100.so (C ABI: include/vit3d.h).

There is no CPU fallback and no alternative backend: if the shared library is missing or a
tensor is not on a CUDA device the call raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libvit3d_sm100.so")

PREC = {"fp32": 0, "tf32": 1, "bf16": 2}
ACT_NONE, ACT_GELU = 0, 1
SHADOW_TILE = 64          # include/vit3d.h VIT3D_SHADOW_TILE: tile edge of the vit3d_refresh_shadows job table


class Vit3dError(RuntimeError):
    pass


def build(verbose: bool = False) -> str:
    """Compile the library in-tree with nvcc for sm_100a (no GPU needed)."""
    r = subprocess.run(["make", "-C", os.path.join(_HERE, "csrc"), "-j8"], capture_output=True, text=True)
    if r.returncode != 0:
        raise Vit3dError("building libvit3d_sm100.so failed:\n" + r.stdout[-4000:] + r.stderr[-4000:])
    if verbose:
        print(r.stdout[-2000:])
    return LIB_PATH


_lib = None

_p, _i, _f, _ll, _u, _ull, _sz = C.c_void_p, C.c_int, C.c_float, C.c_longlong, C.c_uint, C.c_ulonglong, C.c_size_t

# name -> (restype, argtypes); must list every symbol include/vit3d.h declares (checked by tests)
SIGNATURES = {
    "vit3d_version": (_i, []),
    "vit3d_last_error": (C.c_char_p, []),
    "vit3d_device_info": (_i, [C.POINTER(_i), C.POINTER(_i)]),
    "vit3d_launch_count": (_ull, []),
    "vit3d_set_tuning": (_i, [_i, _i]),
    "vit3d_get_tuning": (_i, [_i]),
    "vit3d_act_bytes": (_i, [_i]),
    "vit3d_tc_supported": (_i, [_i, _i, _i, _i]),
    "vit3d_patch_gather": (_i, [_p, _p, _i, _i, _i, _i, _i, _i, _i, _p]),
    "vit3d_patch_embed_ws_bytes": (_sz, [_i] * 9),
    "vit3d_patch_embed_fwd": (_i, [_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _sz, _p]),
    "vit3d_patch_embed_bwd": (_i, [_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _sz, _p]),
    "vit3d_patch_embed_dgrad": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _sz, _p]),
    "vit3d_ln_fwd": (_i, [_p, _p, _p, _p, _i, _p, _p, _i, _i, _f, _p]),
    "vit3d_ln_bwd": (_i, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _i, _i, _p]),
    "vit3d_linear_fwd": (_i, [_p, _i, _i, _p, _p, _p, _p, _p, _i, _p, _i, _i, _i, _i, _i, _p]),
    "vit3d_linear_ln_fwd": (_i, [_p, _p, _p, _p, _p, _p, _p, _f, _p, _p, _p, _i, _i, _i, _p]),
    "vit3d_linear_ln_supported": (_i, [_i, _i, _i]),
    "vit3d_linear_bwd": (_i, [_p, _i, _p, _i, _i, _p, _p, _p, _i, _i, _p, _p, _i, _i, _i, _i, _p]),
    "vit3d_mlp_fwd": (_i, [_p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _p]),
    "vit3d_mlp_supported": (_i, [_i, _i, _i]),
    "vit3d_mlp_ln_fwd": (_i, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _f, _p, _i, _i, _i, _p]),
    "vit3d_mlp_lnf_fwd": (_i, [_p, _p, _p, _p, _p, _p, _p, _p, _f, _p, _i, _i, _i, _p]),
    "vit3d_mlp_ln_supported": (_i, [_i, _i, _i]),
    "vit3d_attn_fwd": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _p]),
    "vit3d_attn_bwd": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _p]),
    "vit3d_attn_fwd_padded": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _p]),
    "vit3d_attn_padded_supported": (_i, [_i, _i, _i]),
    "vit3d_qkv_attn_fwd": (_i, [_p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _p]),
    "vit3d_qkv_attn_supported": (_i, [_i, _i, _i]),
    "vit3d_gelu_fwd": (_i, [_p, _p, _ll, _i, _p]),
    "vit3d_gelu_bwd": (_i, [_p, _p, _p, _ll, _i, _p]),
    "vit3d_gelu_dropout_bwd": (_i, [_p, _p, _p, _ll, _i, _f, _ull, _u, _u, _p, _p]),
    "vit3d_dropout": (_i, [_p, _p, _p, _ll, _i, _f, _ull, _u, _u, _p, _p]),
    "vit3d_dropout_mask": (_i, [_p, _ll, _f, _ull, _u, _u, _p]),
    "vit3d_dropout_masked": (_i, [_p, _p, _p, _p, _ll, _i, _f, _p]),
    "vit3d_cast_f32_to_bf16": (_i, [_p, _p, _ll, _p]),
    "vit3d_cast_bf16_to_f32": (_i, [_p, _p, _ll, _p]),
    "vit3d_round_tf32": (_i, [_p, _p, _ll, _p]),
    "vit3d_cast_f32_to_f16": (_i, [_p, _p, _ll, _p]),
    "vit3d_u8_to_f32": (_i, [_p, _p, _ll, _f, _p]),
    "vit3d_transpose_f32_to_bf16": (_i, [_p, _p, _i, _i, _p]),
    "vit3d_add_inplace": (_i, [_p, _p, _ll, _p]),
    "vit3d_bce_logits_fwd": (_i, [_p, _p, _f, _p, _p, _i, _p]),
    "vit3d_bce_logits_bwd": (_i, [_p, _p, _f, _p, _p, _p, _i, _p]),
    "vit3d_meta_fwd": (_i, [_p, _p, _p, _p, _i, _i, _i, _p]),
    "vit3d_meta_bwd": (_i, [_p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _p]),
    "vit3d_sgd_step": (_i, [_p, _p, _p, _ll, _f, _f, _f, _i, _f, _p, _p]),
    "vit3d_adam_step": (_i, [_p, _p, _p, _p, _ll, _f, _f, _f, _f, _f, _i, _f, _p, _p, _p]),
    "vit3d_memset_zero": (_i, [_p, _sz, _p]),
    "vit3d_train_supported": (_i, [_i, _i, _i, _i, _i]),
    "vit3d_dropout_bits": (_i, [_p, _i, C.POINTER(_u), C.POINTER(_ll), _f, _ull, _u, _p, _p]),
    "vit3d_ln256_fwd": (_i, [_p, _p, _f, _p, _p, _p, _p, _p, _p, _p, _i, _f, _p]),
    "vit3d_ln256_bwd": (_i, [_p, _p, _p, _p, _p, _p, _p, _f, _i, _p, _p, _p, _p, _p, _i, _p]),
    "vit3d_mul_colsum_bwd": (_i, [_p, _p, _p, _p, _i, _i, _p]),
    "vit3d_mlp_bwd": (_i, [_p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _p]),
    "vit3d_mlp_bwd_supported": (_i, [_i, _i, _i]),
    "vit3d_head_bwd": (_i, [_p, _p, _p, _p, _p, _p, _i, _i, _i, _p]),
    "vit3d_refresh_shadows": (_i, [_p, _i, _i, _p, _p]),
    "vit3d_fc1_train_fwd": (_i, [_p, _p, _p, _p, _p, _p, _f, _i, _i, _i, _p]),
    "vit3d_linear_res_train_fwd": (_i, [_p, _p, _p, _p, _p, _p, _f, _p, _p, _f, _p, _p, _p, _i, _i, _i, _p]),
    "vit3d_wgrad": (_i, [_p, _p, _p, _p, _p, _i, _i, _i, _i, _p]),
    "vit3d_wgrad_ws_bytes": (_sz, [_i, _i, _i]),
    "vit3d_wgrad_partial": (_i, [_p, _p, _p, _i, _i, _i, C.POINTER(_i), C.POINTER(_i), _p]),
    "vit3d_wgrad_reduce": (_i, [_p, _i, _p]),
    "vit3d_attn_bwd_bias": (_i, [_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _p]),
}


def lib():
    """The loaded shared library (loads on first use; raises if it has not been built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise Vit3dError(f"{LIB_PATH} not found: run `python -c 'import __graft_entry__ as g; g.build()'` "
                             "(there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = lib().vit3d_last_error().decode("utf-8", "replace")
        raise Vit3dError(f"{what}: error {rc}: {msg}")


def ptr(t):
    """Device pointer of a CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise Vit3dError("vit3d kernels need CUDA tensors (there is no CPU fallback)")
    return t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


def call(name: str, *args):
    check(getattr(lib(), name)(*args), name)
