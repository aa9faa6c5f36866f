"""ctypes binding of libxclip_b200.so - the only way Python reaches the CUDA kernels.

There is deliberately no fallback: if the shared library is missing, or a call
returns a non-zero code, this raises.  Signatures mirror include/xclip_b200.h.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_int64, c_longlong, c_void_p
from pathlib import Path

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libxclip_b200.so"

_lib = None


class XClipB200Error(RuntimeError):
    pass


# name -> (restype, argtypes).  Kept in one table so tests can check that every
# symbol declared in include/xclip_b200.h is exported and bound.
SIGNATURES = {
    "xclip_abi_version": (c_int, []),
    "xclip_last_error": (c_char_p, []),
    "xclip_init": (c_int, []),
    "xclip_launch_count": (c_longlong, []),
    "xclip_launch_count_reset": (None, []),
    "xclip_gemm_set_pair_mode": (c_int, [c_int]),
    "xclip_tune_set": (c_int, [c_int, c_int]),
    "xclip_gemm_bf16": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_int64, c_int, c_void_p,
                                c_int64, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p,
                                c_int64, c_int, c_void_p, c_int, c_void_p]),
    "xclip_patchify_gather": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p,
                                      c_void_p]),
    "xclip_scatter_add_rows": (c_int, [c_void_p, c_int, c_void_p, c_int64, c_void_p, c_int64, c_int, c_int,
                                       c_void_p]),
    "xclip_colsum_rows": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_int, c_void_p]),
    "xclip_layernorm_fwd": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_void_p,
                                    c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_void_p,
                                    c_int, c_int, c_float, c_void_p]),
    "xclip_layernorm_bwd": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p,
                                    c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int, c_int,
                                    c_void_p]),
    "xclip_l2norm_fwd": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                 c_int, c_void_p]),
    "xclip_l2norm_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "xclip_cast_f32_bf16": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "xclip_attn_fwd": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_int,
                               c_int, c_int, c_float, c_int, c_void_p]),
    "xclip_attn_bwd": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_int64,
                               c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int, c_int,
                               c_int, c_float, c_int, c_void_p]),
    "xclip_nce_num_col_blocks": (c_int, [c_int]),
    "xclip_nce_fwd": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_int,
                              c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_void_p]),
    "xclip_nce_bwd": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_int,
                              c_void_p, c_void_p, c_float, c_float, c_float, c_void_p, c_void_p,
                              c_int64, c_void_p, c_void_p]),
    "xclip_text_embed_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                     c_int, c_int, c_void_p]),
    "xclip_text_embed_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                     c_int, c_int, c_void_p]),
    "xclip_ff_permute_cast": (c_int, [c_void_p, c_void_p, c_int, c_void_p]),
    "xclip_ff_scale_cast": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "xclip_ff_up": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p,
                            c_int, c_int, c_void_p]),
    "xclip_ff_down": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p,
                              c_int64, c_void_p, c_int64, c_void_p, c_float, c_int, c_int, c_void_p]),
    "xclip_ff_bwd_prep": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p,
                                  c_void_p, c_int, c_int, c_void_p]),
    "xclip_ff_bwd": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p,
                             c_int64, c_int, c_int, c_void_p]),
    "xclip_ff_w2_grad_post": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "xclip_adamw_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_float, c_float, c_float,
                                 c_float, c_float, c_int, c_float, c_void_p]),
    "xclip_rotary_inplace": (c_int, [c_void_p, c_int64, c_int64, c_int, c_int, c_void_p, c_void_p, c_int,
                                     c_void_p]),
    "xclip_filip_segmax": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_int,
                                   c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "xclip_filip_reduce": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_int,
                                   c_void_p]),
    "xclip_filip_nce_fwd": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_float,
                                    c_void_p]),
    "xclip_filip_nce_bwd": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                    c_void_p]),
    "xclip_filip_expand": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                   c_int, c_int, c_int, c_void_p, c_int64, c_void_p, c_void_p]),
}


def load() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise XClipB200Error(
            f"{LIB_PATH} is missing. Build it with `python -m x_clip_b200.build` "
            "(nvcc, sm_100a). x_clip_b200 has no CPU or eager-PyTorch fallback.")
    lib = ctypes.CDLL(str(LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().xclip_last_error()
        raise XClipB200Error(f"{what} failed (code {rc}): {msg.decode() if msg else '?'}")


def call(name: str, *args) -> None:
    check(getattr(load(), name)(*args), name)
