"""ctypes binding of libmkd_b200.so — the thin boundary between the Python host code and the CUDA kernels.

Mirrors include/mkd_b200.h one to one.  There is no fallback of any kind: if the library is missing, or the device
is not a B200 (sm_100), importing the kernels raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmkd_b200.so")

MKD_BF16, MKD_F32 = 0, 1
ACT_NONE, ACT_SILU, ACT_GEGLU = 0, 1, 2
PATH_AUTO, PATH_GENERIC, PATH_TCGEN05, PATH_TCGEN05_SINGLE, PATH_TCGEN05_PAIR = 0, 1, 2, 3, 4
ABI_VERSION = 13


class ConvDesc(C.Structure):
    """struct mkd_conv_desc (include/mkd_b200.h)"""
    _fields_ = [
        ("dtype", C.c_int),
        ("N", C.c_int), ("H", C.c_int), ("W", C.c_int), ("C", C.c_int),
        ("K", C.c_int), ("R", C.c_int), ("S", C.c_int),
        ("stride", C.c_int), ("pad", C.c_int), ("upsample", C.c_int),
        ("ldx", C.c_int), ("ldy", C.c_int), ("ldr", C.c_int), ("lde", C.c_int),
        ("act", C.c_int), ("geglu_block", C.c_int),
        ("path", C.c_int),
        ("alpha", C.c_float),
        ("x", C.c_void_p), ("w", C.c_void_p), ("y", C.c_void_p),
        ("bias", C.c_void_p), ("emb", C.c_void_p), ("residual", C.c_void_p),
        ("residual_dtype", C.c_int), ("ldy32", C.c_int), ("y32", C.c_void_p),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
        ("stats", C.c_void_p), ("stats_ld", C.c_int),
        ("pad_hi_extra", C.c_int),
        ("x2", C.c_void_p), ("C2", C.c_int), ("ldx2", C.c_int),
        ("wgroups", C.c_int),
        ("gn_y", C.c_void_p), ("gn_ld", C.c_int), ("gn_groups", C.c_int), ("gn_silu", C.c_int), ("gn_eps", C.c_float),
        ("gn_gamma", C.c_void_p), ("gn_beta", C.c_void_p),
    ]


_vp, _i, _f, _i64, _sz = C.c_void_p, C.c_int, C.c_float, C.c_int64, C.c_size_t

# name -> (restype, argtypes); every symbol include/mkd_b200.h declares
PROTOTYPES = {
    "mkd_abi_version": (_i, []),
    "mkd_compiled_arch": (_i, []),
    "mkd_device_ok": (_i, [_i]),
    "mkd_last_error": (C.c_char_p, []),
    "mkd_launch_count": (C.c_longlong, []),
    "mkd_ddim_update": (_i, [_vp, _vp, _i, _f, _vp, _f, _f, _f, _f, _f, _f, _vp, _vp, _i64, _vp]),
    "mkd_ddim_update_peers": (_i, [_vp, _vp, _i, _f, _vp, _f, _f, _f, _f, _f, _f, _vp, _i, _vp, _i64, _vp]),
    "mkd_plms_update": (_i, [_vp, _vp, _i, _f, _vp, _i, _vp, _vp, _vp, _f, _f, _f, _f, _vp, _vp, _i64, _vp]),
    "mkd_plms_update_peers": (_i, [_vp, _vp, _i, _f, _vp, _i, _vp, _vp, _vp, _f, _f, _f, _f, _vp, _i, _vp, _i64, _vp]),
    "mkd_dpm_update": (_i, [_vp, _vp, _i, _f, _f, _f, _vp, _i, _vp, _f, _f, _f, _f, _vp, _i64, _vp]),
    "mkd_dpm_update_peers": (_i, [_vp, _vp, _i, _f, _f, _f, _vp, _i, _vp, _f, _f, _f, _f, _vp, _i, _i64, _vp]),
    "mkd_ddpm_update": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _f, _vp, _vp, _i64, _vp]),
    "mkd_ddpm_update_peers": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _f, _vp, _vp, _i, _i64, _vp]),
    "mkd_nchw_to_nhwc": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "mkd_nhwc_to_nchw": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "mkd_timestep_embedding": (_i, [_vp, _vp, _i, _i, _i, _f, _vp]),
    "mkd_timestep_embedding_f32": (_i, [_vp, _vp, _i, _i, _i, _f, _vp]),
    "mkd_silu": (_i, [_vp, _vp, _i, _i64, _vp]),
    "mkd_geglu": (_i, [_vp, _vp, _i, _i64, _i, _i, _i, _vp]),
    "mkd_add": (_i, [_vp, _vp, _vp, _i, _i64, _i, _i, _i, _i, _vp]),
    "mkd_groupnorm_workspace_bytes": (_sz, [_i, _i]),
    "mkd_groupnorm": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _f, _i, _vp, _sz, _i, _vp]),
    "mkd_groupnorm_apply": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _f, _i, _vp, _i, _i, _i, _vp]),
    "mkd_softmax_rows": (_i, [_vp, _vp, _i, _i, _i64, _i, _i, _i, _f, _vp]),
    "mkd_layernorm": (_i, [_vp, _vp, _i, _i, _i64, _i, _i, _i, _vp, _vp, _f, _i, _vp]),
    "mkd_conv2d": (_i, [C.POINTER(ConvDesc), _vp]),
    "mkd_conv2d_path": (_i, [C.POINTER(ConvDesc)]),
    "mkd_attention": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _f, _vp]),
    "mkd_attention_causal": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _f, _vp]),
    "mkd_embed_tokens": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "mkd_image_grid_u8": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
}

_lib = None


def load() -> C.CDLL:
    """dlopen the library and bind every prototype; raises if it is absent (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: build it with `python -m makeupdiffuse_b200.build` "
            "(or __graft_entry__.build()). makeupdiffuse_b200 has no CPU / PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype, fn.argtypes = res, args
    if lib.mkd_abi_version() != ABI_VERSION:
        raise RuntimeError(f"libmkd_b200 ABI {lib.mkd_abi_version()} != expected {ABI_VERSION}: rebuild")
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().mkd_last_error().decode(errors="replace")
        raise RuntimeError(f"libmkd_b200 {what} failed (rc={rc}): {msg}")
