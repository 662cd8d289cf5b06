"""The C-ABI library loads on a CPU-only box and exports every symbol include/mkd_b200.h declares (no compute calls)."""
import ctypes
import os
import re

from makeupdiffuse_b200 import _lib, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "mkd_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(mkd_[a-z0-9_]+)\s*\(", src)))


def test_header_and_binding_agree():
    syms = declared_symbols()
    assert len(syms) >= 15
    assert sorted(_lib.PROTOTYPES) == syms


def test_library_builds_loads_and_exports_everything():
    build.build()
    lib = _lib.load()
    for s in declared_symbols():
        assert hasattr(lib, s), s
    assert lib.mkd_abi_version() == _lib.ABI_VERSION and lib.mkd_compiled_arch() == 100
    assert lib.mkd_groupnorm_workspace_bytes(16, 32) == 16 * 64 * 32 * 8


def test_conv_desc_struct_layout_matches_header():
    """field order/size of the ctypes mirror == the C struct (probe through mkd_conv2d_path validation)"""
    lib = _lib.load()
    d = _lib.ConvDesc()
    assert lib.mkd_conv2d_path(ctypes.byref(d)) < 0  # null x/w/y rejected, no CUDA call involved
    assert b"null x/w/y" in lib.mkd_last_error()
    d.x = d.w = d.y = 16
    d.dtype, d.N, d.H, d.W, d.C, d.K, d.R, d.S, d.stride, d.pad = 0, 1, 8, 8, 64, 64, 3, 3, 1, 1
    d.ldx = d.ldy = 64
    d.path = 7
    assert lib.mkd_conv2d_path(ctypes.byref(d)) < 0 and b"bad path" in lib.mkd_last_error()
    d.path = _lib.PATH_AUTO
    assert lib.mkd_conv2d_path(ctypes.byref(d)) == _lib.PATH_TCGEN05
    d.stride = 2
    assert lib.mkd_conv2d_path(ctypes.byref(d)) == _lib.PATH_GENERIC
    d.path = _lib.PATH_TCGEN05
    assert lib.mkd_conv2d_path(ctypes.byref(d)) < 0 and b"stride" in lib.mkd_last_error()


def test_fp32_conv_rejects_a_bf16_residual():
    """the generic kernel reads an fp32 conv's residual as fp32: a bf16 residual_dtype there is refused, not misread"""
    MKD_E_INVALID = -1  # include/mkd_b200.h
    lib = _lib.load()
    d = _lib.ConvDesc()
    d.x = d.w = d.y = d.residual = 16
    d.dtype, d.N, d.H, d.W, d.C, d.K, d.R, d.S, d.stride, d.pad = _lib.MKD_F32, 1, 8, 8, 64, 64, 3, 3, 1, 1
    d.ldx = d.ldy = d.ldr = 64
    d.path = _lib.PATH_GENERIC
    d.residual_dtype = _lib.MKD_F32
    assert lib.mkd_conv2d_path(ctypes.byref(d)) == _lib.PATH_GENERIC
    d.residual_dtype = _lib.MKD_BF16
    assert lib.mkd_conv2d_path(ctypes.byref(d)) == MKD_E_INVALID and b"fp32 residual" in lib.mkd_last_error()
    d.path = _lib.PATH_AUTO
    assert lib.mkd_conv2d_path(ctypes.byref(d)) == MKD_E_INVALID
