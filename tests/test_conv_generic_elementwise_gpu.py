"""Element-wise parity of the generic conv kernel (conv_generic.cu: conv_generic_kernel<T, GEGLU>) against float64, on every
descriptor production sends it, in both dtypes.

The generic kernel runs every contraction of the fp32 check mode (UNet, ControlNet, VAE, CLIP text encoder) and, in bf16, the
VAE's quant_conv / post_quant_conv and the layers of non-power-of-two latent maps that the tensor-core kernels decline.  The
checker, the float64 reference, the NaN-guarded buffers and the bounds are those of test_gemm_elementwise_gpu.py, with
dtype = "f32" (fp32 x, w, emb, y and residual; the reference takes the same fp32 values to float64) and generic = True:

    fp32 y with y32:      y == y32 bit for bit (one value stored twice)
    fp32 y alone, y32:    |out - ref| <= tau_g A,   tau_g = 2 u sqrt(K_tot + 4)
    bf16 y:               as in test_gemm_elementwise_gpu (y == bf16(y32), else 2^-8 |ref| + (1 + 2^-8) tau_g A)
    SiLU:                 the tensor-core path's bound (silu_f is the same function), with tau_g
    GEGLU:                gelu_erf_f = 0.5 x (1 + erff(x / sqrt 2)): erff is within 2 ulp, the argument, 1 + erf and the
                          product round once each, <= 3 u |x| in all: GELU_ERFF = 4 u per |g| in place of GELU_APPROX
    exact operands:       small dyadic integers (x, w, bias, emb, residual, alpha in {0.5, 1, 2}) make every partial sum
                          representable: y32 == ref and y == ref rounded to its dtype, whatever the accumulation order

tau_g: the kernel accumulates each output as one serial fmaf chain in k order, then adds bias and embedding, scales by alpha and
adds the residual: n = K_tot + 4 roundings, each at most u times a partial sum bounded by A.  The errors are independent
roundings, so |err| / A behaves like a random walk of n steps; it does not grow like sqrt(K_tot) the way the tensor-core
kernels' per-MMA-step adds do.  At small K_tot the tensor-core tau = u sqrt(K_tot) is then too tight: an fp32 emulation of
this kernel's arithmetic gives max |err| / (A u sqrt(K_tot)) = c = 1.38 at K_tot = 4 (post_quant_conv), 1.21 at 8
(quant_conv), 0.87 at 27, 0.13 at 1152, over 2^16 - 2^20 outputs.  tau_g = 2 u sqrt(K_tot + 4) covers the measured worst case
about 2x and stays far inside the rigorous (K_tot + 4) u A.  A run prints c per case and its maximum; a dropped 16-deep k chunk
or a wrong tap is still thousands of times the bound.
"""
import ctypes
import json
import math
import os
import re
import subprocess
import sys
import zlib

import pytest
import torch
import torch.nn.functional as F

from makeupdiffuse_b200 import _lib as L
from makeupdiffuse_b200 import ops
from test_gemm_elementwise_gpu import (GELU_ERFF, MEASURED, NAN, U, _bits, check_outputs, depth, launched_kernels,
                                       make_operands, out_geometry, reference, spec_of, tau)

BF, F32 = torch.bfloat16, torch.float32

# ---- kernel names -----------------------------------------------------------------------------------------------------------
_GEN = re.compile(r"conv_generic_kernel(?:<\s*(float|__nv_bfloat16)\s*,\s*(true|false|0|1)\s*>|I(f|13__nv_bfloat16)Lb([01])E)")


def generic_name(name):
    """'void (anonymous namespace)::conv_generic_kernel<float, false>(...)' (or its mangled form) ->
    'conv_generic_kernel<float,0>'; None for any other kernel"""
    m = _GEN.search(name)
    if not m:
        return None
    t = m.group(1) or {"f": "float", "13__nv_bfloat16": "__nv_bfloat16"}[m.group(3)]
    g = m.group(2) or m.group(4)
    return f"conv_generic_kernel<{t},{int(g in ('true', '1'))}>"


def want_kernel(s):
    return f"conv_generic_kernel<{'float' if s['dtype'] == 'f32' else '__nv_bfloat16'},{int(s['act'] == 'geglu')}>"


# ---- descriptor signatures: what a case covers and what production sends -------------------------------------------------
def signature(d, residual, y, y32):
    """the properties of a generic-kernel descriptor its correctness can depend on"""
    Hi, Wi = (2 * d.H, 2 * d.W) if d.upsample else (d.H, d.W)
    P = (Hi + 2 * d.pad + d.pad_hi_extra - d.R) // d.stride + 1
    Q = (Wi + 2 * d.pad + d.pad_hi_extra - d.S) // d.stride + 1
    M, kout = d.N * P * Q, d.K // 2 if d.act == L.ACT_GEGLU else d.K
    if residual is None:
        res = "none"
    elif any(o is not None and o.data_ptr() == residual.data_ptr() for o in (y, y32)):
        res = "in place"
    else:
        res = "f32" if residual.dtype == F32 else "bf16"
    outs = "both" if y is not None and y32 is not None else ("y" if y is not None else "y32")
    return (("f32" if d.dtype == L.MKD_F32 else "bf16"), d.R, d.stride, d.pad, d.pad_hi_extra, bool(d.upsample),
            {L.ACT_NONE: "none", L.ACT_SILU: "silu", L.ACT_GEGLU: "geglu"}[d.act],
            "bias" if d.bias else "-", "emb" if d.emb else "-", "res " + res, "alpha 1" if d.alpha == 1.0 else "alpha != 1",
            outs, "x sliced" if d.ldx > d.C else "x whole",
            "out sliced" if (y is not None and d.ldy > kout) or (y32 is not None and d.ldy32 > kout) else "out whole",
            "RSC%16" if (d.R * d.S * d.C) % 16 == 0 else "RSC ragged", "K%64" if kout % 64 == 0 else "K ragged",
            "M%64" if M % 64 == 0 else "M ragged", "tile spans images" if d.N > 1 and (P * Q) % 64 else "-")


def record(census, sig, d, where):
    e = census.setdefault(sig, dict(n=0, where=where, rsc=0, m=0))
    Hi, Wi = (2 * d.H, 2 * d.W) if d.upsample else (d.H, d.W)
    P = (Hi + 2 * d.pad + d.pad_hi_extra - d.R) // d.stride + 1
    Q = (Wi + 2 * d.pad + d.pad_hi_extra - d.S) // d.stride + 1
    e["n"] += 1
    e["rsc"] = max(e["rsc"], d.R * d.S * d.C)
    e["m"] = max(e["m"], d.N * P * Q)


def print_census(census, cover):
    print("\ngeneric-kernel census (signature -> launches, first seen in, covering case):")
    for sig in sorted(census, key=str):
        e = census[sig]
        print(f"  {' | '.join(map(str, sig))}\n      {e['n']:5d} launches, max R*S*C {e['rsc']}, max M {e['m']}, first in "
              f"{e['where']}; case: {cover.get(sig, 'NONE')}")


# ---- the cases ------------------------------------------------------------------------------------------------------------
def gcase(**kw):
    return spec_of(generic=True, **kw)


CASES = {}
for dt in ("f32", "bf16"):
    CASES.update({
        # tiles
        f"{dt} 3x3 C 3 (R*S*C = 27), K 64, ragged M": gcase(dtype=dt, N=1, H=9, W=11, C=3, K=64, R=3),
        f"{dt} 3x3 C 4 -> 320 (conv_in), batch 2, tile spans images": gcase(dtype=dt, N=2, H=10, W=6, C=4, K=320, R=3, tight=True),
        f"{dt} 3x3 C 6 -> 16 + SiLU (hint conv 0), odd map": gcase(dtype=dt, N=2, H=13, W=9, C=6, K=16, R=3, act="silu",
                                                                  spread=8.0),
        f"{dt} 3x3 320 -> 4 (out conv), K < 64": gcase(dtype=dt, N=2, H=8, W=12, C=320, K=4, R=3),
        f"{dt} 1x1 linear 64 -> 1000, ragged channel tile, no bias": gcase(dtype=dt, N=1, H=1, W=77, C=64, K=1000, bias=False),
        f"{dt} 1x1 linear 96 -> 96, ragged channel tile": gcase(dtype=dt, N=1, H=1, W=130, C=96, K=96),
        # geometry
        f"{dt} stride 2 p1 even 16x12 + SiLU": gcase(dtype=dt, N=2, H=16, W=12, C=16, K=32, R=3, stride=2, act="silu", spread=8.0),
        f"{dt} stride 2 p1 odd 15x9": gcase(dtype=dt, N=2, H=15, W=9, C=32, K=96, R=3, stride=2),
        f"{dt} upsample 5x7 -> 10x14": gcase(dtype=dt, N=2, H=5, W=7, C=64, K=64, R=3, up=True),
        f"{dt} ResBlock conv1 + emb, rectangular 5x3, batch 3": gcase(dtype=dt, N=3, H=5, W=3, C=64, K=128, R=3, emb=True),
        # operands
        f"{dt} in-place residual, alpha 0.5 (zero-conv)": gcase(dtype=dt, N=2, H=6, W=10, C=64, K=64, res=dt, inplace=True,
                                                                alpha=0.5),
        f"{dt} fp32 residual -> y + y32": gcase(dtype=dt, N=2, H=8, W=8, C=128, K=128, R=3, res="f32", y32=True),
        f"{dt} y32 only, emb": gcase(dtype=dt, N=2, H=8, W=8, C=64, K=128, R=3, emb=True, y=False, y32=True),
        # epilogue
        f"{dt} SiLU, pre-activations +-100": gcase(dtype=dt, N=1, H=1, W=200, C=64, K=192, act="silu", spread=100.0),
        f"{dt} alpha 1.702 + SiLU (quick_gelu fold)": gcase(dtype=dt, N=1, H=1, W=77, C=128, K=320, alpha=1.702, act="silu"),
        f"{dt} GEGLU [80 | 80], gate +-8": gcase(dtype=dt, N=1, H=1, W=100, C=64, K=640, act="geglu", gb=80, spread=8.0),
        f"{dt} GEGLU [128 | 128], no bias": gcase(dtype=dt, N=1, H=1, W=70, C=96, K=512, act="geglu", gb=128, bias=False),
        # exact operands
        f"{dt} exact: 3x3 + emb + alpha 2, tile spans images": gcase(dtype=dt, N=3, H=6, W=6, C=40, K=72, R=3, emb=True,
                                                                     alpha=2.0, exact=True),
        f"{dt} exact: in-place residual, alpha 0.5": gcase(dtype=dt, N=1, H=1, W=150, C=64, K=100, res=dt, inplace=True,
                                                          alpha=0.5, exact=True),
        f"{dt} exact: fp32 residual, upsample 5x7, y + y32": gcase(dtype=dt, N=1, H=5, W=7, C=24, K=40, R=3, up=True, res="f32",
                                                                   y32=True, exact=True),
        f"{dt} exact: stride 2 p1 odd 9x7, C 6": gcase(dtype=dt, N=2, H=9, W=7, C=6, K=16, R=3, stride=2, exact=True),
        f"{dt} exact: SiLU": gcase(dtype=dt, N=1, H=1, W=300, C=64, K=64, act="silu", exact=True, y32=True),
        f"{dt} exact: GEGLU [80 | 80]": gcase(dtype=dt, N=1, H=1, W=100, C=64, K=320, act="geglu", gb=80, exact=True),
    })
CASES.update({
    "bf16 bf16 residual": gcase(N=2, H=8, W=8, C=64, K=64, R=3, res="bf16"),
    "bf16 exact: bf16 residual + emb, alpha 0.5": gcase(N=2, H=5, W=5, C=32, K=64, R=3, emb=True, res="bf16", alpha=0.5,
                                                        exact=True),
    "f32 exact: stride 2 p0 + far edge, 10x8": gcase(dtype="f32", N=2, H=10, W=8, C=16, K=32, R=3, stride=2, pad=0,
                                                    pad_hi_extra=1, exact=True),
    # production sizes (fp32 check mode)
    "f32 VAE Downsample p0 + far edge, 64x64 128 -> 128": gcase(dtype="f32", N=1, H=64, W=64, C=128, K=128, R=3, stride=2,
                                                               pad=0, pad_hi_extra=1),
    "f32 decoder ResBlock conv1 3x3 2560 -> 1280 at 4x4 + emb": gcase(dtype="f32", N=2, H=4, W=4, C=2560, K=1280, R=3,
                                                                     emb=True),
    "f32 Upsample 3x3 1280, 8 -> 16": gcase(dtype="f32", N=1, H=8, W=8, C=1280, K=1280, R=3, up=True),
    "f32 GEGLU 1280 -> 2 x 5120": gcase(dtype="f32", N=1, H=1, W=64, C=1280, K=10240, act="geglu", gb=5120),
    "f32 3x3 320 -> 320 at 32x32, batch 2": gcase(dtype="f32", N=2, H=32, W=32, C=320, K=320, R=3),
    "f32 hint 6 -> 16 + SiLU at 512^2": gcase(dtype="f32", N=1, H=512, W=512, C=6, K=16, R=3, act="silu", tight=True),
    "f32 VAE conv_out 128 -> 3 at 256^2": gcase(dtype="f32", N=1, H=256, W=256, C=128, K=3, R=3),
    "f32 quant_conv 8 -> 8 at 32x32": gcase(dtype="f32", N=1, H=32, W=32, C=8, K=8, tight=True),
    "f32 post_quant_conv 4 -> 4 at 32x32": gcase(dtype="f32", N=1, H=32, W=32, C=4, K=4, tight=True),
    "bf16 ResBlock conv1 3x3 2560 -> 1280 at 5x3 + emb, y32 only": gcase(N=1, H=5, W=3, C=2560, K=1280, R=3, emb=True, y=False,
                                                                        y32=True, tight=True),
    "bf16 hint 6 -> 16 + SiLU at 320x192": gcase(N=1, H=320, W=192, C=6, K=16, R=3, act="silu", spread=8.0, tight=("y",)),
    "f32 CLIP fc1 768 -> 3072, alpha 1.702 + SiLU": gcase(dtype="f32", N=1, H=1, W=77, C=768, K=3072, alpha=1.702, act="silu",
                                                         tight=True),
})


# every signature the production census finds (test_production_census), one case each, on the smallest map that has it:
# dtype R stride pad pad_hi_extra up(U) act bias(B) emb(E) residual(none / bf16 / f32 / inpl) alpha(1 / a) outputs(y / y32 / both)
# x(xs sliced / xw whole) out(os / ow) R*S*C(16: % 16 == 0 / r) Kout(64 / r) M(64 / r) span(S: a 64-row tile spans two images)
PRODUCTION = [
    "bf16 1 1 0 0 - none B - none 1 y xs os r r 64 -", "bf16 3 1 1 0 - none B - bf16 1 both xw ow 16 64 64 -",
    "bf16 3 1 1 0 - none B - f32 1 both xw os 16 64 r -", "bf16 3 1 1 0 - none B - f32 1 both xw ow 16 64 r -",
    "bf16 3 1 1 0 - none B - f32 1 y xw os 16 64 r -", "bf16 3 1 1 0 - none B - f32 1 y xw ow 16 64 r -",
    "bf16 3 1 1 0 - none B - f32 1 y32 xw ow 16 64 r -", "bf16 3 1 1 0 - none B - f32 1 y32 xw ow 16 64 64 -",
    "bf16 3 1 1 0 - none B - none 1 both xw os 16 64 64 -", "bf16 3 1 1 0 - none B - none 1 y xw os 16 r 64 -",
    "bf16 3 1 1 0 - none B - none 1 y xw ow 16 64 64 -", "bf16 3 1 1 0 - none B E none 1 y32 xw ow 16 64 r -",
    "bf16 3 1 1 0 - none B E none 1 y32 xw ow 16 64 64 -", "bf16 3 1 1 0 - silu B - none 1 y xs ow r r 64 -",
    "bf16 3 1 1 0 - silu B - none 1 y xw ow 16 r 64 -", "bf16 3 1 1 0 U none B - none 1 y xw os 16 64 r -",
    "bf16 3 1 1 0 U none B - none 1 y xw os 16 64 64 -", "bf16 3 2 1 0 - silu B - none 1 y xw ow 16 r 64 -",
    "bf16 3 2 1 0 - silu B - none 1 y xw ow 16 64 64 -", "f32 1 1 0 0 - geglu B - none 1 y xw ow 16 64 r -",
    "f32 1 1 0 0 - geglu B - none 1 y xw ow 16 64 64 -", "f32 1 1 0 0 - none - - none 1 y xw ow 16 64 r -",
    "f32 1 1 0 0 - none - - none 1 y xw ow 16 64 64 -", "f32 1 1 0 0 - none B - f32 1 y xw os 16 64 r -",
    "f32 1 1 0 0 - none B - f32 1 y xw os 16 64 64 -", "f32 1 1 0 0 - none B - f32 1 y xw ow 16 64 r -",
    "f32 1 1 0 0 - none B - f32 1 y xw ow 16 64 r S", "f32 1 1 0 0 - none B - f32 1 y xw ow 16 64 64 -",
    "f32 1 1 0 0 - none B - inpl 1 y xw os 16 64 r -", "f32 1 1 0 0 - none B - inpl 1 y xw os 16 64 r S",
    "f32 1 1 0 0 - none B - inpl 1 y xw os 16 64 64 -", "f32 1 1 0 0 - none B - inpl 1 y xw ow 16 64 r -",
    "f32 1 1 0 0 - none B - inpl 1 y xw ow 16 64 64 -", "f32 1 1 0 0 - none B - none 1 y xs os r r 64 -",
    "f32 1 1 0 0 - none B - none 1 y xs ow 16 64 r -", "f32 1 1 0 0 - none B - none 1 y xs ow 16 64 64 -",
    "f32 1 1 0 0 - none B - none 1 y xw ow r r 64 -", "f32 1 1 0 0 - none B - none 1 y xw ow 16 64 r -",
    "f32 1 1 0 0 - none B - none 1 y xw ow 16 64 r S", "f32 1 1 0 0 - none B - none 1 y xw ow 16 64 64 -",
    "f32 1 1 0 0 - silu B - none a y xw ow 16 64 r -", "f32 1 1 0 0 - silu B - none 1 y xw ow 16 64 r -",
    "f32 3 1 1 0 - none B - f32 1 y xs ow r 64 64 -", "f32 3 1 1 0 - none B - f32 1 y xw os 16 64 r -",
    "f32 3 1 1 0 - none B - f32 1 y xw os 16 64 r S", "f32 3 1 1 0 - none B - f32 1 y xw ow 16 64 r -",
    "f32 3 1 1 0 - none B - f32 1 y xw ow 16 64 r S", "f32 3 1 1 0 - none B - f32 1 y xw ow 16 64 64 -",
    "f32 3 1 1 0 - none B - none 1 y xs os r 64 64 -", "f32 3 1 1 0 - none B - none 1 y xs ow r 64 64 -",
    "f32 3 1 1 0 - none B - none 1 y xw os 16 r 64 -", "f32 3 1 1 0 - none B - none 1 y xw ow 16 r 64 -",
    "f32 3 1 1 0 - none B - none 1 y xw ow 16 64 64 -", "f32 3 1 1 0 - none B E none 1 y xw ow 16 64 r -",
    "f32 3 1 1 0 - none B E none 1 y xw ow 16 64 r S", "f32 3 1 1 0 - none B E none 1 y xw ow 16 64 64 -",
    "f32 3 1 1 0 - silu B - none 1 y xs ow r r 64 -", "f32 3 1 1 0 - silu B - none 1 y xw ow 16 r 64 -",
    "f32 3 1 1 0 U none B - none 1 y xw os 16 64 r -", "f32 3 1 1 0 U none B - none 1 y xw os 16 64 64 -",
    "f32 3 1 1 0 U none B - none 1 y xw ow 16 64 64 -", "f32 3 2 0 1 - none B - none 1 y xw ow 16 64 64 -",
    "f32 3 2 1 0 - none B - none 1 y xs os 16 64 r -", "f32 3 2 1 0 - none B - none 1 y xs os 16 64 r S",
    "f32 3 2 1 0 - none B - none 1 y xs os 16 64 64 -", "f32 3 2 1 0 - none B - none 1 y xw ow 16 64 r -",
    "f32 3 2 1 0 - none B - none 1 y xw ow 16 64 r S", "f32 3 2 1 0 - none B - none 1 y xw ow 16 64 64 -",
    "f32 3 2 1 0 - silu B - none 1 y xw ow 16 r 64 -", "f32 3 2 1 0 - silu B - none 1 y xw ow 16 64 64 -",
]


def from_code(code):
    dt, R, st, pad, phe, up, act, b, e, res, a, outs, xs, os_, rsc, k, m, sp = code.split()
    R, st, pad, phe, up = int(R), int(st), int(pad), int(phe), up == "U"
    N, (P, Q) = (2 if sp == "S" else 1), {("64", "-"): (8, 8), ("r", "-"): (6, 10), ("r", "S"): (6, 4), ("64", "S"): (8, 12)}[m, sp]
    H, W = (P // 2, Q // 2) if up else ((2 * P, 2 * Q) if st == 2 else (P, Q))
    C = (32 if R == 1 else 16) if rsc == "16" else 4
    Ko = 64 if k == "64" else 40
    tight = (("x",) if xs == "xw" else ()) + (("y", "y32", "res") if os_ == "ow" else ())
    return gcase(dtype=dt, N=N, H=H, W=W, C=C, K=2 * Ko if act == "geglu" else Ko, R=R, stride=st, pad=pad, pad_hi_extra=phe,
                 up=up, act=act, gb=Ko // 2, spread=8.0 if act != "none" else 0.0, bias=b == "B", emb=e == "E",
                 res=None if res == "none" else ((dt if outs != "y32" else "f32") if res == "inpl" else res), inplace=res == "inpl",
                 alpha=1.0 if a == "1" else (1.702 if act == "silu" else 0.5), y=outs != "y32", y32=outs != "y", tight=tight)


CASES.update({f"production: {c}": from_code(c) for c in PRODUCTION})


# ---- running a case on the GPU ----------------------------------------------------------------------------------------------
C_MEASURED = {}  # label -> max |err| / (A u sqrt(K_tot)) of the case's fp32 output (act none, random operands)


def case_launch(label):
    """the operands of a case and its ops.conv2d keywords, forced onto the generic kernel"""
    ops_ = make_operands(CASES[label], "cuda", zlib.crc32(label.encode()))
    ops_["kw"]["path"] = L.PATH_GENERIC
    return ops_


def profile_every_case():
    """label -> the CUDA kernels one launch of the case runs, by torch.profiler.  Runs in a child process (kernel_names):
    once CUPTI has started in a process, a later profiler session can lose its kernel records; on the B200 the first
    session after the samplers' CUDA-graph tests recorded no kernel at all, even with 200 ms of idle time around the launch.
    A child keeps this file's ~130 sessions from starting CUPTI in the test process."""
    names = {}
    for label in CASES:
        o = case_launch(label)
        names[label] = launched_kernels(lambda: ops.conv2d(o["x"], o["w"], o["y"], **o["kw"]))
    return names


@pytest.fixture(scope="module")
def kernel_names():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([root] + [p for p in [os.environ.get("PYTHONPATH")] if p]))
    r = subprocess.run([sys.executable, "-s", os.path.abspath(__file__)], env=env, capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, f"profiling child failed:\n{r.stdout[-2000:]}\n{r.stderr[-4000:]}"
    return json.loads(r.stdout.strip().splitlines()[-1])


def run_case(label, s, profiled):
    ops_ = case_launch(label)
    x, w, y, kw = ops_["x"], ops_["w"], ops_["y"], ops_["kw"]
    assert ops.conv2d_path(x, w, y, **kw) == L.PATH_GENERIC, label
    assert [generic_name(n) for n in profiled] == [want_kernel(s)], \
        f"{label}: the profiled launch ran {profiled}, expected [{want_kernel(s)}]"
    guards_before = {k: b.clone() for k, (b, _) in ops_["bufs"].items()}
    refd = reference(s, x, w, ops_["bias"], ops_["emb"], ops_["res"], None)
    inplace_before = ops_["res"].clone() if s["inplace"] else None
    n0 = L.load().mkd_launch_count()
    ops.conv2d(x, w, y, **kw)
    torch.cuda.synchronize()
    assert L.load().mkd_launch_count() - n0 == 1, f"{label}: {L.load().mkd_launch_count() - n0} launches, expected 1"
    guards = [(k, b, guards_before[k], inside if k in ("y", "y32") else None) for k, (b, inside) in ops_["bufs"].items()]
    worst = check_outputs(label, s, refd, y=y, y32=ops_["y32"], guards=guards)
    c = None
    if s["act"] == "none" and not s["exact"]:
        out = ops_["y32"] if ops_["y32"] is not None else (y if y.dtype == F32 else None)
        if out is not None:
            c = float(((out.double() - refd["ref"]).abs() / refd["A"]).max()) / (U * math.sqrt(depth(s)))
            C_MEASURED[label] = c
    # a second identical launch writes bit-identical outputs
    first = [None if t is None else t.clone() for t in (y, ops_["y32"])]
    if s["inplace"]:
        ops_["res"].copy_(inplace_before)
    ops.conv2d(x, w, y, **kw)
    torch.cuda.synchronize()
    for name, a, b in zip(("y", "y32"), first, (y, ops_["y32"])):
        if a is not None:
            assert torch.equal(_bits(a), _bits(b)), f"{label}: second launch differs in {name}"
    extra = "" if c is None else f"  c {c:.3f} (tau_g / (u sqrt(K_tot)) = {tau(s) / (U * math.sqrt(depth(s))):.2f})"
    print(f"{label:<66s} worst err/bound " + "  ".join(f"{k} {v:.3f}" for k, v in worst.items()) + extra +
          f"   [{want_kernel(s)}]")


@pytest.fixture(scope="module", autouse=True)
def _report_margins():
    saved = {k: v for k, v in MEASURED.items()}
    MEASURED.update({k: (0.0, "") for k in MEASURED})
    yield
    if C_MEASURED:
        worst = max(C_MEASURED, key=C_MEASURED.get)
        print(f"\nmeasured c = max |out - ref| / (A u sqrt(K_tot)) = {C_MEASURED[worst]:.3f} (at {worst}); over 1 at: "
              f"{sorted(k for k, v in C_MEASURED.items() if v > 1) or 'none'}")
        r, where = MEASURED["err_over_A"]
        print(f"max |out - ref| / A = {r / U:.2f} u (at {where}); bound tau_g = 2 u sqrt(K_tot + 4) >= {2 * math.sqrt(5):.2f} u")
    if MEASURED["gelu_coef"][0] > 0:
        c, where = MEASURED["gelu_coef"]
        print(f"implied gelu_erf_f error <= {c:.3e} |a| |g| (at {where}); bound GELU_ERFF = {GELU_ERFF:.3e}")
    MEASURED.update(saved)


@pytest.mark.gpu
@pytest.mark.parametrize("label", list(CASES))
def test_generic_elementwise(label, kernel_names):
    run_case(label, CASES[label], kernel_names[label])


@pytest.mark.gpu
def test_fp32_conv_with_a_bf16_residual_is_refused():
    x = torch.randn(64, 16, device="cuda")
    w = torch.randn(16, 16, device="cuda")
    y = torch.empty(64, 16, device="cuda")
    res = torch.randn(64, 16, device="cuda").to(BF)
    with pytest.raises(RuntimeError, match="fp32 residual"):
        ops.conv2d(x, w, y, N=1, H=1, W=64, residual=res, path=L.PATH_GENERIC)
    with pytest.raises(RuntimeError, match="fp32 residual"):
        ops.conv2d(x, w, y, N=1, H=1, W=64, residual=res)


def test_kernel_name_forms():
    assert generic_name("void (anonymous namespace)::conv_generic_kernel<float, false>((anonymous namespace)::ConvP, "
                        "float const*, float const*, float*, float const*, float const*, void const*)") == \
        "conv_generic_kernel<float,0>"
    assert generic_name("void (anonymous namespace)::conv_generic_kernel<__nv_bfloat16, true>(...)") == \
        "conv_generic_kernel<__nv_bfloat16,1>"
    assert generic_name("_ZN12_GLOBAL__N_119conv_generic_kernelI13__nv_bfloat16Lb0EEEvNS_5ConvPEPKT_S6_PS4_PKfS6_PKv") == \
        "conv_generic_kernel<__nv_bfloat16,0>"
    assert generic_name("_ZN12_GLOBAL__N_119conv_generic_kernelIfLb1EEEvNS_5ConvPEPKT_S5_PS3_PKfS5_PKv") == \
        "conv_generic_kernel<float,1>"
    assert generic_name("void (anonymous namespace)::gemm_tcgen05_kernel<160, 1, 4, 10, 0>(...)") is None


# ---- the checker's self-test (CPU): an fp32 case, correct result accepted, each injected fault rejected ----------------------
def _rounded(s, ops_, refd):
    """what a correct kernel stores: the reference rounded once to fp32 (y is the same value)"""
    ops_["y32"].copy_(refd["ref"].float())
    ops_["y"].copy_(ops_["y32"])


def _self_case(geom, exact, fault=None):
    s = gcase(dtype="f32", y32=True, exact=exact, **geom)
    ops_ = make_operands(s, "cpu", 7)
    refd = reference(s, ops_["x"], ops_["w"], ops_["bias"], ops_["emb"], ops_["res"], None)
    before = {k: b.clone() for k, (b, _) in ops_["bufs"].items()}
    if fault is None:
        _rounded(s, ops_, refd)
    else:
        fault(s, ops_, refd)
    guards = [(k, b, before[k], inside if k in ("y", "y32") else None) for k, (b, inside) in ops_["bufs"].items()]
    return lambda: check_outputs("self-test", s, refd, y=ops_["y"], y32=ops_["y32"], guards=guards)


def _faulted(s, ops_, x=None, w=None, bias=None, emb_rows=None, res=None, **geom):
    """store the correctly rounded result of the case computed with a faulty operand / geometry"""
    s2 = dict(s, **geom)
    e = ops_["emb"]
    if emb_rows is not None:  # a per-output-row embedding
        pre = reference(dict(s, emb=False, res=None, act="none", alpha=1.0), ops_["x"], ops_["w"], ops_["bias"], None, None,
                        None)["ref"]
        v = s["alpha"] * (pre + emb_rows.double()) + (0 if ops_["res"] is None else ops_["res"].double())
        ops_["y32"].copy_(v.float())
        ops_["y"].copy_(ops_["y32"])
        return
    r = reference(s2, ops_["x"] if x is None else x, ops_["w"] if w is None else w, ops_["bias"] if bias is None else bias, e,
                  ops_["res"] if res is None else res, None)["ref"]
    ops_["y32"].copy_(r.float())
    ops_["y"].copy_(ops_["y32"])


def fault_far_edge(s, o, r):
    """the far-edge padding tap (pad_hi_extra) reads the neighbouring (last) pixel instead of zero"""
    N, H, W, C = (s[k] for k in "NHWC")
    x = o["x"].reshape(N, H, W, C).permute(0, 3, 1, 2)
    x = F.pad(x, (0, 1, 0, 1), mode="replicate").permute(0, 2, 3, 1).reshape(-1, C)
    _faulted(s, o, x=x, H=H + 1, W=W + 1, pad_hi_extra=0)


def fault_upsample(s, o, r):
    """the nearest-x2 source index rounded up at odd positions: (i + 1) >> 1 instead of i >> 1"""
    N, H, W, C = (s[k] for k in "NHWC")
    x = o["x"].reshape(N, H, W, C)
    ih = torch.clamp((torch.arange(2 * H) + 1) // 2, max=H - 1)
    iw = torch.clamp((torch.arange(2 * W) + 1) // 2, max=W - 1)
    x = x[:, ih][:, :, iw].reshape(-1, C)
    _faulted(s, o, x=x, H=2 * H, W=2 * W, up=False)


def fault_sentinel_tile(s, o, r):
    """the last, ragged 64-row tile never written: it keeps the NaN sentinel"""
    _rounded(s, o, r)
    Mo = o["y32"].shape[0]
    assert Mo % 64
    o["y32"][Mo // 64 * 64:] = NAN
    o["y"][Mo // 64 * 64:] = NAN


def fault_tile_first_image_emb(s, o, r):
    """a 64-row tile that spans two images adds the embedding row of its first image to all its rows"""
    P, Q, Mo = out_geometry(s)
    img = torch.arange(Mo) // (P * Q)
    first = img[(torch.arange(Mo) // 64) * 64]
    assert bool((first != img).any())
    _faulted(s, o, emb_rows=o["emb"][first])


def fault_missing_k_chunk(s, o, r):
    """one 16-deep k chunk (k = 32..47 of R*S*C) missing in the second 64-row tile"""
    _rounded(s, o, r)
    w = o["w"].clone()
    w[:, 32:48] = 0
    rows = slice(64, 128)
    without = reference(s, o["x"], w, o["bias"], o["emb"], o["res"], None)["ref"]
    o["y32"][rows] = without[rows].float()
    o["y"][rows] = o["y32"][rows]


def fault_geglu_swap(s, o, r):
    """the value and gate weight rows of one GEGLU block swapped"""
    gb = s["gb"]
    j = 1  # block 1: weight rows [2 gb, 4 gb)
    perm = torch.arange(s["K"])
    perm[2 * gb * j:2 * gb * j + gb] += gb
    perm[2 * gb * j + gb:2 * gb * (j + 1)] -= gb
    _faulted(s, o, w=o["w"][perm], bias=None if o["bias"] is None else o["bias"][perm])


def fault_residual_pitch(s, o, r):
    """the fp32 residual read with row pitch Kout instead of ldr (reads of a guard column taken as 0)"""
    buf, (rows, cols) = o["bufs"]["res"]
    Mo, Ko = o["res"].shape
    flat = buf.reshape(-1)
    idx = cols.start + torch.arange(Mo)[:, None] * Ko + torch.arange(Ko)[None]
    _faulted(s, o, res=flat[idx].nan_to_num(0.0))


SELF_GEOM = dict(N=2, H=6, W=10, C=24, K=40, R=3, emb=True, res="f32", alpha=0.5)
FAULTS = [("far-edge padding tap reads the neighbouring pixel", fault_far_edge,
           dict(N=2, H=10, W=8, C=8, K=24, R=3, stride=2, pad=0, pad_hi_extra=1)),
          ("upsample index rounded up at odd positions", fault_upsample, dict(N=2, H=5, W=7, C=8, K=24, R=3, up=True)),
          ("last ragged 64-row tile left at the sentinel", fault_sentinel_tile, dict(N=1, H=10, W=10, C=16, K=24, R=3)),
          ("tile spanning two images takes its first image's embedding", fault_tile_first_image_emb, SELF_GEOM),
          ("one 16-deep k chunk missing in one tile", fault_missing_k_chunk, SELF_GEOM),
          ("GEGLU value and gate rows swapped in one block", fault_geglu_swap,
           dict(N=1, H=1, W=70, C=32, K=64, act="geglu", gb=16)),
          ("fp32 residual read with the wrong row pitch", fault_residual_pitch, SELF_GEOM)]


@pytest.mark.parametrize("exact", [False, True], ids=["random", "exact"])
@pytest.mark.parametrize("geom", [g for _, _, g in FAULTS], ids=[n for n, _, _ in FAULTS])
def test_checker_accepts_a_correctly_rounded_fp32_result(geom, exact):
    check = _self_case(geom, exact)
    worst = check()
    assert max(worst.values()) <= (0.0 if exact and geom.get("act") is None else 0.5), worst


@pytest.mark.parametrize("exact", [False, True], ids=["random", "exact"])
@pytest.mark.parametrize("fault,geom", [(f, g) for _, f, g in FAULTS], ids=[n for n, _, _ in FAULTS])
def test_checker_rejects_fault(fault, geom, exact):
    check = _self_case(geom, exact, fault)
    with pytest.raises(AssertionError):
        check()


# ---- production census ------------------------------------------------------------------------------------------------------
def production_runs(dtype, dev):
    """(tag, fn) for every network the census runs at one dtype: UNet + ControlNet apply_model at 256^2 with 1 and 2 rows and
    at a 40x24 latent map, VAE decode and encode at 256^2, the CLIP text encoder on one prompt"""
    from makeupdiffuse_b200 import B200ControlLDM, B200FirstStageDecoder, B200FirstStageEncoder
    from makeupdiffuse_b200.clip import B200FrozenCLIPEmbedder
    from makeupdiffuse_b200.synth import synthetic_first_stage_state_dict, synthetic_state_dict
    from oracle.clip import BOS, EOS, OracleCLIPTextEncoder
    name = "f32" if dtype == F32 else "bf16"
    g = torch.Generator(device=dev).manual_seed(0)
    m = B200ControlLDM(dtype=dtype, device=dev)
    m.load_state_dict(synthetic_state_dict(m, 0, dev))
    for rows, h, w in ((1, 32, 32), (2, 32, 32), (1, 40, 24)):
        cond = {"c_crossattn": [torch.randn(rows, 77, 768, device=dev, generator=g)],
                "c_concat": [torch.rand(rows, 6, 8 * h, 8 * w, device=dev, generator=g)]}
        x = torch.randn(rows, 4, h, w, device=dev, generator=g)
        t = torch.full((rows,), 501, device=dev, dtype=torch.long)
        yield f"{name} apply_model {rows} x {8 * h}x{8 * w}", lambda: m.apply_model(x, t, cond)
    del m
    dec, enc = B200FirstStageDecoder(dtype=dtype), B200FirstStageEncoder(dtype=dtype)
    dec.load_state_dict(synthetic_first_stage_state_dict(dec, 0, dev), device=dev)
    enc.load_state_dict(synthetic_first_stage_state_dict(enc, 0, dev), device=dev)
    z = torch.randn(1, 4, 32, 32, device=dev, generator=g)
    img = torch.rand(1, 3, 256, 256, device=dev, generator=g) * 2 - 1
    yield f"{name} VAE decode 256^2", lambda: dec.decode(z)
    yield f"{name} VAE encode 256^2", lambda: enc.encode(img)
    del dec, enc
    torch.manual_seed(0)
    clip = B200FrozenCLIPEmbedder(device=dev, dtype=dtype).load_state_dict(OracleCLIPTextEncoder().state_dict())
    tok = torch.randint(0, 49406, (1, 77), generator=torch.Generator().manual_seed(0))
    tok[0, 0], tok[0, 12:] = BOS, EOS
    yield f"{name} CLIP text encoder, one prompt", lambda: clip(tok.to(dev))


def case_signatures():
    """signature -> case label, and per dtype the largest R*S*C and M a case runs"""
    sigs, most = {}, {}
    for label, s in CASES.items():
        P, Q, Mo = out_geometry(s)
        o = make_operands(s, "cuda", 0)
        d = ops.make_conv_desc(o["x"], o["w"], o["y"], **o["kw"])
        sigs.setdefault(signature(d, o["res"], o["y"], o["y32"]), label)
        r, m = most.get(s["dtype"], (0, 0))
        most[s["dtype"]] = (max(r, depth(s)), max(m, Mo))
    return sigs, most


@pytest.mark.gpu
def test_production_census(monkeypatch):
    """every descriptor the yaml-size networks send to the generic kernel, in both dtypes, has the signature of a case here, and
    no case is smaller in R*S*C or M than what production sends; the bf16 step at power-of-two sizes sends it nothing"""
    real = ops.conv2d
    census, tag, bf16_step = {}, [""], []

    def recorder(x2d, w, y2d, **kw):
        d = ops.make_conv_desc(x2d, w, y2d, **kw)
        if L.load().mkd_conv2d_path(ctypes.byref(d)) == L.PATH_GENERIC:
            sig = signature(d, kw.get("residual"), y2d, kw.get("y32"))
            record(census, sig, d, tag[0])
            if tag[0].startswith("bf16 apply_model") and tag[0].endswith("256x256"):
                bf16_step.append((tag[0], sig))
        real(x2d, w, y2d, **kw)
    monkeypatch.setattr(ops, "conv2d", recorder)
    for dtype in (F32, BF):
        for tag[0], fn in production_runs(dtype, "cuda"):
            fn()
            torch.cuda.synchronize()
    monkeypatch.undo()
    sigs, most = case_signatures()
    print_census(census, sigs)
    missing = [sig for sig in census if sig not in sigs]
    assert not missing, f"production sends the generic kernel descriptors no case covers: {missing}"
    for dt in ("f32", "bf16"):
        rsc = max((e["rsc"] for sig, e in census.items() if sig[0] == dt), default=0)
        m = max((e["m"] for sig, e in census.items() if sig[0] == dt), default=0)
        assert rsc <= most[dt][0] and m <= most[dt][1], (dt, rsc, m, most[dt])
    print(f"bf16 apply_model at 256x256: {len(bf16_step)} generic launches")
    assert not bf16_step, f"the bf16 step at power-of-two sizes sends the generic kernel {sorted(set(bf16_step), key=str)}"


if __name__ == "__main__":  # the profiling child of kernel_names: one JSON line on stdout
    print(json.dumps(profile_every_case()))
