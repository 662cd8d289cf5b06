"""Element-wise parity of the attention kernels (attention_tcgen05.cu: attn_split_kernel<DN>, attn_tcgen05_kernel<DN, NWG, KST,
VST>; attention.cu: attn_simt_kernel<T>; norm.cu: softmax_rows_kernel<T, TO>) against a float64 statement of the same
operation on the same operands, plus proof of which instantiation each case ran and a census of what production launches.

Why element-wise, and why these inputs: a relative L2 norm over a whole output cannot see a fault confined to a few elements,
and N(0, 1) scores never move the row max after the first key tile.  Here every stored element is held to its own bound, and
the inputs are built so that the path under test holds the probability mass (section "cases"); a CPU restatement of the
tcgen05 algorithm counts, per case, that the declared path is really reached (test_every_case_reaches_its_declared_path).

Reference (float64, the kernel's actual bf16 / fp32 operands): S = q k^T, s = scale S, P = softmax(s) (causal where the entry
is), ref = P v.  A[i, c] = sum_j P_ij |v_jc|.  u = 2^-24.  sl2 = fp32(fp32(scale) * fp32(log2 e)), the host's argument.

tcgen05 kernels (both): bound = 2^-8 |ref| + (1 + 2^-8) E, 2^-8 for the bf16 output, and E the sum of
    bf16 P          2^-8 A.  Every p goes to the PV MMA rounded to bf16 while l sums the unrounded fp32 p: rigorous.
    per-p errors    p_j = 2^(a_j) carries a relative error e_ij; through O / l it moves the output by sum_j P_ij e_ij (v_jc - ref_ic),
                    bounded by sum_j P_ij e_ij |v_jc| + |ref_ic| sum_j P_ij e_ij, with
                      e_ij = EX2 + ln2 (sl2 (dS_ij + dS_max,i) + u (sl2 |S_max,i| + 8 + 4 (|a_ij| + 8)))
                    EX2 = 2^-22: ex2.approx.ftz.f32, at most 2 ulp of its result (PTX ISA, "ex2").
                    dS_ij = u sqrt(dn) sum_c |q_ic| |k_jc|: the tensor-core accumulation of the score (the bound the GEMM test
                    measured, dn = head dim rounded up to 16); dS_max is the error of the row max the kernel subtracts.
                    u (sl2 |S_max| + 8): the rounding of m sl2 (the lazily raised m sits at most 8 / sl2 below the row max);
                    4 u (|a| + 8): the rounding of the FFMA2 argument s sl2 - m sl2 and of sl2 itself (|a| <= |a_ij| + 8 with
                    the lazy max).  This term grows with |s sl2| and is not negligible at |s sl2| ~ 10^3.
    sums            u (Nkv + 4 T + 24) A: l is 16 + 3 fp32 adds per tile plus one per tile and one rescale multiply per tile;
                    O is at most one fp32 add per key (the MMA adds once per 16 keys), one rescale multiply per tile and the
                    final * (1 / l) (two roundings).  T = key tiles (128 keys) or, for the split kernel, 64-key halves.
    merge (split)   (EX2 + 2 ln2 u (D_i + 8)) (A + |ref|) + 8 u A, D_i = sl2 (max_j S_ij - min_j S_ij): a_g = ex2((m_g - m) sl2)
                    carries the ex2 error and the rounding of its argument, and it scales O_g and l_g alike (so it enters as a
                    per-p error); inv = 1 / (l a + l' a'), c = a inv, r c, own + oth round 8 times at most.
    E is multiplied by 1.01 for second-order products (each first-order relative term is below 2^-7) and gets the absolute
    floor Nkv 2^-126 max|v| (ex2.approx.ftz flushes p < 2^-126; l >= 1) + 2^-133 (bf16 subnormal output).

attn_simt_kernel<T> (one warp per query; three serial fmaf chains): tau(n) = 2 u sqrt(n + 4), the serial-chain bound of
test_conv_generic_elementwise_gpu.py, per chain:
    score           qs = q * scale (one rounding) then a d-long fmaf chain: dS_ij = (tau(d) + 2 u) scale sum_c |q_ic| |k_jc|
    per-p errors    x_ij = s_ij - m_i: e_ij = dS_ij + dS_max,i + 2 u |x_ij| (the subtraction and __expf's x log2 e) +
                    (2 + 1.173 |x_ij|) 2^-23 (__expf: 2 + floor(1.173 |x|) ulp, CUDA C Programming Guide, intrinsic functions),
                    entering as above
    sums            (tau(ceil(Nkv / 32) + 5) + tau(Nkv) + 2 u) A: the per-lane sums then the 5-level warp reduction, the
                    Nkv-long PV chain, and acc * inv with inv = 1 / sum
    output          bf16: 2^-8 |ref| + (1 + 2^-8) E; fp32: u |ref| + (1 + u) E; E as above (factor 1.01, floor)
softmax_rows_kernel<T, TO>: y_j = 2^(a_j) / sum, a_j = fmaf(x_j, sl2, -m sl2), per element relative
    eps_j = ln2 u (sl2 |x_max| + 3 |a_j|) + 2^-22 (the rounding of m sl2, of the fmaf and of sl2; exp2f: 2 ulp, CUDA C
    Programming Guide); |y_j - ref_j| <= y_j (eps_j + sum_k y_k eps_k + (8 ceil(C / 256) + 5) u + 2 u) (the fp32 sum: per-lane
    serial adds then the warp reduction; 1 / sum and the product), times 1.01, + C 2^-148 (subnormal exp2f results), plus the
    output rounding (2^-8 or u relative, 2^-133 absolute for bf16).

Exact-operand cases (held to bit equality): scale chosen so that sl2 is a power of two (SIMT: scale itself), small-integer q
and k, every p exactly 0 or 1 (the selected keys score the row max, all others >= 150 / sl2 lower: ex2 underflows to 0), a
power-of-two count of selected keys (1 / l is IEEE division) and small-integer v: the output is an exact bf16 value.  All real
scores are negative, so a zero-filled tail key that escaped the -inf mask would score 0, become the max and take the weight.

Every output sits in a NaN-prefilled buffer at a column offset with ldo > C and guard rows after B Nq; each case runs in the
production layout (q, k, v column slices of one [M, 3C] buffer, or [M, C] + [M_kv, 2C] for cross-attention) and in a guarded
one (each operand in its own buffer with NaN columns on both sides and NaN rows after B N: any read outside a view poisons the
result).  After a call every guard and every input is unchanged bit for bit; a second launch is bit-identical (no atomics).

Out of scope: MKD_ATTN_WHOLE=1 (attn_tcgen05_kernel<48|64, 1, 2, 2>), a debug switch read once per process, and the MKD_ATTN_MMA
kernel of trace builds (attn_mma_kernel), which the shipped library does not contain.
"""
import json
import math
import os
import re
import subprocess
import sys
import zlib

import numpy as np
import pytest
import torch

from makeupdiffuse_b200 import _lib as L
from makeupdiffuse_b200 import ops
from test_gemm_elementwise_gpu import NAN, U, _bits, check_guards, launched_kernels

BF, F32 = torch.bfloat16, torch.float32
DT = {"bf16": BF, "f32": F32}
TN = {"bf16": "__nv_bfloat16", "f32": "float"}
LN2 = math.log(2.0)
EX2 = 2.0 ** -22
BF16_REL = 2.0 ** -8
LOG2E_F = np.float32(1.4426950408889634)

MEASURED = {}  # bound name -> (worst |err| / bound, case label, element)


def host_sl2(scale):
    """the kernels' scale * log2 e, as the host computes it in fp32"""
    return float(np.float32(np.float32(scale) * LOG2E_F))


def exact_scale(sl2):
    """an fp32 scale whose host product scale * 1.4426950408889634f is exactly sl2 (a power of two)"""
    x = np.float32(sl2 / 1.4426950408889634)
    for c in (x, np.nextafter(x, np.float32(0)), np.nextafter(x, np.float32(100))):
        if np.float32(c) * LOG2E_F == np.float32(sl2):
            return float(c)
    raise AssertionError(f"no fp32 scale gives sl2 = {sl2}")


def tau(n):
    return 2 * U * math.sqrt(n + 4)


# ---- kernel names and the instantiation table ------------------------------------------------------------------------------
FAMILY = ("attn_tcgen05_kernel", "attn_split_kernel", "attn_simt_kernel", "softmax_rows_kernel", "attn_mma_kernel")
_FAM = re.compile(r"(?<![A-Za-z_])(" + "|".join(FAMILY) + r")(<[^>]*>|I(?:Li-?\d+E|f|13__nv_bfloat16|S\d*_)+E)?")
_MANGLED_ARG = re.compile(r"Li(-?\d+)E|(f)|13(__nv_bfloat16)|(S\d*_)")


def canonical(name):
    """'void (anonymous namespace)::attn_tcgen05_kernel<80, 2, 2, 1>(...)' (or its mangled form) ->
    'attn_tcgen05_kernel<80,2,2,1>'; None for kernels outside the attention family"""
    m = _FAM.search(name)
    if not m:
        return None
    args = m.group(2)
    if not args:
        return m.group(1)
    if args.startswith("I"):
        vals = []
        for i, f, b, sub in _MANGLED_ARG.findall(args[1:-1]):
            vals.append(i or ("float" if f else b) if not sub else vals[-1])  # S<n>_: a type named earlier
    else:
        vals = [re.sub(r"^\((?:int|unsigned)\)|[uUlL]+$", "", a.strip()) for a in args[1:-1].split(",")]
    return f"{m.group(1)}<{','.join(vals)}>"


def tc(dn, nwg, kst, vst):
    return f"attn_tcgen05_kernel<{dn},{nwg},{kst},{vst}>"


def split(dn):
    return f"attn_split_kernel<{dn}>"


def simt(dt):
    return f"attn_simt_kernel<{TN[dt]}>"


def softmax_k(xdt, ydt):
    return f"softmax_rows_kernel<{TN[xdt]},{TN[ydt]}>"


def instantiation(s):
    """the kernel each entry point reaches with the default switches (attention.cu mkd_attention / mkd_attention_causal,
    attention_tcgen05.cu attention_tcgen05(), norm.cu mkd_softmax_rows)"""
    if s["entry"] == "softmax":
        return softmax_k(s["xdt"], s["ydt"])
    if s["entry"] == "causal" or s["dtype"] == "f32" or s["d"] > 160:
        return simt(s["dtype"])
    dn = -(-s["d"] // 16) * 16
    if dn <= 64:
        return split(dn)
    return tc(80, 2, 2, 1) if dn <= 80 else (tc(128, 2, 2, 1) if dn <= 128 else tc(160, 1, 2, 1))


TABLE = frozenset([split(16), split(32), split(48), split(64), tc(80, 2, 2, 1), tc(128, 2, 2, 1), tc(160, 1, 2, 1),
                   simt("bf16"), simt("f32"), softmax_k("f32", "bf16"), softmax_k("f32", "f32"), softmax_k("bf16", "bf16")])


def bound_name(s):
    k = instantiation(s)
    if s["entry"] == "softmax":
        return f"softmax_rows -> {s['ydt']}"
    return "split" if k.startswith("attn_split") else ("tcgen05" if k.startswith("attn_tcgen05") else f"simt {s['dtype']}")


# ---- the cases -------------------------------------------------------------------------------------------------------------
def acase(d, Nq, Nkv, pat, B=2, heads=2, dtype="bf16", entry="attn", scale=None, sl2=1.0):
    """an attention case; exact patterns take a scale that makes sl2 (tcgen05) or scale (SIMT) a power of two"""
    s = dict(entry=entry, dtype=dtype, B=B, heads=heads, Nq=Nq, Nkv=Nkv, d=d, pat=pat, exact=pat.startswith("exact"))
    if scale is None:
        if s["exact"]:
            simt_ = instantiation(s).startswith("attn_simt")
            scale = (64.0 if entry == "causal" else 1.0) if simt_ else exact_scale(sl2)
        else:
            scale = float(np.float32(d ** -0.5))
    s["scale"] = scale
    return s


def scase(M, C, pat, xdt="f32", ydt="bf16", scale=512 ** -0.5):
    return dict(entry="softmax", xdt=xdt, ydt=ydt, M=M, C=C, pat=pat, scale=float(np.float32(scale)), exact=False)


BUCKETS = {16: (8, 16), 32: (24, 32), 48: (40, 48), 64: (56, 64), 80: (72, 80), 128: (88, 96, 120, 128),
           160: (136, 152, 160)}
# (Nq, Nkv): Nq = 1 / 127 / 128 / 129 / 255 / 300 reach a last CTA whose second warpgroup has zero or one live row (NWG = 2);
# Nkv = 1 / 2 / 15 / 16 / 17 / 63 / 64 / 65 / 77 / 127 / 128 / 129 / 192 / 1000: ragged and whole 16-key steps, 64-key halves
# and 128-key tiles, down to one valid key in the last tile; H = 1, 2, 3 (odd) halves for the split kernel
EXACT_GEOS = [(129, 129), (128, 1), (1, 2), (16, 15), (64, 17), (127, 63), (255, 65), (300, 192), (129, 77), (16, 127),
              (64, 128), (127, 16), (255, 64), (300, 1000)]
BOUNDED = [("staircase", 300, 1000), ("staircase", 129, 4096), ("falling", 255, 1000), ("dominant", 300, 129),
           ("dominant", 64, 192), ("dominant", 129, 77), ("merge", 129, 192), ("merge", 255, 1000), ("warp", 300, 300),
           ("large", 128, 129), ("equal", 64, 4096)]

CASES = {}
for dn, ds in BUCKETS.items():
    for i, (Nq, Nkv) in enumerate(EXACT_GEOS):
        d = ds[i % len(ds)]
        CASES[f"d{d} exact {Nq}x{Nkv}" + (" sl2 2" if i % 2 else "")] = acase(d, Nq, Nkv, "exact", heads=3 if i % 3 == 1 else 2,
                                                                               sl2=2.0 if i % 2 else 1.0)
    for i, (pat, Nq, Nkv) in enumerate(BOUNDED):
        d = ds[(i + 1) % len(ds)]
        CASES[f"d{d} {pat} {Nq}x{Nkv}"] = acase(d, Nq, Nkv, pat, heads=3 if i % 4 == 3 else 2)
# production's regime (nets.py SpatialTransformer at 256^2 and 512^2, yaml heads = 8): self- and cross-attention (Nkv = 77)
for d, n in ((40, 1024), (40, 4096), (80, 256), (80, 1024), (160, 256), (160, 64), (160, 16)):
    B = 32 if (d, n) == (40, 1024) else 2
    CASES[f"production d{d} self {n} B{B} x 8 heads"] = acase(d, n, n, "normal", B=B, heads=8)
    CASES[f"production d{d} cross {n}x77 B{B} x 8 heads"] = acase(d, n, 77, "normal", B=B, heads=8)
# the SIMT kernel: bf16 for head dims > 160 (the VAE's 512-wide head at 512^2), fp32 for the whole check mode
CASES.update({
    "bf16 d512 VAE 512^2 4096x4096": acase(512, 4096, 4096, "normal", heads=2),
    "bf16 d512 exact 129x77": acase(512, 129, 77, "exact"),
    "bf16 d168 exact 127x129": acase(168, 127, 129, "exact", heads=3),
    "bf16 d256 large 64x1000": acase(256, 64, 1000, "large"),
    "bf16 d176 dominant 100x300": acase(176, 100, 300, "dominant"),
})
for d, n in ((40, 1024), (80, 256), (160, 64), (160, 16), (16, 256), (32, 64), (64, 16), (64, 4)):  # yaml and reduced nets
    CASES[f"f32 d{d} self {n}"] = acase(d, n, n, "normal", dtype="f32", heads=4)
    CASES[f"f32 d{d} cross {n}x77"] = acase(d, n, 77, "normal", dtype="f32", heads=4)
CASES.update({
    "f32 d40 exact 129x77": acase(40, 129, 77, "exact", dtype="f32"),
    "f32 d8 exact 16x15": acase(8, 16, 15, "exact", dtype="f32", heads=3),
    "f32 d40 large 64x1000": acase(40, 64, 1000, "large", dtype="f32"),
    "f32 d80 dominant 255x192": acase(80, 255, 192, "dominant", dtype="f32"),
    "f32 d40 equal 64x4096": acase(40, 64, 4096, "equal", dtype="f32"),
})
# causal (the CLIP text encoder: 77 tokens, 12 heads of 64): row i sees keys 0..i exactly
for dt in ("bf16", "f32"):
    CASES.update({
        f"{dt} causal exact 77 d64 x 12 heads": acase(64, 77, 77, "exact causal", dtype=dt, heads=12, entry="causal"),
        f"{dt} causal 77 d64 x 12 heads": acase(64, 77, 77, "normal", dtype=dt, heads=12, entry="causal"),
        f"{dt} causal exact 1 d8": acase(8, 1, 1, "exact causal", dtype=dt, entry="causal"),
        f"{dt} causal large 33 d16": acase(16, 33, 33, "large", dtype=dt, entry="causal"),
    })
# softmax_rows: the VAE's mid attention at 256^2 (S [1024, 1024] fp32 -> P bf16, scale 512^-0.5), ragged C, one-hot, equal and
# large-magnitude rows, every dtype pair
for xdt, ydt in (("f32", "bf16"), ("f32", "f32"), ("bf16", "bf16")):
    CASES.update({
        f"softmax {xdt}->{ydt} VAE 1024x1024": scase(1024, 1024, "normal", xdt, ydt),
        f"softmax {xdt}->{ydt} ragged C 1000": scase(77, 1000, "normal", xdt, ydt, scale=0.125),
        f"softmax {xdt}->{ydt} C 8": scase(300, 8, "normal", xdt, ydt, scale=1.0),
        f"softmax {xdt}->{ydt} C 2048 one-hot": scase(64, 2048, "onehot", xdt, ydt),
        f"softmax {xdt}->{ydt} C 72 equal rows": scase(33, 72, "equal", xdt, ydt),
        f"softmax {xdt}->{ydt} C 264 large": scase(40, 264, "large", xdt, ydt, scale=3.0),
    })
for s in CASES.values():
    s["kernel"] = instantiation(s)


def declared_paths(s):
    """the paths a case is built to reach (checked by test_every_case_reaches_its_declared_path)"""
    k = s["kernel"]
    if not (k.startswith("attn_split") or k.startswith("attn_tcgen05")):
        return ()
    blk = 64 if k.startswith("attn_split") else 128
    out = set()
    if s["pat"] in ("staircase", "warp") or (s["pat"] == "exact" and s["Nkv"] > 128):
        out.add("rescale")
    if k.startswith("attn_split") and (s["pat"] == "merge" or (s["pat"] == "exact" and s["Nkv"] > 64)):
        out.add("merge")
    if s["Nkv"] % blk and s["pat"] in ("exact", "dominant", "large"):
        out.add("mask")
    return tuple(sorted(out))


# ---- operands -----------------------------------------------------------------------------------------------------------
def pow2floor(n):
    return 1 << (n.bit_length() - 1)


def exact_regions(Nkv, cap):
    """key sets (power-of-two sizes) the rows of an exact case select: the first keys, the last valid key(s), a pair that
    straddles a 16-key PV step, the second 64-key half's last key and its first keys, keys of a later 128-key tile"""
    regs = [list(range(min(pow2floor(Nkv), 4))), [Nkv - 1]]
    if Nkv >= 2:
        regs.append([Nkv - 2, Nkv - 1])
    if Nkv > 64:
        regs.append([min(Nkv, 128) - 1])
        regs.append(list(range(64, 64 + pow2floor(min(Nkv - 64, 4)))))
    if Nkv > 128:
        regs.append([128 + (Nkv - 129) // 2])
    if Nkv >= 17:
        regs.append([15, 16])
    out = []
    for r in regs:
        if r not in out:
            out.append(r)
    return out[:cap]


def make_qkv(s, seed):
    """q [B, Nq, heads, d], k / v [B, Nkv, heads, d] (CPU, fp32 values exact in the case's dtype); patterns in log2 units of
    the softmax (a = sl2 s)"""
    g = torch.Generator().manual_seed(seed)
    B, H, Nq, Nkv, d = s["B"], s["heads"], s["Nq"], s["Nkv"], s["d"]
    Lf = host_sl2(s["scale"])
    q, k = torch.zeros(B, Nq, H, d), torch.zeros(B, Nkv, H, d)
    v = torch.randn(B, Nkv, H, d, generator=g)
    i, j = torch.arange(Nq), torch.arange(Nkv)
    b_, h_ = torch.arange(B)[:, None, None], torch.arange(H)[None, None, :]
    pat = s["pat"]

    def noise(nres, log2_std=1.0):
        sig = math.sqrt(log2_std / (Lf * math.sqrt(max(d - nres, 1))))
        q[..., nres:] = torch.randn(B, Nq, H, d - nres, generator=g) * sig
        k[..., nres:] = torch.randn(B, Nkv, H, d - nres, generator=g) * sig
    if pat == "normal":
        q.normal_(generator=g)
        k.normal_(generator=g)
    elif pat == "exact":
        # channel 0: every score -200; channel 1 + r: +180 for the keys of region r, which row i of (b, h) selects
        regs = exact_regions(Nkv, d - 1)
        v = torch.randint(-7, 8, (B, Nkv, H, d), generator=g).float()
        q[..., 0], k[..., 0] = -200.0, 1.0
        for r, keys in enumerate(regs):
            k[:, keys, :, 1 + r] = 1.0
        sel = (i[None, :, None] + 3 * b_ + 5 * h_) % len(regs)
        q.scatter_(3, 1 + sel[..., None].expand(B, Nq, H, 1), 180.0)
    elif pat == "exact causal":
        # score -200 + 2j (odd heads -200 - 2j) times scale 64: every row selects its last visible key (odd heads: key 0)
        v = torch.randint(-7, 8, (B, Nkv, H, d), generator=g).float()
        q[..., 0], k[..., 0] = -200.0, 1.0
        if d > 1:
            q[..., 1] = 1.0
            k[..., 1] = (2.0 * j[None, :, None] * torch.where(h_ % 2 == 1, -1.0, 1.0)).expand(B, Nkv, H)
    elif pat in ("staircase", "falling"):
        noise(1)
        t = j // 128
        lev = (t // 2) * 15 + (t % 2) * 6 if pat == "staircase" else -12 * t  # staircase: +6 (no rescale), +9 (rescale), ...
        q[..., 0] = 1.0
        k[..., 0] = (lev.float() / Lf)[None, :, None]
    elif pat == "dominant":
        G = 4
        noise(1 + G)
        pos = [0, Nkv - 1, min(Nkv, 128) - 1, min(Nkv, 64) - 1]  # first tile, last (ragged) tile, each 64-key half's last key
        for r, p in enumerate(pos):
            k[:, p, :, 1 + r] = 12.0 / Lf
        sel = (i[None, :, None] + b_ + h_) % G
        q.scatter_(3, 1 + sel[..., None].expand(B, Nq, H, 1), 1.0)
    elif pat == "merge":
        noise(1)
        gaps = torch.tensor([-40.0, -12.0, -3.0, 0.0, 3.0, 12.0, 40.0])  # stream 1 max minus stream 0 max, log2 units
        k[..., 0] = (torch.where((j // 64) % 2 == 1, 20.0, -20.0) / Lf)[None, :, None]
        q[..., 0] = (gaps[i % 7] / 40.0)[None, :, None]
    elif pat == "warp":
        noise(1)
        q[..., 0] = (i % 32 == 7).float()[None, :, None]  # one row per 32-row warp sees its max rise by 12 at key 128
        k[..., 0] = (12.0 / Lf * (j >= 128).float())[None, :, None]
    elif pat == "large":
        noise(1, log2_std=8.0)
        q[..., 0] = 1.0
        k[..., 0] = torch.where(b_ % 2 == 0, -1000.0 / Lf, 1000.0 / Lf)
    elif pat == "equal":
        q[..., 0], k[..., 0] = 1.0, -3.0
    else:
        raise ValueError(pat)
    dt = DT[s["dtype"]]
    return q.to(dt).float(), k.to(dt).float(), v.to(dt).float()


def make_x(s, seed):
    """softmax_rows input [M, C] (CPU)"""
    g = torch.Generator().manual_seed(seed)
    M, C = s["M"], s["C"]
    Lf = host_sl2(s["scale"])
    x = torch.randn(M, C, generator=g) * 4
    if s["pat"] == "onehot":
        x[torch.arange(M), (torch.arange(M) * 7) % C] = 4 * 8 + 150.0 / Lf
    elif s["pat"] == "equal":
        x[:] = 0.7
    elif s["pat"] == "large":
        x = (torch.randn(M, C, generator=g) * 8 + torch.where(torch.arange(M)[:, None] % 2 == 0, -1000.0, 1000.0)) / Lf
    return x.to(DT[s["xdt"]]).float()


# ---- float64 reference and bounds -----------------------------------------------------------------------------------------
def reference(s, q, k, v):
    """ref [B Nq, heads d], bound (same shape), exact (the expected bits as float64, or None)"""
    B, H, Nq, Nkv, d = s["B"], s["heads"], s["Nq"], s["Nkv"], s["d"]
    kern, causal = s["kernel"], s["entry"] == "causal"
    tcg = not kern.startswith("attn_simt")
    out_rel = BF16_REL if s["dtype"] == "bf16" else U
    scale, sl2 = s["scale"], host_sl2(s["scale"])
    blk = 64 if kern.startswith("attn_split") else 128
    nblk = -(-Nkv // blk)
    dn = -(-d // 16) * 16
    dev = q.device
    ref = torch.empty(B, Nq, H, d, dtype=torch.float64, device=dev)
    bound, exact = torch.empty_like(ref), (torch.empty_like(ref) if s["exact"] else None)
    hc = max(1, min(H, (1 << 24) // (Nq * Nkv)))
    valid = None
    if causal:
        valid = torch.arange(Nkv, device=dev)[None, :] <= torch.arange(Nq, device=dev)[:, None]
    for b in range(B):
        for h0 in range(0, H, hc):
            Q, K, V = (t[b, :, h0:h0 + hc].permute(1, 0, 2).double() for t in (q, k, v))
            S = Q @ K.transpose(1, 2)
            QK = Q.abs() @ K.abs().transpose(1, 2)
            if valid is not None:
                S = S.masked_fill(~valid, -math.inf)
            Smax = S.amax(-1, keepdim=True)
            E = torch.exp(scale * (S - Smax))
            P = E / E.sum(-1, keepdim=True)
            r = P @ V
            Va = V.abs()
            A = P @ Va
            if tcg:
                dS = U * math.sqrt(dn) * QK
                a = (sl2 * (S - Smax)).abs()
                e = EX2 + LN2 * (sl2 * (dS + dS.amax(-1, keepdim=True)) + U * (sl2 * Smax.abs() + 8 + 4 * (a + 8)))
                sums = U * (Nkv + 4 * nblk + 24) * A
                if kern.startswith("attn_split") and Nkv > 64:
                    D = sl2 * (Smax - S.amin(-1, keepdim=True))
                    sums = sums + (EX2 + 2 * LN2 * U * (D + 8)) * (A + r.abs()) + 8 * U * A
                extra = BF16_REL * A + sums
            else:
                dS = (tau(d) + 2 * U) * scale * QK
                dSm = dS.masked_fill(~valid, 0).amax(-1, keepdim=True) if valid is not None else dS.amax(-1, keepdim=True)
                x = (scale * (S - Smax)).abs()
                if valid is not None:
                    x = x.masked_fill(~valid, 0)
                e = dS + dSm + 2 * U * x + (2 + 1.173 * x) * 2.0 ** -23
                extra = (tau(-(-Nkv // 32) + 5) + tau(Nkv) + 2 * U) * A
            Pe = P * e
            E_ = 1.01 * (Pe @ Va + r.abs() * Pe.sum(-1, keepdim=True) + extra) + Nkv * 2.0 ** -126 * float(Va.max())
            if s["dtype"] == "bf16":
                E_ = E_ + 2.0 ** -133
            ref[b, :, h0:h0 + hc] = r.permute(1, 0, 2)
            bound[b, :, h0:h0 + hc] = (out_rel * r.abs() + (1 + out_rel) * E_).permute(1, 0, 2)
            if exact is not None:  # every p is exactly 0 or 1: the mean of the selected keys' v
                sel = (S == Smax).double()
                cnt = sel.sum(-1)
                assert bool(((cnt.long() & (cnt.long() - 1)) == 0).all()), "exact case: selected key count not a power of two"
                assert float((scale * (S - Smax)).masked_fill(sel.bool() | (S == -math.inf), -1e9).amax()) <= \
                    -(104.0 if not tcg else 150.0 / sl2 * scale), "exact case: unselected key too close to the max"
                exact[b, :, h0:h0 + hc] = ((sel @ V) / cnt[..., None]).permute(1, 0, 2)
    C = H * d
    ref, bound = ref.reshape(B * Nq, C), bound.reshape(B * Nq, C)
    if exact is not None:
        exact = exact.reshape(B * Nq, C).to(DT[s["dtype"]]).double()
    return dict(ref=ref, bound=bound, exact=exact)


def softmax_reference(s, x):
    sl2, C = host_sl2(s["scale"]), s["C"]
    x = x.double()
    xm = x.amax(-1, keepdim=True)
    y = torch.softmax(s["scale"] * x, -1)
    a = (sl2 * (x - xm)).abs()
    eps = LN2 * U * (sl2 * xm.abs() + 3 * a) + 2.0 ** -22
    rel = eps + (y * eps).sum(-1, keepdim=True) + (8 * -(-C // 256) + 5) * U + 2 * U
    E = 1.01 * y * rel + C * 2.0 ** -148
    out_rel = BF16_REL if s["ydt"] == "bf16" else U
    return dict(ref=y, bound=out_rel * y + (1 + out_rel) * E + (2.0 ** -133 if s["ydt"] == "bf16" else 0.0), exact=None)


# ---- the checker ------------------------------------------------------------------------------------------------------------
def check_output(label, s, refd, got, guards=()):
    """raises AssertionError on any changed guard / input, a non-finite element, or an element outside its bound (exact
    cases: any element that is not the expected bits); returns the worst |err| / bound"""
    check_guards(guards)
    got = got.double()
    bad = ~torch.isfinite(got)
    assert not bool(bad.any()), f"{label}: {int(bad.sum())} non-finite output element(s), first at {bad.nonzero()[0].tolist()}"
    if refd["exact"] is not None:
        ne = got != refd["exact"]
        assert not bool(ne.any()), (f"{label}: output != the exact result at {int(ne.sum())} element(s), first "
                                    f"{ne.nonzero()[0].tolist()}: {float(got[ne][0])} vs {float(refd['exact'][ne][0])}")
    r = (got - refd["ref"]).abs() / refd["bound"]
    idx = int(torch.argmax(r))
    worst, at = float(r.reshape(-1)[idx]), divmod(idx, got.shape[1])
    assert worst <= 1.0, (f"{label}: out[{at}] = {float(got[at]):.9g}, reference {float(refd['ref'][at]):.9g}, |err| / bound "
                          f"{worst:.3g}")
    return worst, at


# ---- buffers ------------------------------------------------------------------------------------------------------------------
def guarded(rows, cols, dtype, dev):
    """NaN-filled buffer holding a [rows, cols] view at column 8 (8 NaN columns on each side) with 3 NaN rows after it"""
    buf = torch.full((rows + 3, cols + 16), NAN, dtype=dtype, device=dev)
    return buf, buf[:rows, 8:8 + cols], (slice(0, rows), slice(8, 8 + cols))


def case_buffers(s, layout, dev, seed):
    """operands of a case on dev: views, and every buffer (name -> (buffer, region the call may write or None))"""
    bufs = {}
    if s["entry"] == "softmax":
        x = make_x(s, seed)
        if layout == "guarded":
            xb, xv, _ = guarded(s["M"], s["C"], DT[s["xdt"]], dev)
            xv.copy_(x)
        else:
            xb = xv = x.to(dev, DT[s["xdt"]])
        yb, yv, inside = guarded(s["M"], s["C"], DT[s["ydt"]], dev)
        bufs.update(x=(xb, None), y=(yb, inside))
        return dict(x=xv, y=yv, bufs=bufs, host=(x,))
    q, k, v = make_qkv(s, seed)
    B, H, Nq, Nkv, d, dt = s["B"], s["heads"], s["Nq"], s["Nkv"], s["d"], DT[s["dtype"]]
    C = H * d
    q2, k2, v2 = q.reshape(B * Nq, C), k.reshape(B * Nkv, C), v.reshape(B * Nkv, C)
    if layout == "guarded":
        views = []
        for name, t in (("q", q2), ("k", k2), ("v", v2)):
            buf, view, _ = guarded(t.shape[0], C, dt, dev)
            view.copy_(t)
            bufs[name] = (buf, None)
            views.append(view)
        qv, kv_, vv = views
    elif Nq == Nkv:  # self-attention: one [M, 3C] buffer
        qkv = torch.cat([q2, k2, v2], 1).to(dev, dt)
        bufs["qkv"] = (qkv, None)
        qv, kv_, vv = qkv[:, :C], qkv[:, C:2 * C], qkv[:, 2 * C:]
    else:  # cross-attention (nets.py): q [M, C], kv [M_kv, 2C]
        qb, kvb = q2.to(dev, dt), torch.cat([k2, v2], 1).to(dev, dt)
        bufs.update(q=(qb, None), kv=(kvb, None))
        qv, kv_, vv = qb, kvb[:, :C], kvb[:, C:]
    ob, ov, inside = guarded(B * Nq, C, dt, dev)
    bufs["o"] = (ob, inside)
    return dict(q=qv, k=kv_, v=vv, o=ov, bufs=bufs, host=(q, k, v))


def launch(s, o):
    if s["entry"] == "softmax":
        ops.softmax_rows(o["x"], o["y"], s["scale"])
    elif s["entry"] == "causal":
        ops.attention_causal(o["q"], o["k"], o["v"], o["o"], B=s["B"], heads=s["heads"], N=s["Nq"], d=s["d"], scale=s["scale"])
    else:
        ops.attention(o["q"], o["k"], o["v"], o["o"], B=s["B"], heads=s["heads"], Nq=s["Nq"], Nkv=s["Nkv"], d=s["d"],
                      scale=s["scale"])


def case_reference(s, o, dev):
    if s["entry"] == "softmax":
        return softmax_reference(s, o["host"][0].to(dev))
    return reference(s, *(t.to(dev) for t in o["host"]))


# ---- CPU restatement of the tcgen05 algorithm (and of the causal SIMT visibility) --------------------------------------------
def restate(s, q, k, v, fault=None, counts=None, rows=None):
    """the output the kernel of case s stores (float64 of its bf16 values), computed in fp32 torch the way the kernel orders
    it: 128-key tiles (attn_tcgen05_kernel) or two 64-key streams and their merge (attn_split_kernel), the 2^8 lazy threshold
    decided per 32-row group, bf16 P with l summed from unrounded p, -inf masking.  fault injects one error; counts (a dict)
    receives the rows that rescaled after the first block, the merges of two live streams with maxima > 8 / sl2 apart and the
    rows with a masked tail that carries weight; rows limits the queries restated (for counting)."""
    B, H, Nq, Nkv, d = s["B"], s["heads"], s["Nq"], s["Nkv"], s["d"]
    nq = Nq if rows is None else min(Nq, rows)
    if s["entry"] == "causal":
        delta = {"causal +1": 1, "causal -1": -1}.get(fault, 0)
        out = torch.empty(B, nq, H, d, dtype=torch.float64)
        for b in range(B):
            for h in range(H):
                S = s["scale"] * (q[b, :nq, h].double() @ k[b, :, h].double().T)
                vis = torch.arange(Nkv)[None, :] <= torch.arange(nq)[:, None] + delta
                out[b, :, h] = torch.softmax(S.masked_fill(~vis, -math.inf), -1) @ v[b, :, h].double()
        return out.reshape(B * nq, H * d).to(DT[s["dtype"]]).double()
    is_split = s["kernel"].startswith("attn_split")
    blk = 64 if is_split else 128
    nb = -(-Nkv // blk)
    sl2 = torch.tensor(host_sl2(s["scale"]), dtype=F32)
    nqp = -(-nq // 32) * 32
    out = torch.zeros(B, nq, H, d, dtype=torch.float64)
    for b in range(B):
        for h in range(H):
            Q = torch.zeros(nqp, d)
            Q[:nq] = q[b, :nq, h]
            S = torch.full((nqp, nb * blk), -math.inf)
            S[:, :Nkv] = (Q.double() @ k[b, :, h].double().T).float()
            V = torch.zeros(nb * blk, d)
            V[:Nkv] = v[b, :, h]
            if fault == "first invalid key unmasked" and Nkv < nb * blk:
                S[:, Nkv] = 0.0  # the zero-filled K row scores 0
            if fault == "last valid key masked":
                S[:, Nkv - 1] = -math.inf
            streams = [list(range(0, nb, 2)), list(range(1, nb, 2))] if is_split else [list(range(nb))]
            if fault == "second stream dropped when H is odd" and nb % 2 == 1 and nb > 1:
                streams[1] = []
            res = []
            for blocks in streams:
                m = torch.full((nqp,), -math.inf)
                l, O = torch.zeros(nqp), torch.zeros(nqp, d)
                for u_, t in enumerate(blocks):
                    st = S[:, t * blk:(t + 1) * blk]
                    mx = st.amax(1)
                    need = ((mx - m) * sl2 > 8.0).reshape(-1, 32).any(1).repeat_interleave(32)
                    m_new = torch.maximum(m, mx)
                    corr = torch.exp2((m - m_new) * sl2)
                    if counts is not None and u_ > 0:
                        counts["rescale"] += int((need & (m_new > m))[:nq].sum())
                    if fault != "l not rescaled":
                        l = torch.where(need, l * corr, l)
                    if fault != "O not rescaled":
                        O = torch.where(need[:, None], O * corr[:, None], O)
                    m = torch.where(need, m_new, m)
                    p = torch.exp2(st * sl2 - m[:, None] * sl2)
                    l = l + p.sum(1)
                    pb = p.bfloat16().float()
                    kvalid = Nkv - t * blk
                    if kvalid < blk and fault == "last partial 16-key PV step skipped":
                        pb[:, 16 * ((kvalid - 1) // 16):] = 0
                    O = O + (pb.double() @ V[t * blk:(t + 1) * blk].double()).float()
                res.append((m, l, O))
            if is_split:
                (m0, l0, O0), (m1, l1, O1) = res
                mm = torch.maximum(m0, m1)
                a0, a1 = torch.exp2((m0 - mm) * sl2), torch.exp2((m1 - mm) * sl2)
                inv = 1.0 / (l0 * a0 + l1 * a1)
                c0, c1 = a0 * inv, a1 * inv
                if fault == "merge uses one stream's coefficient for both":
                    c1 = c0
                O = O0 * c0[:, None] + O1 * c1[:, None]
                if counts is not None and len(streams[1]):
                    counts["merge"] += int(((m0 - m1).abs() * sl2 > 8.0)[:nq].sum())
            else:
                m, l, O = res[0]
                O = O * (1.0 / l)[:, None]
            out[b, :, h] = O[:nq].double()
            if counts is not None and Nkv % blk:  # masked tail, and either the tail's block carries >= 1/4 of the row's mass or
                # every real score is negative (an unmasked zero-filled key would take the weight)
                P = torch.softmax(S[:nq, :Nkv].double() * s["scale"], -1)
                counts["mask"] += int(((P[:, (nb - 1) * blk:].sum(1) >= 0.25) | (S[:nq, :Nkv].amax(1) < 0)).sum())
    out = out.reshape(B * nq, H * d)
    if fault == "output rows offset into the next batch":
        out = torch.cat([out[:1], out[:-1]])
    if fault == "head column offset wrong":
        out = out.reshape(B * nq, H, d).roll(1, 1).reshape(B * nq, H * d)
    return out.to(BF).double()


# ---- running a case on the GPU ------------------------------------------------------------------------------------------------
def run_case(label, layout, profiled):
    s = CASES[label]
    dev = "cuda"
    o = case_buffers(s, layout, dev, zlib.crc32(label.encode()))
    assert [c for c in map(canonical, profiled) if c] == [s["kernel"]], \
        f"{label}: the profiled launch ran {profiled}, expected [{s['kernel']}]"
    refd = case_reference(s, o, dev)
    before = {n: b.clone() for n, (b, _) in o["bufs"].items()}
    n0 = L.load().mkd_launch_count()
    launch(s, o)
    torch.cuda.synchronize()
    assert L.load().mkd_launch_count() - n0 == 1, f"{label}: {L.load().mkd_launch_count() - n0} launches, expected 1"
    out = o["y"] if s["entry"] == "softmax" else o["o"]
    guards = [(n, b, before[n], inside) for n, (b, inside) in o["bufs"].items()]
    worst, at = check_output(f"{label} [{layout}]", s, refd, out, guards)
    if not s["exact"] and worst > MEASURED.get(bound_name(s), (-1.0,))[0]:
        MEASURED[bound_name(s)] = (worst, f"{label} [{layout}]", at)
    first = out.clone()
    launch(s, o)
    torch.cuda.synchronize()
    assert torch.equal(_bits(first), _bits(out)), f"{label}: a second launch differs"
    print(f"{label + ' [' + layout + ']':<62s} worst err/bound {worst:.3f}{'  (bits exact)' if s['exact'] else ''}   "
          f"[{s['kernel']}]")


def profile_every_case():
    """label -> the CUDA kernels one launch of the case runs, by torch.profiler (see kernel_names)"""
    names = {}
    for label, s in CASES.items():
        o = case_buffers(s, "guarded", "cuda", zlib.crc32(label.encode()))
        names[label] = launched_kernels(lambda: launch(s, o))
        del o
    return names


@pytest.fixture(scope="module")
def kernel_names():
    """the profiled kernels of every case and the production census, from a child process: once CUPTI has started in a
    process, a later profiler session can lose its kernel records (test_conv_generic_elementwise_gpu.py)"""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([root] + [p for p in [os.environ.get("PYTHONPATH")] if p]))
    r = subprocess.run([sys.executable, "-s", os.path.abspath(__file__)], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, f"profiling child failed:\n{r.stdout[-2000:]}\n{r.stderr[-4000:]}"
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.fixture(scope="module", autouse=True)
def _report_margins():
    yield
    if MEASURED:
        print("\nworst measured |err| / bound per bound:")
        for name, (w, label, at) in sorted(MEASURED.items()):
            print(f"  {name:<22s} {w:.3f}   at {label}, element {at}")


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["production", "guarded"])
@pytest.mark.parametrize("label", list(CASES))
def test_attention_elementwise(label, layout, kernel_names):
    run_case(label, layout, kernel_names["cases"][label])


# ---- the table, the names, the paths (CPU) ----------------------------------------------------------------------------------
def test_cases_cover_exactly_the_instantiation_table():
    """every instantiation reachable with the default switches has exact and bounded cases, and no case reaches another"""
    got = {s["kernel"] for s in CASES.values()}
    assert got == TABLE, (sorted(got - TABLE), sorted(TABLE - got))
    for k in TABLE - {softmax_k(a, b) for a, b in (("f32", "bf16"), ("f32", "f32"), ("bf16", "bf16"))}:
        kinds = {s["exact"] for s in CASES.values() if s["kernel"] == k}
        assert kinds == {True, False}, f"{k}: exact and bounded cases needed, have {kinds}"
    assert instantiation(acase(40, 1, 1, "normal")) == split(48)
    assert instantiation(acase(136, 1, 1, "normal")) == tc(160, 1, 2, 1)
    assert instantiation(acase(168, 1, 1, "normal")) == simt("bf16")
    assert instantiation(acase(40, 1, 1, "normal", dtype="f32")) == simt("f32")


def test_every_case_geometry_rule():
    for label, s in CASES.items():
        if s["entry"] != "softmax":
            assert s["B"] >= 2 and s["heads"] >= 2, label  # cross-batch and cross-head writes are visible
    geos = {(s["Nq"], s["Nkv"]) for s in CASES.values() if s["entry"] == "attn"}
    for n in (1, 16, 64, 127, 128, 129, 255, 300, 1024, 4096):
        assert any(g[0] == n for g in geos), n
    for n in (1, 2, 15, 16, 17, 63, 64, 65, 77, 127, 128, 129, 192, 1000, 4096):
        assert any(g[1] == n for g in geos), n
    ds = {s["d"] for s in CASES.values() if s["entry"] == "attn"}
    assert {8, 24, 40, 56, 72, 88, 120, 136, 152} <= ds


def test_kernel_name_canonical_form():
    assert canonical("void (anonymous namespace)::attn_tcgen05_kernel<80, 2, 2, 1>(CUtensorMap_st, CUtensorMap_st, "
                     "CUtensorMap_st, __nv_bfloat16*, int, int, int, int, float)") == tc(80, 2, 2, 1)
    assert canonical("_ZN53_GLOBAL__N__a66b2dfe_20_attention_tcgen05_cu_79b444c719attn_tcgen05_kernelILi160ELi1ELi2ELi1EEEv14"
                     "CUtensorMap_stS1_S1_P13__nv_bfloat16iiiif") == tc(160, 1, 2, 1)
    assert canonical("void (anonymous namespace)::attn_split_kernel<48>(CUtensorMap_st, ...)") == split(48)
    assert canonical("_ZN53_GLOBAL__N__a66b2dfe_20_attention_tcgen05_cu_79b444c717attn_split_kernelILi16EEEv14CUtensorMap_stS1_"
                     "S1_P13__nv_bfloat16iiiif") == split(16)
    assert canonical("void (anonymous namespace)::attn_simt_kernel<__nv_bfloat16>(__nv_bfloat16 const*, ...)") == simt("bf16")
    assert canonical("_ZN45_GLOBAL__N__f58937f6_12_attention_cu_595359f816attn_simt_kernelIfEEvPKT_S3_S3_PS1_iiiiiiifi") == \
        simt("f32")
    assert canonical("void (anonymous namespace)::softmax_rows_kernel<float, __nv_bfloat16>(float const*, ...)") == \
        softmax_k("f32", "bf16")
    assert canonical("_ZN39_GLOBAL__N__048b5d68_7_norm_cu_5df35a2e19softmax_rows_kernelI13__nv_bfloat16S1_EEvPKT_PT0_liiif") == \
        softmax_k("bf16", "bf16")
    assert canonical("_ZN39_GLOBAL__N__048b5d68_7_norm_cu_5df35a2e19softmax_rows_kernelIffEEvPKT_PT0_liiif") == \
        softmax_k("f32", "f32")
    assert canonical("void (anonymous namespace)::gemm_tcgen05_kernel<160, 1, 4, 10, 0>(...)") is None


def test_exact_scales_give_a_power_of_two_sl2():
    for sl2 in (1.0, 2.0):
        assert host_sl2(exact_scale(sl2)) == sl2


REACH = [lbl for lbl, s in CASES.items() if declared_paths(s)]


@pytest.mark.parametrize("label", REACH)
def test_every_case_reaches_its_declared_path(label):
    """the restatement, on the case's own operands, counts rows that rescaled after the first key block, merges of two live
    streams whose maxima are > 8 / sl2 apart, and rows with a masked tail that carries weight: each declared path is > 0"""
    s = CASES[label]
    q, k, v = make_qkv(s, zlib.crc32(label.encode()))
    got = {"rescale": 0, "merge": 0, "mask": 0}
    B = min(s["B"], 2)  # the first two batches, the first 256 queries of every head
    restate(dict(s, B=B), q[:B], k[:B], v[:B], counts=got, rows=256)
    for path in declared_paths(s):
        assert got[path] > 0, f"{label}: declared path {path} not reached ({got})"


def test_every_tcgen05_instantiation_has_cases_on_every_path():
    for k in TABLE:
        if k.startswith("attn_split") or k.startswith("attn_tcgen05"):
            paths = {p for s in CASES.values() if s["kernel"] == k for p in declared_paths(s)}
            want = {"rescale", "mask"} | ({"merge"} if k.startswith("attn_split") else set())
            assert paths >= want, (k, paths)


# ---- the checker's self-tests (CPU): correct results pass, each injected fault fails ----------------------------------------
SELF = {
    "split staircase": acase(40, 64, 700, "staircase"),
    "tile staircase": acase(80, 64, 700, "staircase"),
    "split dominant ragged": acase(40, 64, 129, "dominant"),
    "tile dominant ragged": acase(88, 64, 129, "dominant"),
    "split merge H 3": acase(40, 64, 192, "merge"),
    "tile large": acase(80, 40, 129, "large"),
    "split large": acase(24, 40, 77, "large"),
    "split normal": acase(40, 70, 77, "normal", heads=3),
    "tile exact": acase(80, 64, 200, "exact", heads=3),
    "split exact": acase(40, 64, 200, "exact", sl2=2.0),
    "causal": acase(16, 77, 77, "normal", entry="causal"),
    "causal exact": acase(16, 77, 77, "exact causal", entry="causal"),
}
for _s in SELF.values():
    _s["kernel"] = instantiation(_s)

FAULTS = [("O not rescaled", ["split staircase", "tile staircase"]),
          ("l not rescaled", ["split staircase", "tile staircase"]),
          ("last valid key masked", ["split dominant ragged", "tile dominant ragged"]),
          ("first invalid key unmasked", ["tile large", "split large"]),
          ("last partial 16-key PV step skipped", ["split dominant ragged", "tile dominant ragged"]),
          ("merge uses one stream's coefficient for both", ["split merge H 3"]),
          ("second stream dropped when H is odd", ["split merge H 3"]),
          ("output rows offset into the next batch", ["split normal", "tile exact"]),
          ("head column offset wrong", ["split normal", "split exact"]),
          ("causal +1", ["causal", "causal exact"]),
          ("causal -1", ["causal", "causal exact"])]


def _self(name, fault=None):
    s = SELF[name]
    q, k, v = make_qkv(s, 11)
    refd = reference(s, q, k, v)
    return s, refd, restate(s, q, k, v, fault=fault)


@pytest.mark.parametrize("name", list(SELF))
def test_checker_accepts_the_restated_kernel(name):
    s, refd, out = _self(name)
    worst, _ = check_output(f"self-test {name}", s, refd, out)
    assert worst < 1.0


@pytest.mark.parametrize("fault,name", [(f, n) for f, names in FAULTS for n in names],
                         ids=[f"{f} ({n})" for f, names in FAULTS for n in names])
def test_checker_rejects_fault(fault, name):
    s, refd, out = _self(name, fault)
    with pytest.raises(AssertionError):
        check_output(f"self-test {name}: {fault}", s, refd, out)


def test_checker_rejects_a_write_past_the_view():
    s = SELF["split normal"]
    o = case_buffers(s, "guarded", "cpu", 3)
    before = {n: b.clone() for n, (b, _) in o["bufs"].items()}
    refd = case_reference(s, o, "cpu")
    q, k, v = o["host"]
    o["o"].copy_(restate(s, q, k, v))
    guards = [(n, b, before[n], inside) for n, (b, inside) in o["bufs"].items()]
    check_output("self-test", s, refd, o["o"], guards)
    buf, inside = o["bufs"]["o"]
    buf[s["B"] * s["Nq"], inside[1].start] = 0.0  # a guard row after B Nq
    with pytest.raises(AssertionError, match="guard"):
        check_output("self-test", s, refd, o["o"], guards)
    buf[s["B"] * s["Nq"], inside[1].start] = NAN
    o["bufs"]["k"][0][5, 3] = 1.0  # an input's guard column
    with pytest.raises(AssertionError, match="guard"):
        check_output("self-test", s, refd, o["o"], guards)


# ---- production census ------------------------------------------------------------------------------------------------------
def production_runs(dev):
    """(tag, fn): UNet + ControlNet apply_model at yaml size (256^2 with 1, 2 and 16 rows, 512^2 with 8 rows), VAE decode and
    encode at 256^2 and 512^2, the CLIP text encoder, one fp32 check-mode apply_model of the reduced networks"""
    from makeupdiffuse_b200 import B200ControlLDM, B200FirstStageDecoder, B200FirstStageEncoder
    from makeupdiffuse_b200.clip import B200FrozenCLIPEmbedder
    from makeupdiffuse_b200.synth import synthetic_first_stage_state_dict, synthetic_state_dict
    from oracle.clip import BOS, EOS, OracleCLIPTextEncoder
    g = torch.Generator(device=dev).manual_seed(0)
    m = B200ControlLDM(dtype=BF, device=dev)
    m.load_state_dict(synthetic_state_dict(m, 0, dev))
    for rows, h in ((1, 32), (2, 32), (16, 32), (8, 64)):
        cond = {"c_crossattn": [torch.randn(rows, 77, 768, device=dev, generator=g)],
                "c_concat": [torch.rand(rows, 6, 8 * h, 8 * h, device=dev, generator=g)]}
        x = torch.randn(rows, 4, h, h, device=dev, generator=g)
        t = torch.full((rows,), 501, device=dev, dtype=torch.long)
        yield f"apply_model {rows} x {8 * h}^2", lambda: m.apply_model(x, t, cond)
    del m
    dec, enc = B200FirstStageDecoder(dtype=BF), B200FirstStageEncoder(dtype=BF)
    dec.load_state_dict(synthetic_first_stage_state_dict(dec, 0, dev), device=dev)
    enc.load_state_dict(synthetic_first_stage_state_dict(enc, 0, dev), device=dev)
    for h in (32, 64):
        z = torch.randn(1, 4, h, h, device=dev, generator=g)
        img = torch.rand(1, 3, 8 * h, 8 * h, device=dev, generator=g) * 2 - 1
        yield f"VAE decode {8 * h}^2", lambda: dec.decode(z)
        yield f"VAE encode {8 * h}^2", lambda: enc.encode(img)
    del dec, enc
    torch.manual_seed(0)
    clip = B200FrozenCLIPEmbedder(device=dev, dtype=BF).load_state_dict(OracleCLIPTextEncoder().state_dict())
    tok = torch.randint(0, 49406, (1, 77), generator=torch.Generator().manual_seed(0))
    tok[0, 0], tok[0, 12:] = BOS, EOS
    yield "CLIP text encoder", lambda: clip(tok.to(dev))
    del clip
    p = dict(model_channels=64, num_heads=4, context_dim=64)
    m32 = B200ControlLDM(p, p, dtype=F32, device=dev)
    m32.load_state_dict(synthetic_state_dict(m32, 0, dev))
    cond = {"c_crossattn": [torch.randn(2, 77, 64, device=dev, generator=g)],
            "c_concat": [torch.rand(2, 6, 128, 128, device=dev, generator=g)]}
    x, t = torch.randn(2, 4, 16, 16, device=dev, generator=g), torch.full((2,), 981, device=dev, dtype=torch.long)
    yield "fp32 check mode, reduced nets, 2 x 128^2", lambda: m32.apply_model(x, t, cond)


def census_run():
    """in the child: every attention-family kernel production launches (by profiler) and every call signature"""
    sigs, kernels = {}, {}
    real = (ops._attention, ops.attention_causal, ops.softmax_rows)
    tag = [""]

    def ld(*ts):
        return "/".join(str(t.stride(0)) for t in ts)

    def rec(key):
        e = sigs.setdefault(json.dumps(key), dict(n=0, where=tag[0]))
        e["n"] += 1

    def att(q2d, k2d, v2d, o2d, *, B, heads, Nq, Nkv, d, scale):
        s = dict(entry="attn", dtype="bf16" if q2d.dtype == BF else "f32", d=d)
        rec([instantiation(s), "attention", s["dtype"], heads, Nq, Nkv, d, f"ld q/k/v/o {ld(q2d, k2d, v2d, o2d)}, C {heads * d}"])
        real[0](q2d, k2d, v2d, o2d, B=B, heads=heads, Nq=Nq, Nkv=Nkv, d=d, scale=scale)

    def causal(q2d, k2d, v2d, o2d, *, B, heads, N, d, scale):
        s = dict(entry="causal", dtype="bf16" if q2d.dtype == BF else "f32", d=d)
        rec([instantiation(s), "attention_causal", s["dtype"], heads, N, N, d, f"ld q/k/v/o {ld(q2d, k2d, v2d, o2d)}, C {heads * d}"])
        real[1](q2d, k2d, v2d, o2d, B=B, heads=heads, N=N, d=d, scale=scale)

    def smx(x2d, y2d, scale=1.0):
        name = {BF: "bf16", F32: "f32"}
        k = softmax_k(name[x2d.dtype], name[y2d.dtype])
        rec([k, "softmax_rows", name[y2d.dtype], 1, x2d.shape[0], x2d.shape[1], x2d.shape[1], f"ld x/y {ld(x2d, y2d)}"])
        real[2](x2d, y2d, scale)
    ops._attention, ops.attention_causal, ops.softmax_rows = att, causal, smx
    try:
        for tag[0], fn in production_runs("cuda"):
            for n in launched_kernels(fn):
                c = canonical(n)
                if c:
                    e = kernels.setdefault(c, dict(n=0, where=tag[0]))
                    e["n"] += 1
            torch.cuda.synchronize()
    finally:
        ops._attention, ops.attention_causal, ops.softmax_rows = real
    return dict(kernels=kernels, sigs=sigs)


def covering_case(key):
    """a case with the same instantiation, head dim and (Nq, Nkv) (softmax_rows: rows and C) as a production signature"""
    kern, _, _, _, nq, nkv, d = key[:7]
    for label, s in CASES.items():
        if s["kernel"] != kern:
            continue
        if s["entry"] == "softmax" and (s["M"], s["C"]) == (nq, nkv):
            return label
        if s["entry"] != "softmax" and (s["Nq"], s["Nkv"], s["d"]) == (nq, nkv, d):
            return label
    return None


@pytest.mark.gpu
def test_production_census(kernel_names):
    """every attention-family kernel the yaml-size networks launch is in the table above, and every (entry, dtype, heads, Nq,
    Nkv, d, leading dimensions) they pass has a case with the same instantiation, d, Nq and Nkv"""
    cen = kernel_names["census"]
    print("\nattention census, kernels (kernel -> launches, first seen in):")
    for k, e in sorted(cen["kernels"].items()):
        print(f"  {k:<40s} {e['n']:6d}   {e['where']:<42s} {'case' if k in TABLE else 'NO CASE'}")
    print("attention census, calls (instantiation | entry dtype heads Nq Nkv d | layout -> calls, first seen in, case):")
    missing = []
    for key_s, e in sorted(cen["sigs"].items()):
        key = json.loads(key_s)
        cover = covering_case(key)
        if cover is None:
            missing.append(key)
        print(f"  {key[0]:<40s} {' '.join(map(str, key[1:7]))} | {key[7]}\n      {e['n']:5d} calls, first in {e['where']}; "
              f"case: {cover or 'NO CASE'}")
    unknown = sorted(k for k in cen["kernels"] if k not in TABLE)
    assert not unknown, f"production launches attention kernels no case here checks: {unknown}"
    assert not missing, f"production passes signatures no case covers: {missing}"


if __name__ == "__main__":  # the profiling child of kernel_names: one JSON line on stdout
    result = dict(cases=profile_every_case())
    torch.cuda.synchronize()
    result["census"] = census_run()
    print(json.dumps(result))
