"""Element-wise parity of the tensor-core conv / GEMM kernels (gemm_tcgen05.cu: single CTA, gemm_pair.cu: CTA pair) against a
float64 statement of mkd_conv_desc on the same bf16 operands, plus proof of which kernel instantiation each case ran.

Why element-wise: a relative L2 norm over a whole output cannot see a fault confined to a few elements (one zeroed row among
30k rows, one 8-channel group without its bias, one image's embedding row).  Here every stored element is held to its own
bound, derived from the magnitude of the terms that produced it:

    A[m, k] = |alpha| * (sum_{r,s,c} |x| |w| + |bias[k]| + |emb[n, k]|) + |residual[m, k]|

    y32:                  |y32 - ref| <= tau * A,   tau = u sqrt(K_tot)   (u = 2^-24, K_tot = R S C + C2: contraction length)
    y (bf16), with y32:   y == bf16(y32) exactly
    y (bf16), alone:      |y - ref| <= 2^-8 |ref| + (1 + 2^-8) tau * A        (2^-8: bf16 keeps 8 significant bits)
    SiLU:                 ref = silu(pre), bound 1.1 tau * A (|silu'| <= 1.1) + the fast-math error of silu_f
    GEGLU:                ref = a * gelu_erf(g), bound 2^-8 |ref| + (1 + 2^-8) [|gelu(g)| tau A_a + 1.13 (|a| + tau A_a) tau A_g
                          + (|a| + tau A_a) GELU_APPROX (|g| + tau A_g)]
    statistics:           every (128-row tile, channel) sum and sum of squares against the float64 sums of the fp32 values
                          the kernel stored, each against its own magnitude (TAU_STATS * sum |v|, TAU_STATS * sum v^2)
    GroupNorm tail:       the normalised output of the split-K reducer against a float64 GroupNorm(+SiLU) of the stored y32

Every output sits in a larger buffer prefilled with a NaN sentinel (rows beyond M, columns outside an ld > K slice, extra
statistics rows / columns); inputs do too, so a read outside a view poisons the result.  After a call every guard and every
input is unchanged bit for bit, and a second identical launch (split-K included) is bit-identical.

tau: the accumulator takes one fp32 add per 16-deep MMA k step, n = K_tot / 16 of them.  Adds rounded to nearest have errors
that cancel like a random walk, and |err| / A would then not grow with depth.  On the B200 it does grow, like sqrt(K_tot):
|err| / A = 6 u at K_tot = 1152, 9 u at 2880, 16 u at 11520 (fp32 output, no split-K).  That is what adds whose errors share a
sign give: the error is ~ u * sum_k |partial sum_k|, partial sums of a random-sign contraction grow like sqrt(k) rms(x w), and
A = sum |x w| like K_tot E|x w|, so |err| / A ~ c u sqrt(K_tot) with a measured c of about 0.15.  tau takes c = 1: within
about 8x of the measured maximum over every case here (a run prints the margin), and far below what one dropped 64-wide
k-block (~8 / (0.64 K_tot) >= 4e-4) or a wrong embedding row produces.

Out of scope: MKD_DUAL=1 (variants 10 / 11) and MKD_CLUSTER=2 (the CL = 2 single-CTA kernel) — opt-in experiments, read once
per process and absent from the shipped library's code path; the generic kernel; weight groups (mkd_conv_desc.wgroups: the
same pair instantiations, compared with two single-group launches in test_kernels_gpu).
"""
import math
import re
import zlib

import pytest
import torch
import torch.nn.functional as F

from makeupdiffuse_b200 import _lib as L
from makeupdiffuse_b200 import ops
from test_kernels_gpu import GN_TAIL_CASES, PAIR_CASES, PAIR_STATS_CASES

U = 2.0 ** -24
TAU_STATS = 2.0 ** -17           # fp32 sum of <= 128 values in any order: |err| <= 127 u sum |v|
GELU_APPROX = 0.75e-7 + 2.0 ** -22  # common.cuh: erf by A-S 7.1.26 (0.75e-7 |x| on gelu) + rcp / ex2.approx and fp32 steps
BF16_REL = 2.0 ** -8             # bf16 unit roundoff: 8 significant bits
WS_BYTES = 64 << 20
NAN = float("nan")

MEASURED = {"err_over_A": (0.0, ""), "c": (0.0, ""), "gelu_coef": (0.0, "")}  # worst |y32 - ref| / A, the same / (u sqrt(K_tot)),
#                                                                            worst GELU approximation error implied per |a| |g|


def tau(s):
    """per-element accumulation bound relative to A (module docstring)"""
    return U * math.sqrt(s["R"] * s["R"] * s["C"] + s["C2"])


# ---- float64 reference ----------------------------------------------------------------------------------------------------
def spec_of(**s):
    """a case: conv geometry + operand set.  res: None / "bf16" / "f32"; inplace: the residual is the output of its dtype"""
    d = dict(N=1, H=1, W=1, C=64, K=64, R=1, stride=1, pad=None, pad_hi_extra=0, up=False, bias=True, spread=0.0, emb=False,
             res=None, inplace=False, alpha=1.0, act="none", gb=80, y=True, y32=False, stats=False, ws=False, C2=0, tight=False,
             gn=None, exact=False)
    d.update(s)
    if d["pad"] is None:
        d["pad"] = d["R"] // 2
    return d


def out_geometry(s):
    Hi, Wi = (2 * s["H"], 2 * s["W"]) if s["up"] else (s["H"], s["W"])
    P = (Hi + 2 * s["pad"] + s["pad_hi_extra"] - s["R"]) // s["stride"] + 1
    Q = (Wi + 2 * s["pad"] + s["pad_hi_extra"] - s["R"]) // s["stride"] + 1
    return P, Q, s["N"] * P * Q


def reference(s, x, w, bias, emb, res, x2):
    """float64: ref [Mo, Ko] and its per-element bounds (b32 for fp32 outputs, b16 for bf16 outputs); pre / A for statistics"""
    N, H, W, C, K, R = (s[k] for k in "NHWCKR")
    P, Q, Mo = out_geometry(s)
    xr = x.double().reshape(N, H, W, C).permute(0, 3, 1, 2)
    if s["up"]:
        xr = xr.repeat_interleave(2, 2).repeat_interleave(2, 3)
    pad = s["pad"]
    if s["pad_hi_extra"]:
        xr = F.pad(xr, (0, s["pad_hi_extra"], 0, s["pad_hi_extra"]))
    wr = w[:, :R * R * C].double().reshape(K, R, R, C).permute(0, 3, 1, 2)
    acc = F.conv2d(xr, wr, stride=s["stride"], padding=pad).permute(0, 2, 3, 1).reshape(Mo, K)
    mag = F.conv2d(xr.abs(), wr.abs(), stride=s["stride"], padding=pad).permute(0, 2, 3, 1).reshape(Mo, K)
    if x2 is not None:
        w2 = w[:, R * R * C:].double()
        acc = acc + x2.double() @ w2.t()
        mag = mag + x2.double().abs() @ w2.abs().t()
    b = bias.double() if bias is not None else torch.zeros(K, dtype=torch.float64, device=acc.device)
    t = 0.0 if s["exact"] else tau(s)  # exact operands: every partial sum is representable, the accumulation is exact
    if s["act"] == "geglu":
        gb, Ko = s["gb"], K // 2
        j = torch.arange(Ko, device=acc.device)
        vrow = (j // gb) * 2 * gb + j % gb
        grow = vrow + gb
        a, g = acc[:, vrow] + b[vrow], acc[:, grow] + b[grow]
        Aa, Ag = mag[:, vrow] + b[vrow].abs(), mag[:, grow] + b[grow].abs()
        ga = F.gelu(g)
        ref = a * ga
        ea, eg = t * Aa, t * Ag
        op = ga.abs() * ea + 1.13 * (a.abs() + ea) * eg              # the operands' own errors, through the product
        b16 = BF16_REL * ref.abs() + (1 + BF16_REL) * (op + (a.abs() + ea) * GELU_APPROX * (g.abs() + eg))
        return dict(ref=ref, b32=None, b16=b16, geglu=(a, g, ea, eg, op))
    pre = acc + b
    A = mag + b.abs()
    if emb is not None:
        e = emb.double()[torch.arange(Mo, device=acc.device) // (P * Q)]
        pre, A = pre + e, A + e.abs()
    pre, A = s["alpha"] * pre, abs(s["alpha"]) * A
    if res is not None:
        pre, A = pre + res.double(), A + res.double().abs()
    if s["act"] == "silu":
        ref = F.silu(pre)
        # __expf: 2 + 1.17 |x| ulp, __fdividef: 2 ulp, the 1 + e rounding: 1/2 ulp (CUDA C Programming Guide, intrinsics)
        b32 = 1.1 * t * A + (5.0 + 1.2 * pre.abs()) * 2.0 ** -23 * ref.abs()
    else:
        ref, b32 = pre, t * A
    return dict(ref=ref, b32=b32, b16=BF16_REL * ref.abs() + (1 + BF16_REL) * b32, A=A, pre=pre)


def tile_sums(v, T):
    """[Mo, K] float64 -> per 128-row tile column sums [T, K] (rows beyond Mo count as absent)"""
    Mo, K = v.shape
    z = torch.zeros(T * 128, K, dtype=v.dtype, device=v.device)
    z[:Mo] = v
    return z.reshape(T, 128, K).sum(1)


# ---- the checker ----------------------------------------------------------------------------------------------------------
def _worst(err, bound):
    r = err / bound.clamp_min(1e-300)
    i = int(torch.argmax(r))
    return float(r.reshape(-1)[i]), divmod(i, err.shape[1]) if err.dim() == 2 else i


def _bits(t):
    return t.view({2: torch.int16, 4: torch.int32}[t.element_size()])


def check_guards(guards):
    """guards: (buffer now, snapshot before the call, index of the region the call may write or None)"""
    for name, buf, snap, inside in guards:
        cur = buf.clone()
        if inside is not None:
            cur[inside] = snap[inside]
        if not torch.equal(_bits(cur), _bits(snap)):
            bad = (_bits(cur) != _bits(snap)).nonzero()
            raise AssertionError(f"{name}: {bad.shape[0]} guard / input element(s) changed, first at {bad[0].tolist()}")


def gn_reference(s, v, gamma, beta, eps, silu, groups=32):
    """float64 GroupNorm(+SiLU) of the stored layer output v [Mo, K] over (pixels of an image, channels of a group), and its
    bound: bf16 rounding + 2^-14 (1 + |xhat|) |gamma| for the fp32 statistics (E[x^2] - mean^2) of the reducer"""
    Mo, K = v.shape
    t = v.reshape(s["N"], Mo // s["N"], groups, K // groups)
    mean, var = t.mean((1, 3), keepdim=True), t.var((1, 3), unbiased=False, keepdim=True)
    xhat = ((t - mean) / (var + eps).sqrt()).reshape(Mo, K)
    r = xhat * gamma.double() + beta.double()
    e = 2.0 ** -14 * gamma.double().abs() * (1 + xhat.abs())
    if silu:
        r, e = F.silu(r), 1.1 * e
    return r, BF16_REL * r.abs() + (1 + BF16_REL) * e


def check_outputs(label, s, refd, y=None, y32=None, stats=None, guards=(), gn=None):
    """raises AssertionError on any element outside its bound; returns {output: worst err / bound}"""
    ref = refd["ref"]
    worst = {}
    check_guards(guards)
    if y32 is not None:
        got = y32.double()
        assert bool(torch.isfinite(got).all()), f"{label}: y32 holds {int((~torch.isfinite(got)).sum())} non-finite values"
        err = (got - ref).abs()
        worst["y32"], at = _worst(err, refd["b32"])
        assert worst["y32"] <= 1.0, (f"{label}: y32[{at}] = {float(got[at]):.9g}, reference {float(ref[at]):.9g}, |err| / bound "
                                     f"{worst['y32']:.3g}")
        if s["act"] == "none":
            r, at = _worst(err, refd["A"])
            if r > MEASURED["err_over_A"][0]:
                MEASURED["err_over_A"] = (r, label)
            if r / tau(s) > MEASURED["c"][0]:
                MEASURED["c"] = (r / tau(s), label)
    if y is not None:
        got = y.double()
        assert bool(torch.isfinite(got).all()), f"{label}: y holds {int((~torch.isfinite(got)).sum())} non-finite values"
        if y32 is not None:
            same = y == y32.to(torch.bfloat16)
            assert bool(same.all()), f"{label}: y != bf16(y32) at {(~same).nonzero()[0].tolist()}"
        else:
            err = (got - ref).abs()
            worst["y"], at = _worst(err, refd["b16"])
            assert worst["y"] <= 1.0, (f"{label}: y[{at}] = {float(got[at]):.6g}, reference {float(ref[at]):.6g}, |err| / bound "
                                       f"{worst['y']:.3g}")
            if "geglu" in refd:  # the GELU approximation error this output implies (what rounding and operands cannot explain)
                a, g, ea, eg, op = refd["geglu"]
                excess = (err - BF16_REL * (ref.abs() + op) - op) / (1 + BF16_REL)
                coef = float((excess / ((a.abs() + ea) * (g.abs() + eg)).clamp_min(1e-30)).max())
                if coef > MEASURED["gelu_coef"][0]:
                    MEASURED["gelu_coef"] = (coef, label)
    if stats is not None:
        Mo, K = ref.shape
        T = stats.shape[0]
        st = stats.double()
        assert bool(torch.isfinite(st).all()), f"{label}: statistics hold non-finite values"
        if y32 is not None:  # the sums of exactly the values stored
            v = y32.double()
            S, Sa, SS = tile_sums(v, T), tile_sums(v.abs(), T), tile_sums(v * v, T)
            bs, bq = TAU_STATS * Sa, TAU_STATS * SS
        else:                # only the bf16 copy was stored: the sums of the fp32 values, each within b32 of the reference
            v, e = ref, refd["b32"]
            S, Sa, SS = tile_sums(v, T), tile_sums(v.abs(), T), tile_sums(v * v, T)
            bs = TAU_STATS * Sa + tile_sums(e, T)
            bq = TAU_STATS * SS + tile_sums(2 * v.abs() * e + e * e, T)
        for i, (name, want, bound) in enumerate((("sum", S, bs), ("sum of squares", SS, bq))):
            worst["stats" if i == 0 else "sumsq"], at = _worst((st[..., i] - want).abs(), bound)
            w_ = worst["stats" if i == 0 else "sumsq"]
            assert w_ <= 1.0, (f"{label}: statistics {name} of (tile, channel) {at} = {float(st[..., i][at]):.9g}, expected "
                               f"{float(want[at]):.9g}, |err| / bound {w_:.3g}")
    if gn is not None:
        out, gamma, beta, eps, silu = gn
        r, bound = gn_reference(s, y32.double(), gamma, beta, eps, silu)
        got = out.double()
        assert bool(torch.isfinite(got).all()), f"{label}: GroupNorm tail holds non-finite values"
        worst["gn"], at = _worst((got - r).abs(), bound)
        assert worst["gn"] <= 1.0, (f"{label}: GroupNorm tail [{at}] = {float(got[at]):.6g}, reference {float(r[at]):.6g}, "
                                    f"|err| / bound {worst['gn']:.3g}")
    return worst


# ---- buffers ----------------------------------------------------------------------------------------------------------------
def guarded(rows, cols, dtype, device, tight=False, extra_rows=3):
    """NaN-filled buffer holding a [rows, cols] view: 8 guard columns on each side (ld a multiple of 8) unless tight"""
    off = 0 if tight else 8
    ld = off + cols + (0 if tight else 8 + (-(off + cols)) % 8)
    if tight and ld % 8:
        ld += (-ld) % 8
    buf = torch.full((rows + extra_rows, ld), NAN, dtype=dtype, device=device)
    return buf, buf[:rows, off:off + cols], (slice(0, rows), slice(off, off + cols))


def make_operands(s, device, seed):
    """every operand of a case, each view in a NaN-guarded buffer (bufs: name -> (buffer, the region its view covers));
    kw: the keywords of ops.conv2d"""
    g = torch.Generator(device=device).manual_seed(seed)
    rnd = lambda *shape, scale=1.0: torch.randn(*shape, device=device, generator=g) * scale  # noqa: E731
    N, H, W, C, K, R = (s[k] for k in "NHWCKR")
    P, Q, Mo = out_geometry(s)
    Ko = K // 2 if s["act"] == "geglu" else K
    BF, F32 = torch.bfloat16, torch.float32
    bufs = {}

    def put(name, rows, cols, dtype, fill, tight=None):
        buf, view, inside = guarded(rows, cols, dtype, device, tight=s["tight"] if tight is None else tight)
        if fill is not None:
            view.copy_(fill)
        bufs[name] = (buf, inside)
        return view
    fan = R * R * C + s["C2"]
    ints = lambda lo, hi, *shape: torch.randint(lo, hi + 1, shape, device=device, generator=g).float()  # noqa: E731
    if s["exact"]:  # x in {-2..2}, w in 2^-7 {-8..8}, bias in 2^-7 {-1024..1024}: every partial sum is k 2^-7, |k| < 2^24
        assert not s["C2"] and not s["emb"] and s["res"] is None and 2 * 8 * fan + 1024 < 2 ** 24
        x = put("x", N * H * W, C, BF, ints(-2, 2, N * H * W, C))
        w = (ints(-8, 8, K, fan) / 128).to(BF)
    else:
        x = put("x", N * H * W, C, BF, rnd(N * H * W, C))
        w = (rnd(K, fan) / math.sqrt(fan)).to(BF)
    x2 = put("x2", N * H * W, s["C2"], BF, rnd(N * H * W, s["C2"])) if s["C2"] else None
    if not s["bias"]:
        bias = None
    elif s["exact"]:
        bias = ints(-1024, 1024, K) / 128
    elif s["spread"]:  # pre-activations spread over about +-spread: the tails of silu_f / gelu_erf_fast
        bias = (torch.rand(K, device=device, generator=g) * 2 - 1) * s["spread"]
    else:
        bias = 0.5 * rnd(K)
    emb = put("emb", N, K, BF, rnd(N, K), tight=False) if s["emb"] else None
    y = put("y", Mo, Ko, BF, rnd(Mo, Ko) if (s["inplace"] and s["res"] == "bf16") else None) if s["y"] else None
    y32 = put("y32", Mo, Ko, F32, rnd(Mo, Ko) if (s["inplace"] and s["res"] == "f32") else None) if s["y32"] else None
    if s["res"] is None:
        res = None
    elif s["inplace"]:
        res = y if s["res"] == "bf16" else y32
        assert res is not None, "an in-place residual needs the output of its dtype"
    else:
        res = put("res", Mo, Ko, BF if s["res"] == "bf16" else F32, rnd(Mo, Ko))
    stats = None
    if s["stats"]:
        T = (Mo + 127) // 128
        off = 0 if s["tight"] else 8
        ld = off + K + (0 if s["tight"] else 8)
        sb = torch.full((T + 2, ld, 2), NAN, device=device)
        stats = sb[:T, off:off + K, :]
        bufs["stats"] = (sb, (slice(0, T), slice(off, off + K), slice(None)))
    gn = None
    if s["gn"]:  # GroupNorm tail of the split-K reducer (mkd_conv_desc.gn_y)
        gamma, beta = 1.0 + 0.3 * rnd(K), 0.2 * rnd(K)
        gn = dict(y=put("gn", Mo, K, BF, None), gamma=gamma, beta=beta, eps=s["gn"]["eps"], silu=s["gn"]["silu"])
    kw = dict(gn=gn) if gn else {}
    kw.update(N=N, H=H, W=W, R=R, S=R, stride=s["stride"], pad=s["pad"], pad_hi_extra=s["pad_hi_extra"], upsample=s["up"],
              bias=bias, emb=emb, residual=res, alpha=s["alpha"], act={"none": L.ACT_NONE, "silu": L.ACT_SILU, "geglu": L.ACT_GEGLU}[s["act"]],
              geglu_block=s["gb"] if s["act"] == "geglu" else 0, y32=y32, stats=stats, x2=x2,
              workspace=torch.empty(WS_BYTES, dtype=torch.uint8, device=device) if s["ws"] else None)
    return dict(x=x, w=w, y=y, kw=kw, bias=bias, emb=emb, res=res, x2=x2, y32=y32, stats=stats, gn=gn, bufs=bufs)


# ---- kernel names ---------------------------------------------------------------------------------------------------------
FAMILY = ("gemm_tcgen05_kernel", "gemm_pair_kernel", "splitk_epilogue_kernel", "splitk_gn_kernel", "im2col_s2_kernel",
          "upsample2x_kernel")
_FAM = re.compile(r"(?<![A-Za-z_])(\d*)(" + "|".join(FAMILY) + r")(<[^>]*>|I(?:Li-?\d+E)+E)?")


def canonical(name):
    """'void (anonymous namespace)::gemm_tcgen05_kernel<160, 1, 4, 10, 0>(...)' (or its mangled form) ->
    'gemm_tcgen05_kernel<160,1,4,10,0>'; None for kernels outside the conv / GEMM family"""
    m = _FAM.search(name)
    if not m:
        return None
    args = m.group(3)
    if not args:
        return m.group(2)
    if args.startswith("I"):
        vals = re.findall(r"Li(-?\d+)E", args)
    else:
        vals = [re.sub(r"^\((?:int|unsigned)\)|[uUlL]+$", "", a.strip()) for a in args[1:-1].split(",")]
    return f"{m.group(2)}<{','.join(vals)}>"


def launched_kernels(fn):
    """run fn under torch.profiler; every CUDA kernel name it launched, canonical ones for the GEMM family"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    return names


def tc(bn, epi, spec=0):
    """gemm_tcgen05_kernel<BN, CL = 1, EPI, SPEC, DUAL = 0>; EPI: 0 plain, 1 SiLU, 2 GEGLU, 3 split-K partials, 4 statistics"""
    return f"gemm_tcgen05_kernel<{bn},1,{epi},{spec},0>"


def splitk(bn):
    return f"splitk_epilogue_kernel<{bn}>"


IM2COL, UPSAMPLE = "im2col_s2_kernel", "upsample2x_kernel"


# ---- the single-CTA kernel: one case per instantiation ----------------------------------------------------------------------
# gemm_tcgen05.cu: pick_bn() chooses the N tile, launch<BN, 1>() the epilogue variant (index into `all`):
#   0 plain, 1 SiLU, 2 GEGLU (BN = 160; EPI_PLAIN elsewhere, never picked: GEGLU always takes 160), 3 split-K partials,
#   4 statistics — run-time operand dispatch; at BN = 160 only, compile-time operand sets (SPEC bits: 1 fp32 residual,
#   2 y32, 4 y, 8 embedding): 5 plain y32 | 6 plain res32 + y32 | 7 plain y | 8 plain res32 + y | 9 stats res32 + y32 + y |
#   12 stats emb + y32 | 13 stats res32 + y32 | 14 stats res32 + y.  (10 / 11: MKD_DUAL only.)  At other N tiles variants
#   5-9 / 12-14 are the SPEC = 0 kernels of 0 / 4.
# Reachable with the default switches, and NOT reachable:
#   BN 160: variants 0-9, 12-14.                 BN 80, 64, 32: plain, SiLU, split-K, statistics.
#   BN 256: plain, SiLU, statistics (>= 148 tiles), split-K only through the wide rule (K % 1280 == 0, >= 4 row tiles,
#           <= 74 tiles of 160, >= 64 k-blocks, workspace, no statistics, act NONE).
#   BN 128: plain, SiLU, statistics.  NOT split-K: BN 128 (and 256 outside the wide rule) needs >= 148 tiles, split-K <= 74.
#   GEGLU at any BN but 160: never (pick_bn returns 160 for GEGLU).  Statistics never split (the reducer emits none).
#   Ragged channel tails (K < 16, scalar epilogue) only at BN 32, never with statistics (K % 8 == 0).
SINGLE_CASES = {
    # ---- BN = 160 -------------------------------------------------------------------------------------------------------
    "160/v0 in-place bf16 residual, alpha 0.5, ragged M": (
        dict(N=1, H=1, W=200, C=640, K=640, res="bf16", inplace=True, alpha=0.5), [tc(160, 0)]),
    "160/v1 SiLU, pre-activations +-8, tiny M": (
        dict(N=1, H=1, W=16, C=1280, K=1280, act="silu", spread=8.0), [tc(160, 1)]),
    "160/v2 GEGLU [80 | 80] blocks, gate +-8, ragged M": (
        dict(N=1, H=1, W=300, C=320, K=2560, act="geglu", gb=80, spread=8.0), [tc(160, 2)]),
    "160/v2 GEGLU, exact operands: gelu_erf_fast's error alone": (
        dict(N=1, H=1, W=1024, C=320, K=2560, act="geglu", gb=80, exact=True), [tc(160, 2)]),
    "160/v1 SiLU, exact operands, fp32 out: silu_f's error alone": (
        dict(N=1, H=1, W=1024, C=320, K=320, act="silu", exact=True, y32=True), [tc(160, 1)]),
    "160/v3 split-K 4x4, box spans 8 images, embedding": (
        dict(N=16, H=4, W=4, C=2560, K=1280, R=3, emb=True, ws=True), [tc(160, 3), splitk(160)]),
    "160/v3 split-K GEGLU (reducer GEGLU epilogue)": (
        dict(N=1, H=1, W=100, C=2048, K=2560, act="geglu", gb=80, spread=8.0, ws=True), [tc(160, 3), splitk(160)]),
    "160/v3 Downsample p1 via im2col + split-K": (
        dict(N=2, H=32, W=32, C=320, K=320, R=3, stride=2, ws=True, y32=True), [IM2COL, tc(160, 3), splitk(160)]),
    "160/v4 statistics, in-place bf16 residual, ragged M": (
        dict(N=1, H=1, W=200, C=320, K=320, res="bf16", inplace=True, alpha=0.5, y32=True, stats=True), [tc(160, 4)]),
    "160/v5 y32 only, ragged M": (
        dict(N=1, H=1, W=1000, C=320, K=960, bias=False, y=False, y32=True), [tc(160, 0, 2)]),
    "160/v6 fp32 residual in place, y32 only": (
        dict(N=1, H=1, W=300, C=320, K=320, res="f32", inplace=True, y=False, y32=True), [tc(160, 0, 3)]),
    "160/v7 y only, input slice": (
        dict(N=1, H=1, W=231, C=768, K=640, bias=False), [tc(160, 0, 4)]),
    "160/v8 fp32 residual -> bf16": (
        dict(N=1, H=1, W=300, C=1280, K=320, res="f32"), [tc(160, 0, 5)]),
    "160/v9 statistics + res32 + y32 + y, 8x8, box spans 2 images, ragged N": (
        dict(N=3, H=8, W=8, C=1280, K=1280, R=3, res="f32", y32=True, stats=True), [tc(160, 4, 7)]),
    "160/v12 statistics + embedding + y32 (ResBlock conv1, batch 2)": (
        dict(N=2, H=32, W=32, C=320, K=320, R=3, emb=True, y=False, y32=True, stats=True, tight=True), [tc(160, 4, 10)]),
    "160/v13 statistics + res32 + y32 (ResBlock conv2, batch 1)": (
        dict(N=1, H=32, W=32, C=320, K=320, R=3, res="f32", y=False, y32=True, stats=True, tight=True), [tc(160, 4, 3)]),
    "160/v14 statistics + res32 + y (proj_out)": (
        dict(N=4, H=16, W=16, C=640, K=640, res="f32", stats=True), [tc(160, 4, 5)]),
    # ---- BN = 256 -------------------------------------------------------------------------------------------------------
    "256 plain, ragged M": (dict(N=1, H=1, W=19000, C=64, K=512), [tc(256, 0)]),
    "256 SiLU +-8": (dict(N=1, H=1, W=19000, C=64, K=256, act="silu", spread=8.0), [tc(256, 1)]),
    "256 statistics, 128x128, res32 + y32 + y": (
        dict(N=2, H=128, W=128, C=256, K=256, R=3, res="f32", y32=True, stats=True), [tc(256, 4)]),
    "256 wide split-K, 8x8 at batch 8, embedding (2 images per box)": (
        dict(N=8, H=8, W=8, C=1280, K=1280, R=3, emb=True, y=False, y32=True, ws=True), [tc(256, 3), splitk(256)]),
    "256 wide split-K, Upsample 8 -> 16": (
        dict(N=2, H=8, W=8, C=1280, K=1280, R=3, up=True, ws=True), [UPSAMPLE, tc(256, 3), splitk(256)]),
    # ---- BN = 128 -------------------------------------------------------------------------------------------------------
    "128 plain, ragged M": (dict(N=1, H=1, W=19000, C=64, K=128), [tc(128, 0)]),
    "128 SiLU +-8": (dict(N=1, H=1, W=19000, C=128, K=128, act="silu", spread=8.0), [tc(128, 1)]),
    "128 statistics, 128x256 (box = half a row)": (
        dict(N=1, H=128, W=256, C=128, K=128, R=3, y32=True, stats=True), [tc(128, 4)]),
    # ---- BN = 80 --------------------------------------------------------------------------------------------------------
    "80 plain": (dict(N=1, H=1, W=500, C=128, K=240), [tc(80, 0)]),
    "80 SiLU +-8, 3x3": (dict(N=2, H=16, W=16, C=64, K=80, R=3, act="silu", spread=8.0), [tc(80, 1)]),
    "80 statistics + embedding": (dict(N=2, H=16, W=16, C=128, K=400, R=3, emb=True, y32=True, stats=True), [tc(80, 4)]),
    "80 split-K, bf16 residual, alpha 0.7": (
        dict(N=1, H=1, W=256, C=2048, K=240, res="bf16", alpha=0.7, ws=True), [tc(80, 3), splitk(80)]),
    # ---- BN = 64 --------------------------------------------------------------------------------------------------------
    "64 plain, ragged N tile (K = 96)": (dict(N=1, H=1, W=300, C=64, K=96), [tc(64, 0)]),
    "64 SiLU +-8, 3x3": (dict(N=2, H=32, W=32, C=64, K=64, R=3, act="silu", spread=8.0), [tc(64, 1)]),
    "64 statistics, 64x64": (dict(N=4, H=64, W=64, C=256, K=128, R=3, y32=True, stats=True), [tc(64, 4)]),
    "64 VAE Downsample p0 + far edge, split-K": (
        dict(N=1, H=64, W=64, C=512, K=512, R=3, stride=2, pad=0, pad_hi_extra=1, ws=True), [IM2COL, tc(64, 3), splitk(64)]),
    "64 VAE Downsample p0 + far edge, 256 -> 128": (
        dict(N=1, H=256, W=256, C=128, K=128, R=3, stride=2, pad=0, pad_hi_extra=1, ws=True), [IM2COL, tc(64, 0)]),
    "64 Downsample p1 + SiLU (hint)": (
        dict(N=2, H=64, W=64, C=64, K=128, R=3, stride=2, act="silu", spread=8.0, ws=True), [IM2COL, tc(64, 1)]),
    "64 VAE Upsample 32 -> 64": (dict(N=1, H=32, W=32, C=512, K=512, R=3, up=True, ws=True), [UPSAMPLE, tc(64, 0)]),
    # ---- BN = 32 (ragged channel counts: scalar tail) ------------------------------------------------------------------
    "32 K = 3 (VAE conv_out) + emb + res32 + y32 + y": (
        dict(N=1, H=64, W=64, C=128, K=3, R=3, emb=True, res="f32", y32=True), [tc(32, 0)]),
    "32 K = 4 (UNet out) SiLU +-8 + emb + bf16 residual, alpha 0.7": (
        dict(N=2, H=32, W=32, C=320, K=4, R=3, emb=True, res="bf16", alpha=0.7, act="silu", spread=8.0), [tc(32, 1)]),
    "32 K = 8 (VAE moments) fp32 only": (dict(N=2, H=32, W=32, C=512, K=8, R=3, y=False, y32=True), [tc(32, 0)]),
    "32 statistics, K = 16": (dict(N=2, H=16, W=16, C=64, K=16, R=3, y32=True, stats=True), [tc(32, 4)]),
    "32 split-K + embedding": (dict(N=2, H=1, W=128, C=2048, K=32, emb=True, ws=True), [tc(32, 3), splitk(32)]),
}


# ---- the CTA-pair kernel: the existing case lists, with the instantiation gemm_pair.cu's plan() picks ------------------------
def from_conv_case(c):
    """test_kernels_gpu.conv_case keywords -> a case here"""
    res = None
    if c.get("residual") or c.get("inplace"):
        res = "f32" if c.get("res32") else "bf16"
    act = {L.ACT_NONE: "none", L.ACT_SILU: "silu", L.ACT_GEGLU: "geglu"}[c.get("act", L.ACT_NONE)]
    y32 = c.get("y32", "")
    return spec_of(N=c["N"], H=c["H"], W=c["W"], C=c["C"], K=c["K"], R=c.get("R", 1), stride=c.get("stride", 1),
                   up=c.get("upsample", False), bias=c.get("bias", True), emb=c.get("emb", False), res=res,
                   inplace=c.get("inplace", False), alpha=c.get("alpha", 1.0), act=act, gb=c.get("gb") or 80,
                   y=y32 != "only", y32=bool(y32), ws=c.get("workspace", False), C2=c.get("C2", 0))


def from_stats_case(c):
    """test_kernels_gpu.test_conv_stats_and_groupnorm_apply keywords -> a case here"""
    res = "bf16" if c.get("inplace") else ("f32" if c.get("residual") else None)
    return spec_of(N=c["N"], H=c["H"], W=c["W"], C=c["C"], K=c["K"], R=c["R"], stride=c.get("stride", 1), up=c.get("up", False),
                   emb=c.get("emb", False), res=res, inplace=c.get("inplace", False), alpha=0.5 if c.get("inplace") else 1.0,
                   y=True, y32=True, stats=True, ws=True, C2=c.get("C2", 0))


def from_gn_case(c):
    """test_kernels_gpu.test_conv_groupnorm_tail keywords -> a case here (3x3, bias, workspace, GroupNorm(+SiLU) tail)"""
    return spec_of(N=c["N"], H=c["H"], W=c["W"], C=c["C"], K=c["K"], R=3, emb=c.get("emb", False), C2=c.get("C2", 0),
                   y=c["y32"] == "both", y32=True, ws=True, gn=dict(silu=c.get("silu", True), eps=c.get("eps", 1e-5)))


def pair_kernels(s):
    """gemm_pair.cu plan() restated: gemm_pair_kernel<UN, NSUB, MODE, STATS> (+ the split-K reducer) of a forced pair launch"""
    N, H, W, C, K, R = (s[k] for k in "NHWCKR")
    P, Q = H // s["stride"], W // s["stride"]
    M = N * P * Q
    kb = (R * R * C + s["C2"]) // 64
    if R == 3:
        Wb = min(Q, 128)
        Hb = min(128 // Wb, P)
        Nb = 128 // (Wb * Hb)
        mt = (Q // Wb) * (P // Hb) * -(-N // Nb)
    else:
        mt = -(-M // 128)
    if s["act"] == "geglu":
        return ["gemm_pair_kernel<256,1,1,0>"]
    mp = (mt + 1) // 2
    u1, u2 = mp * (K // 160), (mp * (K // 320) if K % 320 == 0 else 0)
    can_split = s["ws"] and not s["stats"] and kb >= 32
    nsub = 2 if (u2 >= 48 and kb >= 16) or (u2 > 0 and 16 <= u1 < 37 and can_split and kb >= 64) else 1
    units = u2 if nsub == 2 else u1
    splits = 1
    if units < 37 and can_split:
        sp = min(74 // units, kb // 12, 16)
        while sp > 1 and sp * M * K * 4 > WS_BYTES:
            sp -= 1
        splits = max(sp, 1)
    if splits > 1:
        kps = -(-kb // splits)
        splits = -(-kb // kps)
    reducer = "splitk_gn_kernel" if s["gn"] else splitk(160)
    return [f"gemm_pair_kernel<160,{nsub},0,{int(bool(s['stats']))}>"] + ([reducer] if splits > 1 else [])


PAIR_ALL = {f"pair {i}": (from_conv_case(c), None) for i, c in enumerate(PAIR_CASES)}
PAIR_ALL.update({f"pair-stats {i}": (from_stats_case(c), None) for i, c in enumerate(PAIR_STATS_CASES)})
PAIR_ALL["pair GEGLU [128 | 128], exact operands: gelu_erf_fast2's error alone"] = (
    spec_of(N=1, H=1, W=1024, C=320, K=2560, act="geglu", gb=128, exact=True), None)
PAIR_ALL.update({f"pair-gn-tail {i}": (from_gn_case(c), None) for i, c in enumerate(GN_TAIL_CASES)
                 if not c.get("declined") and c.get("wgroups", 1) == 1})
PAIR_ALL = {k: (s, pair_kernels(s)) for k, (s, _) in PAIR_ALL.items()}

# every conv / GEMM-family kernel some case here launches: production must launch nothing else (test_production_census)
EXPECTED = frozenset(n for _, names in list(SINGLE_CASES.values()) + list(PAIR_ALL.values()) for n in names)


# ---- running a case on the GPU ----------------------------------------------------------------------------------------------
def run_case(label, s, path, want):
    dev = "cuda"
    s = spec_of(**s)
    ops_ = make_operands(s, dev, zlib.crc32(label.encode()))
    x, w, y, kw = ops_["x"], ops_["w"], ops_["y"], ops_["kw"]
    kw["path"] = path
    assert ops.conv2d_path(x, w, y, **kw) == L.PATH_TCGEN05, label
    guards_before = {k: b.clone() for k, (b, _) in ops_["bufs"].items()}
    refd = reference(s, x, w, ops_["bias"], ops_["emb"], ops_["res"], ops_["x2"])
    inplace_view = ops_["res"] if s["inplace"] else None
    inplace_before = None if inplace_view is None else inplace_view.clone()
    names = launched_kernels(lambda: ops.conv2d(x, w, y, **kw))
    got = sorted({c for c in map(canonical, names) if c})
    assert got == sorted(set(want)), f"{label}: launched {got}, expected {sorted(set(want))} (all kernels: {names})"
    writable = {"y", "y32", "stats", "gn"}
    guards = [(k, b, guards_before[k], inside if k in writable else None) for k, (b, inside) in ops_["bufs"].items()]
    gn = ops_["gn"]
    worst = check_outputs(label, s, refd, y=y, y32=ops_["y32"], stats=ops_["stats"], guards=guards,
                          gn=None if gn is None else (gn["y"], gn["gamma"], gn["beta"], gn["eps"], gn["silu"]))
    # a second identical launch writes bit-identical outputs (split-K reducers sum in a fixed order)
    outs = (y, ops_["y32"], ops_["stats"], None if gn is None else gn["y"])
    first = [None if t is None else t.clone() for t in outs]
    if inplace_view is not None:
        inplace_view.copy_(inplace_before)
    ops.conv2d(x, w, y, **kw)
    torch.cuda.synchronize()
    for name, a, b in zip(("y", "y32", "stats", "GroupNorm tail"), first, outs):
        if a is not None:
            assert torch.equal(_bits(a), _bits(b)), f"{label}: second launch differs in {name}"
    print(f"{label:<72s} worst err/bound " + "  ".join(f"{k} {v:.3f}" for k, v in worst.items()) + f"   [{' '.join(got)}]")
    return worst


@pytest.fixture(scope="module", autouse=True)
def _report_margins():
    yield
    if MEASURED["err_over_A"][0] > 0:
        r, where = MEASURED["err_over_A"]
        c, where_c = MEASURED["c"]
        print(f"\nmeasured max |y32 - ref| / A = {r:.3e} = {r / U:.1f} u (at {where}); max |y32 - ref| / (A u sqrt(K_tot)) = "
              f"{c:.3f} (at {where_c}): tau = u sqrt(K_tot) has a margin of {1 / c:.1f}x")
    if MEASURED["gelu_coef"][0] > 0:
        c, where = MEASURED["gelu_coef"]
        print(f"implied GELU approximation error <= {c:.3e} |a| |g| (at {where}); bound GELU_APPROX = {GELU_APPROX:.3e}")


@pytest.mark.gpu
@pytest.mark.parametrize("label", list(SINGLE_CASES))
def test_single_cta_instantiation(label):
    s, want = SINGLE_CASES[label]
    run_case(label, s, L.PATH_TCGEN05_SINGLE, want)


@pytest.mark.gpu
@pytest.mark.parametrize("label", list(PAIR_ALL))
def test_pair_elementwise(label):
    s, want = PAIR_ALL[label]
    run_case(label, s, L.PATH_TCGEN05_PAIR, want)


def test_every_reachable_single_cta_instantiation_has_a_case():
    """the table above names every single-CTA instantiation reachable with the default switches"""
    names = {n for _, want in SINGLE_CASES.values() for n in want}
    reachable = {tc(160, e) for e in range(5)} | {tc(160, 0, sp) for sp in (2, 3, 4, 5)} | {tc(160, 4, sp) for sp in (7, 10, 3, 5)}
    reachable |= {tc(bn, e) for bn in (80, 64, 32) for e in (0, 1, 3, 4)} | {tc(256, e) for e in (0, 1, 3, 4)}
    reachable |= {tc(128, e) for e in (0, 1, 4)}
    assert {n for n in names if n.startswith("gemm_tcgen05_kernel")} == reachable
    assert {splitk(bn) for bn in (256, 160, 80, 64, 32)} <= names and {IM2COL, UPSAMPLE} <= names


def test_kernel_name_canonical_form():
    assert canonical("void (anonymous namespace)::gemm_tcgen05_kernel<160, 1, 4, 10, 0>(CUtensorMap_st, CUtensorMap_st, "
                     "(anonymous namespace)::MainP, (anonymous namespace)::EpiP)") == "gemm_tcgen05_kernel<160,1,4,10,0>"
    assert canonical("_ZN12_GLOBAL__N_119gemm_tcgen05_kernelILi256ELi1ELi3ELi0ELi0EEEv14CUtensorMap_stS1_NS_5MainPENS_4EpiPE") == \
        "gemm_tcgen05_kernel<256,1,3,0,0>"
    assert canonical("void (anonymous namespace)::im2col_s2_kernel(__nv_bfloat16 const*, __nv_bfloat16*, int)") == IM2COL
    assert canonical("void conv_generic_kernel<float>(ConvP, float const*)") is None


# ---- the checker's self-test (CPU): it accepts a correct result and rejects each injected fault ------------------------------
SELF = spec_of(N=2, H=10, W=10, C=192, K=24, emb=True, res="f32", alpha=0.7, y32=True, stats=True)


def _self_case():
    ops_ = make_operands(SELF, "cpu", 5)
    refd = reference(SELF, ops_["x"], ops_["w"], ops_["bias"], ops_["emb"], ops_["res"], None)
    before = {k: b.clone() for k, (b, _) in ops_["bufs"].items()}
    y32 = ops_["y32"]
    y32.copy_(refd["ref"].float())             # what a correct kernel stores: the result rounded once to fp32
    ops_["y"].copy_(y32.to(torch.bfloat16))
    T = ops_["stats"].shape[0]
    v = y32.double()
    ops_["stats"].copy_(torch.stack([tile_sums(v, T), tile_sums(v * v, T)], -1).float())
    return ops_, refd, before


def _check(ops_, refd, before):
    writable = {"y", "y32", "stats"}
    guards = [(k, b, before[k], inside if k in writable else None) for k, (b, inside) in ops_["bufs"].items()]
    return check_outputs("self-test", SELF, refd, y=ops_["y"], y32=ops_["y32"], stats=ops_["stats"], guards=guards)


def _refresh(ops_):
    """recompute y and the statistics from a (faulted) y32, as the kernel would have"""
    y32 = ops_["y32"]
    ops_["y"].copy_(y32.to(torch.bfloat16))
    T = ops_["stats"].shape[0]
    v = y32.double().nan_to_num(0.0)
    ops_["stats"].copy_(torch.stack([tile_sums(v, T), tile_sums(v * v, T)], -1).float())


def test_checker_accepts_a_correctly_rounded_result():
    ops_, refd, before = _self_case()
    worst = _check(ops_, refd, before)
    assert max(worst.values()) < 0.5, worst


def _fault_no_bias(o, r):
    o["y32"][37, 8:16] -= 0.7 * o["bias"][8:16]


def _fault_missing_kblock(o, r):
    x, w = o["x"].double(), o["w"].double()
    rows = slice(128, 200)  # the second (ragged) 128-row tile, k-block 1 of 3
    o["y32"][rows] -= (0.7 * x[rows, 64:128] @ w[:, 64:128].t()).float()


def _fault_neighbour_emb(o, r):
    e = o["emb"].double()
    o["y32"][:100] += (0.7 * (e[1] - e[0])).float()


def _fault_sentinel_row(o, r):
    o["y32"][199] = NAN


def _fault_zero_row(o, r):
    o["y32"][199] = 0.0


FAULTS = [("one row of one 8-channel group without its bias", _fault_no_bias),
          ("one 64-wide k-block missing for one 128-row tile", _fault_missing_kblock),
          ("the embedding row of the neighbouring image", _fault_neighbour_emb),
          ("the last row of a ragged tile left at the sentinel", _fault_sentinel_row),
          ("the last row of a ragged tile zeroed", _fault_zero_row)]


@pytest.mark.parametrize("fault", [f for _, f in FAULTS], ids=[n for n, _ in FAULTS])
def test_checker_rejects_output_fault(fault):
    ops_, refd, before = _self_case()
    fault(ops_, refd)
    _refresh(ops_)
    with pytest.raises(AssertionError):
        _check(ops_, refd, before)


def test_checker_rejects_statistics_from_the_neighbouring_tile():
    ops_, refd, before = _self_case()
    ops_["stats"][0, 5] = ops_["stats"][1, 5]
    with pytest.raises(AssertionError, match="statistics"):
        _check(ops_, refd, before)


def test_checker_rejects_a_write_past_the_slice():
    ops_, refd, before = _self_case()
    buf, inside = ops_["bufs"]["y32"]
    buf[3, inside[1].stop] = ops_["y32"][3, -1]
    with pytest.raises(AssertionError, match="guard"):
        _check(ops_, refd, before)
    ops_, refd, before = _self_case()
    buf, inside = ops_["bufs"]["y"]
    buf[200, inside[1].start] = 0.0  # a row beyond M
    with pytest.raises(AssertionError, match="guard"):
        _check(ops_, refd, before)


def test_checker_rejects_a_bf16_copy_that_is_not_the_rounding_of_y32():
    ops_, refd, before = _self_case()
    ops_["y"][7, 3] = ops_["y"][7, 3] * 1.01
    with pytest.raises(AssertionError, match="bf16"):
        _check(ops_, refd, before)


# ---- production census ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_production_census():
    """every conv / GEMM-family kernel the yaml-size networks launch (UNet + ControlNet at 256^2 with 1, 2 and 16 rows and at
    512^2 with 8 rows; VAE decode and encode at 256^2, batch 1 and 2) is one that a case here runs and checks"""
    from makeupdiffuse_b200 import B200ControlLDM, B200FirstStageDecoder, B200FirstStageEncoder
    from makeupdiffuse_b200.synth import synthetic_first_stage_state_dict, synthetic_state_dict
    dev = "cuda"
    m = B200ControlLDM(dtype=torch.bfloat16, device=dev)
    m.load_state_dict(synthetic_state_dict(m, 0, dev))
    dec, enc = B200FirstStageDecoder(dtype=torch.bfloat16), B200FirstStageEncoder(dtype=torch.bfloat16)
    dec.load_state_dict(synthetic_first_stage_state_dict(dec, 0, dev))
    enc.load_state_dict(synthetic_first_stage_state_dict(enc, 0, dev))
    g = torch.Generator(device=dev).manual_seed(0)
    census, where = {}, {}

    def count(tag, fn):
        for n in launched_kernels(fn):
            c = canonical(n)
            key = c or ("(other) " + (re.findall(r"\w*kernel\w*", n) or [n[:40]])[0])
            if c is None and "conv" not in n:
                continue
            census[key] = census.get(key, 0) + 1
            where.setdefault(key, tag)
    for rows, h in ((1, 32), (2, 32), (16, 32), (8, 64)):
        cond = {"c_crossattn": [torch.randn(rows, 77, 768, device=dev, generator=g)],
                "c_concat": [torch.rand(rows, 6, 8 * h, 8 * h, device=dev, generator=g)]}
        x = torch.randn(rows, 4, h, h, device=dev, generator=g)
        t = torch.full((rows,), 501, device=dev, dtype=torch.long)
        count(f"apply_model {rows} x {8 * h}^2", lambda: m.apply_model(x, t, cond))
    for b in (1, 2):
        z = torch.randn(b, 4, 32, 32, device=dev, generator=g)
        img = torch.rand(b, 3, 256, 256, device=dev, generator=g) * 2 - 1
        count(f"VAE decode {b} x 256^2", lambda: dec.decode(z))
        count(f"VAE encode {b} x 256^2", lambda: enc.encode(img))
    print("\nproduction census (kernel -> launches, first seen in):")
    for k in sorted(census):
        mark = "case" if k in EXPECTED else ("generic kernel, outside this file" if k.startswith("(other)") else "NO CASE")
        print(f"  {k:<48s} {census[k]:6d}   {where[k]:<26s} {mark}")
    missing = sorted(k for k in census if not k.startswith("(other)") and k not in EXPECTED)
    assert not missing, f"production launches conv / GEMM kernels no case here checks: {missing}"
