"""Tensor-level wrappers over the C-ABI: torch is used for device memory and streams only.

Activations are 2-D strided views ``[pixels, channels]`` (NHWC with an explicit row pitch), so a tensor may be a
column slice of a wider concat buffer; spatial sizes travel as plain ints.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib as L

_DT = {torch.bfloat16: L.MKD_BF16, torch.float32: L.MKD_F32}


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _dt(t: torch.Tensor) -> int:
    try:
        return _DT[t.dtype]
    except KeyError:
        raise TypeError(f"unsupported dtype {t.dtype}; the B200 path stores bf16 (or fp32 in check mode)") from None


def _rows(t: torch.Tensor):
    """(data_ptr, row pitch) of a 2-D view whose last dim is contiguous"""
    if t.dim() != 2 or t.stride(1) != 1 or not t.is_cuda:
        raise ValueError(f"expected a CUDA 2-D view with unit inner stride, got shape {tuple(t.shape)} strides {t.stride()}")
    return t.data_ptr(), t.stride(0)


def _p(t):
    return None if t is None else t.data_ptr()


PROFILE = None  # bench.py sets this to a list to time every launch in place (CUDA events on the stream)


def _timed(name, nbytes_fn=None):
    """decorator: when PROFILE is on, bracket the op with CUDA events and record (name, algorithmic bytes)"""
    def deco(fn):
        def wrapper(*a, **kw):
            if PROFILE is None:
                return fn(*a, **kw)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = fn(*a, **kw)
            e1.record()
            PROFILE.append({"op": name, "bytes": nbytes_fn(*a, **kw) if nbytes_fn else 0, "e0": e0, "e1": e1,
                            "replay": (fn, a, kw)})
            return r
        wrapper.__name__ = fn.__name__
        wrapper.__doc__ = fn.__doc__
        return wrapper
    return deco


def _nb(*ts):
    return sum(t.numel() * t.element_size() for t in ts if t is not None)


def device_ok(device: int = 0):
    L.check(L.load().mkd_device_ok(device), "device check")


def ddim_update(x, eps, x_prev, *, sqrt_one_minus_at, sqrt_at, sqrt_a_prev, dir_coef, sigma_t=0.0, temperature=1.0,
                noise=None, pred_x0=None, cfg_scale=None, peer_ptrs=None):
    """eps holds n values, or 2n ([uncond; cond]) when cfg_scale is given  (diffmk/cddim.py:39-40,56-78)."""
    n = x.numel()
    for t in (x, eps, x_prev, noise, pred_x0):
        if t is not None and (t.dtype != torch.float32 or not t.is_contiguous() or not t.is_cuda):
            raise ValueError("ddim_update works on contiguous fp32 CUDA latents")
    cfg = cfg_scale is not None
    if eps.numel() != (2 * n if cfg else n):
        raise ValueError("eps has the wrong number of elements")
    if peer_ptrs is not None:  # x_prev goes to every rank's gather buffer (mkd_ddim_update_peers); x_prev = own slice
        arr = (C.c_void_p * len(peer_ptrs))(*[int(p) for p in peer_ptrs])
        L.check(L.load().mkd_ddim_update_peers(x.data_ptr(), eps.data_ptr(), int(cfg), float(cfg_scale or 0.0), _p(noise),
                                               float(sqrt_one_minus_at), float(sqrt_at), float(sqrt_a_prev), float(dir_coef),
                                               float(sigma_t), float(temperature), arr, len(peer_ptrs), _p(pred_x0), n,
                                               _stream()), "ddim_update_peers")
        return
    L.check(L.load().mkd_ddim_update(x.data_ptr(), eps.data_ptr(), int(cfg), float(cfg_scale or 0.0), _p(noise),
                                     float(sqrt_one_minus_at), float(sqrt_at), float(sqrt_a_prev), float(dir_coef),
                                     float(sigma_t), float(temperature), x_prev.data_ptr(), _p(pred_x0), n, _stream()),
            "ddim_update")


PLMS_HISTORY = (0, 1, 1, 2, 3)  # earlier eps each mode of mkd_plms_update reads


def plms_update(x, eps, x_prev, *, mode, history=(), e_store=None, sqrt_one_minus_at, sqrt_at, sqrt_a_prev, dir_coef,
                pred_x0=None, cfg_scale=None, peer_ptrs=None):
    """One PLMS update (upstream plms.py p_sample_plms after its model call): eps holds n values, or 2n ([uncond; cond]) when
    cfg_scale is given; the combined e_t goes to e_store when given.  history: the earlier eps the mode combines, newest
    first (upstream's old_eps[-1], old_eps[-2], old_eps[-3]); mode 1 averages with history[0] (the pseudo improved Euler
    step), modes 2 / 3 / 4 are the Adams-Bashforth orders, mode 0 is the plain DDIM update."""
    n = x.numel()
    if not 0 <= mode <= 4 or len(history) != PLMS_HISTORY[mode]:
        raise ValueError(f"plms_update mode {mode} takes {PLMS_HISTORY[mode] if 0 <= mode <= 4 else '?'} history tensors")
    for t in (x, eps, x_prev, e_store, pred_x0, *history):
        if t is not None and (t.dtype != torch.float32 or not t.is_contiguous() or not t.is_cuda):
            raise ValueError("plms_update works on contiguous fp32 CUDA latents")
    for t in (x_prev, e_store, pred_x0, *history):
        if t is not None and t.numel() != n:
            raise ValueError("plms_update: every latent-sized tensor must hold x.numel() values")
    cfg = cfg_scale is not None
    if eps.numel() != (2 * n if cfg else n):
        raise ValueError("eps has the wrong number of elements")
    h = [_p(t) for t in history] + [None] * (3 - len(history))
    head = (x.data_ptr(), eps.data_ptr(), int(cfg), float(cfg_scale or 0.0), _p(e_store), int(mode), *h,
            float(sqrt_one_minus_at), float(sqrt_at), float(sqrt_a_prev), float(dir_coef))
    if peer_ptrs is not None:  # x_prev goes to every rank's gather buffer (mkd_plms_update_peers); x_prev = own slice
        arr = (C.c_void_p * len(peer_ptrs))(*[int(p) for p in peer_ptrs])
        L.check(L.load().mkd_plms_update_peers(*head, arr, len(peer_ptrs), _p(pred_x0), n, _stream()), "plms_update_peers")
        return
    L.check(L.load().mkd_plms_update(*head, x_prev.data_ptr(), _p(pred_x0), n, _stream()), "plms_update")


def dpm_update(x, eps, x_prev, *, alpha_s, sigma_s, sigma_ratio, phi, order=1, m_prev=None, half_phi=0.0, inv_r0=0.0,
               m_store=None, cfg_scale=None, peer_ptrs=None):
    """One DPM-Solver++ multistep update (upstream dpm_solver.py, predict_x0=True, after one model call): eps holds n values,
    or 2n ([uncond; cond]) when cfg_scale is given; the data prediction m = (x - sigma_s * e) / alpha_s goes to m_store
    when given; order 1 steps with m alone, order 2 also with the previous data prediction m_prev.  The scalars come from
    upstream's expressions (mkd_dpm_update in include/mkd_b200.h)."""
    n = x.numel()
    if order not in (1, 2) or (order == 2) != (m_prev is not None):
        raise ValueError("dpm_update: order 1 takes no m_prev, order 2 needs it")
    for t in (x, eps, x_prev, m_store, m_prev):
        if t is not None and (t.dtype != torch.float32 or not t.is_contiguous() or not t.is_cuda):
            raise ValueError("dpm_update works on contiguous fp32 CUDA latents")
    for t in (x_prev, m_store, m_prev):
        if t is not None and t.numel() != n:
            raise ValueError("dpm_update: every latent-sized tensor must hold x.numel() values")
    cfg = cfg_scale is not None
    if eps.numel() != (2 * n if cfg else n):
        raise ValueError("eps has the wrong number of elements")
    head = (x.data_ptr(), eps.data_ptr(), int(cfg), float(cfg_scale or 0.0), float(alpha_s), float(sigma_s), _p(m_store),
            int(order), _p(m_prev), float(sigma_ratio), float(phi), float(half_phi), float(inv_r0))
    if peer_ptrs is not None:  # x_prev goes to every rank's gather buffer (mkd_dpm_update_peers); x_prev = own slice
        arr = (C.c_void_p * len(peer_ptrs))(*[int(p) for p in peer_ptrs])
        L.check(L.load().mkd_dpm_update_peers(*head, arr, len(peer_ptrs), n, _stream()), "dpm_update_peers")
        return
    L.check(L.load().mkd_dpm_update(*head, x_prev.data_ptr(), n, _stream()), "dpm_update")


@_timed("nchw_to_nhwc", lambda s, d: _nb(s, d))
def nchw_to_nhwc(src, dst2d):
    N, Cc, H, W = src.shape
    if src.dtype != torch.float32 or not src.is_contiguous():
        raise ValueError("nchw_to_nhwc expects a contiguous fp32 NCHW tensor")
    p, ld = _rows(dst2d)
    assert dst2d.shape == (N * H * W, Cc)
    L.check(L.load().mkd_nchw_to_nhwc(src.data_ptr(), p, _dt(dst2d), N, Cc, H, W, ld, _stream()), "nchw_to_nhwc")


@_timed("nhwc_to_nchw", lambda s, d: _nb(s, d))
def nhwc_to_nchw(src2d, dst):
    N, Cc, H, W = dst.shape
    if dst.dtype != torch.float32 or not dst.is_contiguous():
        raise ValueError("nhwc_to_nchw expects a contiguous fp32 NCHW destination")
    p, ld = _rows(src2d)
    assert src2d.shape == (N * H * W, Cc)
    L.check(L.load().mkd_nhwc_to_nchw(p, dst.data_ptr(), _dt(src2d), N, Cc, H, W, ld, _stream()), "nhwc_to_nchw")


@_timed("timestep_embedding", None)
def timestep_embedding(t, out, max_period=10000.0):
    assert t.dtype == torch.int64 and t.is_contiguous() and out.is_contiguous()
    B, dim = out.shape
    L.check(L.load().mkd_timestep_embedding(t.data_ptr(), out.data_ptr(), _dt(out), B, dim, float(max_period), _stream()),
            "timestep_embedding")


@_timed("timestep_embedding_f32", None)
def timestep_embedding_f32(t, out, max_period=10000.0):
    """upstream timestep_embedding of fp32 timesteps, fractional ones as they are"""
    assert t.dtype == torch.float32 and t.is_contiguous() and out.is_contiguous()
    B, dim = out.shape
    L.check(L.load().mkd_timestep_embedding_f32(t.data_ptr(), out.data_ptr(), _dt(out), B, dim, float(max_period),
                                                _stream()), "timestep_embedding_f32")


@_timed("silu", lambda x, y: _nb(x, y))
def silu(x, y):
    assert x.is_contiguous() and y.is_contiguous() and x.dtype == y.dtype
    L.check(L.load().mkd_silu(x.data_ptr(), y.data_ptr(), _dt(x), x.numel(), _stream()), "silu")


@_timed("geglu", lambda x, y: _nb(x, y))
def geglu(x2d, y2d):
    px, ldx = _rows(x2d)
    py, ldy = _rows(y2d)
    M, inner = y2d.shape
    assert x2d.shape == (M, 2 * inner)
    L.check(L.load().mkd_geglu(px, py, _dt(x2d), M, inner, ldx, ldy, _stream()), "geglu")


@_timed("add", lambda a, b, y: _nb(a, b, y))
def add(a2d, b2d, y2d):
    pa, lda = _rows(a2d)
    pb, ldb = _rows(b2d)
    py, ldy = _rows(y2d)
    M, Cc = y2d.shape
    L.check(L.load().mkd_add(pa, pb, py, _dt(y2d), M, Cc, lda, ldb, ldy, _stream()), "add")


def groupnorm_workspace_bytes(N, groups=32) -> int:
    return int(L.load().mkd_groupnorm_workspace_bytes(N, groups))


@_timed("groupnorm", lambda x, y, *a, **k: _nb(x, y))
def groupnorm(x2d, y2d, N, gamma, beta, eps, silu, workspace, groups=32, wgroups=1):
    """wgroups = 2: gamma / beta hold [2, C]; samples n >= N/2 use the second row (two networks' layer in one launch)"""
    px, ldx = _rows(x2d)
    py, ldy = _rows(y2d)
    M, Cc = x2d.shape
    assert M % N == 0 and y2d.shape == x2d.shape and gamma.dtype == torch.float32 and beta.dtype == torch.float32
    assert gamma.numel() == wgroups * Cc and beta.numel() == wgroups * Cc and gamma.is_contiguous() and beta.is_contiguous()
    L.check(L.load().mkd_groupnorm(px, py, _dt(x2d), _dt(y2d), N, M // N, Cc, groups, ldx, ldy, gamma.data_ptr(), beta.data_ptr(),
                                   float(eps), int(bool(silu)), workspace.data_ptr(),
                                   workspace.numel() * workspace.element_size(), wgroups, _stream()), "groupnorm")


@_timed("groupnorm_apply", lambda x, y, *a, **k: _nb(x, y))
def groupnorm_apply(x2d, y2d, N, gamma, beta, eps, silu, stats, groups=32, wgroups=1):
    """GroupNorm whose statistics were emitted by the producing conv2d(..., stats=): ``stats`` is a
    [N * HW / 128, C, 2] fp32 view (row pitch may exceed C when it is a channel slice of a concat's statistics)."""
    px, ldx = _rows(x2d)
    py, ldy = _rows(y2d)
    M, Cc = x2d.shape
    assert M % N == 0 and (M // N) % 128 == 0 and y2d.shape == x2d.shape
    assert stats.dtype == torch.float32 and stats.dim() == 3 and stats.shape[1:] == (Cc, 2) and stats.stride(2) == 1
    assert stats.stride(1) == 2 and stats.shape[0] == M // 128 and stats.stride(0) % 2 == 0
    assert gamma.numel() == wgroups * Cc and beta.numel() == wgroups * Cc and gamma.is_contiguous() and beta.is_contiguous()
    L.check(L.load().mkd_groupnorm_apply(px, py, _dt(x2d), _dt(y2d), N, M // N, Cc, groups, ldx, ldy, gamma.data_ptr(),
                                         beta.data_ptr(), float(eps), int(bool(silu)), stats.data_ptr(),
                                         stats.stride(0) // 2, (M // N) // 128, wgroups, _stream()), "groupnorm_apply")


@_timed("layernorm", lambda x, y, *a, **k: _nb(x, y))
def layernorm(x2d, y2d, gamma, beta, eps=1e-5, wgroups=1):
    px, ldx = _rows(x2d)
    py, ldy = _rows(y2d)
    M, Cc = x2d.shape
    assert gamma.dtype == torch.float32 and beta.dtype == torch.float32
    assert gamma.numel() == wgroups * Cc and beta.numel() == wgroups * Cc and gamma.is_contiguous() and beta.is_contiguous()
    L.check(L.load().mkd_layernorm(px, py, _dt(x2d), _dt(y2d), M, Cc, ldx, ldy, gamma.data_ptr(), beta.data_ptr(), float(eps),
                                   wgroups, _stream()), "layernorm")


@_timed("softmax_rows", lambda x, y, *a, **k: _nb(x, y))
def softmax_rows(x2d, y2d, scale=1.0):
    """y = softmax(scale * x) over the last dim (fp32 statistics)"""
    px, ldx = _rows(x2d)
    py, ldy = _rows(y2d)
    M, Cc = x2d.shape
    assert y2d.shape == x2d.shape
    L.check(L.load().mkd_softmax_rows(px, py, _dt(x2d), _dt(y2d), M, Cc, ldx, ldy, float(scale), _stream()), "softmax_rows")


def make_conv_desc(x2d, w, y2d, *, N, H, W, R=1, S=1, stride=1, pad=0, upsample=False, bias=None, emb=None,
                   residual=None, alpha=1.0, act=L.ACT_NONE, geglu_block=0, path=L.PATH_AUTO, workspace=None,
                   y32=None, stats=None, pad_hi_extra=0, x2=None, wgroups=1, gn=None) -> L.ConvDesc:
    """y2d: output in the activation dtype (or None); y32: optional fp32 copy of the same result.
    x2: optional second input [N*H*W, C2] of a fused 1x1 term (mkd_conv_desc.x2): w is then [K, R*S*C + C2].
    gn: optional GroupNorm tail (mkd_conv_desc.gn_y): dict(y=, gamma=, beta=, eps=, silu=, groups=32) — the GroupNorm(+SiLU) of
    the layer's output written to ``y`` by the split-K reducer; only launches that split K take it (conv2d_supported)."""
    px, ldx = _rows(x2d)
    Cc = x2d.shape[1]
    K = w.shape[0] // wgroups  # wgroups = 2: w holds the rows of two networks' layer, bias both biases (mkd_conv_desc.wgroups)
    C2 = 0 if x2 is None else x2.shape[1]
    assert x2d.shape[0] == N * H * W, (x2d.shape, N, H, W)
    assert w.is_contiguous() and w.numel() == wgroups * K * (R * S * Cc + C2) and w.dtype == x2d.dtype
    assert bias is None or bias.numel() == wgroups * K
    d = L.ConvDesc()
    d.dtype = _dt(x2d)
    d.residual_dtype = d.dtype
    for out in (y2d, y32):
        if out is not None and out.shape[1] != (K // 2 if act == L.ACT_GEGLU else K):
            raise ValueError(f"output view has {out.shape[1]} channels, the filter bank produces {K}")
    if y2d is None and y32 is None:
        raise ValueError("conv2d needs an output")
    if y2d is not None:
        assert y2d.dtype == x2d.dtype
        d.y, d.ldy = _rows(y2d)
    if y32 is not None:
        assert y32.dtype == torch.float32
        d.y32, d.ldy32 = _rows(y32)
    d.N, d.H, d.W, d.C, d.K, d.R, d.S = N, H, W, Cc, K, R, S
    d.stride, d.pad, d.upsample, d.pad_hi_extra = stride, pad, int(bool(upsample)), int(pad_hi_extra)
    d.ldx = ldx
    d.act, d.geglu_block, d.path, d.alpha = act, geglu_block, path, float(alpha)
    d.x, d.w = px, w.data_ptr()
    if bias is not None:
        assert bias.dtype == torch.float32 and bias.is_contiguous()
        d.bias = bias.data_ptr()
    if emb is not None:
        pe, lde = _rows(emb)
        assert emb.dtype == x2d.dtype
        d.emb, d.lde = pe, lde
    if residual is not None:
        pr, ldr = _rows(residual)
        d.residual, d.ldr, d.residual_dtype = pr, ldr, _dt(residual)
    if workspace is not None:
        d.workspace, d.workspace_bytes = workspace.data_ptr(), workspace.numel() * workspace.element_size()
    if stats is not None:  # [ceil(M_out / 128), K, 2] fp32 view: GroupNorm partials of the output (mkd_conv_desc.stats)
        assert stats.dtype == torch.float32 and stats.dim() == 3 and stats.shape[1:] == (K, 2)
        assert stats.stride(2) == 1 and stats.stride(1) == 2 and stats.stride(0) % 2 == 0
        d.stats, d.stats_ld = stats.data_ptr(), stats.stride(0) // 2
    if x2 is not None:
        assert x2.dtype == x2d.dtype and x2.shape[0] == x2d.shape[0] and stride == 1 and not upsample
        d.x2, d.ldx2 = _rows(x2)
        d.C2 = C2
    d.wgroups = wgroups
    if gn is not None:
        gy, ga, be = gn["y"], gn["gamma"], gn["beta"]
        assert gy.dtype == x2d.dtype and gy.shape[1] == K and ga.dtype == torch.float32 and be.dtype == torch.float32
        assert ga.numel() == wgroups * K and be.numel() == wgroups * K and ga.is_contiguous() and be.is_contiguous()
        d.gn_y, d.gn_ld = _rows(gy)
        d.gn_gamma, d.gn_beta = ga.data_ptr(), be.data_ptr()
        d.gn_eps, d.gn_silu, d.gn_groups = float(gn["eps"]), int(bool(gn["silu"])), int(gn.get("groups", 32))
    return d


def conv2d(x2d, w, y2d, **kw):
    d = make_conv_desc(x2d, w, y2d, **kw)
    if PROFILE is None:
        L.check(L.load().mkd_conv2d(C.byref(d), _stream()), "conv2d")
        return
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    path = L.load().mkd_conv2d_path(C.byref(d))
    e0.record()
    L.check(L.load().mkd_conv2d(C.byref(d), _stream()), "conv2d")
    e1.record()
    Hi, Wi = (2 * d.H, 2 * d.W) if d.upsample else (d.H, d.W)
    P = (Hi + 2 * d.pad + d.pad_hi_extra - d.R) // d.stride + 1
    Q = (Wi + 2 * d.pad + d.pad_hi_extra - d.S) // d.stride + 1
    PROFILE.append({"op": "conv2d", "path": path, "flops": 2.0 * d.N * P * Q * d.K * (d.R * d.S * d.C + d.C2), "M": d.N * P * Q, "K": d.K,
                    "C": d.C, "C2": d.C2, "R": d.R, "stride": d.stride, "up": d.upsample, "e0": e0, "e1": e1, "desc": d})


def conv2d_grouped(x2d, w, y2d, *, N, **kw):
    """The same layer of TWO networks on two stacked batches in one launch (mkd_conv_desc.wgroups = 2): rows [0, M/2) of every
    row-indexed tensor (x, y, y32, residual, x2; emb and stats by image / tile) belong to network 0, the rest to network 1;
    ``w`` / ``bias`` hold network 0's rows followed by network 1's.  Shapes the CTA-pair kernel declines (parts that are not
    whole 256-row tile pairs, tiny problems) run as one launch per part on slices."""
    d = make_conv_desc(x2d, w, y2d, N=N, wgroups=2, **kw)
    if L.load().mkd_conv2d_path(C.byref(d)) >= 0:
        conv2d(x2d, w, y2d, N=N, wgroups=2, **kw)
        return
    assert N % 2 == 0 and w.shape[0] % 2 == 0
    K = w.shape[0] // 2
    out = y2d if y2d is not None else kw.get("y32")
    rows = {"x": x2d.shape[0] // 2, "out": out.shape[0] // 2}

    def part(t, g, n):
        return None if t is None else t[g * n:(g + 1) * n]
    for g in (0, 1):
        k2 = dict(kw)
        k2["bias"] = part(kw.get("bias"), g, K)
        for name in ("residual", "y32"):
            k2[name] = part(kw.get(name), g, rows["out"])
        k2["emb"] = part(kw.get("emb"), g, N // 2)
        k2["x2"] = part(kw.get("x2"), g, rows["x"])
        if kw.get("stats") is not None:
            k2["stats"] = part(kw["stats"], g, kw["stats"].shape[0] // 2)
        if kw.get("gn") is not None:
            k2["gn"] = dict(kw["gn"], y=part(kw["gn"]["y"], g, rows["out"]), gamma=part(kw["gn"]["gamma"], g, K), beta=part(kw["gn"]["beta"], g, K))
        conv2d(part(x2d, g, rows["x"]), w[g * K:(g + 1) * K], part(y2d, g, rows["out"]), N=N // 2, **k2)


def conv2d_path(x2d, w, y2d, **kw) -> int:
    d = make_conv_desc(x2d, w, y2d, **kw)
    rc = L.load().mkd_conv2d_path(C.byref(d))
    if rc < 0:
        L.check(rc, "conv2d_path")
    return rc


def conv2d_supported(x2d, w, y2d, **kw) -> bool:
    """does some kernel take this descriptor?  (False for a fused `x2` term the CTA-pair kernel declines: the caller then
    issues the two layers as two launches)"""
    return L.load().mkd_conv2d_path(C.byref(make_conv_desc(x2d, w, y2d, **kw))) >= 0


def run_conv_desc(d: L.ConvDesc):
    L.check(L.load().mkd_conv2d(C.byref(d), _stream()), "conv2d")


def attention(q2d, k2d, v2d, o2d, *, B, heads, Nq, Nkv, d, scale):
    if PROFILE is None:
        return _attention(q2d, k2d, v2d, o2d, B=B, heads=heads, Nq=Nq, Nkv=Nkv, d=d, scale=scale)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    _attention(q2d, k2d, v2d, o2d, B=B, heads=heads, Nq=Nq, Nkv=Nkv, d=d, scale=scale)
    e1.record()
    PROFILE.append({"op": "attention", "bytes": _nb(q2d, k2d, v2d, o2d), "flops": 4.0 * B * heads * Nq * Nkv * d,
                    "e0": e0, "e1": e1,
                    "replay": (_attention, (q2d, k2d, v2d, o2d), dict(B=B, heads=heads, Nq=Nq, Nkv=Nkv, d=d, scale=scale))})


def _attention(q2d, k2d, v2d, o2d, *, B, heads, Nq, Nkv, d, scale):
    pq, ldq = _rows(q2d)
    pk, ldk = _rows(k2d)
    pv, ldv = _rows(v2d)
    po, ldo = _rows(o2d)
    L.check(L.load().mkd_attention(pq, pk, pv, po, _dt(q2d), B, heads, Nq, Nkv, d, ldq, ldk, ldv, ldo, float(scale),
                                   _stream()), "attention")


def attention_causal(q2d, k2d, v2d, o2d, *, B, heads, N, d, scale):
    """causal self-attention over N tokens per sample (CLIP text encoder); q/k/v may be column slices of one buffer"""
    pq, ldq = _rows(q2d)
    pk, ldk = _rows(k2d)
    pv, ldv = _rows(v2d)
    po, ldo = _rows(o2d)
    L.check(L.load().mkd_attention_causal(pq, pk, pv, po, _dt(q2d), B, heads, N, d, ldq, ldk, ldv, ldo, float(scale),
                                          _stream()), "attention_causal")


def embed_tokens(ids, tok_emb, pos_emb, out2d):
    """out[b*T + t] = tok_emb[ids[b, t]] + pos_emb[t]   (fp32)"""
    B, T = ids.shape
    vocab, Cc = tok_emb.shape
    assert ids.dtype == torch.int64 and ids.is_contiguous() and tok_emb.dtype == pos_emb.dtype == out2d.dtype == torch.float32
    assert pos_emb.shape[0] >= T and pos_emb.shape[1] == Cc and tok_emb.is_contiguous() and pos_emb.is_contiguous()
    if int(ids.min()) < 0 or int(ids.max()) >= vocab:
        raise IndexError(f"token id outside [0, {vocab})")  # nn.Embedding raises IndexError as well
    po, ldo = _rows(out2d)
    L.check(L.load().mkd_embed_tokens(ids.data_ptr(), tok_emb.data_ptr(), pos_emb.data_ptr(), po, B, T, Cc, vocab, ldo,
                                      _stream()), "embed_tokens")


def image_grid_shape(N, H, W, nrow, padding=2):
    if N == 1:
        padding = 0  # torchvision's make_grid returns a single image without the padding frame
    xmaps = min(nrow, N)
    ymaps = (N + xmaps - 1) // xmaps
    return (H + padding) * ymaps + padding, (W + padding) * xmaps + padding


def image_grid_u8(images, nrow, padding=2, clamp=True, rescale=True):
    """images [N, C, H, W] fp32 (C = 1 or 3) -> uint8 [GH, GW, 3] grid (make_grid + rescale + HWC + uint8 in one pass)"""
    assert images.dtype == torch.float32 and images.dim() == 4
    images = images.contiguous()
    N, Cc, H, W = images.shape
    GH, GW = image_grid_shape(N, H, W, nrow, padding)
    out = torch.empty(GH, GW, 3, dtype=torch.uint8, device=images.device)
    L.check(L.load().mkd_image_grid_u8(images.data_ptr(), out.data_ptr(), N, Cc, H, W, int(nrow), int(padding), int(clamp),
                                       int(rescale), _stream()), "image_grid_u8")
    return out
