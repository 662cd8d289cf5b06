"""B200 replacements for the two networks ``apply_model`` drives (SURVEY.md §8(b) level B2).

``B200ControlNet`` / ``B200ControlledUnet`` take the same ``params:`` kwargs as ``cldm.cldm.ControlNet`` /
``cldm.cldm.ControlledUnetModel`` in ``diffmodels/base_diffusion_makeup.yaml:52-84`` and the same keyword call forms as
``diffmk/makeup_diffuse.py:164-168``:

    control_model(x=, hint=, timesteps=, context=)                         -> list of 13 residuals (NCHW fp32)
    diffusion_model(x=, timesteps=, context=, control=, only_mid_control=) -> eps (NCHW fp32)

so they are installed by pointing the yaml's two ``target:`` strings at them.  ``load_state_dict`` accepts upstream
checkpoint keys (``input_blocks.1.0.in_layers.2.weight`` ...) and repacks once: OIHW fp32 -> KRSC bf16, fused q/k/v
and cross k/v projection matrices, GEGLU rows interleaved for the fused epilogue.

Everything below the Python orchestration is a hand-written sm_100a kernel behind the C-ABI (ops.py): activations
are NHWC bf16 (fp32 in check mode), skip tensors are produced directly into the decoder's concat buffers, and the
fused path (``inject=`` / ``B200ControlLDM.apply_model``) lets the ControlNet zero-conv GEMM epilogues accumulate
into those skip slots, so ``hs.pop() + control.pop()`` and ``torch.cat`` never run as separate passes.
There is no PyTorch compute fallback: without the CUDA library these classes cannot run.
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn

from . import _lib as L
from . import ops

_SPLITK_WS_BYTES = 96 << 20


def timesteps_for_embedding(t):
    """the timestep tensor the embedding kernels take: integer timesteps as int64 (mkd_timestep_embedding), floating ones
    as fp32 (mkd_timestep_embedding_f32), so a fractional t is not truncated.  For integers below 2^24 both give the
    same bits."""
    return (t.to(torch.float32) if t.is_floating_point() else t.to(torch.int64)).contiguous()


class Act:
    """A trunk tensor of the bf16 path, stored up to twice:
    ``lo`` — activation dtype (bf16), what tensor-core A operands and the decoder's concat slots read;
    ``hi`` — fp32 copy written by the same epilogue, what norms and residual adds read, so that the residual
             stream is not re-rounded at every block (that rounding, not the bf16 MMAs, dominated the eps error).
    In the fp32 check mode only ``lo`` (fp32) exists.
    ``st`` — optional GroupNorm statistics of the tensor, [rows / 128, C, 2] fp32: per-tile column (sum, sumsq) emitted
             by the epilogue that produced it (mkd_conv_desc.stats), so the consuming GroupNorm is one streaming pass.
             ``None`` means "not produced": the consumer then runs the full (reduce + normalise) GroupNorm kernel."""
    __slots__ = ("lo", "hi", "st")

    def __init__(self, lo=None, hi=None, st=None):
        self.lo, self.hi, self.st = lo, hi, st

    def src(self):
        return self.hi if self.hi is not None else self.lo


def _geglu_block(inner: int) -> int:
    # 128: the CTA-pair kernel's [128 value | 128 gate] tiles (one 256-wide MMA per k-step); 80: the single-CTA kernel's
    for gb in (128, 80, 64, 32, 16, 8):
        if inner % gb == 0:
            return gb
    raise ValueError(f"FF inner dim {inner} not supported")


class _Net(nn.Module):
    """time_embed + input_blocks + middle_block; subclasses add the ControlNet or decoder specific parts."""

    def __init__(self, in_channels=4, model_channels=320, attention_resolutions=(4, 2, 1), num_res_blocks=2,
                 channel_mult=(1, 2, 4, 4), num_heads=8, transformer_depth=1, context_dim=768,
                 dtype=torch.bfloat16, **unused):
        super().__init__()
        if transformer_depth != 1:
            raise NotImplementedError("only transformer_depth=1 (the yaml's value) is implemented")
        self.dtype = dtype
        self.in_channels, self.mc, self.heads, self.context_dim = in_channels, model_channels, num_heads, context_dim
        self.ted = 4 * model_channels
        mc = model_channels
        self.input_blocks = [[("conv_in", "input_blocks.0.0", in_channels, mc)]]
        self.block_chans = [mc]
        self.block_ds = [1]
        ch, ds = mc, 1
        for level, mult in enumerate(channel_mult):
            for _ in range(num_res_blocks):
                i = len(self.input_blocks)
                layers = [("res", f"input_blocks.{i}.0", ch, mult * mc)]
                ch = mult * mc
                if ds in attention_resolutions:
                    layers.append(("st", f"input_blocks.{i}.1", ch))
                self.input_blocks.append(layers)
                self.block_chans.append(ch)
                self.block_ds.append(ds)
            if level != len(channel_mult) - 1:
                i = len(self.input_blocks)
                self.input_blocks.append([("down", f"input_blocks.{i}.0.op", ch)])
                ds *= 2
                self.block_chans.append(ch)
                self.block_ds.append(ds)
        self.middle = [("res", "middle_block.0", ch, ch), ("st", "middle_block.1", ch), ("res", "middle_block.2", ch, ch)]
        self._ch, self._ds = ch, ds
        self._attn_res = tuple(attention_resolutions)
        self.fused_gn_stats = True  # False: always the two-phase GroupNorm (A/B runs)
        self.fuse_skip = True       # False: ResBlock skip projections always as their own GEMM (A/B runs)
        self.fuse_gn_tail = True    # False: out_layers' GroupNorm always as its own launch (A/B runs)
        self._fuse_ok: dict = {}
        # bumped whenever context_kv() / hint_features() refill their (shared, static) arena buffers: a holder of earlier
        # results — B200ControlLDM's cond cache — compares epochs to learn that the buffers now hold another cond's data
        self.arena_epoch = 0
        self._wg = 1  # weight groups of every launch (2 in B200GroupedTrunk: two networks' layer on two stacked batches)
        self._channel_mult, self._nrb = tuple(channel_mult), num_res_blocks
        self.w: dict[str, torch.Tensor] = {}
        self._bufs: dict = {}
        self._loaded = False

    # ---- parameters ------------------------------------------------------------------------------------------
    def _all_layers(self):
        for blk in self.input_blocks:
            yield from blk
        yield from self.middle

    def _res_layers(self):
        return [l for l in self._all_layers() if l[0] == "res"]

    def _put(self, name, t, act_dtype=False):
        t = t.detach().to(device=self._device, dtype=self.dtype if act_dtype else torch.float32).contiguous()
        self.w[name] = t

    @staticmethod
    def _krsc(w):  # OIHW -> [O][R][S][I]
        return w.permute(0, 2, 3, 1).contiguous()

    def load_state_dict(self, sd, strict=True, prefix="", device="cuda"):  # noqa: D401 (upstream-keyed checkpoints)
        """Repack an upstream-keyed state dict (fp32 OIHW / [out,in]) into the layouts the kernels read."""
        self._device = torch.device(device)
        used = set()

        def g(k):
            used.add(prefix + k)
            return sd[prefix + k]

        self._put("te0.w", g("time_embed.0.weight"), True); self._put("te0.b", g("time_embed.0.bias"))
        self._put("te2.w", g("time_embed.2.weight"), True); self._put("te2.b", g("time_embed.2.bias"))
        emb_w, emb_b = [], []
        for layer in self._all_layers():
            kind, key = layer[0], layer[1]
            if kind == "conv_in" and self._hi:
                # bf16 path: the 4 latent channels are zero-padded to 64 so that conv_in runs on the tensor-core kernel
                # (which wants C % 64 == 0) and emits GroupNorm statistics like every other trunk producer
                w = self._krsc(g(key + ".weight"))
                wp = torch.zeros(w.shape[0], 3, 3, 64, dtype=w.dtype)
                wp[..., :w.shape[3]] = w
                self._put(key + ".w", wp, True); self._put(key + ".b", g(key + ".bias"))
            elif kind in ("conv_in", "down", "up"):
                self._put(key + ".w", self._krsc(g(key + ".weight")), True); self._put(key + ".b", g(key + ".bias"))
            elif kind == "res":
                self._put(key + ".gn1.g", g(key + ".in_layers.0.weight")); self._put(key + ".gn1.b", g(key + ".in_layers.0.bias"))
                self._put(key + ".c1.w", self._krsc(g(key + ".in_layers.2.weight")), True); self._put(key + ".c1.b", g(key + ".in_layers.2.bias"))
                emb_w.append(g(key + ".emb_layers.1.weight")); emb_b.append(g(key + ".emb_layers.1.bias"))
                self._put(key + ".gn2.g", g(key + ".out_layers.0.weight")); self._put(key + ".gn2.b", g(key + ".out_layers.0.bias"))
                self._put(key + ".c2.w", self._krsc(g(key + ".out_layers.3.weight")), True); self._put(key + ".c2.b", g(key + ".out_layers.3.bias"))
                if layer[2] != layer[3]:
                    self._put(key + ".sk.w", self._krsc(g(key + ".skip_connection.weight")), True)
                    self._put(key + ".sk.b", g(key + ".skip_connection.bias"))
                    if self._hi:
                        # out_layers conv + skip_connection as ONE contraction (mkd_conv_desc.x2): weight rows
                        # [3][3][cout] followed by the cin columns of the 1x1 projection, biases summed
                        co = layer[3]
                        self._put(key + ".c2sk.w", torch.cat([self._krsc(g(key + ".out_layers.3.weight")).reshape(co, -1),
                                                              g(key + ".skip_connection.weight").reshape(co, -1)], 1), True)
                        self._put(key + ".c2sk.b", g(key + ".out_layers.3.bias") + g(key + ".skip_connection.bias"))
            elif kind == "st":
                tb = key + ".transformer_blocks.0."
                self._put(key + ".gn.g", g(key + ".norm.weight")); self._put(key + ".gn.b", g(key + ".norm.bias"))
                self._put(key + ".pi.w", self._krsc(g(key + ".proj_in.weight")), True); self._put(key + ".pi.b", g(key + ".proj_in.bias"))
                self._put(key + ".po.w", self._krsc(g(key + ".proj_out.weight")), True); self._put(key + ".po.b", g(key + ".proj_out.bias"))
                for n in ("norm1", "norm2", "norm3"):
                    self._put(key + f".{n}.g", g(tb + n + ".weight")); self._put(key + f".{n}.b", g(tb + n + ".bias"))
                self._put(key + ".qkv.w", torch.cat([g(tb + "attn1.to_q.weight"), g(tb + "attn1.to_k.weight"),
                                                     g(tb + "attn1.to_v.weight")], 0), True)
                self._put(key + ".o1.w", g(tb + "attn1.to_out.0.weight"), True); self._put(key + ".o1.b", g(tb + "attn1.to_out.0.bias"))
                self._put(key + ".q2.w", g(tb + "attn2.to_q.weight"), True)
                self._put(key + ".kv2.w", torch.cat([g(tb + "attn2.to_k.weight"), g(tb + "attn2.to_v.weight")], 0), True)
                self._put(key + ".o2.w", g(tb + "attn2.to_out.0.weight"), True); self._put(key + ".o2.b", g(tb + "attn2.to_out.0.bias"))
                wff, bff = g(tb + "ff.net.0.proj.weight"), g(tb + "ff.net.0.proj.bias")
                inner = wff.shape[0] // 2
                gb = _geglu_block(inner)
                # rows: blocks of [gb value rows | gb gate rows]  (mkd_conv_desc GEGLU layout)
                wv, wg = wff[:inner].reshape(inner // gb, gb, -1), wff[inner:].reshape(inner // gb, gb, -1)
                bv, bg = bff[:inner].reshape(inner // gb, gb), bff[inner:].reshape(inner // gb, gb)
                self._put(key + ".ff1.w", torch.stack([wv, wg], 1).reshape(2 * inner, -1), True)
                self._put(key + ".ff1.b", torch.stack([bv, bg], 1).reshape(2 * inner))
                self._put(key + ".ff2.w", g(tb + "ff.net.2.weight"), True); self._put(key + ".ff2.b", g(tb + "ff.net.2.bias"))
        # all ResBlock emb_layers as ONE [sum(Cout), 4*mc] matrix: one skinny GEMM per step instead of 22 / 10
        self._put("emb_all.w", torch.cat(emb_w, 0), True); self._put("emb_all.b", torch.cat(emb_b, 0))
        off = 0
        self._emb_off = {}
        for layer in self._res_layers():
            self._emb_off[layer[1]] = off
            off += layer[3]
        self._emb_total = off
        self._load_extra(g)
        if strict:
            missing = [k for k in sd if k.startswith(prefix) and k not in used]
            if missing:
                raise KeyError(f"unexpected keys in state dict: {missing[:5]} ...")
        self._ws = torch.empty(_SPLITK_WS_BYTES // 4, dtype=torch.float32, device=self._device)
        self._loaded = True
        self._fuse_ok.clear()
        # every holder of something derived from these tensors — captured graphs (raw pointers), the stacked copies of
        # B200GroupedTrunk, the timestep-embedding table — compares this counter (B200ControlLDM._weights_epoch)
        self.load_epoch = getattr(self, "load_epoch", 0) + 1
        return self

    def _load_extra(self, g):
        pass

    def _extra_shapes(self):
        return {}

    def upstream_shapes(self) -> dict:
        """{upstream state-dict key: shape} this network expects (what a ControlNet / SD-1.5 checkpoint holds)"""
        mc, ted, cd = self.mc, self.ted, self.context_dim
        out = {"time_embed.0.weight": (ted, mc), "time_embed.0.bias": (ted,),
               "time_embed.2.weight": (ted, ted), "time_embed.2.bias": (ted,)}

        def conv(k, co, ci, r):
            out[k + ".weight"] = (co, ci, r, r)
            out[k + ".bias"] = (co,)

        def norm(k, c):
            out[k + ".weight"] = (c,)
            out[k + ".bias"] = (c,)

        for layer in self._all_layers():
            kind, key = layer[0], layer[1]
            if kind == "conv_in":
                conv(key, layer[3], layer[2], 3)
            elif kind in ("down", "up"):
                conv(key, layer[2], layer[2], 3)
            elif kind == "res":
                cin, cout = layer[2], layer[3]
                norm(key + ".in_layers.0", cin); conv(key + ".in_layers.2", cout, cin, 3)
                out[key + ".emb_layers.1.weight"] = (cout, ted); out[key + ".emb_layers.1.bias"] = (cout,)
                norm(key + ".out_layers.0", cout); conv(key + ".out_layers.3", cout, cout, 3)
                if cin != cout:
                    conv(key + ".skip_connection", cout, cin, 1)
            elif kind == "st":
                c, tb = layer[2], key + ".transformer_blocks.0."
                norm(key + ".norm", c); conv(key + ".proj_in", c, c, 1); conv(key + ".proj_out", c, c, 1)
                for n in ("norm1", "norm2", "norm3"):
                    norm(tb + n, c)
                for a, kd in (("attn1", c), ("attn2", cd)):
                    out[tb + a + ".to_q.weight"] = (c, c)
                    out[tb + a + ".to_k.weight"] = (c, kd)
                    out[tb + a + ".to_v.weight"] = (c, kd)
                    out[tb + a + ".to_out.0.weight"] = (c, c); out[tb + a + ".to_out.0.bias"] = (c,)
                out[tb + "ff.net.0.proj.weight"] = (8 * c, c); out[tb + "ff.net.0.proj.bias"] = (8 * c,)
                out[tb + "ff.net.2.weight"] = (c, 4 * c); out[tb + "ff.net.2.bias"] = (c,)
        out.update(self._extra_shapes())
        return out

    # ---- buffers ---------------------------------------------------------------------------------------------
    def _buf(self, name, rows, cols, dtype=None):
        key = (name, rows, cols, dtype)
        b = self._bufs.get(key)
        if b is None:
            b = torch.empty(rows, cols, dtype=dtype or self.dtype, device=self._device)
            self._bufs[key] = b
        return b

    def _gn_ws(self, N):
        return self._buf("gn_ws", 1, ops.groupnorm_workspace_bytes(N) // 4, torch.float32)

    def _stats_ok(self, N, H, W):
        """fused GroupNorm statistics: bf16 path, whole 128-row tiles per sample (so a tile never spans two samples), and
        power-of-two maps — the only ones the tensor-core 3x3 kernels (which emit the statistics) take; other sizes
        (48 x 48 for 384^2 images, ...) run the generic conv and the two-phase GroupNorm"""
        pow2 = lambda v: v > 0 and v & (v - 1) == 0  # noqa: E731
        return self._hi and self.fused_gn_stats and (H * W) % 128 == 0 and pow2(H) and pow2(W)

    def _stats(self, name, rows, cols):
        key = ("st_" + name, rows, cols)
        b = self._bufs.get(key)
        if b is None:
            b = torch.zeros(rows // 128, cols, 2, dtype=torch.float32, device=self._device)
            self._bufs[key] = b
        return b

    def _gn(self, x, y, N, gamma, beta, eps, silu):
        """x: Act (or (tensor, stats) via Act); GroupNorm(+SiLU) of x into the bf16 operand buffer y"""
        if x.st is not None:
            ops.groupnorm_apply(x.src(), y, N, gamma, beta, eps, silu, x.st, wgroups=self._wg)
        else:
            ops.groupnorm(x.src(), y, N, gamma, beta, eps, silu, self._gn_ws(N), wgroups=self._wg)

    # ---- building blocks ---------------------------------------------------------------------------------------
    def _conv(self, x, wkey, y, N, H, W, R=1, **kw):
        """y: activation-dtype output view or None; kw may carry y32= (fp32 copy), residual=, emb=, act= ..."""
        if kw.get("stride", 1) == 2 or kw.get("upsample"):
            # the library materialises the im2col matrix (stride 2) / the x2-upsampled input in the workspace
            rows = N * (H // 2) * (W // 2) * 9 if kw.get("stride", 1) == 2 else N * 4 * H * W
            self._grow_ws(rows * x.shape[1] * 2 + _SPLITK_WS_BYTES)
        self._launch(x, self.w[wkey + ".w"], y, N=N, H=H, W=W, R=R, S=R, pad=R // 2 if "pad" not in kw else kw.pop("pad"),
                     bias=self.w.get(wkey + ".b"), workspace=self._ws, **kw)

    def _launch(self, x, w, y, **kw):
        if self._wg == 2:
            ops.conv2d_grouped(x, w, y, **kw)
        else:
            ops.conv2d(x, w, y, **kw)

    def _grow_ws(self, need):
        """large batches outgrow the default workspace; a replaced buffer stays alive (captured graphs of other shapes
        still point into it)"""
        if need > self._ws.numel() * 4:
            self._ws_retired = getattr(self, "_ws_retired", []) + [self._ws]
            self._ws = torch.empty(-(-need // 4), dtype=torch.float32, device=self._device)

    def _linear(self, x, wkey, y, **kw):
        self._launch(x, self.w[wkey + ".w"], y, N=self._wg, H=1, W=x.shape[0] // self._wg, bias=self.w.get(wkey + ".b"),
                     workspace=self._ws, **kw)

    def _time_embedding(self, t, B, out=None):
        """emb = time_embed(timestep_embedding(t)); returns silu(emb) @ W_all + b_all for every ResBlock at once
        (into ``out``, a [B, _emb_total] view, when given).  t: int64 timesteps, or fp32 ones (fractional values as they
        are, as upstream's t.float() takes them) — see timesteps_for_embedding."""
        te = self._buf("t_emb", B, self.mc)
        if t.is_floating_point():
            ops.timestep_embedding_f32(t, te)
        else:
            ops.timestep_embedding(t, te)
        e1 = self._buf("te1", B, self.ted)
        self._linear(te, "te0", e1, act=L.ACT_SILU)
        e2 = self._buf("te2", B, self.ted)
        self._linear(e1, "te2", e2, act=L.ACT_SILU)  # every consumer (ResBlock.emb_layers) starts with SiLU: fused here
        ea = self._buf("emb_all", B, self._emb_total) if out is None else out
        self._linear(e2, "emb_all", ea)
        return ea

    @property
    def _hi(self):
        return self.dtype != torch.float32

    def _side(self, name, rows, cols):
        """a non-operand intermediate: fp32 in the bf16 path (returned as (None, buf32)), plain buffer in check mode"""
        if self._hi:
            return None, self._buf(name + "32", rows, cols, torch.float32)
        return self._buf(name, rows, cols), None

    def _act(self, name, rows, cols, lo=True, hi=True):
        """allocate an Act with the requested forms (check mode: always just lo)"""
        if not self._hi:
            return Act(self._buf(name, rows, cols))
        return Act(self._buf(name, rows, cols) if lo else None,
                   self._buf(name + "32", rows, cols, torch.float32) if hi else None)

    def _res(self, layer, x, y, emb_all, N, H, W):
        """x, y: Act.  h and the skip projection never feed a tensor core directly -> fp32 side buffers."""
        _, key, cin, cout = layer
        M = N * H * W
        t1 = self._buf("gn_a", M, cin)
        self._gn(x, t1, N, self.w[key + ".gn1.g"], self.w[key + ".gn1.b"], 1e-5, True)
        h_lo, h_hi = self._side("res_h", M, cout)
        h_st = self._stats("res_h", M, cout) if self._stats_ok(N, H, W) else None
        e = emb_all[:, self._emb_off[key]:self._emb_off[key] + cout]
        t2 = self._buf("gn_b", M, cout)
        gn2 = dict(y=t2, gamma=self.w[key + ".gn2.g"], beta=self.w[key + ".gn2.b"], eps=1e-5, silu=True)
        if h_st is None and self._gn_tail_ok(key + ".c1", t1, h_lo, h_hi, e, N, H, W, gn2):
            # deep levels: conv1 runs as split-K partials + reducer, and the reducer normalises what it has just summed — out_layers'
            # GroupNorm + SiLU without a launch of its own (mkd_conv_desc.gn_y)
            self._conv(t1, key + ".c1", h_lo, N, H, W, R=3, emb=e, y32=h_hi, gn=gn2)
        else:
            self._conv(t1, key + ".c1", h_lo, N, H, W, R=3, emb=e, y32=h_hi, stats=h_st)
            self._gn(Act(h_lo, h_hi, h_st), t2, N, gn2["gamma"], gn2["beta"], 1e-5, True)
        if cin != cout and self._skip_fuses(key, t2, x.lo, y, N, H, W):
            # h = conv2(...) + skip_connection(x): the 1x1 projection rides as extra k-blocks of the 3x3 conv's GEMM
            self._conv(t2, key + ".c2sk", y.lo, N, H, W, R=3, x2=x.lo, y32=y.hi, stats=y.st)
            return
        if cin != cout:
            s_lo, s_hi = self._side("res_sk", M, cout)
            self._conv(x.lo, key + ".sk", s_lo, N, H, W, R=1, y32=s_hi)
            sk = s_hi if s_hi is not None else s_lo
        else:
            sk = x.src()
        self._conv(t2, key + ".c2", y.lo, N, H, W, R=3, residual=sk, y32=y.hi, stats=y.st)

    def _gn_tail_ok(self, wkey, x, y_lo, y_hi, emb, N, H, W, gn):
        """does this conv take the GroupNorm that follows it as a tail of its split-K reducer?  (bf16 path, launches the library
        runs as split-K: the 8x8 / 4x4 levels at small batch; asked once per (layer, shape))"""
        if not (self._hi and self.fuse_gn_tail):
            return False
        ck = ("gn_tail", wkey, N, H, W, y_lo is None, y_hi is None)
        ok = self._fuse_ok.get(ck)
        if ok is None:
            w, b = self.w[wkey + ".w"], self.w.get(wkey + ".b")
            kw = dict(H=H, W=W, R=3, S=3, pad=1, workspace=self._ws)
            ok = ops.conv2d_supported(x, w, y_lo, N=N, bias=b, emb=emb, y32=y_hi, gn=gn, wgroups=self._wg, **kw)
            # (stacked trunk: only as ONE grouped launch — where that does not split K, two split-K launches per network with tails
            #  would replace one grouped launch + one GroupNorm launch: measured slower at the 8x8 level)
            self._fuse_ok[ck] = ok
        return ok

    def _skip_fuses(self, key, t2, x_lo, y, N, H, W):
        """can this ResBlock's out conv take its skip projection as a second term?  (bf16 path, CTA-pair kernel shapes;
        asked once per (layer, shape))"""
        if not (self._hi and self.fuse_skip and x_lo is not None and key + ".c2sk.w" in self.w):
            return False
        ck = (key, N, H, W, y.lo is None, y.hi is None, y.st is None)
        ok = self._fuse_ok.get(ck)
        if ok is None:
            w, b = self.w[key + ".c2sk.w"], self.w[key + ".c2sk.b"]
            ok = ops.conv2d_supported(t2, w, y.lo, N=N, H=H, W=W, R=3, S=3, pad=1, x2=x_lo, bias=b, workspace=self._ws,
                                      y32=y.hi, stats=y.st, wgroups=self._wg)
            if not ok and self._wg == 2:
                # the grouped launch is declined (parts that are not whole tile pairs): ops.conv2d_grouped then issues one launch
                # per network, each of which may still take the second term
                half = lambda v: None if v is None else v[:v.shape[0] // 2]  # noqa: E731
                ok = ops.conv2d_supported(half(t2), half(w), half(y.lo), N=N // 2, H=H, W=W, R=3, S=3, pad=1, x2=half(x_lo),
                                          bias=half(b), workspace=self._ws, y32=half(y.hi), stats=half(y.st))
            self._fuse_ok[ck] = ok
        return ok

    def _st(self, layer, x, y, ctx_kv, N, H, W):
        """x, y: Act.  The token stream xs (x += attn1, += attn2, += ff) lives in fp32 until its last update, which
        writes the bf16 operand of proj_out directly."""
        _, key, ch = layer
        M, hd = N * H * W, ch // self.heads
        scale = hd ** -0.5
        n = self._buf("st_n", M, ch)
        self._gn(x, n, N, self.w[key + ".gn.g"], self.w[key + ".gn.b"], 1e-6, False)
        x_lo, x_hi = self._side("st_x", M, ch)
        xs = x_hi if x_hi is not None else x_lo           # the stream every LN / residual reads
        o_lo, o_hi = (None, xs) if self._hi else (xs, None)  # how an in-place update of xs is written
        self._conv(n, key + ".pi", o_lo, N, H, W, R=1, y32=o_hi)
        ln = self._buf("st_ln", M, ch)
        # self-attention
        ops.layernorm(xs, ln, self.w[key + ".norm1.g"], self.w[key + ".norm1.b"], wgroups=self._wg)
        qkv = self._buf("st_qkv", M, 3 * ch)
        self._linear(ln, key + ".qkv", qkv)
        att = self._buf("st_att", M, ch)
        ops.attention(qkv[:, :ch], qkv[:, ch:2 * ch], qkv[:, 2 * ch:], att, B=N, heads=self.heads, Nq=H * W, Nkv=H * W,
                      d=hd, scale=scale)
        self._linear(att, key + ".o1", o_lo, residual=xs, y32=o_hi)
        # cross-attention (K/V of the step-invariant context are precomputed: ctx_kv[key] = [N*L, 2*ch])
        ops.layernorm(xs, ln, self.w[key + ".norm2.g"], self.w[key + ".norm2.b"], wgroups=self._wg)
        q2 = self._buf("st_q2", M, ch)
        self._linear(ln, key + ".q2", q2)
        kv = ctx_kv[key]
        Lc = kv.shape[0] // N
        ops.attention(q2, kv[:, :ch], kv[:, ch:], att, B=N, heads=self.heads, Nq=H * W, Nkv=Lc, d=hd, scale=scale)
        self._linear(att, key + ".o2", o_lo, residual=xs, y32=o_hi)
        # GEGLU feed-forward (gate fused into the first GEMM's epilogue)
        ops.layernorm(xs, ln, self.w[key + ".norm3.g"], self.w[key + ".norm3.b"], wgroups=self._wg)
        inner = 4 * ch
        ff = self._buf("st_ff", M, inner)
        self._linear(ln, key + ".ff1", ff, act=L.ACT_GEGLU, geglu_block=_geglu_block(inner))
        xa = self._buf("st_xa", M, ch) if self._hi else xs  # proj_out's A operand (activation dtype)
        self._linear(ff, key + ".ff2", xa, residual=xs)
        self._conv(xa, key + ".po", y.lo, N, H, W, R=1, residual=x.src(), y32=y.hi, stats=y.st)

    def context_kv(self, context):
        """attn2 K/V projections of the (step-invariant) text context for every SpatialTransformer: hoisted out of
        the 50-step loop (SURVEY.md §7 hard part 7).  context: [B, L, context_dim] fp32/bf16."""
        B, Lc, D = context.shape
        self.arena_epoch += 1
        ctx = self._buf("ctx", B * Lc, D)
        ctx.copy_(context.reshape(B * Lc, D))
        out = {}
        for layer in self._all_layers():
            if layer[0] == "st":
                kv = self._buf("kv_" + layer[1], B * Lc, 2 * layer[2])
                self._linear(ctx, layer[1] + ".kv2", kv)
                out[layer[1]] = kv
        return out

    def _x_in(self, x):
        """the latent x_t as conv_in's NHWC operand: [B*H*W, 64] with zero pad channels (bf16 path) or [.., 4] (check mode)"""
        if not self._hi:
            return self._to_nhwc(x, "x_in")
        B, Cc, H, W = x.shape
        key = ("x_in_p", B * H * W, 64)
        if key not in self._bufs:
            self._bufs[key] = torch.zeros(B * H * W, 64, dtype=self.dtype, device=self._device)  # pad columns stay 0
        buf = self._bufs[key]
        ops.nchw_to_nhwc(x.float().contiguous(), buf[:, :Cc])
        return buf

    def _to_nhwc(self, x, name):
        B, Cc, H, W = x.shape
        buf = self._buf(name, B * H * W, (Cc + 7) // 8 * 8)
        v = buf[:, :Cc]
        ops.nchw_to_nhwc(x.float().contiguous(), v)
        return v

    @staticmethod
    def _needs(layer):
        """(lo, hi) forms a layer reads of its input: A operands want lo, norms / identity residuals want hi"""
        kind = layer[0]
        if kind == "res":
            return layer[2] != layer[3], True
        if kind == "st":
            return False, True
        return True, False  # down / up / conv: tensor-core operand only

    def _run_block(self, layers, x, y, emb_all, ctx_kv, N, H, W, conv_in_residual=None):
        """runs a block's layers x -> y (Acts) through ping-pong temporaries; returns the output spatial size"""
        cur = x
        for li, layer in enumerate(layers):
            last = li == len(layers) - 1
            kind = layer[0]
            if not last:
                lo, hi = self._needs(layers[li + 1])
                cout = layer[3] if kind == "res" else layer[2]
                out = self._act(f"pp{li % 2}", N * H * W, cout, lo=lo, hi=hi)
                if hi and kind != "up" and self._stats_ok(N, H, W):  # the next layer starts with a GroupNorm
                    out.st = self._stats(f"pp{li % 2}", N * H * W, cout)
            else:
                out = y
            if kind == "conv_in":
                pow2 = H & (H - 1) == 0 and W & (W - 1) == 0
                if not (self._hi and pow2):
                    out.st = None  # the generic kernel (check mode / odd sizes) emits no statistics
                self._conv(cur.lo, layer[1], out.lo, N, H, W, R=3, residual=conv_in_residual, y32=out.hi, stats=out.st)
            elif kind == "res":
                self._res(layer, cur, out, emb_all, N, H, W)
            elif kind == "st":
                self._st(layer, cur, out, ctx_kv, N, H, W)
            elif kind == "down":
                self._conv(cur.lo, layer[1], out.lo, N, H, W, R=3, stride=2, y32=out.hi, stats=out.st)
                H, W = H // 2, W // 2
            elif kind == "up":
                assert last
                self._conv(cur.lo, layer[1], out.lo, N, H, W, R=3, upsample=True, y32=out.hi, stats=out.st)
                H, W = 2 * H, 2 * W
            cur = out
        return H, W

    def _next_needs_hi(self, j):
        """does the consumer of input block j's output (block j+1, or the middle block) read the fp32 form?"""
        nxt = self.input_blocks[j + 1][0] if j + 1 < len(self.input_blocks) else self.middle[0]
        return self._needs(nxt)[1]


class B200ControlNet(_Net):
    """Drop-in for ``cldm.cldm.ControlNet`` (yaml:52-67)."""

    HINT = ((16, 1), (16, 1), (32, 2), (32, 1), (96, 2), (96, 1), (256, 2))

    def __init__(self, image_size=32, in_channels=4, hint_channels=6, model_channels=320, attention_resolutions=(4, 2, 1),
                 num_res_blocks=2, channel_mult=(1, 2, 4, 4), num_heads=8, use_spatial_transformer=True,
                 transformer_depth=1, context_dim=768, use_checkpoint=False, legacy=False, dtype=torch.bfloat16, **kw):
        super().__init__(in_channels, model_channels, attention_resolutions, num_res_blocks, channel_mult, num_heads,
                         transformer_depth, context_dim, dtype)
        self.hint_channels = hint_channels

    def _load_extra(self, g):
        for i in range(8):
            k = f"input_hint_block.{2 * i}"
            w, b = self._krsc(g(k + ".weight")), g(k + ".bias")
            self._put(k + ".w", w, True); self._put(k + ".b", b)
            if self._hi:
                # bf16 path: the hint block's channel counts (6, 16, 32, 96, 256) are zero-padded to multiples of 64
                # so that every conv of it runs on the tcgen05 kernel (which wants C % 64 == 0) instead of the
                # CUDA-core kernel: padded input channels meet zero weights, padded output channels have zero
                # weights and bias, and SiLU(0) = 0 keeps them zero for the next layer.
                co, _, _, ci = w.shape
                cop, cip = -(-co // 64) * 64, -(-ci // 64) * 64
                wp = torch.zeros(cop, 3, 3, cip, dtype=w.dtype)
                wp[:co, :, :, :ci] = w
                bp = torch.zeros(cop, dtype=b.dtype)
                bp[:co] = b
                self._put(k + ".wp", wp, True); self._put(k + ".bp", bp)
        for j in range(len(self.input_blocks)):
            k = f"zero_convs.{j}.0"
            self._put(k + ".w", self._krsc(g(k + ".weight")), True); self._put(k + ".b", g(k + ".bias"))
        k = "middle_block_out.0"
        self._put(k + ".w", self._krsc(g(k + ".weight")), True); self._put(k + ".b", g(k + ".bias"))

    def _extra_shapes(self):
        out, cin = {}, self.hint_channels
        for i, co in enumerate([c for c, _ in self.HINT] + [self.mc]):
            out[f"input_hint_block.{2 * i}.weight"] = (co, cin, 3, 3)
            out[f"input_hint_block.{2 * i}.bias"] = (co,)
            cin = co
        for j, c in enumerate(self.block_chans):
            out[f"zero_convs.{j}.0.weight"] = (c, c, 1, 1)
            out[f"zero_convs.{j}.0.bias"] = (c,)
        out["middle_block_out.0.weight"] = (self._ch, self._ch, 1, 1)
        out["middle_block_out.0.bias"] = (self._ch,)
        return out

    def hint_features(self, hint):
        """input_hint_block(hint): independent of x and t, so computed once per batch of images, not once per step.
        hint: [B, 6, 8h, 8w] fp32 in [0,1] = cat(source, reference) (makeup_diffuse.py:56).  Returns [B*h*w, mc]."""
        B, Cc, H, W = hint.shape
        self.arena_epoch += 1
        chans = [c for c, _ in self.HINT] + [self.mc]
        strides = [s for _, s in self.HINT] + [1]
        pow2 = lambda v: v > 0 and v & (v - 1) == 0  # noqa: E731
        if self._hi and pow2(H) and pow2(W) and H >= 8 and W >= 8:
            return self._hint_features_padded(hint, chans, strides)
        cur = self._to_nhwc(hint, "hint_in")
        for i, (co, s) in enumerate(zip(chans, strides)):
            Ho, Wo = (H + 2 - 3) // s + 1, (W + 2 - 3) // s + 1
            out = self._buf(f"hint_{i}", B * Ho * Wo, co)
            self._conv(cur, f"input_hint_block.{2 * i}", out, B, H, W, R=3, stride=s,
                       act=L.ACT_SILU if i < 7 else L.ACT_NONE)
            cur, H, W = out, Ho, Wo
        return cur

    def _hint_features_padded(self, hint, chans, strides):
        """the hint block on the tensor cores: channel-padded buffers / weights (see _load_extra)"""
        B, Cc, H, W = hint.shape
        pad = lambda c: -(-c // 64) * 64  # noqa: E731
        key = ("hint_in_p", B * H * W, pad(Cc))
        if key not in self._bufs:
            self._bufs[key] = torch.zeros(B * H * W, pad(Cc), dtype=self.dtype, device=self._device)  # pad columns stay 0
        cur = self._bufs[key]
        ops.nchw_to_nhwc(hint.float().contiguous(), cur[:, :Cc])
        for i, (co, s) in enumerate(zip(chans, strides)):
            Ho, Wo = H // s, W // s
            out = self._buf(f"hint_p{i}", B * Ho * Wo, pad(co))
            ws = self._ws
            if s == 2:  # the stride-2 convs run as im2col + GEMM: the im2col matrix lives in the workspace
                need = B * Ho * Wo * 9 * cur.shape[1] * 2 + (2 << 20)
                ws = self._buf("hint_ws", 1, -(-need // 4), torch.float32) if need > self._ws.numel() * 4 else self._ws
            k = f"input_hint_block.{2 * i}"
            ops.conv2d(cur, self.w[k + ".wp"], out, N=B, H=H, W=W, R=3, S=3, stride=s, pad=1, bias=self.w[k + ".bp"],
                       workspace=ws, act=L.ACT_SILU if i < 7 else L.ACT_NONE)
            cur, H, W = out, Ho, Wo
        return cur[:, :self.mc]

    def run_trunk(self, x_nhwc, guided_hint, t, ctx_kv, N, H, W, emb=None):
        """time embedding + input blocks + middle block.  Returns the 13 pending zero-conv calls
        [(weight key, input view, index, h, w)]: the trunk touches no UNet buffer, so it can run on a second stream
        concurrently with the UNet encoder; the zero-convs (which may inject into UNet skip slots) come after the join.
        emb: the ResBlock embeddings [N, _emb_total] when the caller already holds them (B200ControlLDM.set_step)."""
        emb_all = self._time_embedding(t, N) if emb is None else emb
        pending = []
        cur, h, w = Act(x_nhwc), H, W
        for j, blk in enumerate(self.input_blocks):
            ch = self.block_chans[j]
            ho, wo = (h // 2, w // 2) if blk[0][0] == "down" else (h, w)
            y = self._act(f"cn_h{j}", N * ho * wo, ch, lo=True, hi=self._next_needs_hi(j))
            if self._next_needs_hi(j) and self._stats_ok(N, ho, wo):
                y.st = self._stats(f"cn_h{j}", N * ho * wo, ch)
            # h = input_blocks[0](x) + guided_hint: the add rides in conv_in's epilogue
            self._run_block(blk, cur, y, emb_all, ctx_kv, N, h, w, conv_in_residual=guided_hint if j == 0 else None)
            cur, h, w = y, ho, wo
            pending.append((f"zero_convs.{j}.0", cur.lo, j, h, w))
        y = self._act("cn_mid", N * h * w, self._ch, lo=True, hi=False)
        self._run_block(self.middle, cur, y, emb_all, ctx_kv, N, h, w)
        pending.append(("middle_block_out.0", y.lo, len(self.input_blocks), h, w))
        return pending

    def zero_convs(self, pending, N, inject=None, scales=None, inject_st=None):
        """the 13 zero-convs: into own buffers (inject None), or accumulated as scale_i * zero_conv_i(h) straight into
        the UNet's skip slots / middle output (makeup_diffuse.py:166 + upstream `hs.pop() + control.pop()`).
        inject_st[j]: statistics view of slot j — the injecting epilogue re-emits the GroupNorm partials of the
        values it leaves in the slot (the decoder's GroupNorm reads those)."""
        return [self._zero_conv(key, x, j, N, h, w, inject, scales, None if inject_st is None else inject_st[j])
                for key, x, j, h, w in pending]

    def run(self, x_nhwc, guided_hint, t, ctx_kv, N, H, W, inject=None, scales=None):
        return self.zero_convs(self.run_trunk(x_nhwc, guided_hint, t, ctx_kv, N, H, W), N, inject, scales)

    def _zero_conv(self, key, x, j, N, h, w, inject, scales, st=None):
        ch = x.shape[1]
        if inject is None:
            out = self._buf(f"cn_out{j}", N * h * w, ch)
            self._conv(x, key, out, N, h, w, R=1)
            return (out, h, w)
        if inject[j] is not None:
            self._conv(x, key, inject[j], N, h, w, R=1, residual=inject[j], alpha=1.0 if scales is None else scales[j],
                       stats=st)
        return None

    def forward(self, x, hint, timesteps, context, **kwargs):
        """Reference call form (makeup_diffuse.py:164): returns the 13 control residuals as NCHW fp32 tensors."""
        assert self._loaded, "load_state_dict() first"
        N, _, H, W = x.shape
        xin = self._x_in(x)
        outs = self.run(xin, self.hint_features(hint), timesteps_for_embedding(timesteps), self.context_kv(context), N, H, W)
        res = []
        for o, h, w in outs:
            t = torch.empty(N, o.shape[1], h, w, dtype=torch.float32, device=o.device)
            ops.nhwc_to_nchw(o, t)
            res.append(t)
        return res


class B200ControlledUnet(_Net):
    """Drop-in for ``cldm.cldm.ControlledUnetModel`` (yaml:69-84)."""

    def __init__(self, image_size=32, in_channels=4, out_channels=4, model_channels=320, attention_resolutions=(4, 2, 1),
                 num_res_blocks=2, channel_mult=(1, 2, 4, 4), num_heads=8, use_spatial_transformer=True,
                 transformer_depth=1, context_dim=768, use_checkpoint=False, legacy=False, dtype=torch.bfloat16, **kw):
        super().__init__(in_channels, model_channels, attention_resolutions, num_res_blocks, channel_mult, num_heads,
                         transformer_depth, context_dim, dtype)
        self.out_channels = out_channels
        mc, ch, ds = model_channels, self._ch, self._ds
        chans = list(self.block_chans)
        self.output_blocks, self.cat_split = [], []
        for level, mult in list(enumerate(channel_mult))[::-1]:
            for i in range(num_res_blocks + 1):
                ich = chans.pop()
                k = len(self.output_blocks)
                layers = [("res", f"output_blocks.{k}.0", ch + ich, mc * mult)]
                self.cat_split.append((ch, ich))
                ch = mc * mult
                if ds in self._attn_res:
                    layers.append(("st", f"output_blocks.{k}.1", ch))
                if level and i == num_res_blocks:
                    layers.append(("up", f"output_blocks.{k}.{len(layers)}.conv", ch))
                    ds //= 2
                self.output_blocks.append(layers)
        self._out_ch = ch

    def _all_layers(self):
        yield from super()._all_layers()
        for blk in self.output_blocks:
            yield from blk

    def _extra_shapes(self):
        return {"out.0.weight": (self._out_ch,), "out.0.bias": (self._out_ch,),
                "out.2.weight": (self.out_channels, self._out_ch, 3, 3), "out.2.bias": (self.out_channels,)}

    def _load_extra(self, g):
        self._put("out.gn.g", g("out.0.weight")); self._put("out.gn.b", g("out.0.bias"))
        self._put("out.2.w", self._krsc(g("out.2.weight")), True); self._put("out.2.b", g("out.2.bias"))

    # the decoder's concat buffers: cat_i = [ h (C_h) | hs[11-i] (C_skip) ]
    # row_groups = 2 (set by B200GroupedTrunk): every concat buffer (and its statistics) is allocated with twice the rows.
    # The decoder and the reference call forms use the first half as before; the grouped trunk writes the stacked
    # (UNet | ControlNet) block outputs through the full-height views (full=True), so the UNet half lands in its slot with
    # no copy and the ControlNet half sits below it, where its zero-conv reads it.
    row_groups = 1

    def _cat(self, i, N, H, W, full=False):
        nb = len(self.input_blocks)
        ds = self.block_ds[nb - 1 - i]
        ch, ich = self.cat_split[i]
        rows = N * (H // ds) * (W // ds)
        buf = self._buf(f"cat{i}", self.row_groups * rows, ch + ich)
        return (buf if full else buf[:rows]), ch, ds

    def skip_slots(self, N, H, W, full=False):
        """views the 12 encoder outputs live in + the view of the middle-block output (13 injection targets,
        ordered like ControlNet's outputs)"""
        nb = len(self.input_blocks)
        slots = []
        for j in range(nb):
            cat, ch, _ = self._cat(nb - 1 - j, N, H, W, full)
            slots.append(cat[:, ch:])
        cat0, ch0, _ = self._cat(0, N, H, W, full)
        slots.append(cat0[:, :ch0])
        return slots

    def _cat_stats(self, i, N, H, W, full=False):
        """GroupNorm statistics of concat buffer i ([tiles, C_h + C_skip, 2]) or None when the level has no whole tiles"""
        cat, _, ds = self._cat(i, N, H, W)
        if not self._stats_ok(N, H // ds, W // ds):
            return None
        st = self._stats(f"cat{i}", self.row_groups * cat.shape[0], cat.shape[1])
        return st if full else st[:cat.shape[0] // 128]

    def skip_slot_stats(self, N, H, W, full=False):
        """statistics views matching skip_slots(): the channel slice of the concat statistics each slot owns"""
        nb = len(self.input_blocks)
        out = []
        for j in range(nb):
            st = self._cat_stats(nb - 1 - j, N, H, W, full)
            out.append(None if st is None else st[:, self.cat_split[nb - 1 - j][0]:, :])
        st0 = self._cat_stats(0, N, H, W, full)
        out.append(None if st0 is None else st0[:, :self.cat_split[0][0], :])
        return out

    def note_slots_rewritten(self, js, with_stats):
        """slots js were updated after encode(): by injecting epilogues that re-emitted their statistics (True) or by
        a plain add (False, the reference call form with an explicit `control` list)"""
        for j in js:
            self._slot_ok[j] = bool(with_stats) and self._slot_st[j] is not None

    def encode(self, x_nhwc, t, ctx_kv, N, H, W, emb=None):
        self._emb_cur = self._time_embedding(t, N) if emb is None else emb
        slots = self.skip_slots(N, H, W)
        self._slot_st = self.skip_slot_stats(N, H, W)
        self._slot_ok = [False] * len(slots)
        cur, h, w = Act(x_nhwc), H, W
        for j, blk in enumerate(self.input_blocks):
            # bf16 copy straight into the decoder's concat slot; fp32 copy for the next block's norm / identity skip
            y = Act(slots[j], self._buf(f"enc{j}_32", slots[j].shape[0], slots[j].shape[1], torch.float32)
                    if self._hi and self._next_needs_hi(j) else None, self._slot_st[j])
            h, w = self._run_block(blk, cur, y, self._emb_cur, ctx_kv, N, h, w)
            self._slot_ok[j] = y.st is not None
            cur = y
        y = Act(slots[-1], None, self._slot_st[-1])
        self._run_block(self.middle, cur, y, self._emb_cur, ctx_kv, N, h, w)
        self._slot_ok[-1] = y.st is not None
        return slots

    def decode(self, ctx_kv, N, H, W, before_block=None):
        """before_block(i): optional hook run before output block i is enqueued (stream waits on pending injections)"""
        nb = len(self.output_blocks)
        nslots = len(self.input_blocks)
        h_ok = self._slot_ok[nslots]  # statistics of the h half of concat 0 (= the middle-block output)
        for i, blk in enumerate(self.output_blocks):
            if before_block is not None:
                before_block(i)
            cat, _, ds = self._cat(i, N, H, W)
            cat_st = self._cat_stats(i, N, H, W)
            if not (h_ok and self._slot_ok[nslots - 1 - i]):
                cat_st = None  # some part of the concat was not produced with statistics: full GroupNorm kernel
            if i + 1 < nb:
                nxt, nch, _ = self._cat(i + 1, N, H, W)
                nst = self._cat_stats(i + 1, N, H, W)
                y = Act(nxt[:, :nch], None, None if nst is None else nst[:, :nch, :])
            else:
                y = self._act("dec_out", N * H * W, self._out_ch, lo=False, hi=True)  # only the out GroupNorm reads it
                if self._stats_ok(N, H, W):
                    y.st = self._stats("dec_out", N * H * W, self._out_ch)
            self._run_block(blk, Act(cat, None, cat_st), y, self._emb_cur, ctx_kv, N, H // ds, W // ds)
            h_ok = y.st is not None
        M = N * H * W
        g = self._buf("gn_a", M, self._out_ch)
        self._gn(y, g, N, self.w["out.gn.g"], self.w["out.gn.b"], 1e-5, True)
        eo = self._buf("eps_nhwc", M, 8)
        self._conv(g, "out.2", eo[:, :self.out_channels], N, H, W, R=3)
        return eo[:, :self.out_channels]

    def forward(self, x, timesteps=None, context=None, control=None, only_mid_control=False, **kwargs):
        """Reference call form (makeup_diffuse.py:161-168). ``control``: list of 13 NCHW tensors or None."""
        assert self._loaded, "load_state_dict() first"
        N, _, H, W = x.shape
        ctx_kv = self.context_kv(context)
        xin = self._x_in(x)
        slots = self.encode(xin, timesteps_for_embedding(timesteps), ctx_kv, N, H, W)
        if control is not None:
            idx = [len(slots) - 1] if only_mid_control else range(len(slots))
            for j in idx:
                c = self._to_nhwc(control[j], f"ctl_in{j}")
                ops.add(slots[j], c, slots[j])
            self.note_slots_rewritten(idx, with_stats=False)
        e = self.decode(ctx_kv, N, H, W)
        out = torch.empty(N, self.out_channels, H, W, dtype=torch.float32, device=e.device)
        ops.nhwc_to_nchw(e, out)
        return out


class B200GroupedTrunk(_Net):
    """``input_blocks`` + ``middle_block`` of the UNet AND of its ControlNet copy as ONE network over a stacked batch.

    The ControlNet trunk is a structural copy of the UNet encoder (upstream cldm.py: same blocks, own weights), and both read the
    same (x_t, t, context): ``apply_model`` (makeup_diffuse.py:164-168) evaluates the same layer shapes twice per step.  Here every
    layer is launched once with ``mkd_conv_desc.wgroups = 2`` / ``wgroups`` of the norm kernels: rows [0, M) of each activation
    belong to the UNet, rows [M, 2M) to the ControlNet; each weight tensor holds the UNet's rows followed by the ControlNet's.
    Twice the work units per launch at the under-filled 16x16 / 8x8 / 4x4 levels, half the trunk's launches.  Shapes the grouped
    kernel declines run as one launch per network on the row halves (ops.conv2d_grouped), so results never depend on the path.

    Outputs: block j of the stacked trunk writes through the full-height view of the decoder's concat slot j
    (B200ControlledUnet.row_groups = 2): the UNet half IS ``hs[j]`` in place, the ControlNet half below it is what
    ``zero_convs.j`` reads."""

    def __init__(self, un: "B200ControlledUnet", cn: "B200ControlNet"):
        super().__init__(un.in_channels, un.mc, un._attn_res, un._nrb, un._channel_mult, un.heads, 1, un.context_dim, un.dtype)
        assert un._loaded and cn._loaded and self.block_chans == cn.block_chans == un.block_chans[:len(self.block_chans)]
        self.un, self.cn = un, cn
        self._device = un._device
        self._wg = 2
        for k, wc in cn.w.items():
            if k.startswith(("input_blocks.", "middle_block.")):
                wu = un.w[k]
                assert wu.shape == wc.shape and wu.dtype == wc.dtype, k
                self.w[k] = torch.cat([wu, wc], 0)
        self._emb_off = {l[1]: cn._emb_off[l[1]] for l in self._res_layers()}
        assert all(un._emb_off[k] == o for k, o in self._emb_off.items())
        self._emb_total = un._emb_total
        self._ws = torch.empty(_SPLITK_WS_BYTES // 4, dtype=torch.float32, device=self._device)
        un.row_groups = 2
        self.fused_gn_stats, self.fuse_skip, self.fuse_gn_tail = un.fused_gn_stats, un.fuse_skip, un.fuse_gn_tail
        self._loaded = True

    def stack_x(self, x):
        """x_t twice: conv_in's stacked NHWC operand (both networks read the same latent)"""
        B, Cc, H, W = x.shape
        M = B * H * W
        cols = 64 if self._hi else (Cc + 7) // 8 * 8
        key = ("x_in2", 2 * M, cols)
        if key not in self._bufs:
            self._bufs[key] = torch.zeros(2 * M, cols, dtype=self.dtype, device=self._device)  # pad columns stay 0
        buf = self._bufs[key]
        xf = x.float().contiguous()
        ops.nchw_to_nhwc(xf, buf[:M, :Cc])
        ops.nchw_to_nhwc(xf, buf[M:, :Cc])
        return buf if self._hi else buf[:, :Cc]

    def stack_cond(self, kv_un, kv_cn, hint):
        """per-cond (step-invariant) operands in stacked form: cross-attention K/V of both networks, and the residual of the
        stacked conv_in — zeros for the UNet rows, ``input_hint_block(hint)`` for the ControlNet rows (cldm.py: h += guided_hint)"""
        kv2 = {}
        for key, kc in kv_cn.items():
            ku = kv_un[key]
            b = self._buf("kv2_" + key, 2 * ku.shape[0], ku.shape[1])
            b[:ku.shape[0]].copy_(ku)
            b[ku.shape[0]:].copy_(kc)
            kv2[key] = b
        h2 = self._buf("hint2", 2 * hint.shape[0], hint.shape[1])
        h2[:hint.shape[0]].zero_()
        h2[hint.shape[0]:].copy_(hint)
        return kv2, h2

    def run(self, x, hint2, t, kv2, N, H, W, side=None, emb2=None):
        """both trunks; leaves the UNet ready for decode() (skip slots, statistics flags, time embedding) and returns
        (slots, the ControlNet's 13 pending zero-conv calls) like encode() + run_trunk() did.
        side: optional second stream — the two time-embedding MLPs (eight skinny launches that depend on t only) run there
        while this stream lays out x_t and runs the stacked conv_in; the first ResBlock waits for them.
        emb2: the stacked embeddings [2N, un._emb_total] when the caller already holds them (B200ControlLDM.set_step)."""
        un, cn = self.un, self.cn
        self.fused_gn_stats, self.fuse_skip, self.fuse_gn_tail = un.fused_gn_stats, un.fuse_skip, un.fuse_gn_tail  # A/B switches follow the UNet's
        ea2 = self._buf("emb_all2", 2 * N, un._emb_total) if emb2 is None else emb2
        emb_done = None
        if emb2 is not None:
            pass
        elif side is not None:
            main = torch.cuda.current_stream()
            fork, emb_done = torch.cuda.Event(), torch.cuda.Event()
            fork.record(main)
            side.wait_event(fork)
            with torch.cuda.stream(side):
                un._time_embedding(t, N, out=ea2[:N])
                cn._time_embedding(t, N, out=ea2[N:, :cn._emb_total])
                emb_done.record(side)
        else:
            un._time_embedding(t, N, out=ea2[:N])
            cn._time_embedding(t, N, out=ea2[N:, :cn._emb_total])
        un._emb_cur = ea2[:N]
        slots, slots2 = un.skip_slots(N, H, W), un.skip_slots(N, H, W, full=True)
        un._slot_st, st2 = un.skip_slot_stats(N, H, W), un.skip_slot_stats(N, H, W, full=True)
        un._slot_ok = [False] * len(slots)
        pending = []
        cur, h, w = Act(self.stack_x(x)), H, W
        for j, blk in enumerate(self.input_blocks):
            hi = self._buf(f"enc{j}_32", slots2[j].shape[0], slots2[j].shape[1], torch.float32) \
                if self._hi and self._next_needs_hi(j) else None
            y = Act(slots2[j], hi, st2[j])
            h, w = self._run_block(blk, cur, y, ea2, kv2, 2 * N, h, w, conv_in_residual=hint2 if j == 0 else None)
            un._slot_ok[j] = y.st is not None
            pending.append((f"zero_convs.{j}.0", slots2[j][slots[j].shape[0]:], j, h, w))
            cur = y
            if j == 0 and emb_done is not None:
                main.wait_event(emb_done)  # block 0 is conv_in alone: every later block reads the embeddings
        y = Act(slots2[-1], None, st2[-1])
        self._run_block(self.middle, cur, y, ea2, kv2, 2 * N, h, w)
        un._slot_ok[-1] = y.st is not None
        pending.append(("middle_block_out.0", slots2[-1][slots[-1].shape[0]:], len(self.input_blocks), h, w))
        return slots, pending
