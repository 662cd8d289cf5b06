"""``B200ControlLDM``: the object the sampler holds as ``self.model`` (SURVEY.md §8(b) levels B1/B2).

It exposes exactly what ``diffmk/cddim.py`` reads off the model — ``apply_model``, ``parameterization``,
``alphas_cumprod``, ``alphas_cumprod_prev``, ``sqrt_one_minus_alphas_cumprod``, ``num_timesteps``, ``betas``,
``device`` — plus ``control_model`` / ``model.diffusion_model`` / ``control_scales`` / ``only_mid_control`` with the
reference's names, so ``apply_model(x_noisy, t, cond)`` keeps the signature and semantics of
``diffmk/makeup_diffuse.py:152-170``.

What differs is the execution order inside ``apply_model`` (results are identical): UNet encoder first, then the
ControlNet whose zero-conv epilogues add ``scale_i * residual_i`` into the encoder skip slots, then the UNet decoder.
Step-invariant work is hoisted and cached per ``cond``: the hint block (independent of x and t, identical for both CFG
halves because ``uc_cat = c_cat``, diffusion_makeup.py:401) and every cross-attention K/V projection.
"""
from __future__ import annotations

import numpy as np
import torch

from . import ops
from .nets import B200ControlNet, B200ControlledUnet, B200GroupedTrunk, timesteps_for_embedding


class _Wrapper:
    def __init__(self, unet):
        self.diffusion_model = unet


class B200ControlLDM:
    def __init__(self, control_params=None, unet_params=None, timesteps=1000, linear_start=0.00085,
                 linear_end=0.0120, parameterization="eps", only_mid_control=False, scale_factor=0.18215,
                 dtype=torch.bfloat16, device="cuda"):
        self.dtype = dtype
        self._device = torch.device(device)
        self.control_model = B200ControlNet(dtype=dtype, **(control_params or {}))
        self.model = _Wrapper(B200ControlledUnet(dtype=dtype, **(unet_params or {})))
        self.control_scales = [1.0] * 13
        self.only_mid_control = only_mid_control
        self.parameterization = parameterization
        self.scale_factor = scale_factor
        self.num_timesteps = int(timesteps)
        # yaml:4-8 `linear` schedule (upstream register_schedule): computed in float64, stored fp32
        betas = np.linspace(linear_start ** 0.5, linear_end ** 0.5, timesteps, dtype=np.float64) ** 2
        ac = np.cumprod(1.0 - betas, axis=0)
        f32 = lambda a: torch.tensor(a, dtype=torch.float32, device=self._device)  # noqa: E731
        self.betas = f32(betas)
        self.alphas_cumprod = f32(ac)
        self.alphas_cumprod_prev = f32(np.append(1.0, ac[:-1]))
        self.sqrt_alphas_cumprod = f32(np.sqrt(ac))
        self.sqrt_one_minus_alphas_cumprod = f32(np.sqrt(1.0 - ac))
        self.sqrt_recip_alphas_cumprod = f32(np.sqrt(1.0 / ac))
        self.sqrt_recipm1_alphas_cumprod = f32(np.sqrt(1.0 / ac - 1))
        self._cond_cache = {}
        self._trunk_epoch = None
        # ControlNet trunk on a second stream, concurrent with the UNet encoder (set False to serialise: profiling, A/B runs)
        self.concurrent = True
        self._side = None
        # UNet encoder + ControlNet trunk as one stacked network (nets.B200GroupedTrunk): each layer of the two structurally
        # identical trunks is one launch over both batches.  "auto": when every level's rows per network are whole 256-row tile
        # pairs (what the grouped kernel takes) on the bf16 path; True / False force one form (tests, A/B runs).  Results do
        # not depend on it.
        self.grouped = "auto"
        self._trunk = None
        # ResBlock timestep embeddings of a whole sampling loop, computed ahead of it (precompute_time_embeddings / set_step)
        self._emb_table = None
        self._emb_bufs = {}
        self._emb_rows = None

    @property
    def device(self):
        return self._device

    def load_state_dict(self, sd, strict=True):
        """upstream prefixes: ``control_model.*`` and ``model.diffusion_model.*`` (runs/train.py:61)"""
        if self._device.type == "cuda":
            # one process per GPU: the C-ABI launches on the CURRENT device's stream (ops._stream) and its kernels'
            # one-time attribute setup is per process, so the model's device must be the current one
            idx = self._device.index if self._device.index is not None else torch.cuda.current_device()
            if idx != torch.cuda.current_device():
                raise RuntimeError(f"B200ControlLDM on cuda:{idx} while the current device is cuda:{torch.cuda.current_device()}: "
                                   "this library is one process per GPU — call torch.cuda.set_device() first")
            ops.device_ok(idx)
        cn = {k: v for k, v in sd.items() if k.startswith("control_model.")}
        un = {k: v for k, v in sd.items() if k.startswith("model.diffusion_model.")}
        self.control_model.load_state_dict(cn, strict=strict, prefix="control_model.", device=self._device)
        self.model.diffusion_model.load_state_dict(un, strict=strict, prefix="model.diffusion_model.", device=self._device)
        self._cond_cache.clear()
        return self

    @property
    def _weights_epoch(self):
        """changes whenever either network (re)loads weights — through this object or through the network's own load_state_dict
        (INTEGRATION level 1).  Captured CUDA graphs hold the old weight pointers, the stacked trunk copies of them and the
        timestep-embedding table values computed from them: all three are keyed on it."""
        return (getattr(self.model.diffusion_model, "load_epoch", 0), getattr(self.control_model, "load_epoch", 0))

    # ---- timestep embeddings of a sampling loop ---------------------------------------------------------------------
    # emb = emb_layers(time_embed(timestep_embedding(t))) depends on t alone.  A DDIM loop knows its timesteps up front and
    # uses ONE t for the whole batch (cddim.py:86-89 / upstream ddim_sampling: ts = torch.full((b,), step)), so the sampler
    # asks for all S of them at once — two MLP chains over S rows instead of S x 2 chains over the batch, each streaming
    # ~85 MB of weights for 16 rows — and selects one row per step.  apply_model(x, t, cond) without a selected step
    # computes the embeddings from its t argument as before.  A DPM-Solver loop feeds fractional model times: integer
    # timesteps key the table as ints (the DDIM / PLMS loops, unchanged), every other value as its exact fp32 value.
    @staticmethod
    def _time_key(v):
        if isinstance(v, (int, np.integer)) or (torch.is_tensor(v) and not v.is_floating_point()):
            return int(v)
        return float(np.float32(v))

    def precompute_time_embeddings(self, values):
        vals = tuple(self._time_key(v) for v in values)
        tb = self._emb_table
        if tb is not None and tb["vals"] == vals and tb["epoch"] == self._weights_epoch:
            return
        un, cn = self.model.diffusion_model, self.control_model
        integer = all(isinstance(v, int) for v in vals)
        tv = torch.tensor(vals, dtype=torch.int64 if integer else torch.float32, device=self._device)
        tab = torch.zeros(len(vals), 2, un._emb_total, dtype=self.dtype, device=self._device)
        un._time_embedding(tv, len(vals), out=tab[:, 0])
        cn._time_embedding(tv, len(vals), out=tab[:, 1, :cn._emb_total])
        self._emb_table = {"vals": vals, "row": {v: i for i, v in enumerate(vals)}, "tab": tab, "epoch": self._weights_epoch}

    def set_step(self, t_value, rows=None):
        """select the precomputed embeddings of timestep ``t_value`` (an int, or a float selecting the row of its fp32 value)
        for the next apply_model calls on ``rows`` batch rows (all at that timestep); ``None`` returns to computing them from
        the ``t`` argument.  Returns whether a row is selected."""
        self._emb_rows = None
        tb = self._emb_table
        if t_value is None or tb is None or tb["epoch"] != self._weights_epoch or self._time_key(t_value) not in tb["row"]:
            return False
        tot = tb["tab"].shape[2]
        buf = self._emb_bufs.get(rows)
        if buf is None:
            buf = self._emb_bufs[rows] = torch.empty(2 * rows, tot, dtype=self.dtype, device=self._device)
        buf.view(2, rows, tot).copy_(tb["tab"][tb["row"][self._time_key(t_value)]][:, None, :].expand(2, rows, tot))
        self._emb_rows = rows
        return True

    def _stack_cond(self, prep):
        prep["kv2"], prep["hint2"] = self._grouped_trunk().stack_cond(prep["kv_unet"], prep["kv_cn"], prep["hint"])

    def _use_grouped(self, N, H, W):
        if self.grouped != "auto":
            return bool(self.grouped)
        ds = self.model.diffusion_model._ds  # the deepest level decides: its row count is the smallest
        return self.dtype != torch.float32 and (N * (H // ds) * (W // ds)) % 256 == 0

    def _grouped_trunk(self):
        if self._trunk is None or self._trunk_epoch != self._weights_epoch:  # stacked COPIES of the trunk weights: rebuilt after a reload
            self._trunk = None
            self._trunk = B200GroupedTrunk(self.model.diffusion_model, self.control_model)
            self._trunk_epoch = self._weights_epoch
        return self._trunk

    # ---- step-invariant conditioning ------------------------------------------------------------------------
    # The hoisted tensors (hint features, cross-attention K/V) are reused while the cond is THE SAME tensors holding the
    # same values.  What that rests on, in order of authority:
    #   1. samplers call invalidate_cond_cache() when a loop starts: every sample() / reconstruct() / sample_sharded()
    #      reads its cond afresh, however the caller filled the tensors (raw stream copies, DLPack, this library's own
    #      kernels — none of which move torch's version counter);
    #   2. between those points: identity + shape + torch's version counter of every cond tensor; a tensor without one
    #      (created under torch.inference_mode(), as Lightning >= 1.8 does in trainer.test) is never considered equal;
    #   3. the nets' arena epochs: module-level calls (control_model(x=, hint=, ...), INTEGRATION level 1) refill the same
    #      static buffers the cached dict points into, and must not be mistaken for the cached cond.
    @staticmethod
    def _tkey(t):
        if t is None:
            return None
        return (t.data_ptr(), tuple(t.shape), object() if t.is_inference() else t._version)

    def invalidate_cond_cache(self):
        """forget the hoisted per-cond tensors: the next apply_model recomputes the hint block and the K/V projections"""
        self._cond_cache.clear()

    def _prepare(self, cond, grouped=False):
        ctx_list, cat_list = cond["c_crossattn"], cond["c_concat"]
        un, cn = self.model.diffusion_model, self.control_model
        key = (tuple(self._tkey(t) for t in ctx_list), None if cat_list is None else tuple(self._tkey(t) for t in cat_list))
        hit = self._cond_cache.get("k")
        if hit is not None and hit[0] == key and hit[4] == (un.arena_epoch, cn.arena_epoch) + self._weights_epoch:
            if grouped and "kv2" not in hit[1]:
                self._stack_cond(hit[1])
            return hit[1]
        ctx = ctx_list[0] if len(ctx_list) == 1 else torch.cat(ctx_list, 1)
        prep = {"kv_unet": un.context_kv(ctx)}
        if cat_list is not None:
            hint = cat_list[0] if len(cat_list) == 1 else torch.cat(cat_list, 1)
            prep["kv_cn"] = cn.context_kv(ctx)
            prep["hint"] = cn.hint_features(hint)
            if grouped:
                self._stack_cond(prep)
        # keep the source tensors alive so data_ptr-based keys cannot be recycled
        # (the weights epoch: K/V projections and hint features are functions of the weights too — a network reloaded through its
        #  own load_state_dict must not be served the old ones)
        self._cond_cache["k"] = (key, prep, ctx_list, cat_list, (un.arena_epoch, cn.arena_epoch) + self._weights_epoch)
        return prep

    # ---- diffmk/makeup_diffuse.py:152-170 ---------------------------------------------------------------------
    def apply_model(self, x_noisy, t, cond, return_all=False, *args, **kwargs):
        assert isinstance(cond, dict)
        un, cn = self.model.diffusion_model, self.control_model
        N, _, H, W = x_noisy.shape
        use_cn = cond["c_concat"] is not None
        grouped = use_cn and self._use_grouped(N, H, W)
        prep = self._prepare(cond, grouped)
        t = timesteps_for_embedding(t)
        emb2 = self._emb_bufs[N] if self._emb_rows == N else None  # [UNet rows | ControlNet rows] of the selected step
        emb_un = None if emb2 is None else emb2[:N]
        emb_cn = None if emb2 is None else emb2[N:, :cn._emb_total]
        two_streams = use_cn and self.concurrent and x_noisy.is_cuda
        pending = None
        if grouped:
            # both trunks as one stacked network on this stream; only the injecting zero-convs go to the side stream below
            if two_streams and self._side is None:
                self._side = torch.cuda.Stream(device=x_noisy.device)
            slots, pending = self._grouped_trunk().run(x_noisy, prep["hint2"], t, prep["kv2"], N, H, W,
                                                       side=self._side if two_streams else None, emb2=emb2)
        elif two_streams:
            # The ControlNet trunk depends only on (x, t, hint, ctx): fork it onto a second stream so its many small,
            # latency-bound kernels fill the SMs the UNet encoder's leave idle.  Inside a CUDA-graph capture this
            # becomes a parallel branch of the graph.
            main = torch.cuda.current_stream()
            if self._side is None:
                self._side = torch.cuda.Stream(device=x_noisy.device)
            fork, join = torch.cuda.Event(), torch.cuda.Event()
            fork.record(main)
            self._side.wait_event(fork)
            with torch.cuda.stream(self._side):
                pending = cn.run_trunk(cn._x_in(x_noisy), prep["hint"], t, prep["kv_cn"], N, H, W, emb=emb_cn)
                join.record(self._side)
        if not grouped:
            xin = un._x_in(x_noisy)
            slots = un.encode(xin, t, prep["kv_unet"], N, H, W, emb=emb_un)
        before_block = None
        if use_cn:
            nb = len(un.input_blocks)
            inject = [None] * nb + [slots[nb]] if self.only_mid_control else slots
            inject_st = un.skip_slot_stats(N, H, W)
            if two_streams:
                if self._side is None:
                    self._side = torch.cuda.Stream(device=x_noisy.device)
                # The 13 injecting zero-convs stay on the side stream, issued in the order the decoder consumes the
                # slots (middle output first, then hs.pop() order) with one event each: the decoder's deep, SM-starved
                # blocks start after the first two and overlap the rest.
                main = torch.cuda.current_stream()
                enc_done = torch.cuda.Event()
                enc_done.record(main)
                evs = {}
                with torch.cuda.stream(self._side):
                    self._side.wait_event(enc_done)  # the encoder has written every slot the epilogues add into
                    for item in sorted(pending, key=lambda p: -p[2]):
                        if inject[item[2]] is None:
                            continue
                        cn.zero_convs([item], N, inject=inject, scales=self.control_scales, inject_st=inject_st)
                        evs[item[2]] = torch.cuda.Event()
                        evs[item[2]].record(self._side)
                    tail = torch.cuda.Event()
                    tail.record(self._side)

                def before_block(i):  # decoder block i reads slot nb-1-i (block 0 also the injected middle output)
                    for j in ([nb] if i == 0 else []) + [nb - 1 - i]:
                        if j in evs:
                            main.wait_event(evs.pop(j))
                    if i == nb - 1:
                        main.wait_event(tail)  # joins the side stream whatever was injected
            else:
                if not grouped:
                    pending = cn.run_trunk(cn._x_in(x_noisy), prep["hint"], t, prep["kv_cn"], N, H, W, emb=emb_cn)
                cn.zero_convs(pending, N, inject=inject, scales=self.control_scales, inject_st=inject_st)
            un.note_slots_rewritten([j for j, s in enumerate(inject) if s is not None], with_stats=True)
        e = un.decode(prep["kv_unet"], N, H, W, before_block=before_block)
        eps = torch.empty(N, un.out_channels, H, W, dtype=torch.float32, device=x_noisy.device)
        ops.nhwc_to_nchw(e, eps)
        if not return_all:
            return eps
        return eps, self.predict_start_from_noise(x_noisy, t, eps)

    # ---- first stage (SURVEY.md §8(f) rank 1): diffmk/makeups.py:260-262, diffusion_makeup.py:389,396,409 --------------
    def attach_first_stage_decoder(self, decoder):
        """decoder: a loaded ``B200FirstStageDecoder`` (the reference's ``first_stage_model``, decode side only)"""
        self.first_stage_model = decoder
        return self

    def decode_first_stage(self, z):
        """``first_stage_model.decode(1 / scale_factor * z)`` -> NCHW fp32 images in (about) [-1, 1]"""
        if getattr(self, "first_stage_model", None) is None:
            raise RuntimeError("no first-stage decoder attached (attach_first_stage_decoder)")
        return self.first_stage_model.decode(1.0 / self.scale_factor * z)

    decode_latent_code = decode_first_stage  # the reference's other name for it (makeups.py:260)

    # ---- x_p entry (SURVEY.md §8(f) rank 2): diffmk/makeup_diffuse.py:37-40, diffusion_makeup.py:384-387 -------------
    # ---- conditioning producer (SURVEY.md 8(f) rank 3) ----------------------------------------------------------
    def attach_cond_stage_model(self, encoder):
        """encoder: a loaded ``B200FrozenCLIPEmbedder`` (the reference's ``cond_stage_model``, yaml:109-110)"""
        self.cond_stage_model = encoder
        self._prompt_cache = {}
        return self

    def get_learned_conditioning(self, c):
        """``cond_stage_model.encode(c)``: prompts (list of str) or token ids [B, 77] -> c_crossattn [B, 77, 768].
        The reference's prompt is the constant 'makeup transfer' (datasets.py:772): string prompts are encoded once and
        the result is reused for every later batch (the encoder is frozen)."""
        if getattr(self, "cond_stage_model", None) is None:
            raise RuntimeError("no cond-stage model attached (attach_cond_stage_model)")
        if torch.is_tensor(c):
            return self.cond_stage_model(c)
        key = tuple([c] if isinstance(c, str) else c)
        if key not in self._prompt_cache:
            uniq = sorted(set(key))
            z = self.cond_stage_model.encode(uniq)
            self._prompt_cache[key] = torch.stack([z[uniq.index(p)] for p in key])
        return self._prompt_cache[key]

    def get_unconditional_conditioning(self, N):
        """CLIP encoding of the empty prompt, N times (diffusion_makeup.py:399-402)"""
        return self.get_learned_conditioning([""] * N)

    @staticmethod
    def assemble_hint(src_img, ref_img):
        """c_concat[0] = cat((src_img, ref_img), 1): source first (makeup_diffuse.py:56; images in [0, 1])"""
        return torch.cat((src_img, ref_img), 1)

    def attach_first_stage_encoder(self, encoder):
        """encoder: a loaded ``B200FirstStageEncoder`` (the reference's ``first_stage_model``, encode side only)"""
        self.first_stage_encoder = encoder
        return self

    def encode_first_stage(self, x):
        """posterior moments (mean, logvar) of ``first_stage_model.encode(x)``; x: [B, 3, H, W] in [-1, 1]"""
        if getattr(self, "first_stage_encoder", None) is None:
            raise RuntimeError("no first-stage encoder attached (attach_first_stage_encoder)")
        return self.first_stage_encoder.encode(x)

    def get_first_stage_encoding(self, posterior, noise=None):
        """``scale_factor * posterior.sample()`` with sample = mean + exp(logvar / 2) * randn (upstream
        DiagonalGaussianDistribution.sample); latent-sized, outside the loop"""
        mean, logvar = posterior
        noise = torch.randn_like(mean) if noise is None else noise
        return self.scale_factor * (mean + torch.exp(0.5 * logvar) * noise)

    def get_z(self, x, noise=None):
        """diffmk/makeup_diffuse.py:37-40"""
        return self.get_first_stage_encoding(self.encode_first_stage(x), noise)

    # ---- x_p entry helpers (diffusion_makeup.py:384-389); latent-sized, outside the 50-step loop ---------------
    @staticmethod
    def _extract(a, t, x):
        return a.gather(-1, t).reshape(t.shape[0], *((1,) * (x.dim() - 1)))

    def q_sample(self, x_start, t, noise=None):
        noise = torch.randn_like(x_start) if noise is None else noise
        return (self._extract(self.sqrt_alphas_cumprod, t, x_start) * x_start +
                self._extract(self.sqrt_one_minus_alphas_cumprod, t, x_start) * noise)

    def predict_start_from_noise(self, x_t, t, noise):
        return (self._extract(self.sqrt_recip_alphas_cumprod, t, x_t) * x_t -
                self._extract(self.sqrt_recipm1_alphas_cumprod, t, x_t) * noise)
