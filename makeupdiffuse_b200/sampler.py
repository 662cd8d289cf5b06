"""``B200DDIMSampler``: drop-in for ``MKDDIMSampler`` (diffmk/cddim.py:5-100) and the upstream ``DDIMSampler`` it
extends — same constructor, same ``make_schedule`` / ``sample`` / ``ddim_sampling`` / ``p_sample_ddim`` /
``denoising_step`` / ``reconstruct`` / ``decode`` / ``stochastic_encode`` / ``encode`` (DDIM inversion) signatures and
return values (SURVEY.md §8(b) level B1).

Per step it runs ``model.apply_model`` (one CUDA-graph replay of the fused UNet+ControlNet kernels when
``use_cuda_graph`` is on) followed by ONE fused kernel for the whole x_t -> x_{t-1} update including the
classifier-free-guidance combine (cddim.py:39-40, 56-78), instead of ~12 elementwise launches + 4 ``torch.full``.
The RNG stream is consumed exactly like the reference: one ``randn(x.shape)`` per step even when sigma == 0
(cddim.py:75).  Unlike upstream nothing is force-moved to "cuda": buffers follow ``model.device``.

``B200PLMSSampler`` (below) is the drop-in for upstream ``PLMSSampler`` on the same machinery, with its own fused update
kernel (mkd_plms_update); ``B200DPMSolverSampler`` the drop-in for upstream ``DPMSolverSampler`` (DPM-Solver++(2M) at
fractional model times, one fused mkd_dpm_update per evaluation); ``B200DDPMSampler`` upstream ``LatentDiffusion``'s own
DDPM ancestral loop (``sample`` / ``p_sample_loop`` / ``progressive_denoising``, one fused mkd_ddpm_update per step).
"""
from __future__ import annotations

import numpy as np
import torch

from . import ops


def _uniform_ddim_timesteps(num_ddim, num_ddpm):
    c = num_ddpm // num_ddim
    return np.asarray(list(range(0, num_ddpm, c))) + 1


def _cat_uncond_first(uc, c):
    """cddim.py:20-38 — [uncond; cond] along batch for every tensor leaf"""
    if isinstance(c, dict):
        assert isinstance(uc, dict)
        return {k: ([torch.cat([uc[k][i], c[k][i]]) for i in range(len(c[k]))] if isinstance(c[k], list)
                    else torch.cat([uc[k], c[k]])) for k in c}
    if isinstance(c, list):
        assert isinstance(uc, list)
        return [torch.cat([uc[i], c[i]]) for i in range(len(c))]
    return torch.cat([uc, c])


class B200DDIMSampler:
    def __init__(self, model, schedule="linear", use_cuda_graph=True, **kwargs):
        self.model = model
        self.ddpm_num_timesteps = model.num_timesteps
        self.schedule = schedule
        self.use_cuda_graph = use_cuda_graph
        self._cfg_cache = None
        self._graph = None
        self.graph_launches = 0  # kernels executed through graph replays (they bypass the library's launch counter)

    # ---- schedule (upstream make_schedule / make_ddim_sampling_parameters) -----------------------------------
    def make_schedule(self, ddim_num_steps, ddim_discretize="uniform", ddim_eta=0.0, verbose=True):
        if ddim_discretize != "uniform":
            raise NotImplementedError(f'There is no ddim discretization method called "{ddim_discretize}"')
        m = self.model
        self.ddim_timesteps = _uniform_ddim_timesteps(ddim_num_steps, self.ddpm_num_timesteps)
        ac = m.alphas_cumprod.detach().float()
        assert ac.shape[0] == self.ddpm_num_timesteps, "alphas have to be defined for each timestep"
        dev = m.device
        self.betas = m.betas.float()
        self.alphas_cumprod = ac
        self.alphas_cumprod_prev = m.alphas_cumprod_prev.float()
        self.sqrt_alphas_cumprod = ac.sqrt()
        self.sqrt_one_minus_alphas_cumprod = (1.0 - ac).sqrt()
        acn = ac.cpu().numpy()
        a = acn[self.ddim_timesteps]
        a_prev = np.asarray([acn[0]] + acn[self.ddim_timesteps[:-1]].tolist())
        sig = ddim_eta * np.sqrt((1 - a_prev) / (1 - a) * (1 - a / a_prev))
        f32 = lambda v: torch.as_tensor(np.asarray(v), dtype=torch.float32).to(dev)  # noqa: E731
        self.ddim_sigmas = f32(sig)
        self.ddim_alphas = f32(a)
        self.ddim_alphas_prev = a_prev
        self.ddim_sqrt_one_minus_alphas = f32(np.sqrt(1.0 - a))
        acp = self.alphas_cumprod_prev
        self.ddim_sigmas_for_original_num_steps = ddim_eta * torch.sqrt((1 - acp) / (1 - ac) * (1 - ac / acp))
        # host copies of the four per-step coefficients, rounded exactly like the reference's fp32 torch ops
        self._coef_ddim = self._coefficients(self.ddim_alphas, self.ddim_alphas_prev, self.ddim_sqrt_one_minus_alphas,
                                             self.ddim_sigmas)
        self._coef_orig = None

    @staticmethod
    def _coefficients(A, AP, S1, SG, device=None):
        """per index: (sqrt(1-a_t), sqrt(a_t), sqrt(a_prev), sqrt(1 - a_prev - sigma^2), sigma) as fp32 values
        (cddim.py:56-59 builds fp32 tensors with torch.full; :63,74,78 take fp32 sqrt), evaluated on ``device`` (the CPU
        by default)"""
        f = lambda v: torch.as_tensor(np.asarray(v.cpu() if torch.is_tensor(v) else v), dtype=torch.float32, device=device)  # noqa: E731
        a, ap, s1, sg = f(A), f(AP), f(S1), f(SG)
        return torch.stack([s1, a.sqrt(), ap.sqrt(), (1.0 - ap - sg ** 2).sqrt(), sg], 1).tolist()

    # ---- sampling from noise ----------------------------------------------------------------------------------
    def sample(self, S, batch_size, shape, conditioning=None, callback=None, normals_sequence=None, img_callback=None,
               quantize_x0=False, eta=0.0, mask=None, x0=None, temperature=1.0, noise_dropout=0.0, score_corrector=None,
               corrector_kwargs=None, verbose=True, x_T=None, log_every_t=100, unconditional_guidance_scale=1.0,
               unconditional_conditioning=None, dynamic_threshold=None, ucg_schedule=None, **kwargs):
        self.make_schedule(ddim_num_steps=S, ddim_eta=eta, verbose=verbose)
        C, H, W = shape
        return self.ddim_sampling(conditioning, (batch_size, C, H, W), callback=callback, img_callback=img_callback,
                                  quantize_denoised=quantize_x0, mask=mask, x0=x0, noise_dropout=noise_dropout,
                                  temperature=temperature, score_corrector=score_corrector,
                                  corrector_kwargs=corrector_kwargs, x_T=x_T, log_every_t=log_every_t,
                                  unconditional_guidance_scale=unconditional_guidance_scale,
                                  unconditional_conditioning=unconditional_conditioning,
                                  dynamic_threshold=dynamic_threshold)

    @torch.no_grad()
    def ddim_sampling(self, cond, shape, x_T=None, callback=None, img_callback=None, quantize_denoised=False, mask=None,
                      x0=None, log_every_t=100, temperature=1.0, noise_dropout=0.0, score_corrector=None,
                      corrector_kwargs=None, unconditional_guidance_scale=1.0, unconditional_conditioning=None,
                      dynamic_threshold=None, **kwargs):
        dev = self.model.device
        b = shape[0]
        steps = np.flip(self.ddim_timesteps)
        self.begin_loop(steps)
        img = torch.randn(shape, device=dev) if x_T is None else x_T
        inter = {"x_inter": [img], "pred_x0": [img]}
        total = steps.shape[0]
        for i, step in enumerate(steps):
            index = total - i - 1
            ts = torch.full((b,), int(step), device=dev, dtype=torch.long)
            if mask is not None:
                img = self.model.q_sample(x0, ts) * mask + (1.0 - mask) * img
            img, pred_x0 = self.denoising_step(
                img, cond, ts, index=index, quantize_denoised=quantize_denoised, temperature=temperature,
                noise_dropout=noise_dropout, score_corrector=score_corrector, corrector_kwargs=corrector_kwargs,
                unconditional_guidance_scale=unconditional_guidance_scale,
                unconditional_conditioning=unconditional_conditioning, dynamic_threshold=dynamic_threshold,
                t_value=int(step))
            if callback:
                callback(i)
            if img_callback:
                img_callback(pred_x0, i)
            if index % log_every_t == 0 or index == total - 1:
                inter["x_inter"].append(img)
                inter["pred_x0"].append(pred_x0)
        return img, inter

    def begin_loop(self, steps=None):
        """A sampling loop starts: whatever was hoisted for an earlier cond (the model's hint features and K/V, the
        doubled CFG cond) is dropped, so the loop reads its conditioning tensors as they are NOW — also when the caller
        refilled the same tensors in a way torch's version counter does not see.  Loops driven from outside
        (makeupdiffuse_b200.dist.sample_sharded, a caller's own loop over denoising_step) call this themselves.
        steps: the loop's timesteps, when known: the model computes the timestep embeddings of all of them at once, and
        denoising_step(..., t_value=step) selects one per step.  Integer steps select as ints; fractional model times (the
        DPM-Solver loop) select by their fp32 value."""
        self._cfg_cache = None
        inv = getattr(self.model, "invalidate_cond_cache", None)
        if inv is not None:
            inv()
        pre = getattr(self.model, "precompute_time_embeddings", None)
        if pre is not None and steps is not None and len(steps):
            pre(list(steps))

    def p_sample_ddim(self, *a, **k):
        with torch.no_grad():
            return self.denoising_step(*a, **k)

    def stochastic_encode(self, x0, t, use_original_steps=False, noise=None):
        sa = self.sqrt_alphas_cumprod if use_original_steps else self.ddim_alphas.sqrt()
        s1 = self.sqrt_one_minus_alphas_cumprod if use_original_steps else self.ddim_sqrt_one_minus_alphas
        noise = torch.randn_like(x0) if noise is None else noise
        ex = lambda v: v.gather(-1, t).reshape(-1, 1, 1, 1)  # noqa: E731
        return ex(sa) * x0 + ex(s1) * noise

    def decode(self, x_latent, cond, t_start, **kw):
        with torch.no_grad():
            return self.reconstruct(x_latent, cond, t_start, **kw)

    def _cfg_cond(self, c, uc):
        """[uncond; cond] for the doubled batch; step-invariant, so built once per loop, not once per step"""
        cc = self._cfg_cache
        if cc is None or cc[0] is not c or cc[1] is not uc:
            cc = self._cfg_cache = (c, uc, _cat_uncond_first(uc, c))
        return cc[2]

    # ---- the model call, optionally as a CUDA-graph replay -------------------------------------------------------
    def _eps(self, x, t, c, t_value=None):
        """model.apply_model(x, t, c); with use_cuda_graph the ~10^3 kernel launches of one UNet+ControlNet step are
        captured once per (cond, batch shape) and replayed (launch-bound otherwise: SURVEY.md §7 hard part 6).
        t_value: the loop's timestep as a host int (or float) when every row of ``t`` holds it (the sampler's own loops): the model
        then takes the ResBlock timestep embeddings from the table computed at the start of the loop (begin_loop(steps))
        instead of running the two embedding MLPs again."""
        set_step = getattr(self.model, "set_step", None)
        if set_step is None or t_value is None:
            return self._eps_call(x, t, c, False)
        try:
            return self._eps_call(x, t, c, set_step(t_value, x.shape[0]))
        finally:
            set_step(None)

    def _eps_call(self, x, t, c, emb_selected):
        prepare = getattr(self.model, "_prepare", None)
        if not (self.use_cuda_graph and x.is_cuda and prepare is not None):
            return self.model.apply_model(x, t, c)
        from . import _lib
        g = self._graph
        # the graph only depends on shapes: every per-cond tensor it reads (hint features, cross-attention K/V) lives
        # in a static arena buffer that model._prepare() refills in place when the cond changes
        m = self.model
        nets = [getattr(m, "control_model", None), getattr(getattr(m, "model", None), "diffusion_model", None)]
        key = (tuple(x.shape), c["c_concat"] is None, tuple(tuple(v.shape) for v in c["c_crossattn"]), id(m),
               getattr(m, "only_mid_control", False), tuple(getattr(m, "control_scales", ())),
               # a graph holds raw pointers and the launch structure of the moment it was captured: reloaded weights
               # (new tensors), another stream layout or another GroupNorm path need a new capture
               getattr(m, "_weights_epoch", 0), getattr(m, "concurrent", None), getattr(m, "grouped", None), emb_selected,
               t.dtype,  # the captured copy_ into the graph's t would cast a fractional fp32 t to int64
               tuple((getattr(n, "fused_gn_stats", None), getattr(n, "fuse_gn_tail", None)) for n in nets))
        if g is None or g["key"] != key:
            sx, st = x.clone(), t.clone()
            self.model.apply_model(sx, st, c)  # warm-up: allocates every static buffer, fills the cond cache
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            n0 = _lib.load().mkd_launch_count()
            with torch.cuda.graph(graph):
                out = self.model.apply_model(sx, st, c)
            g = self._graph = {"key": key, "graph": graph, "x": sx, "t": st, "out": out,
                               "launches": _lib.load().mkd_launch_count() - n0}
        # no-op when the cond is unchanged; otherwise recomputes the hoisted tensors eagerly (in the stacked form too when the
        # captured evaluation runs the two trunks as one network)
        ug = getattr(m, "_use_grouped", None)
        if ug is not None:
            prepare(c, c["c_concat"] is not None and ug(x.shape[0], x.shape[2], x.shape[3]))
        else:
            prepare(c)
        g["x"].copy_(x)
        g["t"].copy_(t)
        g["graph"].replay()
        self.graph_launches += g["launches"]
        return g["out"]

    # ---- one x_t -> x_{t-1} update: diffmk/cddim.py:9-79 ---------------------------------------------------------
    def denoising_step(self, x, c, t, index, repeat_noise=False, use_original_steps=False, quantize_denoised=False,
                       temperature=1.0, noise_dropout=0.0, score_corrector=None, corrector_kwargs=None,
                       unconditional_guidance_scale=1.0, unconditional_conditioning=None, dynamic_threshold=None,
                       out=None, peer_ptrs=None, t_value=None):
        """``out`` (extension, optional): tensor that receives x_prev — e.g. this rank's slice of an all-gather
        buffer, so the last update of a sharded run lands directly where the collective reads it.
        ``peer_ptrs`` (extension, optional): device pointers of that same slice inside EVERY rank's gather buffer (peer
        memory); the update kernel then stores x_prev to all of them — the all-gather fused into the kernel.
        ``t_value`` (extension, optional): the timestep as a host int when every row of ``t`` holds it (see _eps)."""
        m = self.model
        if m.parameterization != "eps":
            raise NotImplementedError("B200 path implements the yaml's parameterization: eps (yaml:50)")
        if score_corrector is not None or quantize_denoised:
            raise NotImplementedError("score_corrector / quantize_denoised are unused by the reference path")
        if dynamic_threshold is not None:
            raise NotImplementedError()
        b = x.shape[0]
        x = x.float().contiguous()
        cfg = not (unconditional_conditioning is None or unconditional_guidance_scale == 1.0)
        if not cfg:
            e = self._eps(x, t, c, t_value)
        else:
            e = self._eps(torch.cat([x] * 2), torch.cat([t] * 2), self._cfg_cond(c, unconditional_conditioning), t_value)
        if use_original_steps:
            if self._coef_orig is None:
                # cddim.py:54 reads the sigma table off the MODEL; without that attribute the reference raises
                # AttributeError, and so does this
                self._coef_orig = self._coefficients(m.alphas_cumprod, m.alphas_cumprod_prev,
                                                     m.sqrt_one_minus_alphas_cumprod,
                                                     m.ddim_sigmas_for_original_num_steps)
            s1m, sq_at, sq_ap, dirc, sigma = self._coef_orig[index]
        else:
            s1m, sq_at, sq_ap, dirc, sigma = self._coef_ddim[index]
        # the reference draws the noise every step, also when sigma == 0 (cddim.py:75): keep the RNG stream in step
        shape = (1, *x.shape[1:]) if repeat_noise else x.shape
        draw = torch.randn(shape, device=x.device)
        noise = None
        if sigma != 0.0:
            noise = draw.repeat(b, *((1,) * (x.dim() - 1))) if repeat_noise else draw
            if noise_dropout > 0.0:
                # dropout acts on sigma*noise*temperature in the reference; it commutes with the scalar factors
                noise = torch.nn.functional.dropout(noise, p=noise_dropout)
            noise = noise.contiguous()
        x_prev, pred_x0 = (torch.empty_like(x) if out is None else out), torch.empty_like(x)
        ops.ddim_update(x, e.contiguous(), x_prev, sqrt_one_minus_at=s1m, sqrt_at=sq_at, sqrt_a_prev=sq_ap, dir_coef=dirc,
                        sigma_t=sigma, temperature=temperature, noise=noise, pred_x0=pred_x0,
                        cfg_scale=float(unconditional_guidance_scale) if cfg else None, peer_ptrs=peer_ptrs)
        return x_prev, pred_x0

    # ---- truncated reverse loop from a caller-supplied x_t: diffmk/cddim.py:81-100 -------------------------------
    def reconstruct(self, x_latent, cond, t_start, unconditional_guidance_scale=1.0, unconditional_conditioning=None,
                    use_original_steps=False, callback=None):
        steps = np.arange(self.ddpm_num_timesteps) if use_original_steps else self.ddim_timesteps
        steps = steps[:t_start]
        total = steps.shape[0]
        self.begin_loop(steps)
        x = x_latent
        for i, step in enumerate(np.flip(steps)):
            ts = torch.full((x_latent.shape[0],), int(step), device=x_latent.device, dtype=torch.long)
            x, _ = self.denoising_step(x, cond, ts, index=total - i - 1, use_original_steps=use_original_steps,
                                       unconditional_guidance_scale=unconditional_guidance_scale,
                                       unconditional_conditioning=unconditional_conditioning, t_value=int(step))
            if callback:
                callback(i)
        return x

    # ---- DDIM inversion x_0 -> x_t (upstream DDIMSampler.encode; the loop that produces reconstruct's x_latent) --------
    @staticmethod
    def _encode_coefficients(alphas_next, alphas):
        """per step (c_x, c_e) with x_next = c_x * x + c_e * eps: upstream's expressions on upstream's operands (fp32
        alphas_next on the model's device; fp64 alphas on the CPU for the DDIM schedule, the fp32 device table with
        use_original_steps), each rounded to fp32 once as the multiply with the fp32 latent does.  They are evaluated where
        upstream evaluates them, as 0-dim tensors on the same devices: c_e subtracts two nearly equal square roots, and the
        same expressions evaluated on the CPU instead gave another fp32 update on a B200 (one ulp, step 6 of S = 20 and 50)."""
        cx, ce = [], []
        for an, a in zip(alphas_next, alphas):
            cx.append((an / a).sqrt().float())
            ce.append((an.sqrt() * ((1 / an - 1).sqrt() - (1 / a - 1).sqrt())).float())
        return list(zip(torch.stack(cx).tolist(), torch.stack(ce).tolist())) if cx else []

    @torch.no_grad()
    def encode(self, x0, c, t_enc, use_original_steps=False, return_intermediates=None, unconditional_guidance_scale=1.0,
               unconditional_conditioning=None, callback=None, out=None, peer_ptrs=None):
        """Deterministic DDIM inversion: t_enc steps from the clean latent x0 towards noise, on the schedule set by the last
        make_schedule.  Returns (x_t, {"x_encoded", "intermediate_steps"[, "intermediates"]}) like upstream; draws no noise.
        ``out`` / ``peer_ptrs`` (extensions, optional): as in denoising_step, for the LAST step only."""
        num_reference_steps = self.ddpm_num_timesteps if use_original_steps else self.ddim_timesteps.shape[0]
        assert t_enc <= num_reference_steps
        if use_original_steps:
            alphas_next, alphas = self.alphas_cumprod[:t_enc], self.alphas_cumprod_prev[:t_enc]
        else:
            alphas_next, alphas = self.ddim_alphas[:t_enc], torch.tensor(self.ddim_alphas_prev[:t_enc])
        coef = self._encode_coefficients(alphas_next, alphas)  # once per call, before the loop
        cfg = unconditional_guidance_scale != 1.0
        if cfg:
            assert unconditional_conditioning is not None
        self.begin_loop(range(t_enc))
        x_next = x0
        intermediates, inter_steps = [], []
        for i in range(t_enc):
            x = x_next.float().contiguous()
            t = torch.full((x.shape[0],), i, device=self.model.device, dtype=torch.long)  # the loop index, as upstream
            if not cfg:
                e = self._eps(x, t, c, t_value=i)
            else:
                e = self._eps(torch.cat([x] * 2), torch.cat([t] * 2), self._cfg_cond(c, unconditional_conditioning), t_value=i)
            last = i == t_enc - 1
            x_next = out if (last and out is not None) else torch.empty_like(x)
            c_x, c_e = coef[i]
            # the sampling kernel with sqrt(1-a_t) = 0, sqrt(a_t) = 1 computes fl(c_x * fl(fl(x - 0*e) / 1)) + fl(c_e * e):
            # for finite values that is upstream's fl(c_x * x) + fl(c_e * e), so the inversion needs no kernel of its own
            ops.ddim_update(x, e.contiguous(), x_next, sqrt_one_minus_at=0.0, sqrt_at=1.0, sqrt_a_prev=c_x, dir_coef=c_e,
                            cfg_scale=float(unconditional_guidance_scale) if cfg else None,
                            peer_ptrs=peer_ptrs if last else None)
            if return_intermediates and i % (t_enc // return_intermediates) == 0 and i < t_enc - 1:
                intermediates.append(x_next)
                inter_steps.append(i)
            elif return_intermediates and i >= t_enc - 2:
                intermediates.append(x_next)
                inter_steps.append(i)
            if callback:
                callback(i)
        res = {"x_encoded": x_next, "intermediate_steps": inter_steps}
        if return_intermediates:
            res["intermediates"] = intermediates
        return x_next, res


class B200PLMSSampler(B200DDIMSampler):
    """Drop-in for upstream ``ldm.models.diffusion.plms.PLMSSampler``: DDIM's schedule (eta must be 0), timesteps and
    coefficients, with the eps of each step replaced by a pseudo-linear multistep combination of the current and up to
    three earlier eps.  A run of S steps makes S + 1 model evaluations (step 0 evaluates twice) and draws S + 1
    ``randn(x.shape)`` like upstream.  Per evaluation: one graph-replayed UNet+ControlNet call, then one fused kernel
    (mkd_plms_update) for the CFG combine, the store of e_t into a ring of three device buffers, the combination and the
    DDIM update.  One deliberate superset: the guided call accepts this model's dict-of-lists cond (upstream's
    ``torch.cat([uc, c])`` takes bare tensors only)."""

    def make_schedule(self, ddim_num_steps, ddim_discretize="uniform", ddim_eta=0.0, verbose=True):
        if ddim_eta != 0:
            raise ValueError("ddim_eta must be 0 for PLMS")
        super().make_schedule(ddim_num_steps, ddim_discretize=ddim_discretize, ddim_eta=ddim_eta, verbose=verbose)
        # the square roots on the model's device, where upstream takes them: torch's fp32 sqrt on the CPU is one ulp off the
        # correctly rounded CUDA result at a few entries of the 50-step schedule (sqrt(a_t) at indices 6 and 44)
        self._coef_ddim = self._coefficients(self.ddim_alphas, self.ddim_alphas_prev, self.ddim_sqrt_one_minus_alphas,
                                             self.ddim_sigmas, device=self.model.device)

    def sample(self, S, batch_size, shape, conditioning=None, callback=None, normals_sequence=None, img_callback=None,
               quantize_x0=False, eta=0.0, mask=None, x0=None, temperature=1.0, noise_dropout=0.0, score_corrector=None,
               corrector_kwargs=None, verbose=True, x_T=None, log_every_t=100, unconditional_guidance_scale=1.0,
               unconditional_conditioning=None, dynamic_threshold=None, out=None, peer_ptrs=None, **kwargs):
        """``out`` / ``peer_ptrs`` (extensions, optional): as in denoising_step, for the LAST update only"""
        self.make_schedule(ddim_num_steps=S, ddim_eta=eta, verbose=verbose)
        C, H, W = shape
        return self.plms_sampling(conditioning, (batch_size, C, H, W), callback=callback, img_callback=img_callback,
                                  quantize_denoised=quantize_x0, mask=mask, x0=x0, ddim_use_original_steps=False,
                                  noise_dropout=noise_dropout, temperature=temperature, score_corrector=score_corrector,
                                  corrector_kwargs=corrector_kwargs, x_T=x_T, log_every_t=log_every_t,
                                  unconditional_guidance_scale=unconditional_guidance_scale,
                                  unconditional_conditioning=unconditional_conditioning,
                                  dynamic_threshold=dynamic_threshold, out=out, peer_ptrs=peer_ptrs)

    @torch.no_grad()
    def plms_sampling(self, cond, shape, x_T=None, ddim_use_original_steps=False, callback=None, timesteps=None,
                      quantize_denoised=False, mask=None, x0=None, img_callback=None, log_every_t=100, temperature=1.0,
                      noise_dropout=0.0, score_corrector=None, corrector_kwargs=None, unconditional_guidance_scale=1.0,
                      unconditional_conditioning=None, dynamic_threshold=None, out=None, peer_ptrs=None):
        if ddim_use_original_steps or timesteps is not None:
            raise NotImplementedError("the B200 PLMS loop runs the DDIM schedule set by make_schedule")
        dev = self.model.device
        b = shape[0]
        img = torch.randn(shape, device=dev) if x_T is None else x_T
        time_range = np.flip(self.ddim_timesteps)
        total = time_range.shape[0]
        self.begin_loop(time_range)
        # the eps history: three device buffers reused round-robin, so a step writes no tensor of its own for it; the slot
        # a step writes is the one of the oldest eps, which AB4 reads in the same kernel
        ring = torch.empty((3, *shape), device=dev, dtype=torch.float32)
        inter = {"x_inter": [img], "pred_x0": [img]}
        old_eps = []
        for i, step in enumerate(time_range):
            index = total - i - 1
            step_next = int(time_range[min(i + 1, total - 1)])
            ts = torch.full((b,), int(step), device=dev, dtype=torch.long)
            ts_next = torch.full((b,), step_next, device=dev, dtype=torch.long)
            if mask is not None:
                img = self.model.q_sample(x0, ts) * mask + (1.0 - mask) * img
            last = i == total - 1
            img, pred_x0, e_t = self.p_sample_plms(
                img, cond, ts, index=index, quantize_denoised=quantize_denoised, temperature=temperature,
                noise_dropout=noise_dropout, score_corrector=score_corrector, corrector_kwargs=corrector_kwargs,
                unconditional_guidance_scale=unconditional_guidance_scale,
                unconditional_conditioning=unconditional_conditioning, old_eps=old_eps, t_next=ts_next,
                dynamic_threshold=dynamic_threshold, e_t_out=ring[i % 3], t_value=int(step), t_next_value=step_next,
                out=out if last else None, peer_ptrs=peer_ptrs if last else None)
            old_eps.append(e_t)
            if len(old_eps) >= 4:
                old_eps.pop(0)
            if callback:
                callback(i)
            if img_callback:
                img_callback(pred_x0, i)
            if index % log_every_t == 0 or index == total - 1:
                inter["x_inter"].append(img)
                inter["pred_x0"].append(pred_x0)
        return img, inter

    @torch.no_grad()
    def p_sample_plms(self, x, c, t, index, repeat_noise=False, use_original_steps=False, quantize_denoised=False,
                      temperature=1.0, noise_dropout=0.0, score_corrector=None, corrector_kwargs=None,
                      unconditional_guidance_scale=1.0, unconditional_conditioning=None, old_eps=None, t_next=None,
                      dynamic_threshold=None, e_t_out=None, t_value=None, t_next_value=None, out=None, peer_ptrs=None):
        """upstream p_sample_plms: returns (x_prev, pred_x0, e_t).  With no earlier eps it evaluates the model a second
        time, at ``t_next``, on the plain DDIM update of x (pseudo improved Euler).
        Extensions (optional): ``e_t_out`` receives e_t (a fresh tensor otherwise); ``t_value`` / ``t_next_value`` are the
        timesteps of ``t`` / ``t_next`` as host ints (see _eps); ``out`` / ``peer_ptrs`` as in denoising_step."""
        m = self.model
        if m.parameterization != "eps":
            raise NotImplementedError("B200 path implements the yaml's parameterization: eps (yaml:50)")
        if score_corrector is not None or quantize_denoised:
            raise NotImplementedError("score_corrector / quantize_denoised are unused by the reference path")
        if dynamic_threshold is not None or use_original_steps:
            raise NotImplementedError()
        old_eps = list(old_eps or [])[-3:]  # upstream's ">= 3" branch reads the newest three
        x = x.float().contiguous()
        cfg = not (unconditional_conditioning is None or unconditional_guidance_scale == 1.0)
        cc = self._cfg_cond(c, unconditional_conditioning) if cfg else c
        scale = float(unconditional_guidance_scale) if cfg else None
        s1m, sq_at, sq_ap, dirc, _ = self._coef_ddim[index]  # sigma == 0: make_schedule insists on eta == 0
        coef = dict(sqrt_one_minus_at=s1m, sqrt_at=sq_at, sqrt_a_prev=sq_ap, dir_coef=dirc)

        def model_output(xx, tt, tv):
            if not cfg:
                return self._eps(xx, tt, c, tv).contiguous()
            return self._eps(torch.cat([xx] * 2), torch.cat([tt] * 2), cc, tv).contiguous()

        def draw():
            # upstream draws the noise in every get_x_prev_and_pred_x0, and sigma is 0: keep the RNG stream in step
            torch.randn((1, *x.shape[1:]) if repeat_noise else x.shape, device=x.device)

        e_t = torch.empty_like(x) if e_t_out is None else e_t_out
        x_prev, pred_x0 = (torch.empty_like(x) if out is None else out), torch.empty_like(x)
        eps = model_output(x, t, t_value)
        if not old_eps:
            # e_t lands in its slot before the second evaluation overwrites the graph's output buffer
            ops.plms_update(x, eps, pred_x0, mode=0, e_store=e_t, cfg_scale=scale, **coef)  # x_pred, in pred_x0's buffer
            draw()
            eps = model_output(pred_x0, t_next, t_next_value)
            mode, history, store = 1, (e_t,), None
        else:
            mode, history, store = len(old_eps) + 1, tuple(reversed(old_eps)), e_t
        ops.plms_update(x, eps, x_prev, mode=mode, history=history, e_store=store, cfg_scale=scale, pred_x0=pred_x0,
                        peer_ptrs=peer_ptrs, **coef)
        draw()
        return x_prev, pred_x0, e_t


def _cond_batch(c):
    """rows of the first conditioning tensor (upstream's batch-size check reads conditioning[first key].shape[0]; here
    a list value, as in this model's dict-of-lists cond, gives its first tensor)"""
    v = c[next(iter(c))] if isinstance(c, dict) else c
    if isinstance(v, list):
        v = v[0] if v else None
    return None if v is None else v.shape[0]


def _elementwise(fn, v):
    """fn(v) for an elementwise torch function of a 1-D tensor.  On the CPU it is applied one element at a time: torch's
    vectorised CPU exp / log / expm1 can differ by an ulp from the scalar ones, which are the ones upstream's per-step
    [batch]-sized tensors take (below 16 rows).  On CUDA an element's value does not depend on its position."""
    if v.is_cuda:
        return fn(v)
    return torch.cat([fn(v[k:k + 1]) for k in range(v.shape[0])])


class B200DPMSolverSampler(B200DDIMSampler):
    """Drop-in for upstream ``ldm.models.diffusion.dpm_solver.DPMSolverSampler``: DPM-Solver++(2M) — upstream's fixed
    configuration: ``NoiseScheduleVP('discrete', alphas_cumprod)``, noise model with classifier-free guidance,
    ``predict_x0=True``, ``skip_type='time_uniform'``, ``method='multistep'``, ``order=2``, ``lower_order_final=True``.
    A run of S steps makes S model evaluations at the fractional model times (t - 1/N) * 1000 and draws no noise when
    ``x_T`` is given.  Per evaluation: one graph-replayed UNet+ControlNet call, then one fused kernel (mkd_dpm_update)
    for the CFG combine, the data prediction (kept in a ring of two device buffers) and the order-1 / order-2 step to the
    next time.  One deliberate superset: the guided call and the batch-size check accept this model's dict-of-lists
    cond (upstream's ``torch.cat([uc, c])`` and ``conditioning[key].shape`` take bare tensors only)."""

    order = 2

    # ---- upstream NoiseScheduleVP('discrete', alphas_cumprod=...) ------------------------------------------------------
    def _noise_schedule(self):
        """(t_array [1, N], log_alpha_array [1, N]) on the model's device: log_alpha = 0.5 * log(alphas_cumprod) on the
        fp32 device schedule, t_array = linspace(0, 1, N + 1)[1:] built on the CPU"""
        ac = self.model.alphas_cumprod.detach().to(torch.float32).to(self.model.device)
        N = ac.shape[0]
        t_array = torch.linspace(0., 1., N + 1)[1:].reshape((1, -1)).to(ac.device)
        return t_array, (0.5 * torch.log(ac)).reshape((1, -1))

    @staticmethod
    def _interpolate(x, xp, yp):
        """upstream interpolate_fn: the piecewise-linear function through (xp, yp), extended linearly beyond the ends;
        x [N, 1], xp / yp [1, K]"""
        N, K = x.shape[0], xp.shape[1]
        all_x = torch.cat([x.unsqueeze(2), xp.unsqueeze(0).repeat((N, 1, 1))], dim=2)
        sorted_all_x, x_indices = torch.sort(all_x, dim=2)
        x_idx = torch.argmin(x_indices, dim=2)
        cand_start_idx = x_idx - 1
        start_idx = torch.where(torch.eq(x_idx, 0), torch.tensor(1, device=x.device),
                                torch.where(torch.eq(x_idx, K), torch.tensor(K - 2, device=x.device), cand_start_idx))
        end_idx = torch.where(torch.eq(start_idx, cand_start_idx), start_idx + 2, start_idx + 1)
        start_x = torch.gather(sorted_all_x, dim=2, index=start_idx.unsqueeze(2)).squeeze(2)
        end_x = torch.gather(sorted_all_x, dim=2, index=end_idx.unsqueeze(2)).squeeze(2)
        start_idx2 = torch.where(torch.eq(x_idx, 0), torch.tensor(0, device=x.device),
                                 torch.where(torch.eq(x_idx, K), torch.tensor(K - 2, device=x.device), cand_start_idx))
        y_positions_expanded = yp.unsqueeze(0).expand(N, -1, -1)
        start_y = torch.gather(y_positions_expanded, dim=2, index=start_idx2.unsqueeze(2)).squeeze(2)
        end_y = torch.gather(y_positions_expanded, dim=2, index=(start_idx2 + 1).unsqueeze(2)).squeeze(2)
        return start_y + (x - start_x) * (end_y - start_y) / (end_x - start_x)

    def _loop_scalars(self, S):
        """Everything a run of S steps needs, once per loop and on the model's device, with upstream's expressions:
        the model times and, per evaluation k (at t_k, stepping to t_{k+1}), the arguments of mkd_dpm_update."""
        dev = self.model.device
        t_array, log_alpha_array = self._noise_schedule()
        N = t_array.shape[1]
        # DPMSolver.sample / get_time_steps('time_uniform'): linspace(t_T, t_0, S + 1) on the CPU, then to the device
        times = torch.linspace(1., 1. / N, S + 1).to(dev)
        model_times = (times[:S] - 1. / N) * 1000.  # model_wrapper.get_model_input_time

        def marginals(t):  # marginal_log_mean_coeff -> marginal_alpha, marginal_std, marginal_lambda
            lmc = self._interpolate(t.reshape((-1, 1)), t_array, log_alpha_array).reshape((-1))
            alpha = torch.exp(lmc)
            sigma = torch.sqrt(1. - torch.exp(2. * lmc))
            lam = lmc - 0.5 * torch.log(1. - torch.exp(2. * lmc))
            return torch.stack([alpha, sigma, lam])

        alpha, sigma, lam = _elementwise(lambda t: marginals(t).t(), times).t()
        h = lam[1:] - lam[:-1]                               # h of the step t_k -> t_{k+1}
        ratio = sigma[1:] / sigma[:-1]                       # sigma_t / sigma_s
        phi1 = alpha[1:] * _elementwise(torch.expm1, -h)     # dpm_solver_first_update: alpha_t * expm1(-h)
        phi2 = alpha[1:] * (_elementwise(torch.exp, -h) - 1.)  # multistep_dpm_solver_second_update
        half2 = 0.5 * phi2
        r0 = torch.cat([h[:1], h[:-1] / h[1:]])              # h_0 / h, with h_0 = lambda_prev_0 - lambda_prev_1 (k >= 1)
        inv_r0 = 1. / r0
        cols = torch.stack([alpha[:S], sigma[:S], ratio, phi1, phi2, half2, inv_r0], 1).tolist()
        steps = []
        for k, (a_s, s_s, rt, p1, p2, hp2, ir0) in enumerate(cols):
            # the first step is order 1; with lower_order_final the last one too when S < 15
            order = 1 if k == 0 or (S < 15 and k == S - 1) else self.order
            steps.append(dict(alpha_s=a_s, sigma_s=s_s, sigma_ratio=rt, order=order, phi=p1 if order == 1 else p2,
                              half_phi=0.0 if order == 1 else hp2, inv_r0=0.0 if order == 1 else ir0))
        return model_times.tolist(), steps

    @torch.no_grad()
    def sample(self, S, batch_size, shape, conditioning=None, callback=None, normals_sequence=None, img_callback=None,
               quantize_x0=False, eta=0.0, mask=None, x0=None, temperature=1.0, noise_dropout=0.0, score_corrector=None,
               corrector_kwargs=None, verbose=True, x_T=None, log_every_t=100, unconditional_guidance_scale=1.0,
               unconditional_conditioning=None, out=None, peer_ptrs=None, **kwargs):
        """upstream DPMSolverSampler.sample: returns (x, None).  Arguments upstream ignores (eta, mask, callbacks, ...)
        are ignored.  ``out`` / ``peer_ptrs`` (extensions, optional): as in denoising_step, for the LAST update only."""
        m = self.model
        if m.parameterization != "eps":
            raise NotImplementedError("B200 path implements the yaml's parameterization: eps (yaml:50)")
        if conditioning is not None:
            cbs = _cond_batch(conditioning)
            if cbs is not None and cbs != batch_size:
                print(f"Warning: Got {cbs} conditionings but batch-size is {batch_size}")
        C, H, W = shape
        size = (batch_size, C, H, W)
        if verbose:
            print(f"Data shape for DPM-Solver sampling is {size}, sampling steps {S}")
        dev = m.device
        img = torch.randn(size, device=dev) if x_T is None else x_T
        assert S >= self.order  # upstream DPMSolver.sample: assert steps >= order
        model_times, steps = self._loop_scalars(S)
        self.begin_loop(model_times)
        cfg = not (unconditional_conditioning is None or unconditional_guidance_scale == 1.0)
        cc = self._cfg_cond(conditioning, unconditional_conditioning) if cfg else conditioning
        scale = float(unconditional_guidance_scale) if cfg else None
        x = img.float().contiguous()
        ring = torch.empty((2, *x.shape), device=x.device, dtype=torch.float32)  # data predictions m_k, slot k % 2
        b = x.shape[0]
        for k, (tv, st) in enumerate(zip(model_times, steps)):
            t = torch.full((b,), tv, device=x.device, dtype=torch.float32)
            if not cfg:
                e = self._eps(x, t, conditioning, t_value=tv)
            else:
                e = self._eps(torch.cat([x] * 2), torch.cat([t] * 2), cc, t_value=tv)
            last = k == S - 1
            x_next = out if (last and out is not None) else torch.empty_like(x)
            ops.dpm_update(x, e.contiguous(), x_next, m_store=ring[k % 2],
                           m_prev=ring[(k - 1) % 2] if st["order"] == 2 else None, cfg_scale=scale,
                           peer_ptrs=peer_ptrs if last else None, **st)
            x = x_next
        return x.to(dev), None


def _slice_cond(cond, b):
    """upstream LatentDiffusion.sample's ``cond[:batch_size]`` on every leaf; a None leaf (this model's c_concat may be
    None) stays None"""
    cut = lambda v: None if v is None else v[:b]  # noqa: E731
    if isinstance(cond, dict):
        return {k: list(map(cut, v)) if isinstance(v, list) else cut(v) for k, v in cond.items()}
    if isinstance(cond, list):
        return [cut(v) for v in cond]
    return cut(cond)


class B200DDPMSampler(B200DDIMSampler):
    """DDPM ancestral sampling, upstream ``ldm.models.diffusion.ddpm.LatentDiffusion``'s ``sample`` / ``p_sample_loop`` /
    ``progressive_denoising`` / ``p_sample`` lifted onto the B200 machinery; ``B200ControlLDM`` delegates its methods of
    those names here.  The model supplies upstream's buffers (``sqrt_recip_alphas_cumprod``,
    ``sqrt_recipm1_alphas_cumprod``, ``posterior_mean_coef1`` / ``2``, ``posterior_log_variance_clipped``) and attributes
    (``clip_denoised``, ``log_every_t``, ``channels``, ``image_size``, ``q_sample``).  Per step: one graph-replayed
    UNet+ControlNet call at the integer timestep (the embeddings of all of a loop's timesteps computed up front), one
    ``randn(x.shape)`` as upstream draws it, also at t = 0, then one fused kernel (mkd_ddpm_update) for x_recon, the clamp,
    the posterior mean and the noise term.  No classifier-free guidance: upstream's loop has none."""

    def __init__(self, model, schedule="linear", use_cuda_graph=True, **kwargs):
        super().__init__(model, schedule=schedule, use_cuda_graph=use_cuda_graph, **kwargs)
        self._ddpm_tables = None

    def _tables(self):
        """[5, T] fp32 on the model's device: sqrt_recip_ac, sqrt_recipm1_ac, coef1, coef2 and
        sigma = exp(0.5 * posterior_log_variance_clipped), the last evaluated by torch on the device as upstream does per
        step (one element at a time on the CPU, see _elementwise)"""
        if self._ddpm_tables is None:
            m = self.model
            f = lambda v: v.to(device=m.device, dtype=torch.float32)  # noqa: E731
            sigma = _elementwise(lambda v: (0.5 * v).exp(), f(m.posterior_log_variance_clipped))
            self._ddpm_tables = torch.stack([f(m.sqrt_recip_alphas_cumprod), f(m.sqrt_recipm1_alphas_cumprod),
                                             f(m.posterior_mean_coef1), f(m.posterior_mean_coef2), sigma]).contiguous()
        return self._ddpm_tables

    @staticmethod
    def _randn(shape, device, repeat=False, rows=None):
        """upstream noise_like(shape, device, repeat).  rows (extension) = (batch_global, lo, hi): draw the noise of the
        whole batch and keep rows [lo, hi), so a sharded run consumes the RNG as the single-process run does"""
        if repeat:
            return torch.randn((1, *shape[1:]), device=device).repeat(shape[0], *((1,) * (len(shape) - 1)))
        if rows is not None:
            bg, lo, hi = rows
            return torch.randn((bg, *shape[1:]), device=device)[lo:hi]
        return torch.randn(shape, device=device)

    @torch.no_grad()
    def p_sample(self, x, c, t, clip_denoised=False, repeat_noise=False, return_codebook_ids=False,
                 quantize_denoised=False, return_x0=False, temperature=1., noise_dropout=0., score_corrector=None,
                 corrector_kwargs=None, out=None, peer_ptrs=None, t_value=None, noise_rows=None):
        """upstream p_sample: x_{t-1} (and x_recon when return_x0) from x_t; rows may carry different t.
        Extensions (optional): ``out`` / ``peer_ptrs`` as in denoising_step; ``t_value`` the timestep as a host int when
        every row holds it (see _eps); ``noise_rows`` as in _randn."""
        m = self.model
        if m.parameterization != "eps":
            raise NotImplementedError("B200 path implements the yaml's parameterization: eps (yaml:50)")
        if score_corrector is not None or quantize_denoised or return_codebook_ids:
            raise NotImplementedError("score_corrector / quantize_denoised / codebook ids are unused by the reference path")
        x = x.float().contiguous()
        t = t.to(device=x.device, dtype=torch.int64).contiguous()
        e = self._eps(x, t, c, t_value)
        noise = self._randn(x.shape, x.device, repeat_noise, noise_rows)
        if noise_dropout > 0.:
            # upstream drops out noise * temperature: the kernel then takes the product as it is
            noise, temperature = torch.nn.functional.dropout(noise * temperature, p=noise_dropout), 1.
        x_prev = torch.empty_like(x) if out is None else out
        x0 = torch.empty_like(x) if return_x0 else None
        ops.ddpm_update(x, e.contiguous(), t, x_prev, tables=self._tables(), noise=noise.contiguous(), clip=clip_denoised,
                        temperature=temperature, x0_out=x0, peer_ptrs=peer_ptrs)
        return (x_prev, x0) if return_x0 else x_prev

    def _loop(self, cond, shape, x_T, timesteps, log_every_t, mask, x0, callback, img_callback, progressive, temperature,
              out, peer_ptrs, noise_rows, **step):
        """the loop of p_sample_loop (progressive=False) and progressive_denoising (True); returns (img, intermediates)"""
        m = self.model
        if (out is not None or peer_ptrs is not None) and (mask is not None or timesteps < 1):
            raise ValueError("out= / peer_ptrs= receive the last step's result: they need a step, and no mask blend after it")
        log_every_t = log_every_t or m.log_every_t
        b = shape[0]
        img = self._randn(shape, m.device, rows=noise_rows) if x_T is None else x_T
        intermediates = [] if progressive else [img]
        if progressive and type(temperature) == float:  # noqa: E721  (upstream's test: only a float is expanded)
            temperature = [temperature] * timesteps
        self.begin_loop(range(timesteps - 1, -1, -1))
        for i in reversed(range(0, timesteps)):
            ts = torch.full((b,), i, device=m.device, dtype=torch.long)
            res = self.p_sample(img, cond, ts, clip_denoised=m.clip_denoised, return_x0=progressive,
                                temperature=temperature[i] if progressive else 1., t_value=i, noise_rows=noise_rows,
                                out=out if i == 0 else None, peer_ptrs=peer_ptrs if i == 0 else None, **step)
            img, x0_partial = res if progressive else (res, None)
            if mask is not None:
                assert x0 is not None
                img = m.q_sample(x0, ts) * mask + (1. - mask) * img  # after the step, with its own draw
            if i % log_every_t == 0 or i == timesteps - 1:
                intermediates.append(x0_partial if progressive else img)
            if callback:
                callback(i)
            if img_callback:
                img_callback(img, i)
        return img, intermediates

    @torch.no_grad()
    def p_sample_loop(self, cond, shape, return_intermediates=False, x_T=None, verbose=True, callback=None,
                      timesteps=None, quantize_denoised=False, mask=None, x0=None, img_callback=None, start_T=None,
                      log_every_t=None, out=None, peer_ptrs=None, noise_rows=None):
        """upstream p_sample_loop: img, or (img, intermediates) with the start and every log_every_t-th step.
        Extensions (optional): ``out`` / ``peer_ptrs`` as in denoising_step, for the LAST step only; ``noise_rows`` as in
        _randn, for x_T and every step's noise."""
        if timesteps is None:
            timesteps = self.model.num_timesteps
        if start_T is not None:
            timesteps = min(timesteps, start_T)
        if mask is not None:
            assert x0 is not None
            assert x0.shape[2:3] == mask.shape[2:3]  # sic: upstream compares one spatial dimension
        img, intermediates = self._loop(cond, shape, x_T, timesteps, log_every_t, mask, x0, callback, img_callback, False,
                                        1., out, peer_ptrs, noise_rows, quantize_denoised=quantize_denoised)
        return (img, intermediates) if return_intermediates else img

    @torch.no_grad()
    def progressive_denoising(self, cond, shape, verbose=True, callback=None, quantize_denoised=False, img_callback=None,
                              mask=None, x0=None, temperature=1., noise_dropout=0., score_corrector=None,
                              corrector_kwargs=None, batch_size=None, x_T=None, start_T=None, log_every_t=None):
        """upstream progressive_denoising: (img, the x_recon of every log_every_t-th step); temperature is a float or one
        value per timestep, indexed by the timestep"""
        if batch_size is not None:
            shape = [batch_size] + list(shape)
        else:
            batch_size = shape[0]
        if cond is not None:
            cond = _slice_cond(cond, batch_size)
        timesteps = self.model.num_timesteps
        if start_T is not None:
            timesteps = min(timesteps, start_T)
        return self._loop(cond, shape, x_T, timesteps, log_every_t, mask, x0, callback, img_callback, True, temperature,
                          None, None, None, quantize_denoised=quantize_denoised, noise_dropout=noise_dropout,
                          score_corrector=score_corrector, corrector_kwargs=corrector_kwargs)

    @torch.no_grad()
    def sample(self, cond, batch_size=16, return_intermediates=False, x_T=None, verbose=True, timesteps=None,
               quantize_denoised=False, mask=None, x0=None, shape=None, **kwargs):
        """upstream LatentDiffusion.sample (not DDIM's sample(S, ...)): every cond leaf cut to batch_size rows, the
        default shape (batch_size, model.channels, model.image_size, model.image_size), then p_sample_loop"""
        m = self.model
        if shape is None:
            shape = (batch_size, m.channels, m.image_size, m.image_size)
        if cond is not None:
            cond = _slice_cond(cond, batch_size)
        return self.p_sample_loop(cond, shape, return_intermediates=return_intermediates, x_T=x_T, verbose=verbose,
                                  timesteps=timesteps, quantize_denoised=quantize_denoised, mask=mask, x0=x0)
