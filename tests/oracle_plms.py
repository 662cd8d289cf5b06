"""TEST-ONLY restatement of upstream ``ldm.models.diffusion.plms.PLMSSampler`` on top of the oracle DDIM sampler.

Upstream ``ldm/models/diffusion/plms.py`` (lllyasviel/ControlNet) is not vendored and cannot be read offline: this is
restated from its description (schedule, loop, p_sample_plms), unchecked against the source, and pinned by the known
answers of tests/test_plms.py and the frozen fixture tests/golden/plms_v1.npz (tests/golden/make_golden_plms.py).
One deliberate superset: the doubled CFG cond is built with the oracle's ``_cat_uncond_first`` (upstream's
``torch.cat([unconditional_conditioning, c])`` takes bare tensors only and raises for this model's dict cond).
"""
import numpy as np
import torch

from oracle.ddim import DDIMSampler, _cat_uncond_first


class PLMSSampler(DDIMSampler):
    def make_schedule(self, ddim_num_steps, ddim_discretize="uniform", ddim_eta=0.0, verbose=True):
        if ddim_eta != 0:
            raise ValueError("ddim_eta must be 0 for PLMS")
        super().make_schedule(ddim_num_steps, ddim_discretize=ddim_discretize, ddim_eta=ddim_eta, verbose=verbose)

    @torch.no_grad()
    def sample(self, S, batch_size, shape, conditioning=None, callback=None, normals_sequence=None, img_callback=None,
               quantize_x0=False, eta=0.0, mask=None, x0=None, temperature=1.0, noise_dropout=0.0, score_corrector=None,
               corrector_kwargs=None, verbose=True, x_T=None, log_every_t=100, unconditional_guidance_scale=1.0,
               unconditional_conditioning=None, dynamic_threshold=None, **kwargs):
        self.make_schedule(ddim_num_steps=S, ddim_eta=eta, verbose=verbose)
        C, H, W = shape
        return self.plms_sampling(conditioning, (batch_size, C, H, W), callback=callback, img_callback=img_callback,
                                  quantize_denoised=quantize_x0, mask=mask, x0=x0, ddim_use_original_steps=False,
                                  noise_dropout=noise_dropout, temperature=temperature, score_corrector=score_corrector,
                                  corrector_kwargs=corrector_kwargs, x_T=x_T, log_every_t=log_every_t,
                                  unconditional_guidance_scale=unconditional_guidance_scale,
                                  unconditional_conditioning=unconditional_conditioning,
                                  dynamic_threshold=dynamic_threshold)

    @torch.no_grad()
    def plms_sampling(self, cond, shape, x_T=None, ddim_use_original_steps=False, callback=None, timesteps=None,
                      quantize_denoised=False, mask=None, x0=None, img_callback=None, log_every_t=100, temperature=1.0,
                      noise_dropout=0.0, score_corrector=None, corrector_kwargs=None, unconditional_guidance_scale=1.0,
                      unconditional_conditioning=None, dynamic_threshold=None):
        dev = self.model.device
        b = shape[0]
        img = torch.randn(shape, device=dev) if x_T is None else x_T
        assert timesteps is None and not ddim_use_original_steps  # the only form the sample() entry uses
        intermediates = {"x_inter": [img], "pred_x0": [img]}
        time_range = np.flip(self.ddim_timesteps)
        total_steps = self.ddim_timesteps.shape[0]
        old_eps = []
        for i, step in enumerate(time_range):
            index = total_steps - i - 1
            ts = torch.full((b,), int(step), device=dev, dtype=torch.long)
            ts_next = torch.full((b,), int(time_range[min(i + 1, len(time_range) - 1)]), device=dev, dtype=torch.long)
            if mask is not None:
                assert x0 is not None
                img_orig = self.model.q_sample(x0, ts)
                img = img_orig * mask + (1.0 - mask) * img
            img, pred_x0, e_t = self.p_sample_plms(
                img, cond, ts, index=index, use_original_steps=ddim_use_original_steps,
                quantize_denoised=quantize_denoised, temperature=temperature, noise_dropout=noise_dropout,
                score_corrector=score_corrector, corrector_kwargs=corrector_kwargs,
                unconditional_guidance_scale=unconditional_guidance_scale,
                unconditional_conditioning=unconditional_conditioning, old_eps=old_eps, t_next=ts_next,
                dynamic_threshold=dynamic_threshold)
            old_eps.append(e_t)
            if len(old_eps) >= 4:
                old_eps.pop(0)
            if callback:
                callback(i)
            if img_callback:
                img_callback(pred_x0, i)
            if index % log_every_t == 0 or index == total_steps - 1:
                intermediates["x_inter"].append(img)
                intermediates["pred_x0"].append(pred_x0)
        return img, intermediates

    @torch.no_grad()
    def p_sample_plms(self, x, c, t, index, repeat_noise=False, use_original_steps=False, quantize_denoised=False,
                      temperature=1.0, noise_dropout=0.0, score_corrector=None, corrector_kwargs=None,
                      unconditional_guidance_scale=1.0, unconditional_conditioning=None, old_eps=None, t_next=None,
                      dynamic_threshold=None):
        b, dev = x.shape[0], x.device
        m = self.model

        def get_model_output(x, t):
            if unconditional_conditioning is None or unconditional_guidance_scale == 1.0:
                e_t = m.apply_model(x, t, c)
            else:
                x_in = torch.cat([x] * 2)
                t_in = torch.cat([t] * 2)
                c_in = _cat_uncond_first(unconditional_conditioning, c)
                e_t_uncond, e_t = m.apply_model(x_in, t_in, c_in).chunk(2)
                e_t = e_t_uncond + unconditional_guidance_scale * (e_t - e_t_uncond)
            if score_corrector is not None:
                assert m.parameterization == "eps"
                e_t = score_corrector.modify_score(m, e_t, x, t, c, **corrector_kwargs)
            return e_t

        alphas = m.alphas_cumprod if use_original_steps else self.ddim_alphas
        alphas_prev = m.alphas_cumprod_prev if use_original_steps else self.ddim_alphas_prev
        sqrt_one_minus_alphas = m.sqrt_one_minus_alphas_cumprod if use_original_steps else self.ddim_sqrt_one_minus_alphas
        sigmas = m.ddim_sigmas_for_original_num_steps if use_original_steps else self.ddim_sigmas

        def get_x_prev_and_pred_x0(e_t, index):
            full = lambda v: torch.full((b, 1, 1, 1), float(v[index]), device=dev)  # noqa: E731
            a_t, a_prev, sigma_t, sqrt_one_minus_at = full(alphas), full(alphas_prev), full(sigmas), full(sqrt_one_minus_alphas)
            pred_x0 = (x - sqrt_one_minus_at * e_t) / a_t.sqrt()
            if quantize_denoised:
                pred_x0, _, *_ = m.first_stage_model.quantize(pred_x0)
            if dynamic_threshold is not None:
                raise NotImplementedError()
            dir_xt = (1.0 - a_prev - sigma_t ** 2).sqrt() * e_t
            draw = torch.randn((1, *x.shape[1:]) if repeat_noise else x.shape, device=dev)
            if repeat_noise:
                draw = draw.repeat(b, *((1,) * (len(x.shape) - 1)))
            noise = sigma_t * draw * temperature
            if noise_dropout > 0.0:
                noise = torch.nn.functional.dropout(noise, p=noise_dropout)
            x_prev = a_prev.sqrt() * pred_x0 + dir_xt + noise
            return x_prev, pred_x0

        e_t = get_model_output(x, t)
        if len(old_eps) == 0:
            # pseudo improved Euler (2nd order)
            x_prev, pred_x0 = get_x_prev_and_pred_x0(e_t, index)
            e_t_next = get_model_output(x_prev, t_next)
            e_t_prime = (e_t + e_t_next) / 2
        elif len(old_eps) == 1:
            # 2nd order pseudo linear multistep (Adams-Bashforth)
            e_t_prime = (3 * e_t - old_eps[-1]) / 2
        elif len(old_eps) == 2:
            # 3rd order pseudo linear multistep (Adams-Bashforth)
            e_t_prime = (23 * e_t - 16 * old_eps[-1] + 5 * old_eps[-2]) / 12
        else:
            # 4th order pseudo linear multistep (Adams-Bashforth)
            e_t_prime = (55 * e_t - 59 * old_eps[-1] + 37 * old_eps[-2] - 9 * old_eps[-3]) / 24
        x_prev, pred_x0 = get_x_prev_and_pred_x0(e_t_prime, index)
        return x_prev, pred_x0, e_t
