"""TEST-ONLY restatement of upstream ``ldm.models.diffusion.ddpm``'s DDPM ancestral sampling on ``LatentDiffusion``:
``register_schedule``'s posterior buffers (``v_posterior = 0``), ``noise_like``, ``extract_into_tensor``, ``q_sample``,
``predict_start_from_noise``, ``q_posterior``, ``p_mean_variance``, ``p_sample``, ``p_sample_loop``, ``sample`` and
``progressive_denoising``, limited to the eps parameterization.

Upstream's file (lllyasviel/ControlNet, from CompVis/latent-diffusion) is not vendored and cannot be read offline: this
is restated from its description, unchecked against the source, and pinned by the known answers of tests/test_ddpm.py
and the frozen fixture tests/golden/ddpm_v1.npz (tests/golden/make_golden_ddpm.py).
``DDPM(model)`` wraps anything with ``apply_model`` / ``parameterization`` / ``device`` (``oracle.OracleControlLDM``,
the toy denoiser) and carries the buffers itself, so ``oracle/`` stays as it is.  Deliberate differences: the progress
bars, ``shorten_cond_schedule``, codebook ids, ``quantize_denoised`` and ``score_corrector`` are left out; a None cond
leaf (this model's ``c_concat`` may be None) survives ``sample``'s slicing.
"""
import numpy as np
import torch

from oracle.ldm import linear_beta_alphas_cumprod


def noise_like(shape, device, repeat=False):
    repeat_noise = lambda: torch.randn((1, *shape[1:]), device=device).repeat(shape[0], *((1,) * (len(shape) - 1)))  # noqa: E731
    noise = lambda: torch.randn(shape, device=device)  # noqa: E731
    return repeat_noise() if repeat else noise()


def extract_into_tensor(a, t, x_shape):
    b, *_ = t.shape
    out = a.gather(-1, t)
    return out.reshape(b, *((1,) * (len(x_shape) - 1)))


def _slice(cond, batch_size):
    cut = lambda x: None if x is None else x[:batch_size]  # noqa: E731
    if isinstance(cond, dict):
        return {key: cut(cond[key]) if not isinstance(cond[key], list) else list(map(cut, cond[key])) for key in cond}
    return [cut(c) for c in cond] if isinstance(cond, list) else cut(cond)


class DDPM:
    """upstream LatentDiffusion's sampling methods over ``model``; also a model for B200DDPMSampler (it exposes the
    buffers and attributes that sampler reads)"""

    def __init__(self, model, timesteps=1000, linear_start=0.00085, linear_end=0.0120, clip_denoised=True,
                 log_every_t=100, channels=4, image_size=32):
        self.model = model
        self.parameterization = model.parameterization
        self.num_timesteps = int(timesteps)
        self.clip_denoised = clip_denoised
        self.log_every_t = log_every_t
        self.channels = channels
        self.image_size = image_size
        # register_schedule (given_betas None, beta_schedule "linear"), numpy float64, stored fp32
        betas = np.linspace(linear_start ** 0.5, linear_end ** 0.5, timesteps, dtype=np.float64) ** 2
        alphas = 1. - betas
        alphas_cumprod = linear_beta_alphas_cumprod(timesteps, linear_start, linear_end)
        alphas_cumprod_prev = np.append(1., alphas_cumprod[:-1])
        to_torch = lambda a: torch.tensor(a, dtype=torch.float32, device=model.device)  # noqa: E731
        self.betas = to_torch(betas)
        self.alphas_cumprod = to_torch(alphas_cumprod)
        self.alphas_cumprod_prev = to_torch(alphas_cumprod_prev)
        self.sqrt_alphas_cumprod = to_torch(np.sqrt(alphas_cumprod))
        self.sqrt_one_minus_alphas_cumprod = to_torch(np.sqrt(1. - alphas_cumprod))
        self.sqrt_recip_alphas_cumprod = to_torch(np.sqrt(1. / alphas_cumprod))
        self.sqrt_recipm1_alphas_cumprod = to_torch(np.sqrt(1. / alphas_cumprod - 1))
        v_posterior = 0.
        posterior_variance = (1 - v_posterior) * betas * (1. - alphas_cumprod_prev) / (1. - alphas_cumprod) + v_posterior * betas
        self.posterior_variance = to_torch(posterior_variance)
        self.posterior_log_variance_clipped = to_torch(np.log(np.maximum(posterior_variance, 1e-20)))
        self.posterior_mean_coef1 = to_torch(betas * np.sqrt(alphas_cumprod_prev) / (1. - alphas_cumprod))
        self.posterior_mean_coef2 = to_torch((1. - alphas_cumprod_prev) * np.sqrt(alphas) / (1. - alphas_cumprod))

    @property
    def device(self):
        return self.model.device

    def apply_model(self, x, t, c):
        return self.model.apply_model(x, t, c)

    def q_sample(self, x_start, t, noise=None):
        noise = torch.randn_like(x_start) if noise is None else noise
        return (extract_into_tensor(self.sqrt_alphas_cumprod, t, x_start.shape) * x_start +
                extract_into_tensor(self.sqrt_one_minus_alphas_cumprod, t, x_start.shape) * noise)

    def predict_start_from_noise(self, x_t, t, noise):
        return (extract_into_tensor(self.sqrt_recip_alphas_cumprod, t, x_t.shape) * x_t -
                extract_into_tensor(self.sqrt_recipm1_alphas_cumprod, t, x_t.shape) * noise)

    def q_posterior(self, x_start, x_t, t):
        posterior_mean = (extract_into_tensor(self.posterior_mean_coef1, t, x_t.shape) * x_start +
                          extract_into_tensor(self.posterior_mean_coef2, t, x_t.shape) * x_t)
        posterior_variance = extract_into_tensor(self.posterior_variance, t, x_t.shape)
        posterior_log_variance_clipped = extract_into_tensor(self.posterior_log_variance_clipped, t, x_t.shape)
        return posterior_mean, posterior_variance, posterior_log_variance_clipped

    def p_mean_variance(self, x, c, t, clip_denoised, return_x0=False):
        model_out = self.apply_model(x, t, c)
        assert self.parameterization == "eps"
        x_recon = self.predict_start_from_noise(x, t=t, noise=model_out)
        if clip_denoised:
            x_recon.clamp_(-1., 1.)
        model_mean, posterior_variance, posterior_log_variance = self.q_posterior(x_start=x_recon, x_t=x, t=t)
        if return_x0:
            return model_mean, posterior_variance, posterior_log_variance, x_recon
        return model_mean, posterior_variance, posterior_log_variance

    @torch.no_grad()
    def p_sample(self, x, c, t, clip_denoised=False, repeat_noise=False, return_x0=False, temperature=1.,
                 noise_dropout=0.):
        b, *_, device = *x.shape, x.device
        outputs = self.p_mean_variance(x=x, c=c, t=t, clip_denoised=clip_denoised, return_x0=return_x0)
        if return_x0:
            model_mean, _, model_log_variance, x0 = outputs
        else:
            model_mean, _, model_log_variance = outputs
        noise = noise_like(x.shape, device, repeat_noise) * temperature
        if noise_dropout > 0.:
            noise = torch.nn.functional.dropout(noise, p=noise_dropout)
        # no noise when t == 0
        nonzero_mask = (1 - (t == 0).float()).reshape(b, *((1,) * (len(x.shape) - 1)))
        if return_x0:
            return model_mean + nonzero_mask * (0.5 * model_log_variance).exp() * noise, x0
        return model_mean + nonzero_mask * (0.5 * model_log_variance).exp() * noise

    @torch.no_grad()
    def p_sample_loop(self, cond, shape, return_intermediates=False, x_T=None, verbose=True, callback=None,
                      timesteps=None, quantize_denoised=False, mask=None, x0=None, img_callback=None, start_T=None,
                      log_every_t=None):
        if not log_every_t:
            log_every_t = self.log_every_t
        device = self.betas.device
        b = shape[0]
        img = torch.randn(shape, device=device) if x_T is None else x_T
        intermediates = [img]
        if timesteps is None:
            timesteps = self.num_timesteps
        if start_T is not None:
            timesteps = min(timesteps, start_T)
        if mask is not None:
            assert x0 is not None
            assert x0.shape[2:3] == mask.shape[2:3]  # spatial size has to match
        for i in reversed(range(0, timesteps)):
            ts = torch.full((b,), i, device=device, dtype=torch.long)
            img = self.p_sample(img, cond, ts, clip_denoised=self.clip_denoised)
            if mask is not None:
                img_orig = self.q_sample(x0, ts)
                img = img_orig * mask + (1. - mask) * img
            if i % log_every_t == 0 or i == timesteps - 1:
                intermediates.append(img)
            if callback:
                callback(i)
            if img_callback:
                img_callback(img, i)
        if return_intermediates:
            return img, intermediates
        return img

    @torch.no_grad()
    def sample(self, cond, batch_size=16, return_intermediates=False, x_T=None, verbose=True, timesteps=None,
               quantize_denoised=False, mask=None, x0=None, shape=None, **kwargs):
        if shape is None:
            shape = (batch_size, self.channels, self.image_size, self.image_size)
        if cond is not None:
            cond = _slice(cond, batch_size)
        return self.p_sample_loop(cond, shape, return_intermediates=return_intermediates, x_T=x_T, verbose=verbose,
                                  timesteps=timesteps, quantize_denoised=quantize_denoised, mask=mask, x0=x0)

    @torch.no_grad()
    def progressive_denoising(self, cond, shape, verbose=True, callback=None, quantize_denoised=False, img_callback=None,
                              mask=None, x0=None, temperature=1., noise_dropout=0., score_corrector=None,
                              corrector_kwargs=None, batch_size=None, x_T=None, start_T=None, log_every_t=None):
        if not log_every_t:
            log_every_t = self.log_every_t
        timesteps = self.num_timesteps
        if batch_size is not None:
            b = batch_size if batch_size is not None else shape[0]
            shape = [batch_size] + list(shape)
        else:
            b = batch_size = shape[0]
        img = torch.randn(shape, device=self.device) if x_T is None else x_T
        intermediates = []
        if cond is not None:
            cond = _slice(cond, batch_size)
        if start_T is not None:
            timesteps = min(timesteps, start_T)
        if type(temperature) == float:  # noqa: E721
            temperature = [temperature] * timesteps
        for i in reversed(range(0, timesteps)):
            ts = torch.full((b,), i, device=self.device, dtype=torch.long)
            img, x0_partial = self.p_sample(img, cond, ts, clip_denoised=self.clip_denoised, return_x0=True,
                                            temperature=temperature[i], noise_dropout=noise_dropout)
            if mask is not None:
                assert x0 is not None
                img_orig = self.q_sample(x0, ts)
                img = img_orig * mask + (1. - mask) * img
            if i % log_every_t == 0 or i == timesteps - 1:
                intermediates.append(x0_partial)
            if callback:
                callback(i)
            if img_callback:
                img_callback(img, i)
        return img, intermediates
