"""TEST-ONLY restatement of upstream ``DDIMSampler.encode`` (DDIM inversion, x_0 -> x_t) on top of the oracle sampler.

Upstream ``ldm/models/diffusion/ddim.py`` (lllyasviel/ControlNet) is not vendored and cannot be read offline: this is
restated from memory, unchecked against the source, and pinned only by the known answers of tests/test_inversion.py and
the frozen fixture tests/golden/ddim_invert_v1.npz (tests/golden/make_golden_invert.py).  One deliberate superset: the
doubled CFG cond is built with the oracle's ``_cat_uncond_first`` (upstream's ``torch.cat((uc, c))`` takes bare tensors
only and raises for this model's dict cond).
"""
import torch

from oracle import MKDDIMSampler
from oracle.ddim import _cat_uncond_first


class InvertingDDIMSampler(MKDDIMSampler):
    """``MKDDIMSampler`` plus the ``encode`` it inherits from upstream ``DDIMSampler``"""

    @torch.no_grad()
    def encode(self, x0, c, t_enc, use_original_steps=False, return_intermediates=None,
               unconditional_guidance_scale=1.0, unconditional_conditioning=None, callback=None):
        num_reference_steps = self.ddpm_num_timesteps if use_original_steps else self.ddim_timesteps.shape[0]
        assert t_enc <= num_reference_steps
        num_steps = t_enc
        if use_original_steps:
            alphas_next = self.alphas_cumprod[:num_steps]
            alphas = self.alphas_cumprod_prev[:num_steps]
        else:
            alphas_next = self.ddim_alphas[:num_steps]
            alphas = torch.tensor(self.ddim_alphas_prev[:num_steps])  # float64
        x_next = x0
        intermediates, inter_steps = [], []
        for i in range(num_steps):
            t = torch.full((x0.shape[0],), i, device=self.model.device, dtype=torch.long)  # the loop index, as upstream
            if unconditional_guidance_scale == 1.0:
                noise_pred = self.model.apply_model(x_next, t, c)
            else:
                assert unconditional_conditioning is not None
                e_t_uncond, noise_pred = torch.chunk(self.model.apply_model(
                    torch.cat((x_next, x_next)), torch.cat((t, t)), _cat_uncond_first(unconditional_conditioning, c)), 2)
                noise_pred = e_t_uncond + unconditional_guidance_scale * (noise_pred - e_t_uncond)
            xt_weighted = (alphas_next[i] / alphas[i]).sqrt() * x_next
            weighted_noise_pred = alphas_next[i].sqrt() * ((1 / alphas_next[i] - 1).sqrt() - (1 / alphas[i] - 1).sqrt()) * noise_pred
            x_next = xt_weighted + weighted_noise_pred
            if return_intermediates and i % (num_steps // return_intermediates) == 0 and i < num_steps - 1:
                intermediates.append(x_next)
                inter_steps.append(i)
            elif return_intermediates and i >= num_steps - 2:
                intermediates.append(x_next)
                inter_steps.append(i)
            if callback:
                callback(i)
        out = {"x_encoded": x_next, "intermediate_steps": inter_steps}
        if return_intermediates:
            out.update({"intermediates": intermediates})
        return x_next, out
