"""TEST-ONLY stand-in for makeupdiffuse_b200.ops.ddpm_update (mkd_ddpm_update of include/mkd_b200.h), in the style of
tests/fake_dpm_ops.py: upstream ddpm.py's own torch expressions (extract_into_tensor, predict_start_from_noise, the clamp,
q_posterior, p_sample's noise term) on the CPU, so that B200DDPMSampler's host logic (the loop, the RNG stream, the
tables, the mask blend) can be tested without a GPU.  Never imported by the product."""
import torch

import fake_dpm_ops


def ddpm_update(x, eps, t, x_prev, *, tables, noise, clip, temperature=1.0, x0_out=None, peer_ptrs=None):
    assert peer_ptrs is None, "peer stores need real GPUs"
    assert t.dtype == torch.int64 and t.shape == (x.shape[0],) and tables.shape[0] == 5
    b = x.shape[0]
    ex = lambda k: tables[k].gather(-1, t).reshape(b, *((1,) * (x.dim() - 1)))  # noqa: E731
    x_recon = ex(0) * x - ex(1) * eps
    if clip:
        x_recon = x_recon.clamp(-1., 1.)
    mean = ex(2) * x_recon + ex(3) * x
    nonzero_mask = (1 - (t == 0).float()).reshape(b, *((1,) * (x.dim() - 1)))
    xp = mean + nonzero_mask * ex(4) * (noise * temperature)
    # stores after every read: x_prev may be x, as the kernel allows
    if x0_out is not None:
        x0_out.copy_(x_recon)
    x_prev.copy_(xp)


def install(ops, patch=setattr):
    """replace every C-ABI wrapper of ``ops`` by its torch stand-in (patch: monkeypatch.setattr in the pytest process,
    plain setattr in a spawned worker)"""
    fake_dpm_ops.install(ops, patch)
    patch(ops, "ddpm_update", ddpm_update)
