"""TEST-ONLY stand-ins for makeupdiffuse_b200.ops.dpm_update (mkd_dpm_update) and ops.timestep_embedding_f32
(mkd_timestep_embedding_f32) of include/mkd_b200.h, in the style of tests/fake_ops.py: upstream dpm_solver.py's and
timestep_embedding's own torch expressions on the CPU, so that B200DPMSolverSampler's host logic (the model times, the
data-prediction ring, the order of every step) and the fractional-timestep path through the networks can be tested
without a GPU.  Never imported by the product."""
import math

import torch

import fake_ops
import fake_plms_ops


def dpm_update(x, eps, x_prev, *, alpha_s, sigma_s, sigma_ratio, phi, order=1, m_prev=None, half_phi=0.0, inv_r0=0.0,
               m_store=None, cfg_scale=None, peer_ptrs=None):
    """upstream's expressions (model_wrapper's CFG combine, data_prediction_fn, the order-1 / order-2 multistep update)"""
    assert peer_ptrs is None, "peer stores need real GPUs"
    assert order in (1, 2) and (order == 2) == (m_prev is not None)
    f = lambda v: torch.tensor(v, dtype=torch.float32)  # noqa: E731
    e = eps
    if cfg_scale is not None:
        eu, ec = eps.chunk(2)
        e = eu + f(cfg_scale) * (ec - eu)
    m = (x - f(sigma_s) * e) / f(alpha_s)
    xp = f(sigma_ratio) * x - f(phi) * m
    if order == 2:
        xp = xp - f(half_phi) * (f(inv_r0) * (m - m_prev))
    # stores after every read: x_prev may be x, as the kernel allows
    if m_store is not None:
        m_store.copy_(m)
    x_prev.copy_(xp)


def timestep_embedding_f32(t, out, max_period=10000.0):
    assert t.dtype == torch.float32
    B, dim = out.shape
    half = dim // 2
    freqs = torch.exp(-math.log(max_period) * torch.arange(half, dtype=torch.float32) / half)
    args = t[:, None].float() * freqs[None]
    out.copy_(torch.cat([torch.cos(args), torch.sin(args)], -1))


def timestep_embedding(t, out, max_period=10000.0):
    """the int64 entry point takes integer timesteps only, as mkd_timestep_embedding does"""
    assert t.dtype == torch.int64
    fake_ops.timestep_embedding(t, out, max_period)


def install(ops, patch=setattr):
    """replace every C-ABI wrapper of ``ops`` by its torch stand-in (patch: monkeypatch.setattr in the pytest process,
    plain setattr in a spawned worker)"""
    fake_plms_ops.install(ops, patch)
    patch(ops, "timestep_embedding", timestep_embedding)
    patch(ops, "timestep_embedding_f32", timestep_embedding_f32)
    patch(ops, "dpm_update", dpm_update)
