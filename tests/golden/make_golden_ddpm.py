"""Generates tests/golden/ddpm_v1.npz from the ORACLE's DDPM ancestral loop (CPU, fp32) — run from the repo root:

    python tests/golden/make_golden_ddpm.py

Upstream's LatentDiffusion is not vendored, so tests/oracle_ddpm.py restates its sampling methods; these fixtures freeze
that restatement (any later edit of it that changes a bit trips tests/test_ddpm.py).  The denoiser is the closed-form toy
of tests/toy_denoiser.py (eps depends on x, t and the cond rows).  Each case seeds torch's generator, so the fixture also
pins the RNG stream: one randn(x.shape) per step including t = 0, and the mask blend's own draw after the step.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle_ddpm import DDPM  # noqa: E402
from toy_denoiser import ToyDenoiser, toy_inputs  # noqa: E402

# name -> (clip_denoised, p_sample_loop keyword arguments); "mask" / "x0" are filled in by compute()
CASES = {"full_clip": (True, {}), "full_noclip": (False, {}), "start_T_250": (True, {"start_T": 250}),
         "mask_start_T_50": (True, {"start_T": 50, "mask": None})}


def toy_mask(i):
    """keep the left half of every latent from x0 (1), denoise the right half (0)"""
    m = torch.zeros_like(i["x_T"][:, :1])
    m[..., : m.shape[-1] // 2] = 1.0
    return m


def compute(make_ddpm, device="cpu", seed=1234):
    """{name: final latents} for every case; make_ddpm(clip) returns the DDPM object (oracle or B200 sampler) to run"""
    i = toy_inputs(device)
    cond = {"c_crossattn": [i["ctx"]], "c_concat": [i["hint"]]}
    out = {}
    for name, (clip, kw) in CASES.items():
        kw = dict(kw)
        if "mask" in kw:
            kw["mask"], kw["x0"] = toy_mask(i), 0.5 * torch.tanh(i["x_T"])
        torch.manual_seed(seed)
        out[name] = make_ddpm(clip).p_sample_loop(cond, tuple(i["x_T"].shape), x_T=i["x_T"], verbose=False, **kw)
    return out


def main():
    torch.set_num_threads(4)
    m = ToyDenoiser()
    out = compute(lambda clip: DDPM(m, clip_denoised=clip))
    path = os.path.join(HERE, "ddpm_v1.npz")
    np.savez_compressed(path, **{k: v.numpy() for k, v in out.items()})
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
