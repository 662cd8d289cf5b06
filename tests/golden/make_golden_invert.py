"""Generates tests/golden/ddim_invert_v1.npz from the ORACLE's DDIM inversion (CPU, fp32) — run from the repo root:

    python tests/golden/make_golden_invert.py

Upstream's DDIMSampler.encode is not vendored, so tests/oracle_invert.py restates it; these fixtures freeze that restatement
(any later edit of it that changes a bit trips tests/test_inversion.py).  The denoiser is the closed-form toy of
tests/toy_denoiser.py (eps depends on x, t and the cond rows), so the fixture pins the timesteps fed to the model, the
CFG batching order and the coefficient rounding of every step.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle_invert import InvertingDDIMSampler  # noqa: E402
from toy_denoiser import ToyDenoiser, toy_inputs  # noqa: E402

# (name, S, t_enc, guidance scale, use_original_steps, return_intermediates)
CASES = [("s50_full", 50, 50, 1.0, False, 5), ("s50_cfg5", 50, 50, 5.0, False, None), ("s20_t10", 20, 10, 1.0, False, 3),
         ("orig_t7", 50, 7, 1.0, True, None)]


def compute(make_sampler, device="cpu"):
    """{name: final x_t, name + '_inter': stacked intermediates (when asked for)} for every case"""
    i = toy_inputs(device)
    cond = {"c_crossattn": [i["ctx"]], "c_concat": [i["hint"]]}
    uc = {"c_crossattn": [i["uc_ctx"]], "c_concat": [i["hint"]]}
    x0 = i["x_T"]  # used here as the clean latent x_0
    out = {}
    for name, S, t_enc, scale, orig, ri in CASES:
        s = make_sampler()
        s.make_schedule(S, ddim_eta=0.0, verbose=False)
        x, d = s.encode(x0, cond, t_enc, use_original_steps=orig, return_intermediates=ri, unconditional_guidance_scale=scale,
                        unconditional_conditioning=uc if scale != 1.0 else None)
        out[name] = x
        if ri:
            out[name + "_inter"] = torch.stack(d["intermediates"])
            out[name + "_steps"] = torch.tensor(d["intermediate_steps"])
    return out


def main():
    torch.set_num_threads(4)
    m = ToyDenoiser()
    out = compute(lambda: InvertingDDIMSampler(m))
    path = os.path.join(HERE, "ddim_invert_v1.npz")
    np.savez_compressed(path, **{k: v.numpy() for k, v in out.items()})
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
