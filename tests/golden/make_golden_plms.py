"""Generates tests/golden/plms_v1.npz from the ORACLE's PLMS sampler (CPU, fp32) — run from the repo root:

    python tests/golden/make_golden_plms.py

Upstream's PLMSSampler is not vendored, so tests/oracle_plms.py restates it; these fixtures freeze that restatement (any
later edit of it that changes a bit trips tests/test_plms.py).  The denoiser is the closed-form toy of
tests/toy_denoiser.py (eps depends on x, t and the cond rows), so the fixture pins the timesteps fed to the model (two
evaluations at step 0), the CFG batching order, the multistep coefficients of every history length and their rounding.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle_plms import PLMSSampler  # noqa: E402
from toy_denoiser import ToyDenoiser, toy_inputs  # noqa: E402

# (name, S, guidance scale, log_every_t or None for the final latents only).  S = 4 is the shortest schedule whose steps see
# every history length (0, 1, 2, 3 earlier eps); S = 3 has no uniform schedule here (its fourth timestep would be 1000).
CASES = [("s50", 50, 1.0, 10), ("s20_cfg5", 20, 5.0, None), ("s1", 1, 1.0, None), ("s4", 4, 1.0, 1),
         ("s4_cfg5", 4, 5.0, None)]


def compute(make_sampler, device="cpu"):
    """{name: final latents, name + '_x_inter' / '_pred_x0': stacked intermediates (when logged)} for every case"""
    i = toy_inputs(device)
    cond = {"c_crossattn": [i["ctx"]], "c_concat": [i["hint"]]}
    uc = {"c_crossattn": [i["uc_ctx"]], "c_concat": [i["hint"]]}
    out = {}
    for name, S, scale, log_every in CASES:
        s = make_sampler()
        x, inter = s.sample(S, i["x_T"].shape[0], tuple(i["x_T"].shape[1:]), cond, x_T=i["x_T"], verbose=False,
                            unconditional_guidance_scale=scale, unconditional_conditioning=uc if scale != 1.0 else None,
                            log_every_t=log_every or 100)
        out[name] = x
        if log_every:
            out[name + "_x_inter"] = torch.stack(inter["x_inter"])
            out[name + "_pred_x0"] = torch.stack(inter["pred_x0"])
    return out


def main():
    torch.set_num_threads(4)
    m = ToyDenoiser()
    out = compute(lambda: PLMSSampler(m))
    path = os.path.join(HERE, "plms_v1.npz")
    np.savez_compressed(path, **{k: v.numpy() for k, v in out.items()})
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
