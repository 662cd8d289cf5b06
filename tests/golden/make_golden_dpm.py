"""Generates tests/golden/dpm_v1.npz from the ORACLE's DPM-Solver sampler (CPU, fp32) — run from the repo root:

    python tests/golden/make_golden_dpm.py

Upstream's DPMSolverSampler is not vendored, so tests/oracle_dpm.py restates it; these fixtures freeze that restatement
(any later edit of it that changes a bit trips tests/test_dpm_solver.py).  The denoiser is the closed-form toy of
tests/toy_denoiser.py (eps depends on x, t and the cond rows), so the fixture pins the fractional model times, the CFG
batching order, the order of every step (S = 2: two order-1 steps; S = 14: the last step order 1; S = 15 and 20: order 2
to the end) and the rounding of every update.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle_dpm import DPMSolverSampler  # noqa: E402
from toy_denoiser import ToyDenoiser, toy_inputs  # noqa: E402

# (name, S, guidance scale)
CASES = [("s20", 20, 1.0), ("s20_cfg5", 20, 5.0), ("s2", 2, 1.0), ("s14", 14, 1.0), ("s15", 15, 1.0)]


def compute(make_sampler, device="cpu"):
    """{name: final latents} for every case"""
    i = toy_inputs(device)
    cond = {"c_crossattn": [i["ctx"]], "c_concat": [i["hint"]]}
    uc = {"c_crossattn": [i["uc_ctx"]], "c_concat": [i["hint"]]}
    out = {}
    for name, S, scale in CASES:
        x, _ = make_sampler().sample(S, i["x_T"].shape[0], tuple(i["x_T"].shape[1:]), cond, x_T=i["x_T"], verbose=False,
                                     unconditional_guidance_scale=scale,
                                     unconditional_conditioning=uc if scale != 1.0 else None)
        out[name] = x
    return out


def main():
    torch.set_num_threads(4)
    m = ToyDenoiser()
    out = compute(lambda: DPMSolverSampler(m))
    path = os.path.join(HERE, "dpm_v1.npz")
    np.savez_compressed(path, **{k: v.numpy() for k, v in out.items()})
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
