#!/usr/bin/env python
"""DPM-Solver++ against DDIM sampling throughput on one B200 at BASELINE.json configs[1]'s shape (yaml-size networks,
256^2, batch 16, bf16, synthetic seeded inputs drawn as bench.py draws them), all in one run:

  dpm_20 / dpm_10    images/s of B200DPMSolverSampler.sample(S): S UNet+ControlNet evaluations at fractional times
  ddim_20 / ddim_50  images/s of B200DDIMSampler.sample(S) on the same batch: S evaluations

Each pass is timed alone with CUDA events after warm-up passes; the JSON gives mean / min / max / stdev over the passes,
the ratio of each rate to DDIM-20's, and the card's name and power limit read in the same run.  The four workloads are
timed interleaved pass by pass, so a drift of the shared machine's clocks spreads over all of them.

    python tools/dpm_bench.py [--passes K] [--warmup W] [--batch B] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from invert_bench import card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--passes", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    if args.passes < 2:
        ap.error("--passes must be at least 2 (the spread needs two)")

    import torch
    from makeupdiffuse_b200 import B200ControlLDM, B200DDIMSampler, B200DPMSolverSampler
    from makeupdiffuse_b200.synth import synthetic_batch, synthetic_state_dict

    if not torch.cuda.is_available():
        raise SystemExit("dpm_bench.py needs a B200: the B200 path has no CPU fallback")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    B, size, h = args.batch, args.size, args.size // 8
    model = B200ControlLDM(dtype=torch.bfloat16, device=dev)
    model.load_state_dict(synthetic_state_dict(model, 0, dev))
    data = synthetic_batch(B, size, 768, seed=1234, device=dev)
    cond = {"c_crossattn": [data["ctx"]], "c_concat": [torch.cat([data["src"], data["ref"]], 1)]}
    samplers = {"dpm": B200DPMSolverSampler(model), "ddim": B200DDIMSampler(model)}

    def make(kind, S):
        return lambda: samplers[kind].sample(S, B, (4, h, h), cond, eta=0.0, x_T=data["x_T"], verbose=False)[0]

    work = {f"{k}_{S}": make(k, S) for k, S in (("dpm", 20), ("dpm", 10), ("ddim", 20), ("ddim", 50))}
    for fn in work.values():
        for _ in range(args.warmup):
            fn()
    torch.cuda.synchronize()
    ms = {name: [] for name in work}
    for _ in range(args.passes):
        for name, fn in work.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn()
            e1.record()
            torch.cuda.synchronize()
            ms[name].append(e0.elapsed_time(e1))
            assert torch.isfinite(out).all()
    res = {}
    for name, t in ms.items():
        ips = [B / (m / 1e3) for m in t]
        res[name] = {"images_per_s": statistics.mean(ips), "images_per_s_min": min(ips), "images_per_s_max": max(ips),
                     "images_per_s_stdev": statistics.stdev(ips), "ms_per_pass": [round(m, 3) for m in t]}
    ratio = {f"{name}_over_ddim_20": res[name]["images_per_s"] / res["ddim_20"]["images_per_s"] for name in res}
    line = {"metric": f"DPM-Solver++ vs DDIM sampling images/s at {size}^2", "card": card(), "batch": B, "dtype": "bf16",
            "data": "synthetic (bench.py's synthetic_batch, seed 1234)", "cuda_graph": True, "guidance": "none (scale 1)",
            "timing": f"CUDA events around each pass, {args.warmup} warm-up passes each, {args.passes} timed passes "
                      "interleaved across the four workloads",
            "what": {"dpm_S": "B200DPMSolverSampler.sample(S) (DPM-Solver++(2M)): S model evaluations",
                     "ddim_S": "B200DDIMSampler.sample(S), eta 0: S model evaluations (bench.py's workload at S = 50)"},
            **res, "ratio": ratio, "ratio_if_evaluation_bound": {"dpm_20": 1.0, "dpm_10": 2.0, "ddim_50": 20 / 50}}
    text = json.dumps(line)
    print(text, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(line, indent=1) + "\n")


if __name__ == "__main__":
    main()
