#!/usr/bin/env python
"""PLMS against DDIM sampling throughput on one B200 at BASELINE.json configs[1]'s shape (yaml-size networks, 256^2,
batch 16, bf16, synthetic seeded inputs drawn as bench.py draws them), all in one run:

  plms_50 / plms_20  images/s of B200PLMSSampler.sample(S): S + 1 UNet+ControlNet evaluations
  ddim_50 / ddim_20  images/s of B200DDIMSampler.sample(S) on the same batch: S evaluations

Each pass is timed alone with CUDA events after warm-up passes; the JSON gives mean / min / max / stdev over the passes,
the ratio of each PLMS rate to the DDIM rate of the same S, and the card's name and power limit read in the same run.
The four workloads are timed interleaved pass by pass, so a drift of the shared machine's clocks spreads over all of them.

    python tools/plms_bench.py [--passes K] [--warmup W] [--batch B] [--out FILE]
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
    from makeupdiffuse_b200 import B200ControlLDM, B200DDIMSampler, B200PLMSSampler
    from makeupdiffuse_b200.synth import synthetic_batch, synthetic_state_dict

    if not torch.cuda.is_available():
        raise SystemExit("plms_bench.py needs a B200: the B200 path has no CPU fallback")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    B, size, h = args.batch, args.size, args.size // 8
    model = B200ControlLDM(dtype=torch.bfloat16, device=dev)
    model.load_state_dict(synthetic_state_dict(model, 0, dev))
    data = synthetic_batch(B, size, 768, seed=1234, device=dev)
    cond = {"c_crossattn": [data["ctx"]], "c_concat": [torch.cat([data["src"], data["ref"]], 1)]}
    samplers = {"plms": B200PLMSSampler(model), "ddim": B200DDIMSampler(model)}

    def make(kind, S):
        return lambda: samplers[kind].sample(S, B, (4, h, h), cond, eta=0.0, x_T=data["x_T"], verbose=False)[0]

    work = {f"{k}_{S}": make(k, S) for S in (50, 20) for k in ("plms", "ddim")}
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
    ratio = {f"plms_over_ddim_{S}": res[f"plms_{S}"]["images_per_s"] / res[f"ddim_{S}"]["images_per_s"] for S in (50, 20)}
    line = {"metric": f"PLMS vs DDIM sampling images/s at {size}^2", "card": card(), "batch": B, "dtype": "bf16",
            "data": "synthetic (bench.py's synthetic_batch, seed 1234)", "cuda_graph": True, "guidance": "none (scale 1)",
            "timing": f"CUDA events around each pass, {args.warmup} warm-up passes each, {args.passes} timed passes "
                      "interleaved across the four workloads",
            "what": {"plms_S": "B200PLMSSampler.sample(S): S + 1 model evaluations",
                     "ddim_S": "B200DDIMSampler.sample(S), eta 0: S model evaluations (bench.py's workload at S = 50)"},
            **res, "ratio": ratio, "ratio_if_evaluation_bound": {"50": 50 / 51, "20": 20 / 21}}
    text = json.dumps(line)
    print(text, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(line, indent=1) + "\n")


if __name__ == "__main__":
    main()
