#!/usr/bin/env python
"""DDPM ancestral sampling against DDIM-50 on one B200 at BASELINE.json configs[1]'s shape (yaml-size networks, 256^2,
batch 16, bf16, synthetic seeded inputs drawn as bench.py draws them), all in one run:

  ddpm_1000       images/s of B200DDPMSampler.p_sample_loop: 1000 UNet+ControlNet evaluations
  ddpm_start_250  images/s of the same loop from start_T = 250 (upstream's partial denoise of a noised x_T)
  ddim_50         images/s of B200DDIMSampler.sample(50) on the same batch (bench.py's workload)
  update_kernel   microseconds per mkd_ddpm_update launch at this shape, from CUDA events over many back-to-back launches

Each pass is timed alone with CUDA events after a warm-up pass; the JSON gives mean / min / max / stdev over the passes,
the per-evaluation time of each loop, the size of the per-loop timestep-embedding table at 1000 rows, and the card's name
and power limit read in the same run.  The three loops are timed interleaved pass by pass.

    python tools/ddpm_bench.py [--passes K] [--batch B] [--out FILE]
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
    ap.add_argument("--passes", type=int, default=3)
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--launches", type=int, default=2000, help="update-kernel launches in its timed window")
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    if args.passes < 2:
        ap.error("--passes must be at least 2 (the spread needs two)")

    import torch
    from makeupdiffuse_b200 import B200ControlLDM, B200DDIMSampler, B200DDPMSampler, ops
    from makeupdiffuse_b200.synth import synthetic_batch, synthetic_state_dict

    if not torch.cuda.is_available():
        raise SystemExit("ddpm_bench.py needs a B200: the B200 path has no CPU fallback")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    B, size, h = args.batch, args.size, args.size // 8
    model = B200ControlLDM(dtype=torch.bfloat16, device=dev)
    model.load_state_dict(synthetic_state_dict(model, 0, dev))
    data = synthetic_batch(B, size, 768, seed=1234, device=dev)
    cond = {"c_crossattn": [data["ctx"]], "c_concat": [torch.cat([data["src"], data["ref"]], 1)]}
    ddpm, ddim = B200DDPMSampler(model), B200DDIMSampler(model)
    shape = (B, 4, h, h)

    def loop(start_T):
        def run():
            torch.manual_seed(0)
            return ddpm.p_sample_loop(cond, shape, x_T=data["x_T"], verbose=False, start_T=start_T)
        return run

    work = {"ddpm_1000": (loop(None), 1000), "ddpm_start_250": (loop(250), 250),
            "ddim_50": (lambda: ddim.sample(50, B, shape[1:], cond, eta=0.0, x_T=data["x_T"], verbose=False)[0], 50)}
    for fn, _ in work.values():
        fn()
    ddpm.begin_loop(range(999, -1, -1))
    tab = model._emb_table["tab"]
    table = {"shape": list(tab.shape), "dtype": str(tab.dtype).replace("torch.", ""),
             "mib": round(tab.numel() * tab.element_size() / 2 ** 20, 2)}
    torch.cuda.synchronize()
    ms = {name: [] for name in work}
    for _ in range(args.passes):
        for name, (fn, _) in work.items():
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
                     "images_per_s_stdev": statistics.stdev(ips), "ms_per_pass": [round(m, 3) for m in t],
                     "ms_per_evaluation": statistics.mean(t) / work[name][1]}

    # the update kernel alone: back-to-back launches at the loop's shape, rows at mixed t
    g = torch.Generator(device=dev).manual_seed(0)
    x, eps, noise = (torch.randn(shape, device=dev, generator=g) for _ in range(3))
    t = torch.randint(0, 1000, (B,), device=dev, generator=g)
    out, x0 = torch.empty_like(x), torch.empty_like(x)
    tables = ddpm._tables()
    for _ in range(50):
        ops.ddpm_update(x, eps, t, out, tables=tables, noise=noise, clip=True, x0_out=x0)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.launches):
        ops.ddpm_update(x, eps, t, out, tables=tables, noise=noise, clip=True, x0_out=x0)
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / args.launches
    # x, eps, noise read, x_prev and x0 written: fp32 latents; the tables are a few L1-resident entries per row
    nbytes = 5 * x.numel() * 4
    kernel = {"us_per_launch": us, "launches": args.launches, "bytes_per_launch": nbytes,
              "gb_per_s": nbytes / (us * 1e-6) / 1e9,
              "note": "back-to-back launches from the host, clip on, x0_out on; at this size the launch itself dominates"}

    line = {"metric": f"DDPM ancestral sampling vs DDIM-50 images/s at {size}^2", "card": card(), "batch": B,
            "dtype": "bf16", "data": "synthetic (bench.py's synthetic_batch, seed 1234)", "cuda_graph": True,
            "timing": f"CUDA events around each pass, one warm-up pass each, {args.passes} timed passes interleaved "
                      "across the three loops",
            "what": {"ddpm_1000": "B200DDPMSampler.p_sample_loop, 1000 steps: 1000 model evaluations",
                     "ddpm_start_250": "the same loop with start_T = 250: 250 model evaluations",
                     "ddim_50": "B200DDIMSampler.sample(50), eta 0: 50 model evaluations"},
            **res, "ratio_ddpm_1000_over_ddim_50": res["ddpm_1000"]["images_per_s"] / res["ddim_50"]["images_per_s"],
            "update_kernel": kernel, "embedding_table_1000_rows": table}
    text = json.dumps(line)
    print(text, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(line, indent=1) + "\n")


if __name__ == "__main__":
    main()
