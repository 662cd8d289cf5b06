#!/usr/bin/env python
"""DDIM inversion throughput on one B200 at BASELINE.json configs[1]'s shape (yaml-size networks, 256^2, batch 16, bf16,
synthetic seeded inputs drawn as bench.py draws them):

  encode      images/s of B200DDIMSampler.encode(z, cond, t_enc=50): x_0 -> x_T
  round_trip  images/s of the whole inversion flow of a dataset of stored inverted latents: image -> get_z (first-stage
              encoder) -> encode(t_enc=50) -> decode(t_start=50) (= reconstruct) -> decode_first_stage
  sample      images/s of B200DDIMSampler.sample(50) on the same batch, measured in the same run for comparison

Each pass is timed alone with CUDA events after warm-up passes; the JSON gives mean / min / max / stdev over the passes and
the card's name and power limit read in the same run.

    python tools/invert_bench.py [--passes K] [--warmup W] [--batch B] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    import torch
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": None, "sm_max_mhz": None}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=10).stdout.strip().splitlines()
        if out:
            pl, clk = (c.strip() for c in out[0].split(","))
            info["power_limit_w"], info["sm_max_mhz"] = float(pl), float(clk)
    except (OSError, ValueError, subprocess.SubprocessError):
        pass
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--passes", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--steps", type=int, default=50, help="DDIM schedule length S; encode / decode run all of it")
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    if args.passes < 2:
        ap.error("--passes must be at least 2 (the spread needs two)")

    import torch
    from makeupdiffuse_b200 import B200ControlLDM, B200DDIMSampler, B200FirstStageDecoder, B200FirstStageEncoder
    from makeupdiffuse_b200.synth import synthetic_batch, synthetic_first_stage_state_dict, synthetic_state_dict

    if not torch.cuda.is_available():
        raise SystemExit("invert_bench.py needs a B200: the B200 path has no CPU fallback")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    B, S, size, h = args.batch, args.steps, args.size, args.size // 8
    model = B200ControlLDM(dtype=torch.bfloat16, device=dev)
    model.load_state_dict(synthetic_state_dict(model, 0, dev))
    enc = B200FirstStageEncoder(dtype=torch.bfloat16)
    model.attach_first_stage_encoder(enc.load_state_dict(synthetic_first_stage_state_dict(enc, 0, dev), device=dev))
    dec = B200FirstStageDecoder(dtype=torch.bfloat16)
    model.attach_first_stage_decoder(dec.load_state_dict(synthetic_first_stage_state_dict(dec, 0, dev), device=dev))
    sampler = B200DDIMSampler(model)
    sampler.make_schedule(S, ddim_eta=0.0, verbose=False)

    data = synthetic_batch(B, size, 768, seed=1234, device=dev)
    cond = {"c_crossattn": [data["ctx"]], "c_concat": [torch.cat([data["src"], data["ref"]], 1)]}
    image = data["src"] * 2 - 1                        # the source images in [-1, 1], as the first-stage encoder takes them
    noise = torch.randn(B, 4, h, h, device=dev, generator=torch.Generator(device=dev).manual_seed(99))
    z = model.get_z(image, noise)

    def encode():
        return sampler.encode(z, cond, S)[0]

    def round_trip():
        zz = model.get_z(image, noise)
        xt, _ = sampler.encode(zz, cond, S)
        return model.decode_first_stage(sampler.decode(xt, cond, S))

    def sample():
        return sampler.sample(S, B, (4, h, h), cond, eta=0.0, x_T=data["x_T"], verbose=False)[0]

    def timed(fn):
        for _ in range(args.warmup):
            fn()
        torch.cuda.synchronize()
        ms = []
        for _ in range(args.passes):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn()
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        assert torch.isfinite(out).all()
        ips = [B / (m / 1e3) for m in ms]
        return {"images_per_s": statistics.mean(ips), "images_per_s_min": min(ips), "images_per_s_max": max(ips),
                "images_per_s_stdev": statistics.stdev(ips), "ms_per_pass": [round(m, 3) for m in ms]}

    res = {"encode": timed(encode), "round_trip": timed(round_trip), "sample": timed(sample)}
    line = {"metric": f"DDIM inversion images/s at {size}^2", "card": card(), "batch": B, "ddim_steps": S, "dtype": "bf16",
            "data": "synthetic (bench.py's synthetic_batch, seed 1234)", "cuda_graph": True,
            "timing": f"CUDA events around each pass, {args.warmup} warm-up passes, {args.passes} timed passes",
            "what": {"encode": f"B200DDIMSampler.encode, t_enc = {S}",
                     "round_trip": f"image -> get_z -> encode(t_enc={S}) -> decode(t_start={S}) -> decode_first_stage",
                     "sample": f"B200DDIMSampler.sample, DDIM-{S}, eta 0, no CFG (bench.py's workload, same run)"},
            **res}
    text = json.dumps(line)
    print(text, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(line, indent=1) + "\n")


if __name__ == "__main__":
    main()
