#!/usr/bin/env python
"""bench.py — DDIM-50 makeup images/s at 256^2 (BASELINE.json metric), per the driver contract.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" = one pass of the hot path over one batch: 50-step DDIM sampling (eta 0, no CFG) of a batch of
16 source/reference pairs per GPU with ControlNet conditioning = BASELINE.json configs[1] (at N = 8 the job is
configs[2]'s 128 images).  Per step the hint block and the cross-attention K/V projections are recomputed (new images
every step), then 50 x [UNet + ControlNet eval -> fused DDIM update].
  value     images/s, inputs already in HBM, CUDA-event timed, max over ranks
  e2e       same metric through the public API with HOST (pinned) inputs: H2D of src/ref/ctx/x_T and D2H of the final
            latents inside the timed region
  roofline  tensor-core roofline of the dominant kernel (tcgen05 implicit-GEMM): algorithmic FLOPs of its launches in
            one UNet+ControlNet eval / their summed CUDA-event durations (single-stream pass, launches queued behind
            a blocker so no host gap is timed), vs the measured sustained bf16 peak; `traffic` = average DRAM bytes per
            launch of that kernel from the committed ncu pass (profiles/r02_ncu_families.json); `others` = the same
            for attention (TFLOP/s) and the norm kernels (GB/s against the measured HBM copy bandwidth)
  cpu_baseline  the oracle (a port: the reference's ldm/cldm dependency is not vendored) on the host cores, bounded sample
--impl reference: the reference's CPU path = the same oracle, timed on the box's host cores (rank 0 only).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# algorithmic FLOPs (SURVEY.md §8(d)): per sample per step excluding step-invariant work, and once per sample
F_STEP = {256: 234.788e9, 512: 1067.53e9}
F_ONCE = {256: 8.052e9, 512: 19.26e9}
DUMP_BYTES = 63 * 10**6  # --dump-outputs: data of all arrays together, so that the files with their headers stay under 64 MB


def dump_outputs(out_dir, arrays, budget=DUMP_BYTES):
    """Writes every tensor of `arrays` as out_dir/<name>.npy in float32.  When together they hold more than `budget`
    bytes, each keeps the same share of its flattened elements: a sample drawn with a fixed seed and kept in index
    order, so that runs with the same arguments write the same elements and two builds compare element for element."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    total = 4 * sum(a.numel() for a in arrays.values())
    for name, a in arrays.items():
        a = a.detach().float().cpu()
        if total > budget:
            pick = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:a.numel() * budget // total]
            a = a.flatten()[pick.sort().values]
        np.save(os.path.join(out_dir, f"{name}.npy"), a.numpy())
        print(f"bench: wrote {name}.npy {tuple(a.shape)} to {out_dir}" + (" (sample)" if total > budget else ""), file=sys.stderr)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"tflops": d["bf16_tflops_sustained"], "tflops_burst": d["bf16_tflops"], "gbs": d["hbm_gbs"], "src": "measured"}
    return {"tflops": 1400.0, "tflops_burst": 1590.0, "gbs": 6650.0, "src": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)"""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.stop, self.index = [], threading.Event(), index

    def _run(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop.wait(0.2)

    def __enter__(self):
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.t.join(timeout=6)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "samples": len(sm), "power_w_max": max(float(r[2]) for r in self.rows)}


# ----------------------------------------------------------------------------------------------------------------
class OracleCPU:
    """the reference's CPU path = the fp32 oracle on all host threads: ONE source/reference pair (BASELINE.json configs[0]),
    DDIM-50 schedule; run(n) times the first n steps of the loop, run(50) the whole loop"""

    def __init__(self, size, cfg=1.0, ddim_steps=50):
        import torch
        from oracle import MKDDIMSampler, OracleControlLDM, seeded_state_dict
        self.torch = torch
        self.cores = os.cpu_count() or 1
        torch.set_num_threads(self.cores)
        h = size // 8
        model = OracleControlLDM().eval()
        seeded_state_dict(model, 0)
        for p in model.parameters():
            p.requires_grad_(False)
        g = torch.Generator().manual_seed(1234)
        self.cond = {"c_crossattn": [torch.randn(1, 77, 768, generator=g)], "c_concat": [torch.rand(1, 6, size, size, generator=g)]}
        self.x = torch.randn(1, 4, h, h, generator=g)
        self.guide = {}
        if cfg != 1.0:
            self.guide = dict(unconditional_guidance_scale=cfg, unconditional_conditioning={
                "c_crossattn": [torch.randn(1, 77, 768, generator=g)], "c_concat": self.cond["c_concat"]})
        self.s = MKDDIMSampler(model)
        self.s.make_schedule(ddim_steps, ddim_eta=0.0, verbose=False)

    def run(self, n):
        with self.torch.no_grad():
            t0 = time.perf_counter()
            self.out = self.s.reconstruct(self.x, self.cond, t_start=n, **self.guide)  # the first n steps of the schedule
            return time.perf_counter() - t0


def workload_config(args, world):
    B, S, size = args.batch, args.ddim_steps, args.size
    cfg, sweep, gb = getattr(args, "cfg", 1.0), getattr(args, "sweep", False), getattr(args, "global_batch", 0)
    if sweep:
        which = "BASELINE.json configs[4] (makeup interpolation sweep: 1 source x 8 references x 5 blend weights = 40 samples)"
    elif cfg != 1.0:
        which = "BASELINE.json configs[3]" + ("" if (size, B * world) == (512, 32) else " shape family (quoted: 512^2, global batch 32 on 8 GPUs)")
    elif gb:
        which = "BASELINE.json configs[2]" + ("" if (size, gb) == (256, 128) else " family (quoted: 256^2, global batch 128)")
    else:
        which = "BASELINE.json configs[1]" + ("" if (size, B) == (256, 16) else " family (quoted: 256^2, batch 16)")
    return {"workload": f"{size}x{size}, DDIM-{S} eta 0, ControlNet (6-ch hint) conditioning, "
                        + (f"classifier-free guidance scale {cfg:g} (doubled [uncond; cond] batch), " if cfg != 1.0 else "no CFG, ")
                        + f"batch {B} per GPU (global {B * world}), random-init (seeded non-zero) weights of "
                        f"base_diffusion_makeup.yaml = {which}"
                        + (" + first-stage (VAE) decode of the samples to images" if getattr(args, "decode", False) else "")
                        + (" + CLIP text encoding of the prompt tokens and uint8 image grid in every e2e pass" if getattr(args, "pipeline", False) else ""),
            "parallelism": f"batch-sharded x{world}, one all-gather of final latents"
                           + (" fused into the last DDIM-update kernel (peer stores)" if getattr(args, "fused_gather", False)
                              and world > 1 else " (NCCL)" if world > 1 else ""),
            "cuda_graph": not args.no_graph,
            "l2": "per-step working set (2.44 GB bf16 weights + activations) exceeds the 126 MB L2; no explicit flush"}


def reference_arm(args, rank):
    """--impl reference: the reference's own CPU implementation of the path (the oracle port: ldm / cldm are not vendored)
    on the box's host cores.  Each of the K timed steps is a bounded sample — the first 4 of the 50 DDIM steps of one
    image pair — and ONE untimed-by-the-contract extra pass runs the whole 50-step loop (BASELINE.json configs[0] exactly
    as written), reported next to it as `full_loop`."""
    if rank != 0:
        return
    S = 20 if args.sweep else args.ddim_steps
    o = OracleCPU(args.size, args.cfg, S)
    n = 4  # DDIM steps per bench step
    for _ in range(max(1, min(args.warmup, 2))):
        o.run(1)
    full_s = o.run(S)
    times = [o.run(n) for _ in range(args.steps)]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"latents": o.out})
    sec_per_model_step = statistics.mean(times) / n
    ips = 1.0 / (S * sec_per_model_step)
    cores = o.cores
    line = {"impl": "reference", "metric": f"DDIM-{S} makeup images/sec at {args.size}^2", "value": ips, "unit": "images/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * statistics.mean(times),
            "higher_is_better": True, "scaling": "strong" if args.global_batch else "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(args, int(os.environ.get("WORLD_SIZE", 1))),
            "cpu_baseline": {"value": ips, "unit": "images/s", "cores": cores, "kind": "port",
                             "sample": f"{n} of {S} DDIM steps of ONE {args.size}^2 source/reference pair per bench step (fp32, "
                                       f"all {cores} host threads), images/s = 1 / ({S} x seconds per UNet+ControlNet step); "
                                       "images are independent, so throughput does not depend on the batch; "
                                       "oracle = PyTorch restatement (the reference's ldm/cldm dependency is not vendored)",
                             "full_loop": {"value": 1.0 / full_s, "unit": "images/s", "seconds": full_s,
                                           "what": f"the whole {S}-step loop of one pair, run once (BASELINE.json configs[0] as written)"}},
            "e2e": {"value": ips, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "ms_per_unet_controlnet_step": 1e3 * sec_per_model_step}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=16, help="images per GPU")
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--ddim-steps", type=int, default=50)
    ap.add_argument("--global-batch", type=int, default=0,
                    help="whole-job batch, split evenly over the GPUs (BASELINE.json configs[2]: 128 on 2 / 4 / 8 GPUs = 64 / 32 / 16 "
                         "per GPU; configs[3]: 32); strong scaling.  Default 0: --batch images per GPU (weak scaling)")
    ap.add_argument("--cfg", type=float, default=1.0,
                    help="classifier-free guidance scale (configs[3]: 9): every step runs the doubled [uncond; cond] batch")
    ap.add_argument("--sweep", action="store_true",
                    help="configs[4]: makeup interpolation sweep, 1 source x 8 references x 5 blend weights = 40 samples, "
                         "20-step DDIM, sharded over the GPUs")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--grouped", action="store_true",
                    help="A/B: force the stacked trunk where the default ('auto') would not pick it (levels whose rows per network are "
                         "not whole tile pairs then run one launch per network)")
    ap.add_argument("--no-gn-tail", action="store_true", help="A/B: out_layers' GroupNorm always as its own launch (no mkd_conv_desc.gn_y)")
    ap.add_argument("--no-grouped", action="store_true",
                    help="A/B: UNet encoder and ControlNet trunk as two networks on two streams instead of one stacked network")
    ap.add_argument("--fused-gather", action="store_true",
                    help="N > 1: all-gather the final latents with the last DDIM-update kernel's own peer stores "
                         "(symmetric memory over NVLink) instead of the NCCL collective")
    ap.add_argument("--decode", action="store_true",
                    help="also run the first-stage (VAE) decoder on the sampled latents inside every pass (SURVEY 8(f) rank 1; "
                         "not part of BASELINE.json's metric, so off by default and named in config.workload when on)")
    ap.add_argument("--pipeline", action="store_true",
                    help="widened flow of SURVEY 8(f) ranks 1, 3, 4 inside every e2e pass: prompt token ids -> CLIP text encoder -> "
                         "c_crossattn, DDIM, first-stage decode, uint8 image grid (mkd_image_grid_u8) -> host; implies --decode; "
                         "off by default (not BASELINE.json's metric) and named in config.workload when on")
    ap.add_argument("--profile-out", default=None, help="write the per-layer kernel timing table to this file")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned on rank 0 (the final latents, or the decoded "
                         "images with --decode) as DIR/<name>.npy in float32, at most 64 MB in all (beyond that a fixed "
                         "seeded sample of the elements); the inputs depend only on the arguments, so two builds compare "
                         "output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        return reference_arm(args, rank)
    if args.warmup < 3:
        args.warmup = 3
    if args.pipeline:
        args.decode = True

    import torch
    import torch.distributed as dist
    from makeupdiffuse_b200 import B200ControlLDM, B200DDIMSampler, _lib, ops
    from makeupdiffuse_b200.dist import sample_sharded, shard_bounds
    from makeupdiffuse_b200.synth import synthetic_batch, synthetic_state_dict

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the B200 path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    if args.sweep:
        args.ddim_steps, args.global_batch = 20, 40
    S, size, h = args.ddim_steps, args.size, args.size // 8
    if args.global_batch:
        if args.global_batch % world:
            raise SystemExit(f"--global-batch {args.global_batch} does not divide over {world} GPUs")
        Bg, B = args.global_batch, args.global_batch // world
        args.batch = B
    else:
        B = args.batch
        Bg = B * world
    cfg = args.cfg != 1.0
    rows = 2 * B if cfg else B  # batch rows one UNet+ControlNet evaluation sees

    model = B200ControlLDM(dtype=torch.bfloat16, device=dev)
    model.load_state_dict(synthetic_state_dict(model, 0, dev))
    if args.no_gn_tail:
        model.model.diffusion_model.fuse_gn_tail = model.control_model.fuse_gn_tail = False
    if args.no_grouped or args.grouped:
        model.grouped = bool(args.grouped)
    args.stacked = bool(model._use_grouped(rows, h, h))
    sampler = B200DDIMSampler(model, use_cuda_graph=not args.no_graph)
    if args.decode:
        from makeupdiffuse_b200 import B200FirstStageDecoder
        from makeupdiffuse_b200.synth import synthetic_first_stage_state_dict
        vae = B200FirstStageDecoder(dtype=torch.bfloat16)
        model.attach_first_stage_decoder(vae.load_state_dict(synthetic_first_stage_state_dict(vae, 0, dev), device=dev))
    if args.pipeline:
        from makeupdiffuse_b200 import B200FrozenCLIPEmbedder
        from makeupdiffuse_b200.synth import synthetic_clip_state_dict
        clip = B200FrozenCLIPEmbedder(device=dev, dtype=torch.bfloat16)
        clip.load_state_dict(synthetic_clip_state_dict(clip.cfg, 0, dev))
        model.attach_cond_stage_model(clip)
        tok_host = torch.randint(0, 49406, (B, 77), generator=torch.Generator().manual_seed(7)).pin_memory()
        dtok = torch.empty(B, 77, dtype=torch.long, device=dev)
    lo, hi = shard_bounds(Bg, rank, world)
    if args.sweep:
        # 1 source x 8 references x 5 blend weights (README.md:25; BASELINE.json configs[4]) as one batch of 40 for the
        # unchanged sampler, from one generator; every rank builds the whole (small) job and keeps its shard
        from makeupdiffuse_b200.sweep import interpolation_cond
        one = synthetic_batch(9, size, 768, seed=1234, device=dev)
        cond_all = interpolation_cond(one["src"][:1], one["ref"][1:9], [0.0, 0.25, 0.5, 0.75, 1.0], one["ctx"][:1])
        assert cond_all["c_concat"][0].shape[0] == Bg
        loc = {"hint": cond_all["c_concat"][0][lo:hi].contiguous(), "ctx": cond_all["c_crossattn"][0][lo:hi].contiguous(),
               "x_T": one["x_T"][:1].expand(B, -1, -1, -1).contiguous()}
        del one, cond_all
    else:
        data = synthetic_batch(Bg, size, 768, seed=1234, device=dev)  # whole-job batch from one generator, then sliced
        loc = {k: v[lo:hi].contiguous() for k, v in data.items()}
        loc["hint"] = torch.cat([loc.pop("src"), loc.pop("ref")], 1)  # c_concat = cat(src, ref) (makeup_diffuse.py:56)
        del data
    hint_dev, ctx_dev = loc["hint"], loc["ctx"]
    guide = {}
    uctx_dev = None
    if cfg:
        # the unconditional branch: another context (the reference encodes the empty prompt), the SAME hint
        # (uc_cat = c_cat, diffusion_makeup.py:399-402)
        uctx_dev = torch.randn(B, 77, 768, device=dev, generator=torch.Generator(device=dev).manual_seed(4321 + rank))
        guide = dict(unconditional_guidance_scale=args.cfg,
                     unconditional_conditioning={"c_crossattn": [uctx_dev], "c_concat": [hint_dev]})

    def one_pass_device():
        # a new batch of images every pass: sample_sharded starts a loop, which drops the hoisted hint block + K/V
        cond = {"c_crossattn": [ctx_dev], "c_concat": [hint_dev]}
        lat = sample_sharded(sampler, S, Bg, (4, h, h), cond, loc["x_T"], rank, world, fused_gather=args.fused_gather, **guide)
        if args.decode:  # each rank decodes its own images
            return model.decode_first_stage(lat[lo:hi])
        return lat

    # host-side (pinned) copies for the end-to-end arm
    pin = {k: loc[k].cpu().pin_memory() for k in ("hint", "ctx", "x_T")}
    dhint, dctx, dxt = (torch.empty_like(loc[k]) for k in ("hint", "ctx", "x_T"))
    if cfg:
        pin["uctx"] = uctx_dev.cpu().pin_memory()
        ductx = torch.empty_like(uctx_dev)
    out_host = torch.empty(Bg, 4, h, h, dtype=torch.float32).pin_memory()
    h2d = sum(pin[k].numel() * 4 for k in pin)
    d2h = out_host.numel() * 4
    if args.pipeline:
        gh, gw = ops.image_grid_shape(B, size, size, 8)
        img_host = torch.empty(gh, gw, 3, dtype=torch.uint8).pin_memory()
        h2d += tok_host.numel() * 8 - pin["ctx"].numel() * 4  # token ids travel instead of the context
        d2h += img_host.numel()
    elif args.decode:
        img_host = torch.empty(B, 3, size, size, dtype=torch.float32).pin_memory()
        d2h += img_host.numel() * 4

    def one_pass_e2e():
        """the public API with HOST inputs: H2D of this rank's hint / context / x_T, the sharded sampling call
        (makeupdiffuse_b200.dist.sample_sharded: B200DDIMSampler steps + the all-gather of the final latents; at one GPU it
        is the B200DDIMSampler.sample loop), D2H of the gathered latents"""
        dhint.copy_(pin["hint"], non_blocking=True)
        if args.pipeline:
            dtok.copy_(tok_host, non_blocking=True)
            ctx_e2e = model.get_learned_conditioning(dtok)  # token ids: encoded every pass (no prompt cache)
        else:
            dctx.copy_(pin["ctx"], non_blocking=True)
            ctx_e2e = dctx
        dxt.copy_(pin["x_T"], non_blocking=True)
        cond = {"c_crossattn": [ctx_e2e], "c_concat": [dhint]}
        g2 = {}
        if cfg:
            ductx.copy_(pin["uctx"], non_blocking=True)
            g2 = dict(unconditional_guidance_scale=args.cfg,
                      unconditional_conditioning={"c_crossattn": [ductx], "c_concat": [dhint]})
        if world == 1 and not args.fused_gather:
            out, _ = sampler.sample(S, B, (4, h, h), cond, eta=0.0, x_T=dxt, verbose=False, **g2)  # the public API call
        else:
            out = sample_sharded(sampler, S, Bg, (4, h, h), cond, dxt, rank, world, fused_gather=args.fused_gather, **g2)
        if args.pipeline:
            img_host.copy_(ops.image_grid_u8(model.decode_first_stage(out[lo:hi] if world > 1 else out), nrow=8), non_blocking=True)
        elif args.decode:
            img_host.copy_(model.decode_first_stage(out[lo:hi] if world > 1 else out), non_blocking=True)
        out_host.copy_(out, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return out_host

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        """k passes of fn between two events: (milliseconds, max over ranks; what the last pass returned)"""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            out = fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms), out

    for _ in range(args.warmup):
        one_pass_device()
    n0, g0 = lib.mkd_launch_count(), sampler.graph_launches
    with ClockSampler(local) as clk:
        ms, last = timed(one_pass_device, args.steps)
    launches = (lib.mkd_launch_count() - n0) + (sampler.graph_launches - g0)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"images" if args.decode else "latents": last})
    for _ in range(2):
        one_pass_e2e()
    ms_e2e, _ = timed(one_pass_e2e, args.steps)

    ips = Bg * args.steps / (ms / 1e3)
    ips_e2e = Bg * args.steps / (ms_e2e / 1e3)
    ms_model_step = ms / args.steps / S

    # ---- roofline of the dominant kernel: every conv2d launch of ONE UNet+ControlNet eval timed in place ------------
    pk = peaks()
    roof, table = None, []
    if rank == 0:
        cond = {"c_crossattn": [ctx_dev], "c_concat": [hint_dev]}
        px = loc["x_T"]
        if cfg:  # the evaluation the guided loop runs: [uncond; cond] rows (cddim.py:18-39)
            from makeupdiffuse_b200.sampler import _cat_uncond_first
            cond = _cat_uncond_first(guide["unconditional_conditioning"], cond)
            px = torch.cat([px] * 2)
        t = torch.full((rows,), 501, device=dev, dtype=torch.long)
        was_concurrent, model.concurrent = model.concurrent, False  # one stream: a launch's events bracket it alone
        # as inside the sampler's loop: the timestep embeddings come from the per-loop table (B200ControlLDM.set_step)
        model.precompute_time_embeddings([501])
        model.set_step(501, rows)
        model.apply_model(px, t, cond)
        torch.cuda.synchronize()
        ops.PROFILE = []
        torch.cuda._sleep(int(0.25 * 1.9e9))  # let the host run ahead so launches queue back to back on the GPU
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        model.apply_model(px, t, cond)
        s1.record()
        torch.cuda.synchronize()
        serial_ms = s0.elapsed_time(s1)
        model.concurrent = was_concurrent
        model.set_step(None)
        prof, ops.PROFILE = ops.PROFILE, None
        other, attn_prof = {}, []
        all_prof = prof
        for r in prof:
            r["ms"] = r["e0"].elapsed_time(r["e1"])
            if r["op"] == "attention":
                attn_prof.append(r)
            if r["op"] != "conv2d":
                a = other.setdefault(r["op"], {"n": 0, "ms": 0.0, "bytes": 0})
                a["n"] += 1; a["ms"] += r["ms"]; a["bytes"] += r["bytes"]
        prof = [r for r in prof if r["op"] == "conv2d"]
        agg = {}
        for r in prof:
            key = (r["path"], r["M"], r["K"], r["C"], r["R"], r["stride"], r["up"], r.get("C2", 0))
            a = agg.setdefault(key, {"n": 0, "ms": 0.0, "flops": 0.0})
            a["n"] += 1; a["ms"] += r["ms"]; a["flops"] += r["flops"]
        tc = [r for r in prof if r["path"] == _lib.PATH_TCGEN05]
        gen = [r for r in prof if r["path"] == _lib.PATH_GENERIC]
        tc_ms_inplace, tc_fl = sum(r["ms"] for r in tc), sum(r["flops"] for r in tc)
        gen_ms = sum(r["ms"] for r in gen)
        # A pair of events around every launch costs ~5 us of GPU time per launch (serial_eval_ms vs the real step), which
        # is a large share of a 10-20 us kernel.  So the figure the roofline uses is taken without them: the SAME 293
        # launches (same descriptors, same buffers, in program order) replayed back to back as one CUDA graph on one
        # stream, two events around the whole replay, averaged over 5 replays.
        def replay_ms(calls):
            """the given launches, in program order, as one CUDA graph on one stream: mean time of 5 replays"""
            g = torch.cuda.CUDAGraph()
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for c in calls:
                    c()  # warm-up outside capture
                with torch.cuda.graph(g, stream=side):
                    for c in calls:
                        c()
            torch.cuda.current_stream().wait_stream(side)
            g.replay()
            torch.cuda.synchronize()
            r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            r0.record()
            for _ in range(5):
                g.replay()
            r1.record()
            torch.cuda.synchronize()
            return r0.elapsed_time(r1) / 5

        tc_ms = replay_ms([(lambda d=r["desc"]: ops.run_conv_desc(d)) for r in tc])
        for fam in ("attention", "groupnorm", "groupnorm_apply", "layernorm"):  # same treatment for the other families
            calls = [(lambda f=r["replay"]: f[0](*f[1], **f[2])) for r in all_prof if r["op"] == fam]
            if calls and fam in other:
                other[fam]["ms_events"], other[fam]["ms"] = other[fam]["ms"], replay_ms(calls)
        achieved = tc_fl / (tc_ms / 1e3) / 1e12 if tc_ms else 0.0
        traffic = None
        for fam_path in (os.path.join(ROOT, "profiles", f) for f in ("r02_ncu_families.json", "r01_ncu_families.json")):
            if os.path.exists(fam_path) and rows == 16 and size == 256:  # the ncu pass was taken on this workload
                fams = json.load(open(fam_path))["families"]
                gem = [fams[k] for k in ("gemm_pair_kernel", "gemm_tcgen05_kernel") if k in fams and fams[k].get("dram_bytes_per_launch")]
                if gem:  # average DRAM bytes per launch over the two tensor-core GEMM kernels
                    traffic = round(sum(f["dram_bytes_per_launch"] * f["launches"] for f in gem) / sum(f["launches"] for f in gem))
                    break
        att = other.get("attention")
        att_flops = sum(r["flops"] for r in attn_prof)
        others = {}
        if att and att["ms"]:
            others["attention"] = {"bound": "tensor", "kernel": "attn_tcgen05_kernel", "achieved": att_flops / (att["ms"] / 1e3) / 1e12,
                                   "unit": "TFLOP/s", "launches_per_eval": att["n"], "kernel_ms_per_eval": att["ms"],
                                   "note": "4*B*heads*Nq*Nkv*d FLOPs; exp2 / latency bound at head dim 40 (XU pipe 41 %), "
                                           f"{att['n']} launches per evaluation, most of them sub-10-us maps (16x16 and deeper levels, 77-key cross-attention)"}
        for k in ("groupnorm", "groupnorm_apply", "layernorm"):
            if k in other and other[k]["ms"]:
                gbs = other[k]["bytes"] / (other[k]["ms"] / 1e3) / 1e9
                others[k] = {"bound": "hbm", "achieved": gbs, "peak": pk["gbs"], "unit": "GB/s", "frac": gbs / pk["gbs"],
                             "launches_per_eval": other[k]["n"], "kernel_ms_per_eval": other[k]["ms"],
                             "note": "1 read + 1 write per element; inputs were just written by the producer (L2-resident)"}
        roof = {"bound": "tensor", "kernel": "gemm_pair_kernel + gemm_tcgen05_kernel (tcgen05 implicit-GEMM conv / linear: CTA-pair and "
                                             "single-CTA forms)", "achieved": achieved,
                "peak": pk["tflops"], "unit": "TFLOP/s", "frac": achieved / pk["tflops"], "traffic": traffic,
                "peak_source": f"{pk['src']} sustained bf16 ({pk['tflops_burst']} burst)", "launches_per_eval": len(tc),
                "kernel_ms_per_eval": tc_ms, "kernel_ms_per_eval_event_pairs": tc_ms_inplace,
                "share_of_serial_eval_event_pairs": tc_ms_inplace / serial_ms if serial_ms else None,
                "timing": "the eval's tcgen05 launches replayed back to back as one CUDA graph, 2 events, mean of 5",
                "generic_conv_ms_per_eval": gen_ms,
                "whole_step_frac": (F_STEP.get(size, 0) * rows / (ms_model_step / 1e3) / 1e12) / pk["tflops"],
                "others": others}
        for key, a in sorted(agg.items(), key=lambda kv: -kv[1]["ms"]):
            table.append({"path": "tcgen05" if key[0] == _lib.PATH_TCGEN05 else "generic", "M": key[1], "N": key[2],
                          "C": key[3], "R": key[4], "stride": key[5], "up": key[6], "C2": key[7], "count": a["n"], "ms": round(a["ms"], 4),
                          "tflops": round(a["flops"] / (a["ms"] / 1e3) / 1e12, 1) if a["ms"] else None})
        if args.profile_out:
            with open(args.profile_out, "w") as f:
                json.dump({"ms_per_unet_controlnet_step": ms_model_step, "conv_table": table,
                           "other_ops": {k: {"count": v["n"], "ms": round(v["ms"], 4),
                                             "GBps": round(v["bytes"] / (v["ms"] / 1e3) / 1e9, 1) if v["ms"] else None}
                                         for k, v in other.items()}}, f, indent=1)

    # ---- CPU baseline (rank 0, N = 1 only): bounded sample of configs[0] ----------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        o = OracleCPU(size, args.cfg, S)
        o.run(1)
        full_s = o.run(S)  # BASELINE.json configs[0] as written: the whole loop of one pair, not an extrapolation
        cpu = {"value": 1.0 / full_s, "unit": "images/s", "cores": o.cores, "kind": "port",
               "sample": f"the full {S}-step DDIM loop of ONE {size}^2 source/reference pair (BASELINE.json configs[0]), fp32 oracle on "
                         f"{o.cores} host threads, run once after a one-step warm-up: {full_s:.1f} s = "
                         f"{1e3 * full_s / S:.0f} ms per UNet+ControlNet step"}

    if rank == 0:
        line = {"metric": f"DDIM-{S} makeup images/sec at {size}^2", "value": ips, "unit": "images/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
                "scaling": "strong" if args.global_batch else "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": workload_config(args, world),
                "trunks": "UNet encoder + ControlNet trunk as one stacked network (two weight groups per launch)" if args.stacked
                          else "UNet encoder and ControlNet trunk as two networks on two streams",
                "ms_per_unet_controlnet_step": ms_model_step,
                "e2e": {"value": ips_e2e, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": ms_e2e / args.steps},
                "gpu_launches": int(launches), "clocks": clk.summary(), "roofline": roof, "cpu_baseline": cpu}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
