"""Batch sharding across the GPUs of one box (SURVEY.md §8(e)).

Every (source, reference, noise) sample denoises independently — nothing in diffmk/cddim.py:9-100 or apply_model mixes
batch rows — so ranks take contiguous batch chunks, weights are replicated (re-generated / loaded per rank) and the
only data-path collective is ONE all-gather of the final latents over NVLink 5 / NVSwitch, done in one of two ways:

* NCCL (default): the last DDIM update kernel writes x_0 directly into this rank's slice of the gather buffer
  (``out=``), and ``all_gather_into_tensor`` runs in place on it — no staging copy.
* fused (``fused_gather=True``): the gather buffer is torch symmetric memory (every rank's copy is mapped into every
  other rank); the last DDIM update kernel stores its x_0 slice into ALL ranks' buffers itself
  (``mkd_ddim_update_peers``: plain stores to peer addresses over NVLink), and a signal barrier between the ranks
  replaces the collective launch.  Same bits as the NCCL path (tests/test_sharding.py, 2 GPUs).

``sample_sharded`` runs the DDIM sampling loop this way; ``encode_sharded`` the DDIM inversion (x_0 -> x_t) of a
dataset's latents, whose last inversion step writes into the gather buffer the same way; ``sample_plms_sharded`` the PLMS
sampling loop (B200PLMSSampler), whose last update kernel (``mkd_plms_update[_peers]``) does the same;
``sample_dpm_sharded`` the DPM-Solver++ loop (B200DPMSolverSampler, ``mkd_dpm_update[_peers]``) likewise.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.distributed as dist

_symm_cache: dict = {}


def shard_bounds(n_global: int, rank: int, world: int):
    """contiguous chunk [lo, hi) of rank; the first n_global % world ranks take one extra sample"""
    base, extra = divmod(n_global, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def _symmetric_gather_buffer(shape, device, group):
    """persistent symmetric-memory gather buffer + its rendezvous handle for this shape (collective on first use)"""
    import torch.distributed._symmetric_memory as symm_mem
    group = group or dist.group.WORLD
    key = (tuple(shape), str(device), group.group_name)
    hit = _symm_cache.get(key)
    if hit is None:
        buf = symm_mem.empty(shape, dtype=torch.float32, device=device)
        hit = _symm_cache[key] = (buf, symm_mem.rendezvous(buf, group.group_name))
    return hit


def _gather_begin(batch_global, lo, hi, shape, device, world, group, fused_gather):
    """the [batch_global, *shape] fp32 gather buffer, this rank's slice [lo, hi) of it, and for the fused gather the
    rendezvous handle and the device pointers of that slice inside every rank's buffer.  The loop's last update writes
    its result into the slice (``out=``) or into every rank's copy of it (``peer_ptrs=``)."""
    if world > 1 and batch_global % world:
        raise ValueError("sharded runs need batch_global % world == 0")
    fused = bool(fused_gather) and world > 1
    hdl = peer_ptrs = None
    if fused:
        gathered, hdl = _symmetric_gather_buffer((batch_global, *shape), device, group)
        off = lo * int(np.prod(shape)) * 4
        peer_ptrs = [int(p) + off for p in hdl.buffer_ptrs]  # this rank's slice inside every rank's buffer
        hdl.barrier()  # nobody still reads the previous result out of the buffers we are about to overwrite
    else:
        gathered = torch.empty(batch_global, *shape, dtype=torch.float32, device=device)
    return gathered, gathered[lo:hi], hdl, peer_ptrs


def _gather_end(gathered, mine, hdl, world, group):
    """completes the gather once the last update of every rank has been enqueued; returns the whole batch"""
    if hdl is not None:
        hdl.barrier()  # every rank's final update kernel has stored its slice everywhere
        return gathered.clone()  # the symmetric buffer is reused by the next call
    if world > 1:
        dist.all_gather_into_tensor(gathered, mine, group=group)  # in place: input is the rank's own slice
    return gathered


def sample_sharded(sampler, S, batch_global, shape, cond_local, x_T_local, rank=0, world=1, group=None,
                   fused_gather=False, **kw):
    """DDIM-sample this rank's chunk and all-gather the final latents.

    cond_local / x_T_local hold this rank's rows only.  Returns the [batch_global, C, H, W] latents on every rank.
    Requires equal chunk sizes when world > 1."""
    lo, hi = shard_bounds(batch_global, rank, world)
    b = hi - lo
    gathered, mine, hdl, peer_ptrs = _gather_begin(batch_global, lo, hi, tuple(shape), x_T_local.device, world, group,
                                                   fused_gather)
    sampler.make_schedule(ddim_num_steps=S, ddim_eta=kw.pop("eta", 0.0), verbose=False)
    steps = np.flip(sampler.ddim_timesteps)
    own = hasattr(sampler, "begin_loop")
    if own:
        sampler.begin_loop(steps)  # this loop reads its cond afresh, timestep embeddings of all steps at once (B200DDIMSampler)
        kw = dict(kw)
    x = x_T_local
    for i, step in enumerate(steps):
        ts = torch.full((b,), int(step), device=x.device, dtype=torch.long)
        last = i == len(steps) - 1
        if own:
            kw["t_value"] = int(step)
        x, _ = sampler.denoising_step(x, cond_local, ts, index=len(steps) - i - 1, out=mine if last else None,
                                      peer_ptrs=peer_ptrs if last else None, **kw)
    return _gather_end(gathered, mine, hdl, world, group)


def _sample_with_sharded(sampler, S, batch_global, shape, cond_local, x_T_local, rank, world, group, fused_gather, kw):
    """run ``sampler.sample`` on this rank's chunk with its last update writing into the gather buffer; the samplers whose
    ``sample`` takes ``out=`` / ``peer_ptrs=`` (B200PLMSSampler, B200DPMSolverSampler)"""
    lo, hi = shard_bounds(batch_global, rank, world)
    gathered, mine, hdl, peer_ptrs = _gather_begin(batch_global, lo, hi, tuple(shape), x_T_local.device, world, group,
                                                   fused_gather)
    kw.setdefault("verbose", False)
    sampler.sample(S, hi - lo, tuple(shape), cond_local, x_T=x_T_local, out=mine, peer_ptrs=peer_ptrs, **kw)
    return _gather_end(gathered, mine, hdl, world, group)


def sample_plms_sharded(sampler, S, batch_global, shape, cond_local, x_T_local, rank=0, world=1, group=None,
                        fused_gather=False, **kw):
    """PLMS-sample this rank's chunk (B200PLMSSampler.sample) and all-gather the final latents.

    Arguments as sample_sharded; kw goes to sample (eta, guidance, callbacks).  Returns the [batch_global, C, H, W] latents
    on every rank.  Requires equal chunk sizes when world > 1."""
    return _sample_with_sharded(sampler, S, batch_global, shape, cond_local, x_T_local, rank, world, group, fused_gather, kw)


def sample_dpm_sharded(sampler, S, batch_global, shape, cond_local, x_T_local, rank=0, world=1, group=None,
                       fused_gather=False, **kw):
    """DPM-Solver-sample this rank's chunk (B200DPMSolverSampler.sample) and all-gather the final latents.

    Arguments as sample_sharded; kw goes to sample (guidance).  Returns the [batch_global, C, H, W] latents on every rank.
    Requires equal chunk sizes when world > 1."""
    return _sample_with_sharded(sampler, S, batch_global, shape, cond_local, x_T_local, rank, world, group, fused_gather, kw)


def encode_sharded(sampler, t_enc, batch_global, x0_local, cond_local, rank=0, world=1, group=None, fused_gather=False,
                   **kw):
    """DDIM-invert this rank's chunk (B200DDIMSampler.encode on the schedule already set) and all-gather the x_t.

    x0_local / cond_local hold this rank's rows only; kw goes to encode (guidance, use_original_steps, callback).
    Returns the [batch_global, C, H, W] inverted latents on every rank.  Requires equal chunk sizes when world > 1."""
    if t_enc < 1:
        raise ValueError("encode_sharded needs t_enc >= 1: the last inversion step writes the gathered result")
    lo, hi = shard_bounds(batch_global, rank, world)
    gathered, mine, hdl, peer_ptrs = _gather_begin(batch_global, lo, hi, tuple(x0_local.shape[1:]), x0_local.device, world,
                                                   group, fused_gather)
    sampler.encode(x0_local, cond_local, t_enc, out=mine, peer_ptrs=peer_ptrs, **kw)
    return _gather_end(gathered, mine, hdl, world, group)
