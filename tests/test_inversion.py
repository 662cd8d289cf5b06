"""DDIM inversion (upstream DDIMSampler.encode: x_0 -> x_t) — oracle restatement, B200 sampler and the sharded form.

The oracle side is tests/oracle_invert.py (upstream encode restated over oracle.MKDDIMSampler).
CPU: known answers, the exact-inverse property against reconstruct, the timesteps / RNG / CFG batching upstream's loop
implies, its return value and guards, the frozen fixture tests/golden/ddim_invert_v1.npz, the B200 sampler against the
oracle bit for bit (C-ABI calls replaced by the torch fakes of tests/fake_ops.py), and 2-rank gloo encode_sharded.
GPU (-m gpu): the update kernel against upstream's literal arithmetic on CUDA, reduced and yaml-size networks against
the fp32 oracle, the image -> latent -> inversion -> reconstruction -> image flow, and 2-GPU encode_sharded."""
import math
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

import fake_ops  # noqa: E402
from golden.make_golden_invert import CASES, compute  # noqa: E402
from makeupdiffuse_b200 import B200ControlLDM, B200DDIMSampler, ops  # noqa: E402
from makeupdiffuse_b200.dist import shard_bounds  # noqa: E402
from oracle import OracleControlLDM, seeded_state_dict  # noqa: E402
from oracle_invert import InvertingDDIMSampler  # noqa: E402
from toy_denoiser import ToyDenoiser, toy_inputs  # noqa: E402

GOLDEN = os.path.join(HERE, "golden", "ddim_invert_v1.npz")


@pytest.fixture()
def faked(monkeypatch):
    for name in fake_ops.ALL:
        monkeypatch.setattr(ops, name, getattr(fake_ops, name))


def rel(a, b):
    a, b = torch.as_tensor(a).float().cpu(), torch.as_tensor(b).float().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-20))


def psnr(a, b):
    peak = float(b.abs().max())
    return 10 * math.log10(peak * peak / float(((a.float() - b.float()) ** 2).mean()))


def toy_cond(i, kind="dict"):
    """the toy's cond in the three forms _cat_uncond_first accepts: (cond, uncond)"""
    if kind == "dict":
        return ({"c_crossattn": [i["ctx"]], "c_concat": [i["hint"]]}, {"c_crossattn": [i["uc_ctx"]], "c_concat": [i["hint"]]})
    if kind == "list":
        return [i["ctx"], i["hint"]], [i["uc_ctx"], i["hint"]]
    return i["ctx"], i["uc_ctx"]


class Recording(ToyDenoiser):
    """the toy denoiser that also keeps the timesteps and the cond rows of every call"""

    def __init__(self, device="cpu", eps=None):
        super().__init__(device)
        self.ts, self.conds, self.eps = [], [], eps

    def apply_model(self, x, t, c):
        self.ts.append(t.tolist())
        self.conds.append(self._leaves(c)[0].clone())
        if self.eps is not None:  # a fixed eps: depends neither on x nor on t
            return self.eps.expand_as(x).contiguous() if self.eps.shape[0] == x.shape[0] else torch.cat([self.eps] * 2)
        return super().apply_model(x, t, c)


def samplers(model, S):
    so, sb = InvertingDDIMSampler(model), B200DDIMSampler(model)
    so.make_schedule(S, ddim_eta=0.0, verbose=False)
    sb.make_schedule(S, ddim_eta=0.0, verbose=False)
    return so, sb


# ---- CPU: oracle and B200 sampler host logic --------------------------------------------------------------------------
@pytest.mark.parametrize("S,t_enc,gain", [(50, 50, 0.0760290), (20, 20, 0.0903435), (50, 10, 0.885054)])
def test_kat_eps_zero(faked, S, t_enc, gain):
    """eps == 0  =>  x_t = x_0 * sqrt(abar[t_enc - 1] / abar_prev[0]): the inverse of K2's 13.152870 / 11.068869"""
    m = ToyDenoiser()
    m.apply_model = lambda x, t, c: torch.zeros_like(x)
    x0 = toy_inputs()["x_T"]
    for s in samplers(m, S):
        x, d = s.encode(x0, None, t_enc)
        torch.testing.assert_close(x, x0 * gain, rtol=2e-6, atol=0)
        assert d["x_encoded"] is x and d["intermediate_steps"] == [] and "intermediates" not in d


@pytest.mark.parametrize("S,k", [(50, 50), (50, 17), (20, 20), (20, 6)])
def test_exact_inverse_of_reconstruct(faked, S, k):
    """eps independent of x and t: encode and reconstruct use the same coefficients in mirror order, so
    reconstruct(encode(x0, k), k) == x0 up to fp32 rounding, for the whole schedule and a truncated one"""
    i = toy_inputs()
    eps = torch.randn(3, 4, 8, 8, generator=torch.Generator().manual_seed(5))
    m = Recording(eps=eps)
    cond, _ = toy_cond(i)
    for s in samplers(m, S):
        xt, _ = s.encode(i["x_T"], cond, k)
        assert rel(xt, i["x_T"]) > 1e-2
        back = s.reconstruct(xt, cond, k)
        assert rel(back, i["x_T"]) < 1e-5, rel(back, i["x_T"])


def test_timesteps_rng_and_cfg_batching(faked):
    i = toy_inputs()
    for kind in ("dict", "list", "tensor"):
        cond, uc = toy_cond(i, kind)
        for s_name in ("oracle", "b200"):
            m = Recording()
            so, sb = samplers(m, 50)
            s = so if s_name == "oracle" else sb
            state = torch.get_rng_state()
            s.encode(i["x_T"], cond, 12)
            assert torch.equal(torch.get_rng_state(), state)               # no noise is drawn
            # the model sees the loop index, not ddim_timesteps[i]: one un-doubled call per step
            assert m.ts == [[j] * 3 for j in range(12)] and m.calls == [3] * 12
            for rec in (m.ts, m.calls, m.conds):
                rec.clear()
            s.encode(i["x_T"], cond, 4, unconditional_guidance_scale=3.0, unconditional_conditioning=uc)
            assert torch.equal(torch.get_rng_state(), state)
            assert m.ts == [[j] * 6 for j in range(4)] and m.calls == [6] * 4
            lead = lambda c: ToyDenoiser._leaves(c)[0]  # noqa: E731
            assert all(torch.equal(c, torch.cat([lead(uc), lead(cond)])) for c in m.conds)   # [uncond; cond]
            m.calls.clear()
            s.encode(i["x_T"], cond, 2, unconditional_guidance_scale=1.0, unconditional_conditioning=uc)
            assert m.calls == [3, 3]                                          # scale 1: uc is ignored
            with pytest.raises(AssertionError):
                s.encode(i["x_T"], cond, 2, unconditional_guidance_scale=3.0, unconditional_conditioning=None)


def test_return_value_and_guards(faked):
    i = toy_inputs()
    cond, _ = toy_cond(i)
    m = ToyDenoiser()
    so, sb = samplers(m, 50)
    for s in (so, sb):
        seen = []
        x, d = s.encode(i["x_T"], cond, 10, return_intermediates=3, callback=seen.append)
        assert sorted(d) == ["intermediate_steps", "intermediates", "x_encoded"]
        assert d["intermediate_steps"] == [0, 3, 6, 8, 9] and len(d["intermediates"]) == 5 and seen == list(range(10))
        assert d["intermediates"][-1] is x and d["x_encoded"] is x
        ptrs = {t.data_ptr() for t in d["intermediates"]}
        assert len(ptrs) == 5                                                # fresh tensors, no aliasing
        x, d = s.encode(i["x_T"], cond, 0)
        assert x is i["x_T"] and d == {"x_encoded": x, "intermediate_steps": []}
        with pytest.raises(AssertionError):
            s.encode(i["x_T"], cond, 51)
        with pytest.raises(AssertionError):
            s.encode(i["x_T"], cond, 1001, use_original_steps=True)
    # use_original_steps reads alphas_cumprod / alphas_cumprod_prev: eps == 0 gives sqrt(abar[k-1] / abar_prev[0])
    mz = ToyDenoiser()
    mz.apply_model = lambda x, t, c: torch.zeros_like(x)
    for s in samplers(mz, 50):
        x, _ = s.encode(i["x_T"], cond, 7, use_original_steps=True)
        gain = math.sqrt(float(mz.alphas_cumprod[6]) / float(mz.alphas_cumprod_prev[0]))
        torch.testing.assert_close(x, i["x_T"] * gain, rtol=2e-6, atol=0)


@pytest.mark.parametrize("kind", ["dict", "list", "tensor"])
def test_b200_equals_oracle_on_the_toy_bitwise(faked, kind):
    i = toy_inputs()
    cond, uc = toy_cond(i, kind)
    m = ToyDenoiser()
    for S, t_enc, orig in ((50, 50, False), (20, 13, False), (50, 9, True)):
        so, sb = samplers(m, S)
        for g in ({}, dict(unconditional_guidance_scale=7.5, unconditional_conditioning=uc)):
            a, da = so.encode(i["x_T"], cond, t_enc, use_original_steps=orig, return_intermediates=4, **g)
            b, db = sb.encode(i["x_T"], cond, t_enc, use_original_steps=orig, return_intermediates=4, **g)
            assert torch.equal(a, b) and da["intermediate_steps"] == db["intermediate_steps"]
            assert all(torch.equal(u, v) for u, v in zip(da["intermediates"], db["intermediates"]))


def test_b200_equals_oracle_on_reduced_networks(faked, tiny_params, monkeypatch):
    """the B200 sampler over B200ControlLDM (C-ABI faked) against the oracle networks, numerically; and against the oracle
    sampler driving the SAME model bit for bit once the per-loop timestep-embedding table is off (its embeddings come from
    a matrix product over all the loop's timesteps at once, whose fp32 rounding differs from the per-call product)"""
    o = OracleControlLDM(control_params=tiny_params, unet_params=tiny_params).eval()
    sd = seeded_state_dict(o, 0)
    m = B200ControlLDM(tiny_params, tiny_params, dtype=torch.float32, device="cpu").load_state_dict(sd)
    g = torch.Generator().manual_seed(3)
    cond = {"c_crossattn": [torch.randn(2, 77, 64, generator=g)], "c_concat": [torch.rand(2, 6, 64, 64, generator=g)]}
    uc = {"c_crossattn": [torch.randn(2, 77, 64, generator=g)], "c_concat": cond["c_concat"]}
    x0 = torch.randn(2, 4, 8, 8, generator=g)
    for guide in ({}, dict(unconditional_guidance_scale=4.0, unconditional_conditioning=uc)):
        sb = B200DDIMSampler(m)
        sm = InvertingDDIMSampler(m)
        so = InvertingDDIMSampler(o)
        for s in (sb, sm, so):
            s.make_schedule(6, ddim_eta=0.0, verbose=False)
        with torch.no_grad():
            b, _ = sb.encode(x0, cond, 6, **guide)
            a, _ = sm.encode(x0, cond, 6, **guide)
            r, _ = so.encode(x0, cond, 6, **guide)
        assert rel(b, r) < 1e-4 and rel(a, b) < 1e-5, (rel(b, r), rel(a, b))
        with monkeypatch.context() as mp_:
            mp_.setattr(m, "precompute_time_embeddings", lambda values: None)
            m._emb_table = None
            with torch.no_grad():
                assert torch.equal(sb.encode(x0, cond, 6, **guide)[0], sm.encode(x0, cond, 6, **guide)[0])


def test_oracle_and_b200_reproduce_the_frozen_fixture(faked):
    G = np.load(GOLDEN)
    assert sorted(G.files) == sorted(set(sum(([n] + ([n + "_inter", n + "_steps"] if ri else []) for n, *_, ri in CASES), [])))
    m = ToyDenoiser()
    for make in (lambda: InvertingDDIMSampler(m), lambda: B200DDIMSampler(m)):
        got = compute(make)
        for k in G.files:
            assert np.array_equal(got[k].numpy(), G[k]), k


# ---- CPU: 2-rank gloo encode_sharded ---------------------------------------------------------------------------------
PARAMS = dict(model_channels=32, num_heads=2, context_dim=32)
BG, H, T_ENC = 4, 8, 5


def _setup(patch=setattr):
    """patch: plain setattr in a spawned worker; monkeypatch.setattr in the pytest process"""
    from makeupdiffuse_b200.synth import synthetic_state_dict
    for name in fake_ops.ALL:
        patch(ops, name, getattr(fake_ops, name))
    m = B200ControlLDM(PARAMS, PARAMS, dtype=torch.float32, device="cpu")
    m.load_state_dict(synthetic_state_dict(m, 0, device="cpu"))
    s = B200DDIMSampler(m)
    s.make_schedule(10, ddim_eta=0.0, verbose=False)
    return s


def _data():
    g = torch.Generator().manual_seed(11)
    return {"ctx": torch.randn(BG, 77, 32, generator=g), "uctx": torch.randn(BG, 77, 32, generator=g),
            "hint": torch.rand(BG, 6, 8 * H, 8 * H, generator=g), "x0": torch.randn(BG, 4, H, H, generator=g)}


def _guide(d, lo, hi):
    return dict(unconditional_guidance_scale=3.0,
                unconditional_conditioning={"c_crossattn": [d["uctx"][lo:hi]], "c_concat": [d["hint"][lo:hi]]})


def _worker(rank, world, port, out_dir):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(2)
    from makeupdiffuse_b200.dist import encode_sharded
    s = _setup()
    d = _data()
    lo, hi = shard_bounds(BG, rank, world)
    cond = {"c_crossattn": [d["ctx"][lo:hi]], "c_concat": [d["hint"][lo:hi]]}
    res = {"plain": encode_sharded(s, T_ENC, BG, d["x0"][lo:hi].contiguous(), cond, rank, world),
           "cfg": encode_sharded(s, T_ENC, BG, d["x0"][lo:hi].contiguous(), cond, rank, world, **_guide(d, lo, hi))}
    torch.save(res, os.path.join(out_dir, f"r{rank}.pt"))
    dist.destroy_process_group()


def test_two_rank_gloo_encode_sharded_equals_single_process(tmp_path, monkeypatch):
    import torch.multiprocessing as mp
    port = 31500 + os.getpid() % 2000
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = torch.load(tmp_path / "r0.pt"), torch.load(tmp_path / "r1.pt")
    s = _setup(monkeypatch.setattr)
    d = _data()
    cond = {"c_crossattn": [d["ctx"]], "c_concat": [d["hint"]]}
    ref = {"plain": s.encode(d["x0"], cond, T_ENC)[0], "cfg": s.encode(d["x0"], cond, T_ENC, **_guide(d, 0, BG))[0]}
    for k in ("plain", "cfg"):
        assert torch.equal(r0[k], r1[k]) and r0[k].shape == (BG, 4, H, H)
        assert float((r0[k] - ref[k]).abs().max()) < 1e-4 * float(ref[k].abs().max()), k
    from makeupdiffuse_b200.dist import encode_sharded
    with pytest.raises(ValueError):
        encode_sharded(s, 0, BG, d["x0"], cond)


# ---- GPU ----------------------------------------------------------------------------------------------------------------
DEV = "cuda"


def _no_tf32():
    # the oracle must be TRUE fp32 on the GPU: cuDNN convolutions default to TF32 otherwise
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


@pytest.mark.gpu
@pytest.mark.parametrize("S", [50, 20])
def test_update_bitexact_against_upstream_arithmetic_on_cuda(S):
    """every index of the schedule: the product's update through mkd_ddim_update (sqrt(1-a_t) = 0, sqrt(a_t) = 1, the
    sampler's coefficients) against upstream's literal expression evaluated on CUDA with upstream's dtypes (fp32 alphas_next on
    the device, fp64 alphas on the CPU), plain and with the CFG combine; also use_original_steps (all fp32)"""
    m = ToyDenoiser(DEV)
    s = B200DDIMSampler(m)
    s.make_schedule(S, ddim_eta=0.0, verbose=False)
    g = torch.Generator(device=DEV).manual_seed(S)
    n = (16, 4, 32, 32)
    for orig in (False, True):
        if orig:
            an_dev, a_up = s.alphas_cumprod[:S], s.alphas_cumprod_prev[:S]
        else:
            an_dev, a_up = s.ddim_alphas[:S], torch.tensor(s.ddim_alphas_prev[:S])
        coef = s._encode_coefficients(an_dev, a_up)
        assert an_dev.is_cuda and (a_up.dtype == torch.float32) == orig
        for i in range(S):
            x = torch.randn(n, device=DEV, generator=g) * (1 + 3 * i / S)
            e2 = torch.randn((2 * n[0],) + n[1:], device=DEV, generator=g)
            for cfg in (None, 7.5):
                e = e2[:n[0]].contiguous() if cfg is None else e2
                if cfg is None:
                    noise_pred = e
                else:
                    e_u, e_c = torch.chunk(e, 2)
                    noise_pred = e_u + cfg * (e_c - e_u)
                ref = (an_dev[i] / a_up[i]).sqrt() * x + an_dev[i].sqrt() * ((1 / an_dev[i] - 1).sqrt() - (1 / a_up[i] - 1).sqrt()) * noise_pred
                out = torch.empty_like(x)
                ops.ddim_update(x, e, out, sqrt_one_minus_at=0.0, sqrt_at=1.0, sqrt_a_prev=coef[i][0], dir_coef=coef[i][1],
                                cfg_scale=cfg)
                assert torch.equal(out, ref), (orig, i, cfg, float((out - ref).abs().max()))
    # and the whole loop: the B200 sampler against the oracle over the same (CUDA) toy denoiser, bit for bit
    i = toy_inputs(DEV)
    cond, uc = toy_cond(i)
    so = InvertingDDIMSampler(m)
    so.make_schedule(S, ddim_eta=0.0, verbose=False)
    for guide in ({}, dict(unconditional_guidance_scale=7.5, unconditional_conditioning=uc)):
        assert torch.equal(s.encode(i["x_T"], cond, S, **guide)[0], so.encode(i["x_T"], cond, S, **guide)[0])


class Bundle:
    def __init__(self, params, f32=True):
        with torch.device(DEV):
            self.oracle = OracleControlLDM(control_params=params, unet_params=params).eval()
        sd = seeded_state_dict(self.oracle, 0)
        for p in self.oracle.parameters():
            p.requires_grad_(False)
        self.bf16 = B200ControlLDM(params, params, dtype=torch.bfloat16).load_state_dict(sd)
        self.f32 = B200ControlLDM(params, params, dtype=torch.float32).load_state_dict(sd) if f32 else None


@pytest.fixture(scope="module")
def tiny(tiny_params):
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    _no_tf32()
    return Bundle(tiny_params)


def make_cond(B, h, cdim, seed=0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    c = {"c_crossattn": [torch.randn(B, 77, cdim, device=DEV, generator=g)],
         "c_concat": [torch.rand(B, 6, 8 * h, 8 * h, device=DEV, generator=g)]}
    uc = {"c_crossattn": [torch.randn(B, 77, cdim, device=DEV, generator=g)], "c_concat": c["c_concat"]}
    # a clean latent scaled like get_z's output (scale_factor 0.18215 x the VAE posterior: about unit variance)
    return c, uc, torch.randn(B, 4, h, h, device=DEV, generator=g)


def _teacher_forced_encode(bundle, models, B, h, cdim, S, cfg_scale=1.0, seed=0):
    """the fp32 oracle's inversion records every (x_i, t = i, eps); each B200 model evaluates eps on the oracle's x_i through
    the sampler's own per-step call (embedding table, graph replay).  Returns {name: [rel-L2 per step]}"""
    cond, uc, x0 = make_cond(B, h, cdim, seed)
    so = InvertingDDIMSampler(bundle.oracle)
    so.make_schedule(S, ddim_eta=0.0, verbose=False)
    rec = []
    orig = bundle.oracle.apply_model
    bundle.oracle.apply_model = lambda x, t, c: (lambda e: (rec.append((x.clone(), t.clone(), e.clone())), e)[1])(orig(x, t, c))
    try:
        guide = dict(unconditional_guidance_scale=cfg_scale, unconditional_conditioning=uc) if cfg_scale != 1.0 else {}
        so.encode(x0, cond, S, **guide)
    finally:
        bundle.oracle.apply_model = orig
    assert [int(t[0]) for _, t, _ in rec] == list(range(S))
    out = {}
    for name, m in models.items():
        s = B200DDIMSampler(m, use_cuda_graph=True)
        s.make_schedule(S, ddim_eta=0.0, verbose=False)
        s.begin_loop(range(S))
        cc = s._cfg_cond(cond, uc) if cfg_scale != 1.0 else cond
        out[name] = [rel(s._eps(x, t, cc, t_value=k), e) for k, (x, t, e) in enumerate(rec)]
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("cfg_scale", [1.0, 9.0])
def test_teacher_forced_eps_reduced_networks(tiny, cfg_scale):
    r = _teacher_forced_encode(tiny, {"f32": tiny.f32, "bf16": tiny.bf16}, 2, 16, 64, S=10, cfg_scale=cfg_scale, seed=1)
    print(f"inversion teacher-forced eps rel-L2 (reduced nets, CFG {cfg_scale:g}): fp32-check max {max(r['f32']):.2e}, "
          f"bf16 max {max(r['bf16']):.2e}")
    assert max(r["f32"]) < 1e-4 and max(r["bf16"]) < 2e-2, r


@pytest.mark.gpu
def test_free_running_graph_and_loop_switches_reduced_networks(tiny):
    B, h, S = 2, 16, 10
    cond, uc, x0 = make_cond(B, h, 64, seed=2)
    with torch.no_grad():
        so = InvertingDDIMSampler(tiny.oracle)
        so.make_schedule(S, ddim_eta=0.0, verbose=False)
        ref, _ = so.encode(x0, cond, S)

    def fresh(m, graph=True):
        s = B200DDIMSampler(m, use_cuda_graph=graph)
        s.make_schedule(S, ddim_eta=0.0, verbose=False)
        return s

    a = fresh(tiny.f32, graph=False).encode(x0, cond, S)[0]
    g = fresh(tiny.f32).encode(x0, cond, S)[0]
    b = fresh(tiny.bf16).encode(x0, cond, S)[0]
    assert torch.equal(a, g)                                           # graph replay == eager
    assert torch.equal(fresh(tiny.bf16, graph=False).encode(x0, cond, S)[0], b)
    p32, p16 = psnr(a, ref), psnr(b, ref)
    print(f"inversion free-running {S} steps PSNR vs oracle: fp32-check {p32:.1f} dB, bf16 {p16:.1f} dB")
    assert p32 > 111 and p16 > 37, (p32, p16)  # measured 120.9 / 46.5 dB: gates within 10 dB of the measurement
    # one sampler: encode -> reconstruct -> encode equals fresh samplers (time-embedding table and graph switch loops)
    for m in (tiny.f32, tiny.bf16):
        s = fresh(m)
        e1 = s.encode(x0, cond, S, unconditional_guidance_scale=3.0, unconditional_conditioning=uc)[0].clone()
        r1 = s.reconstruct(e1, cond, S).clone()
        e2 = s.encode(r1, cond, 6)[0]
        assert torch.equal(e1, fresh(m).encode(x0, cond, S, unconditional_guidance_scale=3.0, unconditional_conditioning=uc)[0])
        assert torch.equal(r1, fresh(m).reconstruct(e1, cond, S))
        assert torch.equal(e2, fresh(m).encode(r1, cond, 6)[0])


@pytest.mark.gpu
def test_full_size_batch16_teacher_forced_all_50_inversion_steps():
    """yaml networks, batch 16, 256^2, bf16 (the benchmarked configuration) over all 50 inversion steps, teacher-forced
    against the fp32 oracle (TF32 off): eps at t = 0..49 on nearly clean latents"""
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    _no_tf32()
    full = Bundle({}, f32=False)
    r = _teacher_forced_encode(full, {"bf16": full.bf16}, 16, 32, 768, S=50, seed=3)["bf16"]
    print("full-size batch-16 inversion teacher-forced 50 steps: eps rel-L2 bf16 max %.2e (step %d) mean %.2e, first %.2e last %.2e"
          % (max(r), int(np.argmax(r)), sum(r) / len(r), r[0], r[-1]))
    del full
    torch.cuda.empty_cache()
    assert len(r) == 50 and max(r) < 1e-2, r


@pytest.mark.gpu
def test_invrec_round_trip_fp32_check():
    """the inversion flow a dataset of stored inverted latents is made with, end to end in fp32 check mode (reduced nets
    and VAE): image -> get_z -> encode -> reconstruct -> decode_first_stage, every stage against the oracle pipeline"""
    from makeupdiffuse_b200 import B200FirstStageDecoder, B200FirstStageEncoder
    from oracle.vae import OracleFirstStageDecoder, OracleFirstStageEncoder, decode_first_stage, get_z
    _no_tf32()
    params = dict(model_channels=64, num_heads=4, context_dim=64)
    dd = dict(ch=64, ch_mult=(1, 2, 4, 4), num_res_blocks=1)
    with torch.device(DEV):
        ol = OracleControlLDM(control_params=params, unet_params=params).eval()
        oe, od = OracleFirstStageEncoder(ddconfig=dd).eval(), OracleFirstStageDecoder(ddconfig=dd).eval()
    sd = seeded_state_dict(ol, 0)
    sde, sdd = seeded_state_dict(oe, 0, prefix="first_stage_model."), seeded_state_dict(od, 0, prefix="first_stage_model.")
    m = B200ControlLDM(params, params, dtype=torch.float32).load_state_dict(sd)
    m.attach_first_stage_encoder(B200FirstStageEncoder(ddconfig=dd, dtype=torch.float32).load_state_dict(sde))
    m.attach_first_stage_decoder(B200FirstStageDecoder(ddconfig=dd, dtype=torch.float32).load_state_dict(sdd))
    g = torch.Generator(device=DEV).manual_seed(8)
    B, hw, S = 2, 128, 10
    img = torch.rand(B, 3, hw, hw, device=DEV, generator=g) * 2 - 1
    cond = {"c_crossattn": [torch.randn(B, 77, 64, device=DEV, generator=g)],
            "c_concat": [torch.rand(B, 6, hw, hw, device=DEV, generator=g)]}
    n1 = torch.randn(B, 4, hw // 8, hw // 8, device=DEV, generator=g)
    so, sb = InvertingDDIMSampler(ol), B200DDIMSampler(m)
    so.make_schedule(S, ddim_eta=0.0, verbose=False)
    sb.make_schedule(S, ddim_eta=0.0, verbose=False)
    with torch.no_grad():
        z_ref = get_z(oe, img, n1)
        xt_ref, _ = so.encode(z_ref, cond, S)
        x_ref = so.decode(xt_ref, cond, S)
        img_ref = decode_first_stage(od, x_ref)
    z = m.get_z(img, n1)
    xt, _ = sb.encode(z, cond, S)
    x = sb.decode(xt, cond, S)
    out = m.decode_first_stage(x)
    r = (rel(z, z_ref), rel(xt, xt_ref), rel(x, x_ref), rel(out, img_ref))
    print("inversion round trip (fp32 check mode): rel-L2 z %.2e, inverted latents %.2e, reconstructed latents %.2e, image %.2e" % r)
    assert max(r) < 1e-3, r


def _gpu_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    from makeupdiffuse_b200.dist import encode_sharded
    from makeupdiffuse_b200.synth import synthetic_state_dict
    params = dict(model_channels=64, num_heads=4, context_dim=64)
    m = B200ControlLDM(params, params, dtype=torch.bfloat16, device=dev)
    m.load_state_dict(synthetic_state_dict(m, 0, dev))
    s = B200DDIMSampler(m)
    s.make_schedule(10, ddim_eta=0.0, verbose=False)
    g = torch.Generator(device=dev).manual_seed(7)
    bg, h = 4, 16
    ctx = torch.randn(bg, 77, 64, device=dev, generator=g)
    hint = torch.rand(bg, 6, 8 * h, 8 * h, device=dev, generator=g)
    x0 = torch.randn(bg, 4, h, h, device=dev, generator=g)
    lo, hi = shard_bounds(bg, rank, world)
    cond = {"c_crossattn": [ctx[lo:hi].contiguous()], "c_concat": [hint[lo:hi].contiguous()]}
    res = {}
    for name, fused in (("nccl", False), ("fused", True), ("fused_again", True)):
        res[name] = encode_sharded(s, 10, bg, x0[lo:hi].contiguous(), cond, rank, world, fused_gather=fused).cpu()
    res["single"] = s.encode(x0, {"c_crossattn": [ctx], "c_concat": [hint]}, 10)[0].cpu()
    torch.save(res, os.path.join(out_dir, f"g{rank}.pt"))
    dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs of one box")
def test_two_gpu_encode_sharded_fused_gather_equals_nccl(tmp_path):
    import torch.multiprocessing as mp
    port = 31600 + os.getpid() % 2000
    mp.spawn(_gpu_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = torch.load(tmp_path / "g0.pt"), torch.load(tmp_path / "g1.pt")
    for r in (r0, r1):
        assert torch.equal(r["nccl"], r["fused"]) and torch.equal(r["fused"], r["fused_again"])
    assert torch.equal(r0["fused"], r1["fused"])
    # a rank's kernels see another batch size than the single-process run (tile / split-K choices differ): numerical
    assert float((r0["fused"] - r0["single"]).abs().max()) < 0.05 * float(r0["single"].abs().max())
