"""PLMS sampling (upstream ldm PLMSSampler) — oracle restatement, B200PLMSSampler, its update kernel and the sharded form.

The oracle side is tests/oracle_plms.py (upstream PLMSSampler restated over oracle.ddim.DDIMSampler).
CPU: known answers, PLMS == DDIM when eps depends neither on x nor on t, the timesteps / RNG / CFG batching upstream's loop
implies, guards, the B200 sampler against the oracle bit for bit (C-ABI calls replaced by the torch fakes of
tests/fake_ops.py and tests/fake_plms_ops.py), the frozen fixture tests/golden/plms_v1.npz, 2-rank gloo sample_plms_sharded
and log_results.
GPU (-m gpu): mkd_plms_update against upstream's torch expressions on CUDA, reduced and yaml-size networks against the fp32
oracle, and the 2-GPU gather paths."""
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

import fake_plms_ops  # noqa: E402
from golden.make_golden_plms import CASES, compute  # noqa: E402
from makeupdiffuse_b200 import B200ControlLDM, B200DDIMSampler, B200PLMSSampler, ops  # noqa: E402
from makeupdiffuse_b200.dist import shard_bounds  # noqa: E402
from oracle import MKDDIMSampler, OracleControlLDM, seeded_state_dict  # noqa: E402
from oracle_plms import PLMSSampler  # noqa: E402
from toy_denoiser import ToyDenoiser, toy_inputs  # noqa: E402

GOLDEN = os.path.join(HERE, "golden", "plms_v1.npz")


@pytest.fixture()
def faked(monkeypatch):
    fake_plms_ops.install(ops, monkeypatch.setattr)


def rel(a, b):
    a, b = torch.as_tensor(a).float().cpu(), torch.as_tensor(b).float().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-20))


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
            self.calls.append(int(x.shape[0]))
            return self.eps.clone() if self.eps.shape[0] == x.shape[0] else torch.cat([self.eps] * 2)
        return super().apply_model(x, t, c)


def run(s, S, i, cond, **kw):
    return s.sample(S, i["x_T"].shape[0], tuple(i["x_T"].shape[1:]), cond, x_T=i["x_T"], verbose=False, **kw)


# ---- CPU: oracle and B200 sampler host logic --------------------------------------------------------------------------
@pytest.mark.parametrize("S,gain", [(50, 13.152870), (20, 11.068869)])
def test_kat_eps_zero(faked, S, gain):
    """K2: eps == 0 makes every combination 0, so x_0 = x_T * sqrt(a_prev[0] / a[last]) as for DDIM"""
    m = ToyDenoiser()
    m.apply_model = lambda x, t, c: torch.zeros_like(x)
    i = toy_inputs()
    for s in (PLMSSampler(m), B200PLMSSampler(m)):
        x, _ = run(s, S, i, None)
        torch.testing.assert_close(x, i["x_T"] * gain, rtol=2e-6, atol=0)


@pytest.mark.parametrize("S", [50, 20, 4, 1])
def test_eps_independent_of_x_and_t_equals_ddim(faked, S):
    """every PLMS coefficient set sums to 1, so with one fixed eps PLMS takes DDIM's steps up to fp32 rounding"""
    i = toy_inputs()
    eps = torch.randn(3, 4, 8, 8, generator=torch.Generator().manual_seed(5))
    m = Recording(eps=eps)
    cond, _ = toy_cond(i)
    ddim = run(MKDDIMSampler(m), S, i, cond)[0]
    for s in (PLMSSampler(m), B200PLMSSampler(m)):
        x = run(s, S, i, cond)[0]
        assert rel(x, ddim) < 2e-6, rel(x, ddim)
    assert rel(ddim, i["x_T"]) > 1e-2


@pytest.mark.parametrize("S", [50, 4, 1])
def test_timesteps_rng_and_cfg_batching(faked, S):
    i = toy_inputs()
    steps = [int(v) for v in np.flip(np.asarray(list(range(0, 1000, 1000 // S))) + 1)]
    seen = [steps[0]] + [steps[min(1, S - 1)]] + steps[1:]           # t0, t1 (t0 again when S == 1), t1, t2, ...
    for kind in ("dict", "list", "tensor"):
        cond, uc = toy_cond(i, kind)
        for make in (PLMSSampler, B200PLMSSampler):
            m = Recording()
            s = make(m)
            torch.manual_seed(7)
            run(s, S, i, cond)
            after = torch.get_rng_state()
            torch.manual_seed(7)
            for _ in range(S + 1):
                torch.randn(i["x_T"].shape)
            assert torch.equal(after, torch.get_rng_state())             # S + 1 draws of randn(x.shape)
            assert m.ts == [[v] * 3 for v in seen] and m.calls == [3] * (S + 1)
            for rec in (m.ts, m.calls, m.conds):
                rec.clear()
            run(s, S, i, cond, unconditional_guidance_scale=3.0, unconditional_conditioning=uc)
            assert m.ts == [[v] * 6 for v in seen] and m.calls == [6] * (S + 1)
            lead = lambda c: ToyDenoiser._leaves(c)[0]  # noqa: E731
            assert all(torch.equal(c, torch.cat([lead(uc), lead(cond)])) for c in m.conds)   # [uncond; cond]
            m.calls.clear()
            run(s, S, i, cond, unconditional_guidance_scale=1.0, unconditional_conditioning=uc)
            assert m.calls == [3] * (S + 1)                                 # scale 1: uc is ignored, no doubling


def test_guards(faked):
    i = toy_inputs()
    cond, _ = toy_cond(i)
    m = ToyDenoiser()
    for s in (PLMSSampler(m), B200PLMSSampler(m)):
        with pytest.raises(ValueError, match="ddim_eta must be 0 for PLMS"):
            s.make_schedule(10, ddim_eta=0.5, verbose=False)
        with pytest.raises(ValueError, match="ddim_eta must be 0 for PLMS"):
            run(s, 10, i, cond, eta=1.0)
    s = B200PLMSSampler(m)
    for kw in (dict(dynamic_threshold=0.9), dict(score_corrector=object()), dict(quantize_x0=True)):
        with pytest.raises(NotImplementedError):
            run(s, 4, i, cond, **kw)
    s.make_schedule(4, verbose=False)
    with pytest.raises(NotImplementedError):
        s.plms_sampling(cond, tuple(i["x_T"].shape), x_T=i["x_T"], ddim_use_original_steps=True)
    with pytest.raises(NotImplementedError):
        s.p_sample_plms(i["x_T"], cond, torch.full((3,), 1), 0, use_original_steps=True)


def test_noise_options_at_sigma_zero(faked):
    """temperature and noise_dropout act on sigma * noise, which is 0 for PLMS: results unchanged; repeat_noise draws one
    sample's noise per call (the B200 loop handles all three as denoising_step does at sigma == 0)"""
    i = toy_inputs()
    cond, _ = toy_cond(i)
    m = ToyDenoiser()
    base = run(B200PLMSSampler(m), 4, i, cond)[0]
    for kw in (dict(temperature=0.3), dict(noise_dropout=0.5)):
        assert torch.equal(run(B200PLMSSampler(m), 4, i, cond, **kw)[0], base)
    s = B200PLMSSampler(m)
    s.make_schedule(4, verbose=False)
    t = torch.full((3,), 751, dtype=torch.long)
    torch.manual_seed(3)
    x1, p1, e1 = s.p_sample_plms(i["x_T"], cond, t, 3, repeat_noise=True, t_next=torch.full((3,), 501, dtype=torch.long))
    after = torch.get_rng_state()
    torch.manual_seed(3)
    torch.randn(1, 4, 8, 8)
    torch.randn(1, 4, 8, 8)
    assert torch.equal(after, torch.get_rng_state())
    x2, p2, e2 = s.p_sample_plms(i["x_T"], cond, t, 3, t_next=torch.full((3,), 501, dtype=torch.long))
    assert torch.equal(x1, x2) and torch.equal(p1, p2) and torch.equal(e1, e2)


@pytest.mark.parametrize("kind", ["dict", "list", "tensor"])
def test_b200_equals_oracle_on_the_toy_bitwise(faked, kind):
    i = toy_inputs()
    cond, uc = toy_cond(i, kind)
    m = ToyDenoiser()
    for S in (50, 20, 4, 1):
        for g in ({}, dict(unconditional_guidance_scale=7.5, unconditional_conditioning=uc)):
            got = []
            for make in (PLMSSampler, B200PLMSSampler):
                cb, icb = [], []
                x, inter = run(make(m), S, i, cond, log_every_t=3, callback=cb.append,
                               img_callback=lambda p, k: icb.append((p.clone(), k)), **g)
                got.append((x, inter, cb, icb))
            (a, ia, ca, ja), (b, ib, cb_, jb) = got
            assert torch.equal(a, b) and ca == cb_ == list(range(S))
            assert len(ia["x_inter"]) == len(ib["x_inter"]) and len(ia["pred_x0"]) == len(ib["pred_x0"])
            for key in ("x_inter", "pred_x0"):
                assert all(torch.equal(u, v) for u, v in zip(ia[key], ib[key])), key
            assert all(torch.equal(u, v) and k == l for (u, k), (v, l) in zip(ja, jb))


def test_p_sample_plms_returns_upstreams_triple(faked):
    """called directly with a caller-held history (upstream's old_eps list), as a loop outside the sampler would"""
    i = toy_inputs()
    cond, uc = toy_cond(i)
    m = ToyDenoiser()
    g = dict(unconditional_guidance_scale=4.0, unconditional_conditioning=uc)
    so, sb = PLMSSampler(m), B200PLMSSampler(m)
    for s in (so, sb):
        s.make_schedule(20, verbose=False)
    steps = np.flip(so.ddim_timesteps)
    xo = xb = i["x_T"]
    ho, hb = [], []
    for k, step in enumerate(steps[:6]):
        t = torch.full((3,), int(step), dtype=torch.long)
        tn = torch.full((3,), int(steps[k + 1]), dtype=torch.long)
        xo, po, eo = so.p_sample_plms(xo, cond, t, 19 - k, old_eps=ho, t_next=tn, **g)
        xb, pb, eb = sb.p_sample_plms(xb, cond, t, 19 - k, old_eps=hb, t_next=tn, **g)
        assert torch.equal(xo, xb) and torch.equal(po, pb) and torch.equal(eo, eb)
        ho.append(eo)
        hb.append(eb)  # a longer history than three: the newest three count, as upstream's ">= 3" branch
    assert len({t.data_ptr() for t in hb}) == 6


def test_oracle_and_b200_reproduce_the_frozen_fixture(faked):
    G = np.load(GOLDEN)
    assert sorted(G.files) == sorted(sum(([n] + ([n + "_x_inter", n + "_pred_x0"] if le else []) for n, _, _, le in CASES), []))
    m = ToyDenoiser()
    for make in (lambda: PLMSSampler(m), lambda: B200PLMSSampler(m)):
        got = compute(make)
        for k in G.files:
            assert np.array_equal(got[k].numpy(), G[k]), k


def test_b200_equals_oracle_on_reduced_networks(faked, tiny_params):
    """B200PLMSSampler over B200ControlLDM (C-ABI faked) against the oracle sampler over the oracle networks"""
    o = OracleControlLDM(control_params=tiny_params, unet_params=tiny_params).eval()
    sd = seeded_state_dict(o, 0)
    m = B200ControlLDM(tiny_params, tiny_params, dtype=torch.float32, device="cpu").load_state_dict(sd)
    g = torch.Generator().manual_seed(3)
    cond = {"c_crossattn": [torch.randn(2, 77, 64, generator=g)], "c_concat": [torch.rand(2, 6, 64, 64, generator=g)]}
    uc = {"c_crossattn": [torch.randn(2, 77, 64, generator=g)], "c_concat": cond["c_concat"]}
    x_T = torch.randn(2, 4, 8, 8, generator=g)
    for guide in ({}, dict(unconditional_guidance_scale=4.0, unconditional_conditioning=uc)):
        with torch.no_grad():
            b, _ = B200PLMSSampler(m).sample(5, 2, (4, 8, 8), cond, x_T=x_T, verbose=False, **guide)
            r, _ = PLMSSampler(o).sample(5, 2, (4, 8, 8), cond, x_T=x_T, verbose=False, **guide)
        assert rel(b, r) < 1e-4, rel(b, r)


def test_log_results_runs_with_the_plms_sampler(faked):
    """harness.log_results(..., sampler=B200PLMSSampler(model)) unchanged: its sample panels are PLMS samples (S + 1
    evaluations per run, doubled under guidance) and differ from the DDIM panels of the same seeds"""
    from makeupdiffuse_b200 import B200FirstStageDecoder, B200FirstStageEncoder, harness
    from oracle.vae import OracleFirstStageDecoder, OracleFirstStageEncoder
    params = dict(model_channels=32, num_heads=2, context_dim=32)
    dd = dict(ch=32, ch_mult=(1, 2, 4, 4), num_res_blocks=1)                    # 8x down / up, as the harness assumes
    ol = OracleControlLDM(control_params=params, unet_params=params).eval()
    oe, od = OracleFirstStageEncoder(ddconfig=dd).eval(), OracleFirstStageDecoder(ddconfig=dd).eval()
    m = B200ControlLDM(params, params, dtype=torch.float32, device="cpu").load_state_dict(seeded_state_dict(ol, 0))
    m.attach_first_stage_encoder(B200FirstStageEncoder(ddconfig=dd, dtype=torch.float32).load_state_dict(
        seeded_state_dict(oe, 0, prefix="first_stage_model."), device="cpu"))
    m.attach_first_stage_decoder(B200FirstStageDecoder(ddconfig=dd, dtype=torch.float32).load_state_dict(
        seeded_state_dict(od, 0, prefix="first_stage_model."), device="cpu"))
    m.get_unconditional_conditioning = lambda n: torch.zeros(n, 77, 32)  # no text encoder attached to this small model
    B, hw, S = 2, 64, 4
    g = torch.Generator().manual_seed(5)
    batch = {"pgt_sr": torch.rand(B, 3, hw, hw, generator=g) * 2 - 1, "src_img": torch.rand(B, 3, hw, hw, generator=g),
             "ref_img": torch.rand(B, 3, hw, hw, generator=g), "c_crossattn": torch.randn(B, 77, 32, generator=g)}
    calls = []
    orig = m.apply_model
    m.apply_model = lambda x, t, c, *a, **k: (calls.append(int(x.shape[0])), orig(x, t, c, *a, **k))[1]
    logs = {}
    for name, make in (("plms", B200PLMSSampler), ("ddim", B200DDIMSampler)):
        calls.clear()
        torch.manual_seed(0)
        logs[name] = harness.log_results(m, batch, 0, ddim_steps=S, unconditional_guidance_scale=9.0, sampler=make(m),
                                         generator=torch.Generator().manual_seed(11))
        n = S + 1 if name == "plms" else S
        assert calls == [B] + [B] * n + [2 * B] * n, (name, calls)
    a, b = logs["plms"], logs["ddim"]
    assert list(a) == list(b) and "samples_cfg_scale_9.00" in a
    for k in a:
        assert a[k].shape == b[k].shape and bool(torch.isfinite(a[k]).all())
    assert torch.equal(a["reconstruction"], b["reconstruction"]) and not torch.equal(a["samples"], b["samples"])


# ---- CPU: 2-rank gloo sample_plms_sharded ----------------------------------------------------------------------------
PARAMS = dict(model_channels=32, num_heads=2, context_dim=32)
BG, H, STEPS = 4, 8, 5


def _setup(patch=setattr):
    """patch: plain setattr in a spawned worker; monkeypatch.setattr in the pytest process"""
    from makeupdiffuse_b200.synth import synthetic_state_dict
    fake_plms_ops.install(ops, patch)
    m = B200ControlLDM(PARAMS, PARAMS, dtype=torch.float32, device="cpu")
    m.load_state_dict(synthetic_state_dict(m, 0, device="cpu"))
    return B200PLMSSampler(m)


def _data():
    g = torch.Generator().manual_seed(12)
    return {"ctx": torch.randn(BG, 77, 32, generator=g), "uctx": torch.randn(BG, 77, 32, generator=g),
            "hint": torch.rand(BG, 6, 8 * H, 8 * H, generator=g), "x_T": torch.randn(BG, 4, H, H, generator=g)}


def _guide(d, lo, hi):
    return dict(unconditional_guidance_scale=3.0,
                unconditional_conditioning={"c_crossattn": [d["uctx"][lo:hi]], "c_concat": [d["hint"][lo:hi]]})


def _worker(rank, world, port, out_dir):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(2)
    from makeupdiffuse_b200.dist import sample_plms_sharded
    s = _setup()
    d = _data()
    lo, hi = shard_bounds(BG, rank, world)
    cond = {"c_crossattn": [d["ctx"][lo:hi]], "c_concat": [d["hint"][lo:hi]]}
    x_T = d["x_T"][lo:hi].contiguous()
    res = {"plain": sample_plms_sharded(s, STEPS, BG, (4, H, H), cond, x_T, rank, world),
           "cfg": sample_plms_sharded(s, STEPS, BG, (4, H, H), cond, x_T, rank, world, **_guide(d, lo, hi))}
    torch.save(res, os.path.join(out_dir, f"r{rank}.pt"))
    dist.destroy_process_group()


def test_two_rank_gloo_sample_plms_sharded_equals_single_process(tmp_path, monkeypatch):
    import torch.multiprocessing as mp
    port = 33500 + os.getpid() % 2000
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = torch.load(tmp_path / "r0.pt"), torch.load(tmp_path / "r1.pt")
    s = _setup(monkeypatch.setattr)
    d = _data()
    cond = {"c_crossattn": [d["ctx"]], "c_concat": [d["hint"]]}
    ref = {"plain": s.sample(STEPS, BG, (4, H, H), cond, x_T=d["x_T"], verbose=False)[0],
           "cfg": s.sample(STEPS, BG, (4, H, H), cond, x_T=d["x_T"], verbose=False, **_guide(d, 0, BG))[0]}
    for k in ("plain", "cfg"):
        assert torch.equal(r0[k], r1[k]) and r0[k].shape == (BG, 4, H, H)
        assert float((r0[k] - ref[k]).abs().max()) < 1e-4 * float(ref[k].abs().max()), k
    # one process, world 1: the gather buffer is the result itself
    from makeupdiffuse_b200.dist import sample_plms_sharded
    assert torch.equal(sample_plms_sharded(s, STEPS, BG, (4, H, H), cond, d["x_T"]), ref["plain"])


# ---- GPU ----------------------------------------------------------------------------------------------------------------
DEV = "cuda"


def _no_tf32():
    # the oracle must be TRUE fp32 on the GPU: cuDNN convolutions default to TF32 otherwise
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


def _upstream_update(x, eps, cfg, hist, mode, coef_tensors):
    """upstream p_sample_plms's torch expressions after the model call, evaluated on CUDA"""
    if cfg is None:
        e_t = eps
    else:
        e_t_uncond, e_t = eps.chunk(2)
        e_t = e_t_uncond + cfg * (e_t - e_t_uncond)
    o = hist
    if mode == 0:
        ep = e_t
    elif mode == 1:
        ep = (o[0] + e_t) / 2
    elif mode == 2:
        ep = (3 * e_t - o[0]) / 2
    elif mode == 3:
        ep = (23 * e_t - 16 * o[0] + 5 * o[1]) / 12
    else:
        ep = (55 * e_t - 59 * o[0] + 37 * o[1] - 9 * o[2]) / 24
    a_t, a_prev, sigma_t, sqrt_one_minus_at = coef_tensors
    pred_x0 = (x - sqrt_one_minus_at * ep) / a_t.sqrt()
    dir_xt = (1.0 - a_prev - sigma_t ** 2).sqrt() * ep
    noise = sigma_t * torch.randn(x.shape, device=x.device) * 1.0
    return a_prev.sqrt() * pred_x0 + dir_xt + noise, pred_x0, e_t


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 65539])
def test_plms_update_bitexact_against_upstream_torch_on_cuda(n):
    """every mode, CFG on and off, several schedule indices: x_prev, pred_x0 and the stored e_t against upstream's literal
    expressions on CUDA fp32 tensors; the in-place forms the sampler uses (x_prev == x, e_store == the oldest history
    slot); and the peers entry (one and two destinations) against the local one"""
    m = ToyDenoiser(DEV)
    s = B200PLMSSampler(m)
    s.make_schedule(50, verbose=False)
    g = torch.Generator(device=DEV).manual_seed(n)
    shape = (n, 1, 1, 1)
    r = lambda k=1: torch.randn((k * n, 1, 1, 1), device=DEV, generator=g)  # noqa: E731
    for index in (49, 44, 31, 7, 6, 0):  # 44, 7 and 6: entries where torch's fp32 sqrt on the CPU is one ulp off
        full = lambda v: torch.full(shape, float(v[index]), device=DEV)  # noqa: E731
        ct = (full(s.ddim_alphas), full(s.ddim_alphas_prev), full(s.ddim_sigmas), full(s.ddim_sqrt_one_minus_alphas))
        a_t, a_prev, sigma_t, s1 = (v[0].reshape(()) for v in ct)
        coef = dict(sqrt_one_minus_at=float(s1), sqrt_at=float(a_t.sqrt()), sqrt_a_prev=float(a_prev.sqrt()),
                    dir_coef=float((1.0 - a_prev - sigma_t ** 2).sqrt()))
        # the sampler's table holds the same values: it takes the square roots on the model's device, as upstream does
        assert s._coef_ddim[index] == [coef["sqrt_one_minus_at"], coef["sqrt_at"], coef["sqrt_a_prev"], coef["dir_coef"], 0.0]
        for mode in range(5):
            for cfg in (None, 7.5):
                x = r() * 3
                eps = r(1 if cfg is None else 2)
                hist = [r() for _ in range(ops.PLMS_HISTORY[mode])]
                ref_x, ref_p, ref_e = _upstream_update(x, eps, cfg, hist, mode, ct)
                out, p0, es = torch.empty_like(x), torch.empty_like(x), torch.empty_like(x)
                ops.plms_update(x, eps, out, mode=mode, history=tuple(hist), e_store=es, pred_x0=p0, cfg_scale=cfg, **coef)
                what = (index, mode, cfg)
                assert torch.equal(out, ref_x), (what, float((out - ref_x).abs().max()))
                assert torch.equal(p0, ref_p) and torch.equal(es, ref_e), what
                # in place: x_prev over x, and the newest e_t over the oldest history slot it reads
                xi, h = x.clone(), [t.clone() for t in hist]
                ops.plms_update(xi, eps, xi, mode=mode, history=tuple(h), e_store=h[-1] if h else None, cfg_scale=cfg, **coef)
                assert torch.equal(xi, ref_x), ("in place", what)
                if h:
                    assert torch.equal(h[-1], ref_e) and all(torch.equal(u, v) for u, v in zip(h[:-1], hist[:-1])), what
                # peers: one destination, then two
                o1, o2 = torch.empty_like(x), torch.empty_like(x)
                ops.plms_update(x, eps, o1, mode=mode, history=tuple(hist), cfg_scale=cfg, peer_ptrs=[o1.data_ptr()], **coef)
                assert torch.equal(o1, ref_x), ("peers", what)
                o1.zero_()
                ops.plms_update(x, eps, o1, mode=mode, history=tuple(hist), cfg_scale=cfg, pred_x0=p0,
                                peer_ptrs=[o1.data_ptr(), o2.data_ptr()], **coef)
                assert torch.equal(o1, ref_x) and torch.equal(o2, ref_x) and torch.equal(p0, ref_p), ("2 peers", what)
    with pytest.raises(ValueError):
        ops.plms_update(x, eps, out, mode=3, history=(x,), **coef)


@pytest.mark.gpu
def test_b200_equals_oracle_on_the_toy_on_cuda():
    """the whole loop over the CUDA toy denoiser: B200PLMSSampler (the kernel) against the oracle (upstream's torch on CUDA),
    bit for bit, with and without guidance"""
    i = toy_inputs(DEV)
    cond, uc = toy_cond(i)
    m = ToyDenoiser(DEV)
    for S in (50, 4, 1):
        for guide in ({}, dict(unconditional_guidance_scale=7.5, unconditional_conditioning=uc)):
            a, ia = run(PLMSSampler(m), S, i, cond, log_every_t=5, **guide)
            b, ib = run(B200PLMSSampler(m), S, i, cond, log_every_t=5, **guide)
            assert torch.equal(a, b), (S, guide.keys(), float((a - b).abs().max()))
            assert all(torch.equal(u, v) for u, v in zip(ia["pred_x0"], ib["pred_x0"]))


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
    return c, uc, torch.randn(B, 4, h, h, device=DEV, generator=g)


@pytest.mark.gpu
@pytest.mark.parametrize("cfg_scale", [1.0, 5.0])
def test_free_running_reduced_networks_against_oracle(tiny, cfg_scale):
    B, h, S = 2, 16, 10
    cond, uc, x_T = make_cond(B, h, 64, seed=2)
    guide = dict(unconditional_guidance_scale=cfg_scale, unconditional_conditioning=uc) if cfg_scale != 1.0 else {}
    with torch.no_grad():
        ref, _ = PLMSSampler(tiny.oracle).sample(S, B, (4, h, h), cond, x_T=x_T, verbose=False, **guide)

    def go(m, graph):
        return B200PLMSSampler(m, use_cuda_graph=graph).sample(S, B, (4, h, h), cond, x_T=x_T, verbose=False, **guide)[0]

    a, g = go(tiny.f32, False), go(tiny.f32, True)
    b, bg = go(tiny.bf16, False), go(tiny.bf16, True)
    assert torch.equal(a, g) and torch.equal(b, bg)                    # graph replay == eager
    r32, r16 = rel(a, ref), rel(b, ref)
    print(f"PLMS-{S} free-running final latents rel-L2 vs oracle (reduced nets, CFG {cfg_scale:g}): fp32-check {r32:.2e}, "
          f"bf16 {r16:.2e}")
    assert r32 < 1e-4 and r16 < 5e-2, (r32, r16)
    # one sampler reused: a DDIM-length change and a second run reproduce fresh samplers (ring, table and graph per loop)
    s = B200PLMSSampler(tiny.bf16)
    s.sample(4, B, (4, h, h), cond, x_T=x_T, verbose=False)
    assert torch.equal(s.sample(S, B, (4, h, h), cond, x_T=x_T, verbose=False, **guide)[0], bg)


@pytest.mark.gpu
def test_full_size_batch16_teacher_forced_all_51_plms_evaluations():
    """yaml networks, batch 16, 256^2, bf16 (the benchmarked configuration): every one of PLMS-50's 51 evaluations,
    teacher-forced against the fp32 oracle (TF32 off) through the sampler's own per-step call (embedding table, graph)"""
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    _no_tf32()
    full = Bundle({}, f32=False)
    S, B, h = 50, 16, 32
    cond, _, x_T = make_cond(B, h, 768, seed=3)
    so = PLMSSampler(full.oracle)
    rec = []
    orig = full.oracle.apply_model
    full.oracle.apply_model = lambda x, t, c: (lambda e: (rec.append((x.clone(), t.clone(), e.clone())), e)[1])(orig(x, t, c))
    try:
        so.sample(S, B, (4, h, h), cond, x_T=x_T, verbose=False)
    finally:
        full.oracle.apply_model = orig
    assert len(rec) == S + 1
    s = B200PLMSSampler(full.bf16, use_cuda_graph=True)
    s.make_schedule(S, verbose=False)
    s.begin_loop(np.flip(s.ddim_timesteps))
    r = [rel(s._eps(x, t, cond, t_value=int(t[0])), e) for x, t, e in rec]
    print("full-size batch-16 PLMS-50 teacher-forced 51 evaluations: eps rel-L2 bf16 max %.2e (evaluation %d) mean %.2e"
          % (max(r), int(np.argmax(r)), sum(r) / len(r)))
    del full
    torch.cuda.empty_cache()
    assert max(r) <= 1e-2, r


def _gpu_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    from makeupdiffuse_b200.dist import sample_plms_sharded
    from makeupdiffuse_b200.synth import synthetic_state_dict
    params = dict(model_channels=64, num_heads=4, context_dim=64)
    m = B200ControlLDM(params, params, dtype=torch.bfloat16, device=dev)
    m.load_state_dict(synthetic_state_dict(m, 0, dev))
    s = B200PLMSSampler(m)
    g = torch.Generator(device=dev).manual_seed(7)
    bg, h = 4, 16
    ctx = torch.randn(bg, 77, 64, device=dev, generator=g)
    hint = torch.rand(bg, 6, 8 * h, 8 * h, device=dev, generator=g)
    x_T = torch.randn(bg, 4, h, h, device=dev, generator=g)
    lo, hi = shard_bounds(bg, rank, world)
    cond = {"c_crossattn": [ctx[lo:hi].contiguous()], "c_concat": [hint[lo:hi].contiguous()]}
    res = {}
    for name, fused in (("nccl", False), ("fused", True), ("fused_again", True)):
        res[name] = sample_plms_sharded(s, 10, bg, (4, h, h), cond, x_T[lo:hi].contiguous(), rank, world,
                                        fused_gather=fused).cpu()
    res["single"] = s.sample(10, bg, (4, h, h), {"c_crossattn": [ctx], "c_concat": [hint]}, x_T=x_T, verbose=False)[0].cpu()
    torch.save(res, os.path.join(out_dir, f"g{rank}.pt"))
    dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs of one box")
def test_two_gpu_sample_plms_sharded_fused_gather_equals_nccl(tmp_path):
    import torch.multiprocessing as mp
    port = 33700 + os.getpid() % 2000
    mp.spawn(_gpu_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = torch.load(tmp_path / "g0.pt"), torch.load(tmp_path / "g1.pt")
    for r in (r0, r1):
        assert torch.equal(r["nccl"], r["fused"]) and torch.equal(r["fused"], r["fused_again"])
    assert torch.equal(r0["fused"], r1["fused"])
    # a rank's kernels see another batch size than the single-process run (tile / split-K choices differ): numerical
    assert float((r0["fused"] - r0["single"]).abs().max()) < 0.05 * float(r0["single"].abs().max())
