"""DPM-Solver++ sampling (upstream ldm DPMSolverSampler) — oracle restatement, B200DPMSolverSampler, its update kernel, the
fractional-timestep embedding and the sharded form.

The oracle side is tests/oracle_dpm.py (upstream DPMSolverSampler / NoiseScheduleVP / model_wrapper / DPMSolver restated).
CPU: known answers (eps == 0, S = 2 as two DDIM steps, a perfect denoiser), the model times / CFG batching / RNG upstream's
loop implies, guards, the frozen fixture tests/golden/dpm_v1.npz, the B200 sampler against the oracle over the reduced
networks (C-ABI calls replaced by the torch fakes of tests/fake_ops.py, tests/fake_plms_ops.py and tests/fake_dpm_ops.py),
the fractional keys of the embedding table, 2-rank gloo sample_dpm_sharded and log_results.
GPU (-m gpu): mkd_timestep_embedding_f32 against the int64 kernel and torch, mkd_dpm_update against upstream's torch
expressions on CUDA, the whole loop over the CUDA toy, reduced and yaml-size networks against the fp32 oracle, and the
2-GPU gather paths."""
import math
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

import fake_dpm_ops  # noqa: E402
from golden.make_golden_dpm import CASES, compute  # noqa: E402
from makeupdiffuse_b200 import B200ControlLDM, B200DDIMSampler, B200DPMSolverSampler, ops  # noqa: E402
from makeupdiffuse_b200.dist import shard_bounds  # noqa: E402
from oracle import MKDDIMSampler, OracleControlLDM, seeded_state_dict  # noqa: E402
from oracle_dpm import DPMSolverSampler, NoiseScheduleVP  # noqa: E402
from toy_denoiser import ToyDenoiser, toy_inputs  # noqa: E402

GOLDEN = os.path.join(HERE, "golden", "dpm_v1.npz")
GAIN_EPS_ZERO = 14.6425866  # sqrt(abar[0] / abar[999]) of the fp32-stored yaml schedule


@pytest.fixture()
def faked(monkeypatch):
    fake_dpm_ops.install(ops, monkeypatch.setattr)


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


def run(s, S, i, cond, **kw):
    return s.sample(S, i["x_T"].shape[0], tuple(i["x_T"].shape[1:]), cond, x_T=i["x_T"], verbose=False, **kw)


def model_times(S, N=1000):
    """upstream's model input times of an S-step run: (linspace(1, 1/N, S + 1)[:-1] - 1/N) * 1000 in fp32"""
    return ((torch.linspace(1., 1. / N, S + 1)[:-1] - 1. / N) * 1000.).tolist()


class Recording(ToyDenoiser):
    """the toy denoiser that also keeps the timesteps (with their dtype) and the cond rows of every call"""

    def __init__(self, device="cpu"):
        super().__init__(device)
        self.ts, self.dtypes, self.conds = [], [], []

    def apply_model(self, x, t, c):
        self.ts.append(t.tolist())
        self.dtypes.append(t.dtype)
        self.conds.append(self._leaves(c)[0].clone())
        return super().apply_model(x, t, c)


# ---- CPU: oracle and B200 sampler host logic --------------------------------------------------------------------------
def test_eps_zero_gain_is_the_schedule_ratio():
    ac = ToyDenoiser().alphas_cumprod.double()
    assert abs(float((ac[0] / ac[999]).sqrt()) - GAIN_EPS_ZERO) < 1e-6


@pytest.mark.parametrize("S", [2, 14, 15, 20])
def test_kat_eps_zero(faked, S):
    """eps == 0: every data prediction is x / alpha, D1 = 0, and the steps telescope to x_T * alpha(t_0) / alpha(1)"""
    m = ToyDenoiser()
    m.apply_model = lambda x, t, c: torch.zeros_like(x)
    i = toy_inputs()
    cond, _ = toy_cond(i)  # upstream's model_wrapper passes the cond as a third argument only when there is one
    for s in (DPMSolverSampler(m), B200DPMSolverSampler(m)):
        x, none = run(s, S, i, cond)
        assert none is None
        torch.testing.assert_close(x, i["x_T"] * GAIN_EPS_ZERO, rtol=4e-6, atol=0)


def _marginals(t):
    """alpha(t), sigma(t) of upstream's discrete schedule in float64 (the same piecewise-linear log alpha)"""
    ns = NoiseScheduleVP("discrete", alphas_cumprod=ToyDenoiser().alphas_cumprod.double())
    ns.t_array = ns.t_array.double()
    lmc = float(ns.marginal_log_mean_coeff(torch.tensor([t], dtype=torch.float64)))
    return math.exp(lmc), math.sqrt(1.0 - math.exp(2.0 * lmc))


@pytest.mark.parametrize("guide", [False, True])
def test_kat_two_steps_are_ddim_steps(faked, guide):
    """S = 2: both steps are order 1 (the first by construction, the last by lower_order_final), and DPM-Solver++ of order
    1 is DDIM (eta 0) on the interpolated alpha / sigma: x' = alpha_t * x0 + sigma_t * eps, x0 = (x - sigma_s eps) / alpha_s"""
    i = toy_inputs()
    cond, uc = toy_cond(i)
    m = ToyDenoiser()
    g = dict(unconditional_guidance_scale=4.0, unconditional_conditioning=uc) if guide else {}
    times = torch.linspace(1., 1. / 1000, 3).tolist()
    x = i["x_T"].double()
    for k in range(2):
        tau = torch.full((3,), model_times(2)[k])
        if guide:
            eu = m.apply_model(x.float(), tau, uc).double()
            e = eu + 4.0 * (m.apply_model(x.float(), tau, cond).double() - eu)
        else:
            e = m.apply_model(x.float(), tau, cond).double()
        (a_s, s_s), (a_t, s_t) = _marginals(times[k]), _marginals(times[k + 1])
        x = a_t * (x - s_s * e) / a_s + s_t * e
    for s in (DPMSolverSampler(m), B200DPMSolverSampler(m)):
        got = run(s, 2, i, cond, **g)[0]
        assert rel(got, x) < 1e-5, rel(got, x)


@pytest.mark.parametrize("S", [2, 10, 14, 15, 20])
def test_kat_perfect_denoiser(faked, S):
    """a model whose eps is exact for one fixed x0*: every data prediction is x0*, so each step keeps
    (x - alpha x0*) / sigma and the result is alpha_0 x0* + sigma_0 / sigma_T (x_T - alpha_T x0*)"""
    i = toy_inputs()
    x0 = torch.randn(i["x_T"].shape, generator=torch.Generator().manual_seed(9))
    m = ToyDenoiser()

    def eps(x, t, c):
        t_cont = float(t[0]) / 1000.0 + 1.0 / 1000  # the model input time back to continuous time
        a, s = _marginals(t_cont)
        return ((x.double() - a * x0.double()) / s).float()
    m.apply_model = eps
    (a0, s0), (aT, sT) = _marginals(1.0 / 1000), _marginals(1.0)
    want = a0 * x0.double() + s0 / sT * (i["x_T"].double() - aT * x0.double())
    cond, _ = toy_cond(i)
    for s in (DPMSolverSampler(m), B200DPMSolverSampler(m)):
        got = run(s, S, i, cond)[0]
        assert rel(got, want) < 1e-5, (S, rel(got, want))


@pytest.mark.parametrize("S", [20, 14, 2])
def test_model_times_rng_and_cfg_batching(faked, S):
    """the model sees S calls at upstream's fractional model times (never t = 0), as fp32; doubled [uncond; cond] under
    guidance, un-doubled at scale 1; no random numbers are drawn when x_T is given"""
    i = toy_inputs()
    want = model_times(S)
    assert want[0] == 999.0 and all(v > 0 for v in want)
    if S == 20:
        assert abs(want[1] - 949.05) < 1e-3 and abs(want[-1] - 49.95) < 1e-3 and want[1] != int(want[1])
    for kind in ("dict", "list", "tensor"):
        cond, uc = toy_cond(i, kind)
        for make in (DPMSolverSampler, B200DPMSolverSampler):
            m = Recording()
            s = make(m)
            torch.manual_seed(7)
            before = torch.get_rng_state()
            run(s, S, i, cond)
            assert torch.equal(before, torch.get_rng_state())
            assert m.ts == [[v] * 3 for v in want] and m.calls == [3] * S
            assert set(m.dtypes) == {torch.float32}
            for rec in (m.ts, m.calls, m.conds):
                rec.clear()
            run(s, S, i, cond, unconditional_guidance_scale=3.0, unconditional_conditioning=uc)
            assert m.ts == [[v] * 6 for v in want] and m.calls == [6] * S
            lead = lambda c: ToyDenoiser._leaves(c)[0]  # noqa: E731
            assert all(torch.equal(c, torch.cat([lead(uc), lead(cond)])) for c in m.conds)   # [uncond; cond]
            m.calls.clear()
            run(s, S, i, cond, unconditional_guidance_scale=1.0, unconditional_conditioning=uc)
            assert m.calls == [3] * S                                        # scale 1: uc is ignored, no doubling


def test_guards(faked, capsys):
    i = toy_inputs()
    cond, _ = toy_cond(i)
    m = ToyDenoiser()
    for s in (DPMSolverSampler(m), B200DPMSolverSampler(m)):
        with pytest.raises(AssertionError):
            run(s, 1, i, cond)                                 # upstream's assert steps >= order
    v = ToyDenoiser()
    v.parameterization = "v"
    with pytest.raises(NotImplementedError):
        run(B200DPMSolverSampler(v), 10, i, cond)
    # ignored as upstream ignores them; the batch-size check reads this model's dict-of-lists cond and only warns
    base = run(B200DPMSolverSampler(m), 4, i, cond)[0]
    got = run(B200DPMSolverSampler(m), 4, i, cond, eta=0.5, mask=torch.zeros(1), callback=lambda k: 1 / 0,
              img_callback=lambda *a: 1 / 0, temperature=0.1, noise_dropout=0.5, log_every_t=1)[0]
    assert torch.equal(base, got)
    capsys.readouterr()
    m.apply_model = lambda x, t, c: torch.zeros_like(x)
    B200DPMSolverSampler(m).sample(4, 2, (4, 8, 8), cond, x_T=i["x_T"][:2], verbose=False)
    assert "Got 3 conditionings but batch-size is 2" in capsys.readouterr().out


@pytest.mark.parametrize("kind", ["dict", "list", "tensor"])
def test_b200_equals_oracle_on_the_toy_bitwise(faked, kind):
    i = toy_inputs()
    cond, uc = toy_cond(i, kind)
    m = ToyDenoiser()
    for S in (20, 15, 14, 10, 3, 2):
        for g in ({}, dict(unconditional_guidance_scale=7.5, unconditional_conditioning=uc)):
            a = run(DPMSolverSampler(m), S, i, cond, **g)[0]
            b = run(B200DPMSolverSampler(m), S, i, cond, **g)[0]
            assert torch.equal(a, b), (S, g.keys())


def test_oracle_and_b200_reproduce_the_frozen_fixture(faked):
    G = np.load(GOLDEN)
    assert sorted(G.files) == sorted(n for n, _, _ in CASES)
    m = ToyDenoiser()
    for make in (lambda: DPMSolverSampler(m), lambda: B200DPMSolverSampler(m)):
        got = compute(make)
        for k in G.files:
            assert np.array_equal(got[k].numpy(), G[k]), k


def test_embedding_table_holds_fractional_times(faked, tiny_params):
    """the per-loop table keys fractional model times by their fp32 value; integer timesteps select the rows they select
    today (an int and the float of the same integer are one key)"""
    o = OracleControlLDM(control_params=tiny_params, unet_params=tiny_params).eval()
    m = B200ControlLDM(tiny_params, tiny_params, dtype=torch.float32, device="cpu").load_state_dict(seeded_state_dict(o, 0))
    times = model_times(20)
    m.precompute_time_embeddings(times)
    tab = m._emb_table
    assert tab["tab"].shape[0] == 20 and tab["vals"] == tuple(times)
    assert m.set_step(times[1], 2) and not m.set_step(int(times[1]), 2)      # 949.05 is not truncated to 949
    assert m.set_step(np.float32(times[3]), 2) and m.set_step(999, 2)          # 999 == 999.0
    un = m.model.diffusion_model
    rows = un._time_embedding(torch.tensor(times), 20).clone()                # the same 20 rows, computed directly
    m.set_step(times[1], 2)
    assert torch.equal(m._emb_bufs[2][0], rows[1]) and torch.equal(m._emb_bufs[2][1], rows[1])
    m.precompute_time_embeddings(np.flip(np.arange(1, 1000, 50)))            # a DDIM loop: int keys, the int64 path
    assert all(isinstance(v, int) for v in m._emb_table["vals"]) and m.set_step(951, 2) and not m.set_step(950.5, 2)
    m.set_step(None)


def test_b200_equals_oracle_on_reduced_networks(faked, tiny_params):
    """B200DPMSolverSampler over B200ControlLDM (C-ABI faked) against the oracle sampler over the oracle networks; the
    model sees fractional times, and the int64 embedding stand-in refuses them, so a layer that still truncated t, or sent
    a float t down the int64 path, fails here"""
    o = OracleControlLDM(control_params=tiny_params, unet_params=tiny_params).eval()
    sd = seeded_state_dict(o, 0)
    m = B200ControlLDM(tiny_params, tiny_params, dtype=torch.float32, device="cpu").load_state_dict(sd)
    g = torch.Generator().manual_seed(3)
    cond = {"c_crossattn": [torch.randn(2, 77, 64, generator=g)], "c_concat": [torch.rand(2, 6, 64, 64, generator=g)]}
    uc = {"c_crossattn": [torch.randn(2, 77, 64, generator=g)], "c_concat": cond["c_concat"]}
    x_T = torch.randn(2, 4, 8, 8, generator=g)
    for guide in ({}, dict(unconditional_guidance_scale=4.0, unconditional_conditioning=uc)):
        with torch.no_grad():
            b, _ = B200DPMSolverSampler(m).sample(5, 2, (4, 8, 8), cond, x_T=x_T, verbose=False, **guide)
            r, _ = DPMSolverSampler(o).sample(5, 2, (4, 8, 8), cond, x_T=x_T, verbose=False, **guide)
        assert rel(b, r) < 1e-5, rel(b, r)
    # one evaluation at a fractional time against the same network fed the truncated time: the embeddings differ enough
    # that the comparison above would see a truncation
    t = torch.full((2,), model_times(5)[1])
    with torch.no_grad():
        e_frac = m.apply_model(x_T, t, cond)
        e_trunc = o.apply_model(x_T, t.long().float(), cond)
        e_ref = o.apply_model(x_T, t, cond)
    assert rel(e_frac, e_ref) < 1e-5 < 100 * rel(e_trunc, e_ref), (rel(e_frac, e_ref), rel(e_trunc, e_ref))


def test_log_results_runs_with_the_dpm_sampler(faked):
    """harness.log_results(..., sampler=B200DPMSolverSampler(model)) unchanged: its sample panels are DPM-Solver samples
    (S evaluations per run at fractional times, doubled under guidance) and differ from the DDIM panels of the same seeds"""
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
    m.apply_model = lambda x, t, c, *a, **k: (calls.append((int(x.shape[0]), t.dtype)), orig(x, t, c, *a, **k))[1]
    logs = {}
    for name, make in (("dpm", B200DPMSolverSampler), ("ddim", B200DDIMSampler)):
        calls.clear()
        torch.manual_seed(0)
        logs[name] = harness.log_results(m, batch, 0, ddim_steps=S, unconditional_guidance_scale=9.0, sampler=make(m),
                                         generator=torch.Generator().manual_seed(11))
        dt = torch.float32 if name == "dpm" else torch.int64
        assert calls == [(B, torch.int64)] + [(B, dt)] * S + [(2 * B, dt)] * S, (name, calls)
    a, b = logs["dpm"], logs["ddim"]
    assert list(a) == list(b) and "samples_cfg_scale_9.00" in a
    for k in a:
        assert a[k].shape == b[k].shape and bool(torch.isfinite(a[k]).all())
    assert torch.equal(a["reconstruction"], b["reconstruction"]) and not torch.equal(a["samples"], b["samples"])


# ---- CPU: 2-rank gloo sample_dpm_sharded ------------------------------------------------------------------------------
PARAMS = dict(model_channels=32, num_heads=2, context_dim=32)
BG, H, STEPS = 4, 8, 5


def _setup(patch=setattr):
    """patch: plain setattr in a spawned worker; monkeypatch.setattr in the pytest process"""
    from makeupdiffuse_b200.synth import synthetic_state_dict
    fake_dpm_ops.install(ops, patch)
    m = B200ControlLDM(PARAMS, PARAMS, dtype=torch.float32, device="cpu")
    m.load_state_dict(synthetic_state_dict(m, 0, device="cpu"))
    return B200DPMSolverSampler(m)


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
    from makeupdiffuse_b200.dist import sample_dpm_sharded
    s = _setup()
    d = _data()
    lo, hi = shard_bounds(BG, rank, world)
    cond = {"c_crossattn": [d["ctx"][lo:hi]], "c_concat": [d["hint"][lo:hi]]}
    x_T = d["x_T"][lo:hi].contiguous()
    res = {"plain": sample_dpm_sharded(s, STEPS, BG, (4, H, H), cond, x_T, rank, world),
           "cfg": sample_dpm_sharded(s, STEPS, BG, (4, H, H), cond, x_T, rank, world, **_guide(d, lo, hi))}
    torch.save(res, os.path.join(out_dir, f"r{rank}.pt"))
    dist.destroy_process_group()


def test_two_rank_gloo_sample_dpm_sharded_equals_single_process(tmp_path, monkeypatch):
    import torch.multiprocessing as mp
    port = 35500 + os.getpid() % 2000
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
    from makeupdiffuse_b200.dist import sample_dpm_sharded
    assert torch.equal(sample_dpm_sharded(s, STEPS, BG, (4, H, H), cond, d["x_T"]), ref["plain"])


# ---- GPU ----------------------------------------------------------------------------------------------------------------
DEV = "cuda"


def _no_tf32():
    # the oracle must be TRUE fp32 on the GPU: cuDNN convolutions default to TF32 otherwise
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


@pytest.mark.gpu
@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float32])
def test_timestep_embedding_f32_kernel(dt):
    """integer t: the same bits as the int64 kernel for every t in [0, 999]; fractional t: upstream's torch expression
    within the bound of the int64 kernel's test"""
    ti = torch.arange(1000, device=DEV)
    a, b = torch.empty(1000, 320, device=DEV, dtype=dt), torch.empty(1000, 320, device=DEV, dtype=dt)
    ops.timestep_embedding(ti, a)
    ops.timestep_embedding_f32(ti.float(), b)
    assert torch.equal(a, b)
    tf = torch.tensor(model_times(20) + [0.5, 12.25, 998.75], device=DEV)
    out = torch.empty(tf.shape[0], 320, device=DEV, dtype=dt)
    ops.timestep_embedding_f32(tf, out)
    freqs = torch.exp(-math.log(10000.0) * torch.arange(160, dtype=torch.float32, device=DEV) / 160)
    args = tf[:, None].float() * freqs[None]
    ref = torch.cat([torch.cos(args), torch.sin(args)], -1)
    assert float((out.float() - ref).abs().max()) < (1e-2 if dt == torch.bfloat16 else 2e-4)
    trunc = torch.empty_like(out)
    ops.timestep_embedding(tf.long(), trunc)
    assert float((trunc.float() - ref).abs().max()) > 0.1  # what a truncating path would have produced


def _upstream_update(x, eps, cfg, m_prev, order, ns, s, t, t_prev):
    """upstream's torch expressions after one model call, evaluated on CUDA on [B]-sized time vectors: model_wrapper's CFG
    combine, data_prediction_fn at s, and the order-1 / order-2 multistep update from s to t"""
    dims = x.dim()
    ex = lambda v: v[(...,) + (None,) * (dims - 1)]  # noqa: E731
    if cfg is None:
        e = eps
    else:
        noise_uncond, noise = eps.chunk(2)
        e = noise_uncond + cfg * (noise - noise_uncond)
    m = (x - ex(ns.marginal_std(s)) * e) / ex(ns.marginal_alpha(s))
    lambda_s, lambda_t = ns.marginal_lambda(s), ns.marginal_lambda(t)
    h = lambda_t - lambda_s
    sigma_s, sigma_t = ns.marginal_std(s), ns.marginal_std(t)
    alpha_t = torch.exp(ns.marginal_log_mean_coeff(t))
    if order == 1:
        return ex(sigma_t / sigma_s) * x - ex(alpha_t * torch.expm1(-h)) * m, m
    h_0 = lambda_s - ns.marginal_lambda(t_prev)
    r0 = h_0 / h
    D1_0 = ex(1. / r0) * (m - m_prev)
    x_t = (ex(sigma_t / sigma_s) * x - ex(alpha_t * (torch.exp(-h) - 1.)) * m
           - 0.5 * ex(alpha_t * (torch.exp(-h) - 1.)) * D1_0)
    return x_t, m


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 65539])
def test_dpm_update_bitexact_against_upstream_torch_on_cuda(n):
    """both orders, CFG on and off, every step of S = 20 and 14: x_prev and the stored data prediction against upstream's
    literal expressions on CUDA fp32 tensors, with the scalars the sampler computes for its loop; the in-place form
    (x_prev is x); and the peers entry (one and two destinations) against the local one"""
    m = ToyDenoiser(DEV)
    ns = NoiseScheduleVP("discrete", alphas_cumprod=m.alphas_cumprod)
    g = torch.Generator(device=DEV).manual_seed(n)
    B = 1  # one batch row of n values: upstream's time vectors have one entry per row
    r = lambda k=1: torch.randn((k, n, 1, 1), device=DEV, generator=g)  # noqa: E731
    checked = set()
    for S in (20, 14):
        s = B200DPMSolverSampler(m)
        _, steps = s._loop_scalars(S)
        times = torch.linspace(1., 1. / 1000, S + 1).to(DEV)
        for k, st in enumerate(steps):
            vt = lambda j: times[j].expand(B)  # noqa: E731
            for cfg in (None, 7.5):
                x, eps, mp = r() * 3, r(1 if cfg is None else 2), r()
                order = st["order"]
                ref_x, ref_m = _upstream_update(x, eps, cfg, mp, order, ns, vt(k), vt(k + 1), vt(max(k - 1, 0)))
                out, ms = torch.empty_like(x), torch.empty_like(x)
                prev = mp if order == 2 else None
                ops.dpm_update(x, eps, out, m_store=ms, m_prev=prev, cfg_scale=cfg, **st)
                what = (S, k, order, cfg)
                assert torch.equal(out, ref_x), (what, float((out - ref_x).abs().max()))
                assert torch.equal(ms, ref_m), what
                xi = x.clone()
                ops.dpm_update(xi, eps, xi, m_prev=prev, cfg_scale=cfg, **st)
                assert torch.equal(xi, ref_x), ("in place", what)
                o1, o2 = torch.empty_like(x), torch.empty_like(x)
                ops.dpm_update(x, eps, o1, m_prev=prev, cfg_scale=cfg, peer_ptrs=[o1.data_ptr()], **st)
                assert torch.equal(o1, ref_x), ("peers", what)
                o1.zero_()
                ops.dpm_update(x, eps, o1, m_store=ms, m_prev=prev, cfg_scale=cfg,
                               peer_ptrs=[o1.data_ptr(), o2.data_ptr()], **st)
                assert torch.equal(o1, ref_x) and torch.equal(o2, ref_x) and torch.equal(ms, ref_m), ("2 peers", what)
                checked.add((order, cfg))
    assert checked == {(1, None), (1, 7.5), (2, None), (2, 7.5)}
    with pytest.raises(ValueError):
        ops.dpm_update(x, eps, out, order=2, **{k: v for k, v in steps[1].items() if k != "order"})


@pytest.mark.gpu
def test_b200_equals_oracle_on_the_toy_on_cuda():
    """the whole loop over the CUDA toy denoiser: B200DPMSolverSampler (the kernel, scalars evaluated on the device) against
    the oracle (upstream's torch on CUDA), bit for bit, with and without guidance"""
    i = toy_inputs(DEV)
    cond, uc = toy_cond(i)
    m = ToyDenoiser(DEV)
    for S in (20, 14, 15, 2):
        for guide in ({}, dict(unconditional_guidance_scale=7.5, unconditional_conditioning=uc)):
            a = run(DPMSolverSampler(m), S, i, cond, **guide)[0]
            b = run(B200DPMSolverSampler(m), S, i, cond, **guide)[0]
            assert torch.equal(a, b), (S, guide.keys(), float((a - b).abs().max()))


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
        ref, _ = DPMSolverSampler(tiny.oracle).sample(S, B, (4, h, h), cond, x_T=x_T, verbose=False, **guide)

    def go(m, graph):
        return B200DPMSolverSampler(m, use_cuda_graph=graph).sample(S, B, (4, h, h), cond, x_T=x_T, verbose=False,
                                                                    **guide)[0]

    a, g = go(tiny.f32, False), go(tiny.f32, True)
    b, bg = go(tiny.bf16, False), go(tiny.bf16, True)
    assert torch.equal(a, g) and torch.equal(b, bg)                    # graph replay == eager
    r32, r16 = rel(a, ref), rel(b, ref)
    print(f"DPM-{S} free-running final latents rel-L2 vs oracle (reduced nets, CFG {cfg_scale:g}): fp32-check {r32:.2e}, "
          f"bf16 {r16:.2e}")
    assert r32 < 1e-4 and r16 < 5e-2, (r32, r16)
    # one sampler reused, after a DDIM loop on the same model (int64 graph and table): reproduces a fresh sampler
    B200DDIMSampler(tiny.bf16).sample(4, B, (4, h, h), cond, x_T=x_T, verbose=False)
    s = B200DPMSolverSampler(tiny.bf16)
    s.sample(4, B, (4, h, h), cond, x_T=x_T, verbose=False)
    assert torch.equal(s.sample(S, B, (4, h, h), cond, x_T=x_T, verbose=False, **guide)[0], bg)


@pytest.mark.gpu
def test_full_size_batch16_teacher_forced_all_20_dpm_evaluations():
    """yaml networks, batch 16, 256^2, bf16 (the benchmarked configuration): every one of DPM-20's 20 evaluations at
    fractional model times, teacher-forced against the fp32 oracle (TF32 off) through the sampler's own per-step call
    (embedding table, graph)"""
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    _no_tf32()
    full = Bundle({}, f32=False)
    S, B, h = 20, 16, 32
    cond, _, x_T = make_cond(B, h, 768, seed=3)
    so = DPMSolverSampler(full.oracle)
    rec = []
    orig = full.oracle.apply_model
    full.oracle.apply_model = lambda x, t, c: (lambda e: (rec.append((x.clone(), t.clone(), e.clone())), e)[1])(orig(x, t, c))
    try:
        so.sample(S, B, (4, h, h), cond, x_T=x_T, verbose=False)
    finally:
        full.oracle.apply_model = orig
    assert len(rec) == S and all(t.dtype == torch.float32 for _, t, _ in rec)
    assert sum(float(t[0]) != int(float(t[0])) for _, t, _ in rec) == S - 1   # all but t = 999 are fractional
    s = B200DPMSolverSampler(full.bf16, use_cuda_graph=True)
    s.begin_loop(model_times(S))
    r = [rel(s._eps(x, t, cond, t_value=float(t[0])), e) for x, t, e in rec]
    print("full-size batch-16 DPM-20 teacher-forced 20 evaluations: eps rel-L2 bf16 max %.2e (evaluation %d) mean %.2e"
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
    from makeupdiffuse_b200.dist import sample_dpm_sharded
    from makeupdiffuse_b200.synth import synthetic_state_dict
    params = dict(model_channels=64, num_heads=4, context_dim=64)
    m = B200ControlLDM(params, params, dtype=torch.bfloat16, device=dev)
    m.load_state_dict(synthetic_state_dict(m, 0, dev))
    s = B200DPMSolverSampler(m)
    g = torch.Generator(device=dev).manual_seed(7)
    bg, h = 4, 16
    ctx = torch.randn(bg, 77, 64, device=dev, generator=g)
    hint = torch.rand(bg, 6, 8 * h, 8 * h, device=dev, generator=g)
    x_T = torch.randn(bg, 4, h, h, device=dev, generator=g)
    lo, hi = shard_bounds(bg, rank, world)
    cond = {"c_crossattn": [ctx[lo:hi].contiguous()], "c_concat": [hint[lo:hi].contiguous()]}
    res = {}
    for name, fused in (("nccl", False), ("fused", True), ("fused_again", True)):
        res[name] = sample_dpm_sharded(s, 10, bg, (4, h, h), cond, x_T[lo:hi].contiguous(), rank, world,
                                       fused_gather=fused).cpu()
    res["single"] = s.sample(10, bg, (4, h, h), {"c_crossattn": [ctx], "c_concat": [hint]}, x_T=x_T, verbose=False)[0].cpu()
    torch.save(res, os.path.join(out_dir, f"g{rank}.pt"))
    dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs of one box")
def test_two_gpu_sample_dpm_sharded_fused_gather_equals_nccl(tmp_path):
    import torch.multiprocessing as mp
    port = 35700 + os.getpid() % 2000
    mp.spawn(_gpu_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = torch.load(tmp_path / "g0.pt"), torch.load(tmp_path / "g1.pt")
    for r in (r0, r1):
        assert torch.equal(r["nccl"], r["fused"]) and torch.equal(r["fused"], r["fused_again"])
    assert torch.equal(r0["fused"], r1["fused"])
    # a rank's kernels see another batch size than the single-process run (tile / split-K choices differ): numerical
    assert float((r0["fused"] - r0["single"]).abs().max()) < 0.05 * float(r0["single"].abs().max())
