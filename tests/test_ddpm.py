"""DDPM ancestral sampling (upstream LatentDiffusion.sample / p_sample_loop / progressive_denoising / p_sample) — oracle
restatement, B200DDPMSampler, the model's methods, its update kernel and the sharded form.

The oracle side is tests/oracle_ddpm.py.  CPU: known answers (eps == 0, a perfect denoiser, the clamp), upstream's loop
semantics (timesteps, RNG stream, mask blend, callbacks, intermediates, start_T, cond slicing, per-step temperature),
guards, the frozen fixture tests/golden/ddpm_v1.npz, the B200 sampler against the oracle over the toy and the reduced
networks (C-ABI calls replaced by the torch fakes of tests/fake_ddpm_ops.py and the modules it installs), and 2-rank gloo
sample_ddpm_sharded.  GPU (-m gpu): mkd_ddpm_update against upstream's torch expressions on CUDA, the whole loop over the
CUDA toy, reduced and yaml-size networks against the fp32 oracle, and the 2-GPU gather paths."""
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

import fake_ddpm_ops  # noqa: E402
from golden.make_golden_ddpm import CASES, compute, toy_mask  # noqa: E402
from makeupdiffuse_b200 import B200ControlLDM, B200DDPMSampler, ops  # noqa: E402
from makeupdiffuse_b200.dist import shard_bounds  # noqa: E402
from oracle import OracleControlLDM, seeded_state_dict  # noqa: E402
from oracle_ddpm import DDPM  # noqa: E402
from toy_denoiser import ToyDenoiser, toy_inputs  # noqa: E402

GOLDEN = os.path.join(HERE, "golden", "ddpm_v1.npz")
BUFFERS = ("betas", "alphas_cumprod", "alphas_cumprod_prev", "sqrt_alphas_cumprod", "sqrt_one_minus_alphas_cumprod",
           "sqrt_recip_alphas_cumprod", "sqrt_recipm1_alphas_cumprod", "posterior_variance",
           "posterior_log_variance_clipped", "posterior_mean_coef1", "posterior_mean_coef2")


@pytest.fixture()
def faked(monkeypatch):
    fake_ddpm_ops.install(ops, monkeypatch.setattr)


def rel(a, b):
    a, b = torch.as_tensor(a).float().cpu(), torch.as_tensor(b).float().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-20))


def toy_cond(i):
    return {"c_crossattn": [i["ctx"]], "c_concat": [i["hint"]]}


def pair(model=None, device="cpu", **kw):
    """(oracle, B200 sampler) over the same toy-backed DDPM object: the B200 sampler reads its buffers and attributes"""
    d = DDPM(model or ToyDenoiser(device), **kw)
    return d, B200DDPMSampler(d)


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


# ---- CPU: known answers -------------------------------------------------------------------------------------------------
def test_posterior_buffers_match_the_oracle_and_upstream_identities():
    """the model's buffers are the oracle's register_schedule bit for bit; coef1[0] = 1 and coef2[0] = 0 (so the last
    step returns x_recon), and the posterior variance of t = 0 is clipped"""
    m = B200ControlLDM(dict(model_channels=32, num_heads=2, context_dim=32), dict(model_channels=32, num_heads=2, context_dim=32),
                       dtype=torch.float32, device="cpu")
    d = DDPM(ToyDenoiser())
    for name in BUFFERS:
        assert torch.equal(getattr(m, name), getattr(d, name)), name
    assert float(m.posterior_mean_coef1[0]) == pytest.approx(1.0, abs=1e-6) and float(m.posterior_mean_coef2[0]) == 0.0
    assert float(m.posterior_variance[0]) == 0.0 and float(m.posterior_log_variance_clipped[0]) == pytest.approx(-46.0517, abs=1e-3)
    assert (m.clip_denoised, m.log_every_t, m.channels, m.image_size) == (True, 100, 4, 32)


@pytest.mark.parametrize("start_T", [1000, 250])
def test_kat_eps_zero(faked, start_T):
    """eps == 0, no clip, temperature 0: each step multiplies x by (coef1 * sqrt_recip_ac + coef2)[t]"""
    i = toy_inputs()
    m = ToyDenoiser()
    m.apply_model = lambda x, t, c: torch.zeros_like(x)
    d = DDPM(ToyDenoiser())
    gain = np.prod([(float(d.posterior_mean_coef1[t]) * float(d.sqrt_recip_alphas_cumprod[t]) + float(d.posterior_mean_coef2[t]))
                    for t in range(start_T)])
    for s in pair(m, clip_denoised=False):
        x, inter = s.progressive_denoising(toy_cond(i), tuple(i["x_T"].shape), x_T=i["x_T"], verbose=False, temperature=0.,
                                           start_T=start_T)
        assert rel(x, i["x_T"].double() * gain) < 2e-5, rel(x, i["x_T"].double() * gain)


def _perfect(x0):
    """eps exact for one fixed x0: x_recon = x0 whatever x"""
    d = DDPM(ToyDenoiser())

    def eps(x, t, c):
        ex = lambda a: a[t].reshape(-1, 1, 1, 1).double()  # noqa: E731
        return ((x.double() - ex(d.sqrt_alphas_cumprod) * x0.double()) / ex(d.sqrt_one_minus_alphas_cumprod)).float()
    m = ToyDenoiser()
    m.apply_model = eps
    return m


@pytest.mark.parametrize("clip", [True, False])
def test_kat_perfect_denoiser(faked, clip):
    """|x0*| < 1, temperature 0: the loop returns x0* (coef1[0] = 1, coef2[0] = 0), clamp or not"""
    i = toy_inputs()
    x0 = 0.9 * torch.tanh(torch.randn(i["x_T"].shape, generator=torch.Generator().manual_seed(9)))
    for s in pair(_perfect(x0), clip_denoised=clip):
        got, _ = s.progressive_denoising(toy_cond(i), tuple(x0.shape), x_T=i["x_T"], verbose=False, temperature=0.)
        assert rel(got, x0) < 1e-5, rel(got, x0)


def test_kat_clip(faked):
    """a denoiser whose x_recon leaves [-1, 1]: with clip on the loop returns the clamped x0*, off x0* itself"""
    i = toy_inputs()
    x0 = 2.5 * torch.randn(i["x_T"].shape, generator=torch.Generator().manual_seed(4))
    assert float(x0.abs().max()) > 2
    for clip, want in ((True, x0.clamp(-1, 1)), (False, x0)):
        for s in pair(_perfect(x0), clip_denoised=clip):
            got, _ = s.progressive_denoising(toy_cond(i), tuple(x0.shape), x_T=i["x_T"], verbose=False, temperature=0.)
            assert rel(got, want) < 1e-5, (clip, rel(got, want))
    # one step, rows at different t: x_recon is clamped before the posterior mean
    d, s = pair(_perfect(x0))
    t = torch.tensor([999, 0, 400])
    x = i["x_T"]
    torch.manual_seed(0)
    xp, xr = s.p_sample(x, toy_cond(i), t, clip_denoised=True, return_x0=True, temperature=0.)
    assert rel(xr, x0.clamp(-1, 1)) < 1e-5
    mean, _, _ = d.q_posterior(xr, x, t)
    assert torch.equal(xp, mean)


# ---- CPU: upstream's loop semantics -------------------------------------------------------------------------------------
@pytest.mark.parametrize("kw,T", [({}, 1000), ({"start_T": 30}, 30), ({"timesteps": 20}, 20),
                                  ({"timesteps": 20, "start_T": 30}, 20), ({"timesteps": 40, "start_T": 7}, 7)])
def test_timesteps_rng_and_callbacks(faked, kw, T):
    """the model sees int64 t = T-1 ... 0 over the batch (no doubling); one randn(x.shape) per step, t = 0 included;
    callback(i) and img_callback(img, i) receive the timestep"""
    i = toy_inputs()
    for make in (lambda m: DDPM(m), lambda m: B200DDPMSampler(DDPM(m))):
        m = Recording()
        s = make(m)
        cbs, imgs = [], []
        torch.manual_seed(5)
        x = s.p_sample_loop(toy_cond(i), tuple(i["x_T"].shape), x_T=i["x_T"], verbose=False, callback=cbs.append,
                            img_callback=lambda img, t: imgs.append((img, t)), **kw)
        after = torch.get_rng_state()
        torch.manual_seed(5)
        for _ in range(T):
            torch.randn(i["x_T"].shape)
        assert torch.equal(after, torch.get_rng_state())
        assert m.ts == [[t] * 3 for t in reversed(range(T))] and set(m.dtypes) == {torch.int64} and m.calls == [3] * T
        assert cbs == list(reversed(range(T))) and [t for _, t in imgs] == cbs and imgs[-1][0] is x


def test_mask_blend_follows_the_step_with_its_own_draw(faked):
    """mask == 1: the result is q_sample(x0, 0) with the LAST of 2T draws (step noise, then the blend's noise, per step)"""
    i = toy_inputs()
    x0 = 0.5 * torch.tanh(i["x_T"])
    T = 6
    for s in pair():
        torch.manual_seed(3)
        got = s.p_sample_loop(toy_cond(i), tuple(x0.shape), x_T=i["x_T"], verbose=False, start_T=T,
                              mask=torch.ones_like(x0[:, :1]), x0=x0)
        torch.manual_seed(3)
        draws = [torch.randn(x0.shape) for _ in range(2 * T)]
        d = DDPM(ToyDenoiser())
        assert torch.equal(got, d.q_sample(x0, torch.zeros(3, dtype=torch.long), noise=draws[-1]))
    with pytest.raises(AssertionError):
        pair()[1].p_sample_loop(toy_cond(i), tuple(x0.shape), x_T=i["x_T"], verbose=False, start_T=2, mask=x0)  # no x0


def test_intermediates_follow_log_every_t(faked):
    """p_sample_loop logs the start and img at i % log_every_t == 0 or i == timesteps - 1; progressive_denoising logs
    x_recon at the same steps; B200 == oracle entry by entry"""
    i = toy_inputs()
    shape = tuple(i["x_T"].shape)
    res = []
    for s in pair():
        torch.manual_seed(8)
        a = s.p_sample_loop(toy_cond(i), shape, x_T=i["x_T"], verbose=False, start_T=250, return_intermediates=True)
        torch.manual_seed(8)
        b = s.p_sample_loop(toy_cond(i), shape, x_T=i["x_T"], verbose=False, start_T=25, return_intermediates=True,
                            log_every_t=10)
        torch.manual_seed(8)
        c = s.progressive_denoising(toy_cond(i), shape, x_T=i["x_T"], verbose=False, start_T=250)
        torch.manual_seed(8)
        n = s.p_sample_loop(toy_cond(i), shape, x_T=i["x_T"], verbose=False, start_T=250)
        res.append((a, b, c, n))
        assert len(a[1]) == 1 + 4 and a[1][0] is i["x_T"] and a[1][-1] is a[0]    # start, 249, 200, 100, 0
        assert len(b[1]) == 1 + 4 and len(c[1]) == 4                               # start, 24, 20, 10, 0; 249, 200, 100, 0
        assert torch.equal(n, a[0])
    (a, b, c, _), (a2, b2, c2, _) = res
    for u, v in zip(a[1] + b[1] + c[1] + [a[0], b[0], c[0]], a2[1] + b2[1] + c2[1] + [a2[0], b2[0], c2[0]]):
        assert torch.equal(u, v)


def test_sample_slices_cond_and_defaults_its_shape(faked):
    i = toy_inputs()
    cond = {"c_crossattn": [i["ctx"]], "c_concat": [i["hint"]]}
    for make in (lambda m: DDPM(m, image_size=8), lambda m: B200DDPMSampler(DDPM(m, image_size=8))):
        m = Recording()
        torch.manual_seed(2)
        x = make(m).sample(cond, batch_size=2, timesteps=3, verbose=False)
        assert x.shape == (2, 4, 8, 8) and m.calls == [2] * 3
        assert all(torch.equal(c, i["ctx"][:2]) for c in m.conds)
    d, s = pair()
    torch.manual_seed(2)
    a = d.sample(cond, batch_size=2, timesteps=3, verbose=False, shape=(2, 4, 8, 8), return_intermediates=True)
    torch.manual_seed(2)
    b = s.sample(cond, batch_size=2, timesteps=3, verbose=False, shape=(2, 4, 8, 8), return_intermediates=True)
    assert torch.equal(a[0], b[0]) and len(a[1]) == len(b[1]) == 3


def test_progressive_denoising_per_step_temperature(faked):
    """temperature as a list is indexed by the timestep; a float is expanded; batch_size prepends the batch dimension"""
    i = toy_inputs()
    T = 12
    temps = [0.1 * (k % 4) for k in range(T)]
    for s in pair():
        torch.manual_seed(6)
        a = s.progressive_denoising(toy_cond(i), (4, 8, 8), batch_size=3, x_T=i["x_T"], verbose=False, start_T=T,
                                    temperature=temps)
        torch.manual_seed(6)
        z = s.progressive_denoising(toy_cond(i), (4, 8, 8), batch_size=3, x_T=i["x_T"], verbose=False, start_T=T,
                                    temperature=[0.] * T)
        torch.manual_seed(6)
        f = s.progressive_denoising(toy_cond(i), (4, 8, 8), batch_size=3, x_T=i["x_T"], verbose=False, start_T=T,
                                    temperature=0.)
        assert torch.equal(z[0], f[0]) and not torch.equal(a[0], z[0])
    d, b = pair()
    torch.manual_seed(6)
    ra = d.progressive_denoising(toy_cond(i), (4, 8, 8), batch_size=3, x_T=i["x_T"], verbose=False, start_T=T,
                                 temperature=temps, noise_dropout=0.3)
    torch.manual_seed(6)
    rb = b.progressive_denoising(toy_cond(i), (4, 8, 8), batch_size=3, x_T=i["x_T"], verbose=False, start_T=T,
                                 temperature=temps, noise_dropout=0.3)
    assert torch.equal(ra[0], rb[0]) and all(torch.equal(u, v) for u, v in zip(ra[1], rb[1]))


def test_guards(faked):
    i = toy_inputs()
    d, s = pair()
    x, t = i["x_T"], torch.full((3,), 5)
    with pytest.raises(NotImplementedError):
        s.p_sample(x, toy_cond(i), t, quantize_denoised=True)
    with pytest.raises(NotImplementedError):
        s.p_sample(x, toy_cond(i), t, score_corrector=object())
    with pytest.raises(NotImplementedError):
        s.p_sample_loop(toy_cond(i), tuple(x.shape), x_T=x, start_T=2, quantize_denoised=True)
    v = ToyDenoiser()
    v.parameterization = "x0"
    with pytest.raises(NotImplementedError):
        B200DDPMSampler(DDPM(v)).p_sample(x, toy_cond(i), t)
    with pytest.raises(ValueError):
        s.p_sample_loop(toy_cond(i), tuple(x.shape), x_T=x, start_T=2, mask=torch.ones_like(x), x0=x, out=torch.empty_like(x))
    with pytest.raises(TypeError):
        s.progressive_denoising(toy_cond(i), tuple(x.shape), x_T=x, start_T=2, temperature=1)  # upstream expands floats only


# ---- CPU: the B200 sampler against the oracle, the frozen fixture ---------------------------------------------------------
def test_b200_equals_oracle_on_the_toy_bitwise(faked):
    """p_sample with mixed per-row t, return_x0, repeat_noise, temperature, noise_dropout; and whole loops"""
    i = toy_inputs()
    d, s = pair()
    t = torch.tensor([0, 999, 317])
    for kw in ({}, dict(clip_denoised=True), dict(return_x0=True, temperature=0.5), dict(repeat_noise=True),
               dict(noise_dropout=0.25, temperature=0.7, clip_denoised=True, return_x0=True)):
        torch.manual_seed(1)
        a = d.p_sample(i["x_T"], toy_cond(i), t, **kw)
        torch.manual_seed(1)
        b = s.p_sample(i["x_T"], toy_cond(i), t, **kw)
        for u, v in zip(a if isinstance(a, tuple) else (a,), b if isinstance(b, tuple) else (b,)):
            assert torch.equal(u, v), kw
    for clip in (True, False):
        d, s = pair(clip_denoised=clip)
        torch.manual_seed(4)
        a = d.p_sample_loop(toy_cond(i), tuple(i["x_T"].shape), verbose=False, start_T=300)  # x_T drawn too
        torch.manual_seed(4)
        b = s.p_sample_loop(toy_cond(i), tuple(i["x_T"].shape), verbose=False, start_T=300)
        assert torch.equal(a, b), clip


def test_oracle_and_b200_reproduce_the_frozen_fixture(faked):
    G = np.load(GOLDEN)
    assert sorted(G.files) == sorted(CASES)
    m = ToyDenoiser()
    for make in (lambda clip: DDPM(m, clip_denoised=clip), lambda clip: B200DDPMSampler(DDPM(m, clip_denoised=clip))):
        got = compute(make)
        for k in G.files:
            assert np.array_equal(got[k].numpy(), G[k]), k


def test_contrast_the_fixture_catches_a_missing_clamp_and_a_skipped_final_mask():
    """the bitwise gate above would see either mistake: an unclipped x_recon, or a loop that skips the blend at t = 0"""
    G = np.load(GOLDEN)
    m = ToyDenoiser()
    unclipped = compute(lambda clip: DDPM(m, clip_denoised=False))["full_clip"]
    assert rel(unclipped, torch.from_numpy(G["full_clip"])) > 1e-2
    i = toy_inputs()
    _, kw = CASES["mask_start_T_50"]
    mask, x0, d = toy_mask(i), 0.5 * torch.tanh(i["x_T"]), DDPM(m)
    outs = {}
    for skip in (False, True):
        torch.manual_seed(1234)
        img = i["x_T"]
        for k in reversed(range(kw["start_T"])):
            ts = torch.full((3,), k, dtype=torch.long)
            img = d.p_sample(img, toy_cond(i), ts, clip_denoised=True)
            if not (skip and k == 0):
                img = d.q_sample(x0, ts) * mask + (1. - mask) * img
        outs[skip] = img
    assert np.array_equal(outs[False].numpy(), G["mask_start_T_50"])
    assert not np.array_equal(outs[True].numpy(), G["mask_start_T_50"]) and rel(outs[True], outs[False]) > 1e-3


def test_b200_equals_oracle_on_reduced_networks(faked, tiny_params):
    """B200ControlLDM's own methods (buffers, q_posterior, p_mean_variance, and sample / p_sample_loop /
    progressive_denoising through its kept sampler) against the oracle over the oracle networks, on a shortened loop"""
    o = OracleControlLDM(control_params=tiny_params, unet_params=tiny_params).eval()
    m = B200ControlLDM(tiny_params, tiny_params, dtype=torch.float32, device="cpu").load_state_dict(seeded_state_dict(o, 0))
    d = DDPM(o)
    g = torch.Generator().manual_seed(3)
    cond = {"c_crossattn": [torch.randn(3, 77, 64, generator=g)], "c_concat": [torch.rand(3, 6, 64, 64, generator=g)]}
    x = torch.randn(2, 4, 8, 8, generator=g)
    t = torch.tensor([999, 0])
    c2 = {k: [v[0][:2]] for k, v in cond.items()}
    with torch.no_grad():
        for a, b in zip(m.p_mean_variance(x, c2, t, True, return_x0=True), d.p_mean_variance(x, c2, t, True, return_x0=True)):
            assert rel(a, b) < 1e-5
        torch.manual_seed(0)
        a = m.sample(cond, batch_size=2, shape=(2, 4, 8, 8), timesteps=4, verbose=False, x_T=x)
        torch.manual_seed(0)
        b = d.sample(cond, batch_size=2, shape=(2, 4, 8, 8), timesteps=4, verbose=False, x_T=x)
        assert rel(a, b) < 1e-5, rel(a, b)
        s = m._ddpm_sampler()
        torch.manual_seed(0)
        a = m.progressive_denoising(c2, (2, 4, 8, 8), x_T=x, start_T=3, verbose=False)[0]
        torch.manual_seed(0)
        b = d.progressive_denoising(c2, (2, 4, 8, 8), x_T=x, start_T=3, verbose=False)[0]
        assert rel(a, b) < 1e-5 and m._ddpm_sampler() is s
        torch.manual_seed(0)
        a = m.p_sample(x, c2, t, clip_denoised=True)
        torch.manual_seed(0)
        b = d.p_sample(x, c2, t, clip_denoised=True)
        assert rel(a, b) < 1e-5


# ---- CPU: 2-rank gloo sample_ddpm_sharded -------------------------------------------------------------------------------
PARAMS = dict(model_channels=32, num_heads=2, context_dim=32)
BG, H, START_T = 4, 8, 4


def _setup(patch=setattr):
    """patch: plain setattr in a spawned worker; monkeypatch.setattr in the pytest process"""
    from makeupdiffuse_b200.synth import synthetic_state_dict
    fake_ddpm_ops.install(ops, patch)
    m = B200ControlLDM(PARAMS, PARAMS, dtype=torch.float32, device="cpu")
    m.load_state_dict(synthetic_state_dict(m, 0, device="cpu"))
    return B200DDPMSampler(m)


def _data():
    g = torch.Generator().manual_seed(12)
    return {"ctx": torch.randn(BG, 77, 32, generator=g), "hint": torch.rand(BG, 6, 8 * H, 8 * H, generator=g),
            "x_T": torch.randn(BG, 4, H, H, generator=g)}


def _worker(rank, world, port, out_dir):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(2)
    from makeupdiffuse_b200.dist import sample_ddpm_sharded
    s = _setup()
    d = _data()
    lo, hi = shard_bounds(BG, rank, world)
    cond = {"c_crossattn": [d["ctx"][lo:hi]], "c_concat": [d["hint"][lo:hi]]}
    torch.manual_seed(21)  # every rank alike
    res = {"x_T": sample_ddpm_sharded(s, BG, (4, H, H), cond, d["x_T"][lo:hi].contiguous(), rank, world, start_T=START_T)}
    torch.manual_seed(21)
    res["drawn"] = sample_ddpm_sharded(s, BG, (4, H, H), cond, None, rank, world, start_T=START_T)
    torch.save(res, os.path.join(out_dir, f"r{rank}.pt"))
    dist.destroy_process_group()


def test_two_rank_gloo_sample_ddpm_sharded_equals_single_process(tmp_path, monkeypatch):
    import torch.multiprocessing as mp
    port = 36100 + os.getpid() % 2000
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = torch.load(tmp_path / "r0.pt"), torch.load(tmp_path / "r1.pt")
    s = _setup(monkeypatch.setattr)
    d = _data()
    cond = {"c_crossattn": [d["ctx"]], "c_concat": [d["hint"]]}
    torch.manual_seed(21)
    ref = {"x_T": s.p_sample_loop(cond, (BG, 4, H, H), x_T=d["x_T"], verbose=False, start_T=START_T)}
    torch.manual_seed(21)
    ref["drawn"] = s.p_sample_loop(cond, (BG, 4, H, H), verbose=False, start_T=START_T)
    for k in ("x_T", "drawn"):
        assert torch.equal(r0[k], r1[k]) and r0[k].shape == (BG, 4, H, H)
        assert float((r0[k] - ref[k]).abs().max()) < 1e-4 * float(ref[k].abs().max()), k
    from makeupdiffuse_b200.dist import sample_ddpm_sharded
    torch.manual_seed(21)
    assert torch.equal(sample_ddpm_sharded(s, BG, (4, H, H), cond, d["x_T"], start_T=START_T), ref["x_T"])


# ---- GPU ----------------------------------------------------------------------------------------------------------------
DEV = "cuda"


def _no_tf32():
    # the oracle must be TRUE fp32 on the GPU: cuDNN convolutions default to TF32 otherwise
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


def _upstream_step(d, x, eps, t, noise, clip, temperature):
    """upstream p_mean_variance after apply_model, and p_sample's return, on CUDA tensors"""
    x_recon = d.predict_start_from_noise(x, t=t, noise=eps)
    if clip:
        x_recon.clamp_(-1., 1.)
    mean, _, logvar = d.q_posterior(x_start=x_recon, x_t=x, t=t)
    noise = noise * temperature
    nonzero_mask = (1 - (t == 0).float()).reshape(x.shape[0], *((1,) * (len(x.shape) - 1)))
    return mean + nonzero_mask * (0.5 * logvar).exp() * noise, x_recon


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 65539])
def test_ddpm_update_bitexact_against_upstream_torch_on_cuda(n):
    """clip on / off, temperature 0 / 0.5 / 1, rows at t = 0, 999 and between, x0_out on / off, in place, 1 and 2 peer
    destinations: bit for bit against upstream's expressions on CUDA fp32 tensors"""
    d = DDPM(ToyDenoiser(DEV))
    tables = B200DDPMSampler(d)._tables()
    g = torch.Generator(device=DEV).manual_seed(n)
    t = torch.tensor([0, 999, 1, 500, 0, 250], device=DEV)
    r = lambda s=1.0: torch.randn((t.shape[0], n, 1, 1), device=DEV, generator=g) * s  # noqa: E731
    checked = 0
    for clip in (True, False):
        for temp in (0.0, 0.5, 1.0):
            x, eps, noise = r(3.0), r(), r()
            ref, ref0 = _upstream_step(d, x, eps, t, noise, clip, temp)
            out, x0 = torch.empty_like(x), torch.empty_like(x)
            ops.ddpm_update(x, eps, t, out, tables=tables, noise=noise, clip=clip, temperature=temp, x0_out=x0)
            what = (clip, temp)
            assert torch.equal(out, ref), (what, float((out - ref).abs().max()))
            assert torch.equal(x0, ref0), what
            o2 = torch.empty_like(x)
            ops.ddpm_update(x, eps, t, o2, tables=tables, noise=noise, clip=clip, temperature=temp)
            assert torch.equal(o2, ref), ("no x0_out", what)
            xi = x.clone()
            ops.ddpm_update(xi, eps, t, xi, tables=tables, noise=noise, clip=clip, temperature=temp, x0_out=x0)
            assert torch.equal(xi, ref) and torch.equal(x0, ref0), ("in place", what)
            p1, p2 = torch.empty_like(x), torch.empty_like(x)
            ops.ddpm_update(x, eps, t, p1, tables=tables, noise=noise, clip=clip, temperature=temp,
                            peer_ptrs=[p1.data_ptr()])
            assert torch.equal(p1, ref), ("peers", what)
            p1.zero_()
            ops.ddpm_update(x, eps, t, p1, tables=tables, noise=noise, clip=clip, temperature=temp, x0_out=x0,
                            peer_ptrs=[p1.data_ptr(), p2.data_ptr()])
            assert torch.equal(p1, ref) and torch.equal(p2, ref) and torch.equal(x0, ref0), ("2 peers", what)
            checked += 1
    assert checked == 6
    with pytest.raises(ValueError):
        ops.ddpm_update(x, eps, t.int(), out, tables=tables, noise=noise, clip=True)


@pytest.mark.gpu
def test_b200_equals_oracle_on_the_toy_on_cuda():
    """the whole 1000-step loop (and the fixture's other cases) over the CUDA toy: B200DDPMSampler against the oracle on
    CUDA, bit for bit"""
    m = ToyDenoiser(DEV)
    a = compute(lambda clip: DDPM(m, clip_denoised=clip), device=DEV)
    b = compute(lambda clip: B200DDPMSampler(DDPM(m, clip_denoised=clip)), device=DEV)
    for k in CASES:
        assert torch.equal(a[k], b[k]), (k, float((a[k] - b[k]).abs().max()))
    i = toy_inputs(DEV)
    d, s = pair(device=DEV)
    torch.manual_seed(3)
    ra = d.progressive_denoising(toy_cond(i), (4, 8, 8), batch_size=3, x_T=i["x_T"], verbose=False, start_T=100,
                                 temperature=[0.01 * k for k in range(100)], noise_dropout=0.2)
    torch.manual_seed(3)
    rb = s.progressive_denoising(toy_cond(i), (4, 8, 8), batch_size=3, x_T=i["x_T"], verbose=False, start_T=100,
                                 temperature=[0.01 * k for k in range(100)], noise_dropout=0.2)
    assert torch.equal(ra[0], rb[0]) and all(torch.equal(u, v) for u, v in zip(ra[1], rb[1]))


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
    return c, torch.randn(B, 4, h, h, device=DEV, generator=g)


@pytest.mark.gpu
def test_reduced_networks_against_oracle_and_graph_equals_eager(tiny):
    """a start_T = 20 loop over the reduced networks with the same seed: fp32 check mode within the 1e-4 gate of the
    oracle; CUDA-graph replay and eager runs give the same bits; the model's kept sampler reproduces them"""
    B, h, T = 2, 16, 20
    cond, x_T = make_cond(B, h, 64, seed=2)
    torch.manual_seed(11)
    ref = DDPM(tiny.oracle).p_sample_loop(cond, (B, 4, h, h), x_T=x_T, verbose=False, start_T=T)

    def go(m, graph):
        torch.manual_seed(11)
        return B200DDPMSampler(m, use_cuda_graph=graph).p_sample_loop(cond, (B, 4, h, h), x_T=x_T, verbose=False,
                                                                      start_T=T)

    a, g = go(tiny.f32, False), go(tiny.f32, True)
    b, bg = go(tiny.bf16, False), go(tiny.bf16, True)
    assert torch.equal(a, g) and torch.equal(b, bg)
    r32, r16 = rel(a, ref), rel(b, ref)
    print(f"DDPM start_T={T} final latents rel-L2 vs oracle (reduced nets): fp32-check {r32:.2e}, bf16 {r16:.2e}")
    assert r32 < 1e-4 and r16 < 5e-2, (r32, r16)
    torch.manual_seed(11)
    assert torch.equal(tiny.bf16.p_sample_loop(cond, (B, 4, h, h), x_T=x_T, verbose=False, start_T=T), bg)


@pytest.mark.gpu
def test_full_size_batch16_teacher_forced_and_start_T_100():
    """yaml networks, batch 16, 256^2, bf16: eps at timesteps spread over 0 ... 999, teacher-forced against the fp32
    oracle (TF32 off) through the sampler's own per-step call (embedding table of 1000 rows, graph), within the 1e-2 gate;
    and a start_T = 100 loop's final latent against the oracle's with the same seed (reported)"""
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    _no_tf32()
    full = Bundle({}, f32=False)
    B, h = 16, 32
    cond, x_T = make_cond(B, h, 768, seed=3)
    s = B200DDPMSampler(full.bf16, use_cuda_graph=True)
    s.begin_loop(range(999, -1, -1))
    tab = full.bf16._emb_table["tab"]
    print(f"per-loop embedding table at 1000 rows: {list(tab.shape)} {tab.dtype}, {tab.numel() * tab.element_size() / 2**20:.1f} MiB")
    r = []
    g = torch.Generator(device=DEV).manual_seed(5)
    for tv in (999, 900, 750, 500, 250, 100, 10, 0):
        t = torch.full((B,), tv, device=DEV, dtype=torch.long)
        x = full.oracle.q_sample(x_T, t, noise=torch.randn(x_T.shape, device=DEV, generator=g))
        with torch.no_grad():
            ref = full.oracle.apply_model(x, t, cond)
        r.append(rel(s._eps(x.contiguous(), t, cond, t_value=tv), ref))
    print("full-size batch-16 DDPM teacher-forced eps rel-L2 bf16 at t = 999 ... 0: " + " ".join(f"{v:.2e}" for v in r))
    assert max(r) <= 1e-2, r
    torch.manual_seed(7)
    a = s.p_sample_loop(cond, (B, 4, h, h), x_T=x_T, verbose=False, start_T=100)
    torch.manual_seed(7)
    b = DDPM(full.oracle).p_sample_loop(cond, (B, 4, h, h), x_T=x_T, verbose=False, start_T=100)
    print(f"full-size batch-16 DDPM start_T=100 final latent rel-L2 bf16 vs fp32 oracle: {rel(a, b):.2e}")
    assert bool(torch.isfinite(a).all())
    del full
    torch.cuda.empty_cache()


def _gpu_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    from makeupdiffuse_b200.dist import sample_ddpm_sharded
    from makeupdiffuse_b200.synth import synthetic_state_dict
    params = dict(model_channels=64, num_heads=4, context_dim=64)
    m = B200ControlLDM(params, params, dtype=torch.bfloat16, device=dev)
    m.load_state_dict(synthetic_state_dict(m, 0, dev))
    s = B200DDPMSampler(m)
    g = torch.Generator(device=dev).manual_seed(7)
    bg, h = 4, 16
    ctx = torch.randn(bg, 77, 64, device=dev, generator=g)
    hint = torch.rand(bg, 6, 8 * h, 8 * h, device=dev, generator=g)
    x_T = torch.randn(bg, 4, h, h, device=dev, generator=g)
    lo, hi = shard_bounds(bg, rank, world)
    cond = {"c_crossattn": [ctx[lo:hi].contiguous()], "c_concat": [hint[lo:hi].contiguous()]}
    res = {}
    for name, fused in (("nccl", False), ("fused", True), ("fused_again", True)):
        torch.manual_seed(9)
        res[name] = sample_ddpm_sharded(s, bg, (4, h, h), cond, x_T[lo:hi].contiguous(), rank, world,
                                        fused_gather=fused, start_T=10).cpu()
    torch.manual_seed(9)
    res["single"] = s.p_sample_loop({"c_crossattn": [ctx], "c_concat": [hint]}, (bg, 4, h, h), x_T=x_T, verbose=False,
                                    start_T=10).cpu()
    torch.save(res, os.path.join(out_dir, f"g{rank}.pt"))
    dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs of one box")
def test_two_gpu_sample_ddpm_sharded_fused_gather_equals_nccl(tmp_path):
    import torch.multiprocessing as mp
    port = 36300 + os.getpid() % 2000
    mp.spawn(_gpu_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = torch.load(tmp_path / "g0.pt"), torch.load(tmp_path / "g1.pt")
    for r in (r0, r1):
        assert torch.equal(r["nccl"], r["fused"]) and torch.equal(r["fused"], r["fused_again"])
    assert torch.equal(r0["fused"], r1["fused"])
    # a rank's kernels see another batch size than the single-process run (tile / split-K choices differ): numerical
    assert float((r0["fused"] - r0["single"]).abs().max()) < 0.05 * float(r0["single"].abs().max())
