"""TEST-ONLY restatement of upstream ``ldm.models.diffusion.dpm_solver`` (``DPMSolverSampler`` in ``sampler.py``;
``NoiseScheduleVP``, ``model_wrapper``, ``DPMSolver`` and ``interpolate_fn`` in ``dpm_solver.py``), limited to what
``DPMSolverSampler.sample`` reaches: the discrete schedule, the noise model with classifier-free guidance, DPM-Solver++
(``predict_x0=True``, no thresholding), ``skip_type='time_uniform'``, ``method='multistep'``, ``order=2``,
``lower_order_final=True``, ``solver_type='dpm_solver'``.

Upstream's files (lllyasviel/ControlNet, from Stability-AI/stablediffusion) are not vendored and cannot be read offline:
this is restated from their description, unchecked against the source, and pinned by the known answers of
tests/test_dpm_solver.py and the frozen fixture tests/golden/dpm_v1.npz (tests/golden/make_golden_dpm.py).
Deliberate differences: the doubled CFG cond is built with the oracle's ``_cat_uncond_first`` and the batch-size check
reads the first tensor of a list value (upstream's ``torch.cat([uc, c])`` and ``conditioning[key].shape`` take bare
tensors only and raise for this model's dict-of-lists cond); buffers follow ``model.device`` instead of being moved to
"cuda"; the progress bars and the 'v' model type are left out.
"""
import torch

from oracle.ddim import _cat_uncond_first

MODEL_TYPES = {"eps": "noise"}


def interpolate_fn(x, xp, yp):
    """piecewise-linear interpolation through (xp, yp), extended linearly beyond the ends.  x [N, C], xp / yp [C, K]"""
    N, K = x.shape[0], xp.shape[1]
    all_x = torch.cat([x.unsqueeze(2), xp.unsqueeze(0).repeat((N, 1, 1))], dim=2)
    sorted_all_x, x_indices = torch.sort(all_x, dim=2)
    x_idx = torch.argmin(x_indices, dim=2)
    cand_start_idx = x_idx - 1
    start_idx = torch.where(
        torch.eq(x_idx, 0),
        torch.tensor(1, device=x.device),
        torch.where(torch.eq(x_idx, K), torch.tensor(K - 2, device=x.device), cand_start_idx),
    )
    end_idx = torch.where(torch.eq(start_idx, cand_start_idx), start_idx + 2, start_idx + 1)
    start_x = torch.gather(sorted_all_x, dim=2, index=start_idx.unsqueeze(2)).squeeze(2)
    end_x = torch.gather(sorted_all_x, dim=2, index=end_idx.unsqueeze(2)).squeeze(2)
    start_idx2 = torch.where(
        torch.eq(x_idx, 0),
        torch.tensor(0, device=x.device),
        torch.where(torch.eq(x_idx, K), torch.tensor(K - 2, device=x.device), cand_start_idx),
    )
    y_positions_expanded = yp.unsqueeze(0).expand(N, -1, -1)
    start_y = torch.gather(y_positions_expanded, dim=2, index=start_idx2.unsqueeze(2)).squeeze(2)
    end_y = torch.gather(y_positions_expanded, dim=2, index=(start_idx2 + 1).unsqueeze(2)).squeeze(2)
    cand = start_y + (x - start_x) * (end_y - start_y) / (end_x - start_x)
    return cand


def expand_dims(v, dims):
    return v[(...,) + (None,) * (dims - 1)]


class NoiseScheduleVP:
    def __init__(self, schedule="discrete", betas=None, alphas_cumprod=None):
        assert schedule == "discrete"
        self.schedule = schedule
        if betas is not None:
            log_alphas = 0.5 * torch.log(1 - betas).cumsum(dim=0)
        else:
            assert alphas_cumprod is not None
            log_alphas = 0.5 * torch.log(alphas_cumprod)
        self.total_N = len(log_alphas)
        self.T = 1.
        self.t_array = torch.linspace(0., 1., self.total_N + 1)[1:].reshape((1, -1))
        self.log_alpha_array = log_alphas.reshape((1, -1,))

    def marginal_log_mean_coeff(self, t):
        return interpolate_fn(t.reshape((-1, 1)), self.t_array.to(t.device), self.log_alpha_array.to(t.device)).reshape((-1))

    def marginal_alpha(self, t):
        return torch.exp(self.marginal_log_mean_coeff(t))

    def marginal_std(self, t):
        return torch.sqrt(1. - torch.exp(2. * self.marginal_log_mean_coeff(t)))

    def marginal_lambda(self, t):
        log_mean_coeff = self.marginal_log_mean_coeff(t)
        log_std = 0.5 * torch.log(1. - torch.exp(2. * log_mean_coeff))
        return log_mean_coeff - log_std


def model_wrapper(model, noise_schedule, model_type="noise", model_kwargs=None, guidance_type="uncond", condition=None,
                  unconditional_condition=None, guidance_scale=1.):
    model_kwargs = model_kwargs or {}
    assert model_type == "noise" and guidance_type == "classifier-free"

    def get_model_input_time(t_continuous):
        return (t_continuous - 1. / noise_schedule.total_N) * 1000.

    def noise_pred_fn(x, t_continuous, cond=None):
        if t_continuous.reshape((-1,)).shape[0] == 1:
            t_continuous = t_continuous.expand((x.shape[0]))
        t_input = get_model_input_time(t_continuous)
        if cond is None:
            output = model(x, t_input, **model_kwargs)
        else:
            output = model(x, t_input, cond, **model_kwargs)
        return output

    def model_fn(x, t_continuous):
        if t_continuous.reshape((-1,)).shape[0] == 1:
            t_continuous = t_continuous.expand((x.shape[0]))
        if guidance_scale == 1. or unconditional_condition is None:
            return noise_pred_fn(x, t_continuous, cond=condition)
        x_in = torch.cat([x] * 2)
        t_in = torch.cat([t_continuous] * 2)
        c_in = _cat_uncond_first(unconditional_condition, condition)
        noise_uncond, noise = noise_pred_fn(x_in, t_in, cond=c_in).chunk(2)
        return noise_uncond + guidance_scale * (noise - noise_uncond)

    return model_fn


class DPMSolver:
    def __init__(self, model_fn, noise_schedule, predict_x0=False, thresholding=False):
        assert not thresholding
        self.model = model_fn
        self.noise_schedule = noise_schedule
        self.predict_x0 = predict_x0

    def noise_prediction_fn(self, x, t):
        return self.model(x, t)

    def data_prediction_fn(self, x, t):
        noise = self.noise_prediction_fn(x, t)
        dims = x.dim()
        alpha_t, sigma_t = self.noise_schedule.marginal_alpha(t), self.noise_schedule.marginal_std(t)
        x0 = (x - expand_dims(sigma_t, dims) * noise) / expand_dims(alpha_t, dims)
        return x0

    def model_fn(self, x, t):
        if self.predict_x0:
            return self.data_prediction_fn(x, t)
        return self.noise_prediction_fn(x, t)

    def get_time_steps(self, skip_type, t_T, t_0, N, device):
        assert skip_type == "time_uniform"
        return torch.linspace(t_T, t_0, N + 1).to(device)

    def dpm_solver_first_update(self, x, s, t, model_s=None):
        ns = self.noise_schedule
        dims = x.dim()
        lambda_s, lambda_t = ns.marginal_lambda(s), ns.marginal_lambda(t)
        h = lambda_t - lambda_s
        log_alpha_s, log_alpha_t = ns.marginal_log_mean_coeff(s), ns.marginal_log_mean_coeff(t)
        sigma_s, sigma_t = ns.marginal_std(s), ns.marginal_std(t)
        alpha_t = torch.exp(log_alpha_t)
        assert self.predict_x0
        phi_1 = torch.expm1(-h)
        if model_s is None:
            model_s = self.model_fn(x, s)
        x_t = (
            expand_dims(sigma_t / sigma_s, dims) * x
            - expand_dims(alpha_t * phi_1, dims) * model_s
        )
        return x_t

    def multistep_dpm_solver_second_update(self, x, model_prev_list, t_prev_list, t, solver_type="dpm_solver"):
        assert solver_type == "dpm_solver" and self.predict_x0
        ns = self.noise_schedule
        dims = x.dim()
        model_prev_1, model_prev_0 = model_prev_list
        t_prev_1, t_prev_0 = t_prev_list
        lambda_prev_1, lambda_prev_0, lambda_t = ns.marginal_lambda(t_prev_1), ns.marginal_lambda(t_prev_0), \
            ns.marginal_lambda(t)
        log_alpha_prev_0, log_alpha_t = ns.marginal_log_mean_coeff(t_prev_0), ns.marginal_log_mean_coeff(t)
        sigma_prev_0, sigma_t = ns.marginal_std(t_prev_0), ns.marginal_std(t)
        alpha_t = torch.exp(log_alpha_t)

        h_0 = lambda_prev_0 - lambda_prev_1
        h = lambda_t - lambda_prev_0
        r0 = h_0 / h
        D1_0 = expand_dims(1. / r0, dims) * (model_prev_0 - model_prev_1)
        x_t = (
            expand_dims(sigma_t / sigma_prev_0, dims) * x
            - expand_dims(alpha_t * (torch.exp(-h) - 1.), dims) * model_prev_0
            - 0.5 * expand_dims(alpha_t * (torch.exp(-h) - 1.), dims) * D1_0
        )
        return x_t

    def multistep_dpm_solver_update(self, x, model_prev_list, t_prev_list, t, order, solver_type="dpm_solver"):
        if order == 1:
            return self.dpm_solver_first_update(x, t_prev_list[-1], t, model_s=model_prev_list[-1])
        elif order == 2:
            return self.multistep_dpm_solver_second_update(x, model_prev_list, t_prev_list, t, solver_type=solver_type)
        raise ValueError("Solver order must be 1 or 2 here, got {}".format(order))

    def sample(self, x, steps=20, t_start=None, t_end=None, order=3, skip_type="time_uniform", method="singlestep",
               lower_order_final=True, denoise_to_zero=False, solver_type="dpm_solver"):
        t_0 = 1. / self.noise_schedule.total_N if t_end is None else t_end
        t_T = self.noise_schedule.T if t_start is None else t_start
        device = x.device
        assert method == "multistep" and not denoise_to_zero
        assert steps >= order
        timesteps = self.get_time_steps(skip_type=skip_type, t_T=t_T, t_0=t_0, N=steps, device=device)
        assert timesteps.shape[0] - 1 == steps
        with torch.no_grad():
            vec_t = timesteps[0].expand((x.shape[0]))
            model_prev_list = [self.model_fn(x, vec_t)]
            t_prev_list = [vec_t]
            # Init the first `order` values by lower order multistep DPM-Solver.
            for init_order in range(1, order):
                vec_t = timesteps[init_order].expand(x.shape[0])
                x = self.multistep_dpm_solver_update(x, model_prev_list, t_prev_list, vec_t, init_order,
                                                     solver_type=solver_type)
                model_prev_list.append(self.model_fn(x, vec_t))
                t_prev_list.append(vec_t)
            # Compute the remaining values by `order`-th order multistep DPM-Solver.
            for step in range(order, steps + 1):
                vec_t = timesteps[step].expand(x.shape[0])
                if lower_order_final and steps < 15:
                    step_order = min(order, steps + 1 - step)
                else:
                    step_order = order
                x = self.multistep_dpm_solver_update(x, model_prev_list, t_prev_list, vec_t, step_order,
                                                     solver_type=solver_type)
                for i in range(order - 1):
                    t_prev_list[i] = t_prev_list[i + 1]
                    model_prev_list[i] = model_prev_list[i + 1]
                t_prev_list[-1] = vec_t
                # We do not need to evaluate the final model value.
                if step < steps:
                    model_prev_list[-1] = self.model_fn(x, vec_t)
        return x


class DPMSolverSampler:
    def __init__(self, model, **kwargs):
        self.model = model
        self.alphas_cumprod = model.alphas_cumprod.clone().detach().to(torch.float32).to(model.device)

    @torch.no_grad()
    def sample(self, S, batch_size, shape, conditioning=None, callback=None, normals_sequence=None, img_callback=None,
               quantize_x0=False, eta=0., mask=None, x0=None, temperature=1., noise_dropout=0., score_corrector=None,
               corrector_kwargs=None, verbose=True, x_T=None, log_every_t=100, unconditional_guidance_scale=1.,
               unconditional_conditioning=None, **kwargs):
        if conditioning is not None:
            if isinstance(conditioning, dict):
                first = conditioning[list(conditioning.keys())[0]]
                cbs = (first[0] if isinstance(first, list) else first).shape[0]
                if cbs != batch_size:
                    print(f"Warning: Got {cbs} conditionings but batch-size is {batch_size}")
            elif torch.is_tensor(conditioning) and conditioning.shape[0] != batch_size:
                print(f"Warning: Got {conditioning.shape[0]} conditionings but batch-size is {batch_size}")
        C, H, W = shape
        size = (batch_size, C, H, W)
        device = self.model.betas.device
        img = torch.randn(size, device=device) if x_T is None else x_T
        ns = NoiseScheduleVP("discrete", alphas_cumprod=self.alphas_cumprod)
        model_fn = model_wrapper(
            lambda x, t, c: self.model.apply_model(x, t, c),
            ns,
            model_type=MODEL_TYPES[self.model.parameterization],
            guidance_type="classifier-free",
            condition=conditioning,
            unconditional_condition=unconditional_conditioning,
            guidance_scale=unconditional_guidance_scale,
        )
        dpm_solver = DPMSolver(model_fn, ns, predict_x0=True, thresholding=False)
        x = dpm_solver.sample(img, steps=S, skip_type="time_uniform", method="multistep", order=2, lower_order_final=True)
        return x.to(device), None
