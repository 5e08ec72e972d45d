"""Drop-in multistep DPM-Solver++ (reference: CompVis/stable-diffusion ldm/models/diffusion/dpm_solver/, the
`--dpm_solver` sampler of scripts/txt2img.py): `NoiseScheduleVP`, `model_wrapper`, `DPM_Solver` and `DPMSolverSampler`,
whose per-evaluation arithmetic (guidance combine, data prediction and the order-1/2/3 update) runs as ONE fused sm_100a
kernel (sdb_dpm_solver_step).

What runs: the discrete noise schedule, noise-prediction models with or without classifier-free guidance, and
`DPM_Solver.sample(method='multistep')` with `predict_x0=True` (DPM-Solver++), `solver_type='dpm_solver'`, orders 1-3 and
the three skip types.  Singlestep and adaptive methods, the noise-prediction form, thresholding, the 'taylor' solver type,
continuous schedules, other model types and classifier guidance raise NotImplementedError.

Every per-step scalar (the schedule's alpha, sigma and lambda at each time, h, r0, r1 and the update coefficients) is
evaluated with the reference's own torch expressions on one-element host fp32 tensors before the first model call, so
the loop makes no host synchronisation; they are cached on the noise schedule per (steps, order, time grid), so a
sampler's later calls with the same settings start the GPU at once.  The reference evaluates them on its [B] batch of equal
times wherever the model lives; on the CPU with a batch below 16 (torch's scalar kernel path) that gives these values bit
for bit, while on CUDA, or with torch's vectorised CPU exp / log / expm1, a value may differ in the last ulp.
"""
import torch

from . import engine, ops
from .ddim import DDIMSampler, _f32_contiguous


def interpolate_fn(x, xp, yp):
    """dpm_solver.py interpolate_fn: piecewise-linear interpolation of x [N, 1] on the keypoints xp, yp [1, K] (linear
    extrapolation outside them), differentiable, as the reference writes it."""
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


class NoiseScheduleVP:
    """The discrete-time VP schedule of a DDPM (dpm_solver.py NoiseScheduleVP('discrete', ...)): log alpha_t is the
    piecewise-linear interpolation of 0.5 * log(alphas_cumprod) on t_n = n / N, n = 1..N.  The tables are host fp32 tensors
    (DPMSolverSampler's alphas_cumprod is fp32), so the sampler's per-step scalars are computed on the host."""

    def __init__(self, schedule='discrete', betas=None, alphas_cumprod=None, continuous_beta_0=0.1, continuous_beta_1=20.):
        if schedule not in ['discrete', 'linear', 'cosine']:
            raise ValueError("Unsupported noise schedule {}. The schedule needs to be 'discrete' or 'linear' or 'cosine'".format(
                schedule))
        if schedule != 'discrete':
            raise NotImplementedError("NoiseScheduleVP: only the 'discrete' schedule of a DDPM is implemented, not %r" % schedule)
        self.schedule = schedule
        host = lambda v: torch.as_tensor(v).detach().to("cpu", torch.float32)
        if betas is not None:
            log_alphas = 0.5 * torch.log(1 - host(betas)).cumsum(dim=0)
        else:
            assert alphas_cumprod is not None
            log_alphas = 0.5 * torch.log(host(alphas_cumprod))
        self.total_N = len(log_alphas)
        self.T = 1.
        self.t_array = torch.linspace(0., 1., self.total_N + 1)[1:].reshape((1, -1))
        self.log_alpha_array = log_alphas.reshape((1, -1,))

    def marginal_log_mean_coeff(self, t):
        """log(alpha_t)."""
        return interpolate_fn(t.reshape((-1, 1)), self.t_array.to(t.device), self.log_alpha_array.to(t.device)).reshape((-1))

    def marginal_alpha(self, t):
        return torch.exp(self.marginal_log_mean_coeff(t))

    def marginal_std(self, t):
        return torch.sqrt(1. - torch.exp(2. * self.marginal_log_mean_coeff(t)))

    def marginal_lambda(self, t):
        """lambda_t = log(alpha_t) - log(sigma_t), the half-logSNR."""
        log_mean_coeff = self.marginal_log_mean_coeff(t)
        log_std = 0.5 * torch.log(1. - torch.exp(2. * log_mean_coeff))
        return log_mean_coeff - log_std

    def inverse_lambda(self, lamb):
        """The t whose lambda_t is `lamb`."""
        log_alpha = -0.5 * torch.logaddexp(torch.zeros((1,)).to(lamb), -2. * lamb)
        t = interpolate_fn(log_alpha.reshape((-1, 1)), torch.flip(self.log_alpha_array.to(lamb.device), [1]),
                           torch.flip(self.t_array.to(lamb.device), [1]))
        return t.reshape((-1,))


class _OnceEach:
    """A view of a NoiseScheduleVP that interpolates log(alpha_t) once per time value and derives alpha, sigma and lambda
    from it with the schedule's own expressions: the same values, without repeating the interpolation's sort for every
    expression of every update that reads the same time."""
    marginal_alpha = NoiseScheduleVP.marginal_alpha
    marginal_std = NoiseScheduleVP.marginal_std
    marginal_lambda = NoiseScheduleVP.marginal_lambda

    def __init__(self, ns):
        self.ns, self._lmc = ns, {}

    def marginal_log_mean_coeff(self, t):
        key = float(t)
        if key not in self._lmc:
            self._lmc[key] = self.ns.marginal_log_mean_coeff(t)
        return self._lmc[key]


class _GuidedNoise:
    """The model_fn of model_wrapper without its final guidance combine: model_fn(x, t_continuous) -> (e, e_uncond).  The
    model is evaluated by DDIMSampler's `_model_eps` (one 2B call with classifier-free guidance, the (uc, c) concatenation
    built once per conditioning pair, tensor and dict conditionings); e_uncond is None without guidance, and otherwise
    sdb_dpm_solver_step forms e_uncond + guidance_scale * (e - e_uncond)."""
    _model_eps = DDIMSampler._model_eps
    _cfg_dict_pairable = staticmethod(DDIMSampler._cfg_dict_pairable)
    _cfg_dict_in = DDIMSampler._cfg_dict_in

    def __init__(self, model, noise_schedule, condition, unconditional_condition, guidance_scale):
        self.model = model
        self.noise_schedule = noise_schedule
        self.condition = condition
        self.unconditional_condition = unconditional_condition
        self.guidance_scale = guidance_scale
        self._cfg_ctx = engine.TensorMemo(1)

    def get_model_input_time(self, t_continuous):
        """Discrete-time models take t_input = (t - 1/N) * 1000, e.g. 999 at t = 1 (a float: 979.02... between knots)."""
        return (t_continuous - 1. / self.noise_schedule.total_N) * 1000.

    def __call__(self, x, t_continuous):
        """x: the device latent; t_continuous: a one-element host fp32 tensor."""
        t_input = torch.full((x.shape[0],), float(self.get_model_input_time(t_continuous)), device=x.device)
        return self._model_eps(x, self.condition, t_input, None, None, self.guidance_scale, self.unconditional_condition)


def model_wrapper(model, noise_schedule, model_type="noise", guidance_type="uncond", condition=None,
                  unconditional_condition=None, guidance_scale=1.):
    """dpm_solver.py model_wrapper for a noise-prediction model, without guidance ("uncond") or with classifier-free
    guidance.  `model` has the LatentDiffusion interface `apply_model(x, t, c)` (the reference takes the function
    `lambda x, t, c: model.apply_model(x, t, c)`).  The returned model_fn(x, t_continuous) gives (e, e_uncond); DPM_Solver
    leaves the guidance combine to its update kernel."""
    if model_type != "noise":
        raise NotImplementedError("model_wrapper: only model_type='noise' is implemented, not %r" % (model_type,))
    if guidance_type == "classifier":
        raise NotImplementedError("model_wrapper: classifier guidance is not implemented; use 'uncond' or 'classifier-free'")
    if guidance_type not in ("uncond", "classifier-free"):
        raise ValueError("model_wrapper: guidance_type must be 'uncond' or 'classifier-free', not %r" % (guidance_type,))
    if guidance_type == "uncond":
        condition, unconditional_condition, guidance_scale = None, None, 1.
    return _GuidedNoise(model, noise_schedule, condition, unconditional_condition, guidance_scale)


class DPM_Solver:
    """dpm_solver.py DPM_Solver, multistep DPM-Solver++: each model evaluation is followed by ONE sdb_dpm_solver_step launch
    that forms the data prediction at the evaluated time and the update to the next time."""

    def __init__(self, model_fn, noise_schedule, predict_x0=True, thresholding=False, max_val=1.):
        if not predict_x0:
            raise NotImplementedError("DPM_Solver: only the data-prediction form (predict_x0=True, DPM-Solver++) is implemented")
        if thresholding:
            raise NotImplementedError("DPM_Solver: dynamic thresholding is not implemented")
        self.model = model_fn
        self.noise_schedule = noise_schedule
        self.predict_x0 = predict_x0
        self.thresholding = thresholding
        self.max_val = max_val

    def get_time_steps(self, skip_type, t_T, t_0, N):
        """The N + 1 times from t_T to t_0 (host fp32), spaced uniformly in logSNR, in time, or in sqrt(time)."""
        if skip_type == 'logSNR':
            lambda_T = self.noise_schedule.marginal_lambda(torch.tensor(t_T))
            lambda_0 = self.noise_schedule.marginal_lambda(torch.tensor(t_0))
            logSNR_steps = torch.linspace(lambda_T.item(), lambda_0.item(), N + 1)
            return self.noise_schedule.inverse_lambda(logSNR_steps)
        elif skip_type == 'time_uniform':
            return torch.linspace(t_T, t_0, N + 1)
        elif skip_type == 'time_quadratic':
            t_order = 2
            return torch.linspace(t_T ** (1. / t_order), t_0 ** (1. / t_order), N + 1).pow(t_order)
        else:
            raise ValueError("Unsupported skip_type {}, need to be 'logSNR' or 'time_uniform' or 'time_quadratic'".format(skip_type))

    @staticmethod
    def step_orders(steps, order, lower_order_final=True):
        """The order of updates k = 1..steps: k for the warm-up updates k < order, then `order`, or with lower_order_final
        and fewer than 15 steps min(order, steps + 1 - k)."""
        return [k if k < order else (min(order, steps + 1 - k) if lower_order_final and steps < 15 else order)
                for k in range(1, steps + 1)]

    def update_coefficients(self, t_prev_list, t, order, ns=None):
        """The ten fp32 scalars of sdb_dpm_solver_step for the order-`order` update from t_prev_list[-1] to t:
        (sigma_s, alpha_s) of data_prediction_fn at s = t_prev_list[-1], then (c_x, c_0, c_1, c_2, inv_r0, inv_r1, c_r, c_d2)
        as dpm_solver_first_update / multistep_dpm_solver_second_update / _third_update form them (0 where the order
        reads none).  Times are one-element host fp32 tensors; ns (default: the solver's schedule) evaluates them."""
        ns = self.noise_schedule if ns is None else ns
        s = t_prev_list[-1]
        head = (ns.marginal_std(s), ns.marginal_alpha(s))
        if order == 1:
            lambda_s, lambda_t = ns.marginal_lambda(s), ns.marginal_lambda(t)
            h = lambda_t - lambda_s
            log_alpha_t = ns.marginal_log_mean_coeff(t)
            sigma_s, sigma_t = ns.marginal_std(s), ns.marginal_std(t)
            alpha_t = torch.exp(log_alpha_t)
            phi_1 = torch.expm1(-h)
            body = (sigma_t / sigma_s, alpha_t * phi_1, 0., 0., 0., 0., 0., 0.)
        elif order == 2:
            t_prev_1, t_prev_0 = t_prev_list[-2], t_prev_list[-1]
            lambda_prev_1, lambda_prev_0, lambda_t = ns.marginal_lambda(t_prev_1), ns.marginal_lambda(t_prev_0), ns.marginal_lambda(t)
            log_alpha_t = ns.marginal_log_mean_coeff(t)
            sigma_prev_0, sigma_t = ns.marginal_std(t_prev_0), ns.marginal_std(t)
            alpha_t = torch.exp(log_alpha_t)
            h_0 = lambda_prev_0 - lambda_prev_1
            h = lambda_t - lambda_prev_0
            r0 = h_0 / h
            c_0 = alpha_t * (torch.exp(-h) - 1.)
            body = (sigma_t / sigma_prev_0, c_0, 0.5 * c_0, 0., 1. / r0, 0., 0., 0.)
        elif order == 3:
            t_prev_2, t_prev_1, t_prev_0 = t_prev_list[-3], t_prev_list[-2], t_prev_list[-1]
            lambda_prev_2, lambda_prev_1 = ns.marginal_lambda(t_prev_2), ns.marginal_lambda(t_prev_1)
            lambda_prev_0, lambda_t = ns.marginal_lambda(t_prev_0), ns.marginal_lambda(t)
            log_alpha_t = ns.marginal_log_mean_coeff(t)
            sigma_prev_0, sigma_t = ns.marginal_std(t_prev_0), ns.marginal_std(t)
            alpha_t = torch.exp(log_alpha_t)
            h_1 = lambda_prev_1 - lambda_prev_2
            h_0 = lambda_prev_0 - lambda_prev_1
            h = lambda_t - lambda_prev_0
            r0, r1 = h_0 / h, h_1 / h
            body = (sigma_t / sigma_prev_0, alpha_t * (torch.exp(-h) - 1.), alpha_t * ((torch.exp(-h) - 1.) / h + 1.),
                    alpha_t * ((torch.exp(-h) - 1. + h) / h ** 2 - 0.5), 1. / r0, 1. / r1, r0 / (r0 + r1), 1. / (r0 + r1))
        else:
            raise ValueError("Solver order must be 1 or 2 or 3, got {}".format(order))
        return tuple(float(v) for v in head + body)

    def _plan(self, steps, t_T, t_0, order, skip_type, lower_order_final):
        """Every scalar of one sample loop, on the host, before the first launch: the times (one-element tensors), the
        order of each update and its coefficients.  Cached on the noise schedule, whose tables are fixed at construction."""
        key = (steps, t_T, t_0, order, skip_type, lower_order_final)
        plans = self.noise_schedule.__dict__.setdefault("_dpm_plans", {})
        if key not in plans:
            timesteps = self.get_time_steps(skip_type=skip_type, t_T=t_T, t_0=t_0, N=steps)
            assert timesteps.shape[0] - 1 == steps
            ts = [timesteps[i].reshape(1) for i in range(steps + 1)]
            orders = self.step_orders(steps, order, lower_order_final)
            ns = _OnceEach(self.noise_schedule)
            coefs = [self.update_coefficients(ts[max(k - order, 0):k], ts[k], orders[k - 1], ns) for k in range(1, steps + 1)]
            plans[key] = (ts, orders, coefs)
        return plans[key]

    def sample(self, x, steps=20, t_start=None, t_end=None, order=2, skip_type='time_uniform', method='multistep',
               lower_order_final=True, solver_type='dpm_solver'):
        """dpm_solver.py DPM_Solver.sample, method='multistep': `steps` model evaluations (the first at t_T, none after the
        last update) from x at t_start (default T = 1) to t_end (default 1/N).  x: the fp32 device latent."""
        if method != 'multistep':
            raise NotImplementedError("DPM_Solver.sample: only method='multistep' is implemented, not %r" % (method,))
        if solver_type == 'taylor':
            raise NotImplementedError("DPM_Solver.sample: only solver_type='dpm_solver' is implemented, not 'taylor'")
        if solver_type != 'dpm_solver':
            raise ValueError("'solver_type' must be either 'dpm_solver' or 'taylor', got {}".format(solver_type))
        if order not in (1, 2, 3):
            raise ValueError("Solver order must be 1 or 2 or 3, got {}".format(order))
        t_0 = 1. / self.noise_schedule.total_N if t_end is None else t_end
        t_T = self.noise_schedule.T if t_start is None else t_start
        assert steps >= order
        ts, orders, coefs = self._plan(steps, t_T, t_0, order, skip_type, lower_order_final)
        x = _f32_contiguous(x)
        hist = []           # data predictions of the previous evaluations, newest last (model_prev_list[:-1])
        for k in range(1, steps + 1):
            p = orders[k - 1]
            e, e_uncond = self.model(x, ts[k - 1])
            # fresh outputs every launch: nothing the kernel reads is written by it
            x, m0 = ops.dpm_solver_step(x, _f32_contiguous(e), p, coefs[k - 1], e_uncond=_f32_contiguous(e_uncond),
                                        cfg_scale=self.model.guidance_scale, m1=hist[-1] if p >= 2 else None,
                                        m2=hist[-2] if p >= 3 else None, want_m0=k < steps and order > 1)
            if order > 1:
                hist = (hist + [m0])[-(order - 1):]
        return x


class DPMSolverSampler(object):
    """CompVis DPMSolverSampler: DPM-Solver++(2M), i.e. DPM_Solver.sample(order=2, skip_type='time_uniform',
    method='multistep', lower_order_final=True) on the model's discrete schedule, with classifier-free guidance.

    `sample` takes DDIMSampler.sample's parameters.  As in the reference, S, batch_size, shape, conditioning, x_T,
    unconditional_guidance_scale and unconditional_conditioning are used; every other argument (eta, temperature, mask, x0,
    callbacks, quantize_x0, noise_dropout, score_corrector, ...) is accepted and ignored.  The sampler has none of
    DDIMSampler's other methods."""

    def __init__(self, model, **kwargs):
        super().__init__()
        self.model = model
        # the schedule on the host (one copy here): every per-step scalar is computed there, with no sync in the loop
        self.alphas_cumprod = model.alphas_cumprod.detach().to("cpu", torch.float32)
        self.noise_schedule = NoiseScheduleVP('discrete', alphas_cumprod=self.alphas_cumprod)
        self._cfg_ctx = engine.TensorMemo(1)

    @torch.no_grad()
    def sample(self, S, batch_size, shape, conditioning=None, callback=None, normals_sequence=None, img_callback=None,
               quantize_x0=False, eta=0., mask=None, x0=None, temperature=1., noise_dropout=0., score_corrector=None,
               corrector_kwargs=None, verbose=True, x_T=None, log_every_t=100, unconditional_guidance_scale=1.,
               unconditional_conditioning=None, **kwargs):
        """(samples, None)."""
        DDIMSampler._warn_conditioning_batch(conditioning, batch_size)
        C, H, W = shape
        size = (batch_size, C, H, W)
        device = self.model.betas.device
        img = torch.randn(size, device=device) if x_T is None else x_T
        model_fn = model_wrapper(self.model, self.noise_schedule, model_type="noise", guidance_type="classifier-free",
                                 condition=conditioning, unconditional_condition=unconditional_conditioning,
                                 guidance_scale=unconditional_guidance_scale)
        model_fn._cfg_ctx = self._cfg_ctx        # one 2B conditioning for every sample call with the same (uc, c)
        dpm_solver = DPM_Solver(model_fn, self.noise_schedule, predict_x0=True, thresholding=False)
        x = dpm_solver.sample(img, steps=S, skip_type="time_uniform", method="multistep", order=2, lower_order_final=True)
        return x.to(device), None
