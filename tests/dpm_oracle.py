"""Eager CPU restatement of CompVis's multistep DPM-Solver++ (ldm/models/diffusion/dpm_solver/dpm_solver.py:
NoiseScheduleVP('discrete'), model_wrapper(model_type='noise', guidance 'uncond' / 'classifier-free'),
DPM_Solver(predict_x0=True).sample(method='multistep', solver_type='dpm_solver')), in fp32 (the reference's dtype) or fp64.

It is written from the reference's formulas and is not pinned to a checkout.  Times, alphas and sigmas are [B] tensors as
the reference's `vec_t = timesteps[i].expand(B)` makes them.  interpolate_fn is the one sdb200.dpm_solver carries (a verbatim
copy of the reference's function; tests/test_dpm_solver_host.py checks it against np.interp in fp64).
"""
import torch

from sdb200.dpm_solver import interpolate_fn


def expand_dims(v, dims):
    return v[(...,) + (None,) * (dims - 1)]


class NoiseScheduleOracle:
    def __init__(self, alphas_cumprod, dtype=torch.float32):
        log_alphas = 0.5 * torch.log(torch.as_tensor(alphas_cumprod).to(dtype))
        self.total_N = len(log_alphas)
        self.T = 1.
        self.t_array = torch.linspace(0., 1., self.total_N + 1, dtype=dtype)[1:].reshape((1, -1))
        self.log_alpha_array = log_alphas.reshape((1, -1))
        self.dtype = dtype

    def marginal_log_mean_coeff(self, t):
        return interpolate_fn(t.reshape((-1, 1)), self.t_array, self.log_alpha_array).reshape((-1))

    def marginal_alpha(self, t):
        return torch.exp(self.marginal_log_mean_coeff(t))

    def marginal_std(self, t):
        return torch.sqrt(1. - torch.exp(2. * self.marginal_log_mean_coeff(t)))

    def marginal_lambda(self, t):
        log_mean_coeff = self.marginal_log_mean_coeff(t)
        log_std = 0.5 * torch.log(1. - torch.exp(2. * log_mean_coeff))
        return log_mean_coeff - log_std

    def inverse_lambda(self, lamb):
        log_alpha = -0.5 * torch.logaddexp(torch.zeros((1,)).to(lamb), -2. * lamb)
        t = interpolate_fn(log_alpha.reshape((-1, 1)), torch.flip(self.log_alpha_array, [1]), torch.flip(self.t_array, [1]))
        return t.reshape((-1,))


class DPMSolverOracle:
    """`model(x, t_input, c)` returns the noise prediction.  `record` receives (x, t_input[0], batch rows) of every model
    call; `evals` receives (x, noise after the guidance combine) of every model evaluation."""

    def __init__(self, model, alphas_cumprod, dtype=torch.float32, condition=None, unconditional_condition=None,
                 guidance_scale=1.):
        self.model = model
        self.ns = NoiseScheduleOracle(alphas_cumprod, dtype)
        self.condition, self.uc, self.scale = condition, unconditional_condition, guidance_scale
        self.record, self.evals = [], []

    # model_wrapper
    def noise_fn(self, x, t_continuous):
        t_input = (t_continuous - 1. / self.ns.total_N) * 1000.
        if self.scale == 1. or self.uc is None:
            out = self.model(x, t_input, self.condition)
            self.record.append((x, float(t_input[0]), x.shape[0]))
        else:
            x_in, t_in = torch.cat([x] * 2), torch.cat([t_input] * 2)
            c, uc = self.condition, self.uc
            if isinstance(c, dict):
                c_in = {k: [torch.cat([uc[k][i], c[k][i]]) for i in range(len(c[k]))] for k in c}
            else:
                c_in = torch.cat([uc, c])
            noise_uncond, noise = self.model(x_in, t_in, c_in).chunk(2)
            self.record.append((x, float(t_input[0]), x_in.shape[0]))
            out = noise_uncond + self.scale * (noise - noise_uncond)
        self.evals.append((x, out))
        return out

    # DPM_Solver.data_prediction_fn
    def model_fn(self, x, t):
        noise = self.noise_fn(x, t)
        dims = x.dim()
        alpha_t, sigma_t = self.ns.marginal_alpha(t), self.ns.marginal_std(t)
        return (x - expand_dims(sigma_t, dims) * noise) / expand_dims(alpha_t, dims)

    def get_time_steps(self, skip_type, t_T, t_0, N):
        dt = self.ns.dtype
        if skip_type == 'logSNR':
            lambda_T = self.ns.marginal_lambda(torch.tensor(t_T, dtype=dt))
            lambda_0 = self.ns.marginal_lambda(torch.tensor(t_0, dtype=dt))
            return self.ns.inverse_lambda(torch.linspace(lambda_T.item(), lambda_0.item(), N + 1, dtype=dt))
        if skip_type == 'time_uniform':
            return torch.linspace(t_T, t_0, N + 1, dtype=dt)
        if skip_type == 'time_quadratic':
            return torch.linspace(t_T ** 0.5, t_0 ** 0.5, N + 1, dtype=dt).pow(2)
        raise ValueError(skip_type)

    def first_update(self, x, s, t, model_s):
        ns, dims = self.ns, x.dim()
        lambda_s, lambda_t = ns.marginal_lambda(s), ns.marginal_lambda(t)
        h = lambda_t - lambda_s
        log_alpha_t = ns.marginal_log_mean_coeff(t)
        sigma_s, sigma_t = ns.marginal_std(s), ns.marginal_std(t)
        alpha_t = torch.exp(log_alpha_t)
        phi_1 = torch.expm1(-h)
        return expand_dims(sigma_t / sigma_s, dims) * x - expand_dims(alpha_t * phi_1, dims) * model_s

    def second_update(self, x, model_prev_list, t_prev_list, t):
        ns, dims = self.ns, x.dim()
        model_prev_1, model_prev_0 = model_prev_list[-2], model_prev_list[-1]
        t_prev_1, t_prev_0 = t_prev_list[-2], t_prev_list[-1]
        lambda_prev_1, lambda_prev_0, lambda_t = ns.marginal_lambda(t_prev_1), ns.marginal_lambda(t_prev_0), ns.marginal_lambda(t)
        log_alpha_t = ns.marginal_log_mean_coeff(t)
        sigma_prev_0, sigma_t = ns.marginal_std(t_prev_0), ns.marginal_std(t)
        alpha_t = torch.exp(log_alpha_t)
        h_0 = lambda_prev_0 - lambda_prev_1
        h = lambda_t - lambda_prev_0
        r0 = h_0 / h
        D1_0 = expand_dims(1. / r0, dims) * (model_prev_0 - model_prev_1)
        return (expand_dims(sigma_t / sigma_prev_0, dims) * x
                - expand_dims(alpha_t * (torch.exp(-h) - 1.), dims) * model_prev_0
                - 0.5 * expand_dims(alpha_t * (torch.exp(-h) - 1.), dims) * D1_0)

    def third_update(self, x, model_prev_list, t_prev_list, t):
        ns, dims = self.ns, x.dim()
        model_prev_2, model_prev_1, model_prev_0 = model_prev_list
        t_prev_2, t_prev_1, t_prev_0 = t_prev_list
        lambda_prev_2, lambda_prev_1, lambda_prev_0, lambda_t = (ns.marginal_lambda(t_prev_2), ns.marginal_lambda(t_prev_1),
                                                                 ns.marginal_lambda(t_prev_0), ns.marginal_lambda(t))
        log_alpha_t = ns.marginal_log_mean_coeff(t)
        sigma_prev_0, sigma_t = ns.marginal_std(t_prev_0), ns.marginal_std(t)
        alpha_t = torch.exp(log_alpha_t)
        h_1 = lambda_prev_1 - lambda_prev_2
        h_0 = lambda_prev_0 - lambda_prev_1
        h = lambda_t - lambda_prev_0
        r0, r1 = h_0 / h, h_1 / h
        D1_0 = expand_dims(1. / r0, dims) * (model_prev_0 - model_prev_1)
        D1_1 = expand_dims(1. / r1, dims) * (model_prev_1 - model_prev_2)
        D1 = D1_0 + expand_dims(r0 / (r0 + r1), dims) * (D1_0 - D1_1)
        D2 = expand_dims(1. / (r0 + r1), dims) * (D1_0 - D1_1)
        return (expand_dims(sigma_t / sigma_prev_0, dims) * x
                - expand_dims(alpha_t * (torch.exp(-h) - 1.), dims) * model_prev_0
                + expand_dims(alpha_t * ((torch.exp(-h) - 1.) / h + 1.), dims) * D1
                - expand_dims(alpha_t * ((torch.exp(-h) - 1. + h) / h ** 2 - 0.5), dims) * D2)

    def multistep_update(self, x, model_prev_list, t_prev_list, t, order):
        if order == 1:
            return self.first_update(x, t_prev_list[-1], t, model_prev_list[-1])
        if order == 2:
            return self.second_update(x, model_prev_list, t_prev_list, t)
        return self.third_update(x, model_prev_list, t_prev_list, t)

    def sample(self, x, steps=20, order=2, skip_type='time_uniform', lower_order_final=True):
        t_0, t_T = 1. / self.ns.total_N, self.ns.T
        assert steps >= order
        timesteps = self.get_time_steps(skip_type, t_T, t_0, steps)
        B = x.shape[0]
        vec_t = timesteps[0].expand((B))
        model_prev_list = [self.model_fn(x, vec_t)]
        t_prev_list = [vec_t]
        for init_order in range(1, order):
            vec_t = timesteps[init_order].expand(B)
            x = self.multistep_update(x, model_prev_list, t_prev_list, vec_t, init_order)
            model_prev_list.append(self.model_fn(x, vec_t))
            t_prev_list.append(vec_t)
        for step in range(order, steps + 1):
            vec_t = timesteps[step].expand(B)
            step_order = min(order, steps + 1 - step) if lower_order_final and steps < 15 else order
            x = self.multistep_update(x, model_prev_list, t_prev_list, vec_t, step_order)
            for i in range(order - 1):
                t_prev_list[i] = t_prev_list[i + 1]
                model_prev_list[i] = model_prev_list[i + 1]
            t_prev_list[-1] = vec_t
            if step < steps:
                model_prev_list[-1] = self.model_fn(x, vec_t)
        return x
