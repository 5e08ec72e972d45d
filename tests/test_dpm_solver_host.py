"""CPU: the DPM-Solver++ host side (noise schedule, time grids, order schedule, per-step scalars, interface, rejected
options) and the host-side argument checks of sdb_dpm_solver_step (every check runs before any launch, so none of them
needs a GPU).  The solver's formulas are checked independently of any restatement on Gaussian data, whose exact
probability-flow solution is known in closed form."""
import inspect
import math

import numpy as np
import pytest
import torch

from dpm_oracle import DPMSolverOracle, NoiseScheduleOracle
from oracle import restate as R

AC = R.sd_alphas_cumprod()


def _ns():
    from sdb200.dpm_solver import NoiseScheduleVP
    return NoiseScheduleVP('discrete', alphas_cumprod=torch.tensor(AC, dtype=torch.float32))


def _solver(model_fn=None):
    from sdb200.dpm_solver import DPM_Solver
    return DPM_Solver(model_fn, _ns(), predict_x0=True)


# ---- noise schedule -------------------------------------------------------------------------------------------------------
def test_noise_schedule_against_fp64():
    ns = _ns()
    assert ns.total_N == 1000 and ns.T == 1.
    t64 = np.concatenate([np.linspace(1e-3, 1., 997), [0.0015, 0.5005, 0.9995]])
    la64 = np.interp(t64, np.arange(1, 1001) / 1000., 0.5 * np.log(AC))
    a64 = np.exp(la64)
    s64 = np.sqrt(1. - a64 ** 2)
    t = torch.tensor(t64, dtype=torch.float32)
    assert np.allclose(ns.marginal_log_mean_coeff(t).double().numpy(), la64, rtol=1e-5, atol=1e-6)
    assert np.allclose(ns.marginal_alpha(t).double().numpy(), a64, rtol=1e-5)
    assert np.allclose(ns.marginal_std(t).double().numpy(), s64, rtol=1e-5, atol=2e-6)      # sqrt(1 - a^2): cancellation
    assert np.allclose(ns.marginal_lambda(t).double().numpy(), np.log(a64) - np.log(s64), rtol=1e-4, atol=1e-4)
    # the knots: alpha_{t_n}^2 is alphas_cumprod[n - 1]
    knots = torch.arange(1, 1001, dtype=torch.float32) / 1000.
    assert np.allclose(ns.marginal_alpha(knots).double().numpy() ** 2, AC, rtol=2e-6)


def test_inverse_lambda_round_trip():
    ns = _ns()
    t = torch.linspace(1e-3, 1., 2001)
    back = ns.inverse_lambda(ns.marginal_lambda(t))
    assert float((back - t).abs().max()) <= 2e-5            # fp32: lambda is steep near t = 0, flat near t = 1
    # and the other way round, on the logSNR grid of the solver
    lam = torch.linspace(float(ns.marginal_lambda(torch.tensor(1.))), float(ns.marginal_lambda(torch.tensor(1e-3))), 50)
    assert float((ns.marginal_lambda(ns.inverse_lambda(lam)) - lam).abs().max()) <= 1e-4


@pytest.mark.parametrize("skip_type", ["time_uniform", "logSNR", "time_quadratic"])
@pytest.mark.parametrize("steps", [1, 2, 10, 20])
def test_time_steps(skip_type, steps):
    ts = _solver().get_time_steps(skip_type, 1., 1. / 1000, steps)
    assert ts.dtype == torch.float32 and ts.device.type == "cpu" and ts.shape == (steps + 1,)
    assert abs(float(ts[0]) - 1.) <= 1e-6 and abs(float(ts[-1]) - 1e-3) <= 1e-6
    assert bool((ts[1:] < ts[:-1]).all())


def test_noise_schedule_options():
    from sdb200.dpm_solver import NoiseScheduleVP
    betas = torch.tensor(1. - AC / np.append(1., AC[:-1]), dtype=torch.float32)
    from_betas = NoiseScheduleVP('discrete', betas=betas)
    assert torch.allclose(from_betas.log_alpha_array, _ns().log_alpha_array, rtol=1e-5, atol=1e-6)
    for sched in ("linear", "cosine"):
        with pytest.raises(NotImplementedError):
            NoiseScheduleVP(sched)
    with pytest.raises(ValueError):
        NoiseScheduleVP("sigmoid")


# ---- the order schedule -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("steps,order,lof,want", [
    (2, 2, True, [1, 1]), (2, 1, True, [1, 1]),
    (3, 2, True, [1, 2, 1]), (3, 3, True, [1, 2, 1]), (3, 3, False, [1, 2, 3]),
    (14, 2, True, [1] + [2] * 12 + [1]), (14, 3, True, [1, 2] + [3] * 10 + [2, 1]), (14, 3, False, [1, 2] + [3] * 12),
    (15, 2, True, [1] + [2] * 14), (15, 3, True, [1, 2] + [3] * 13),
    (20, 2, True, [1] + [2] * 19), (20, 3, True, [1, 2] + [3] * 18), (20, 1, True, [1] * 20),
])
def test_step_orders(steps, order, lof, want):
    from sdb200.dpm_solver import DPM_Solver
    assert DPM_Solver.step_orders(steps, order, lof) == want


# ---- the formulas against the exact solution on Gaussian data ---------------------------------------------------------
MU, SD = 0.5, 0.5         # data N(MU, SD^2 I)


def _gaussian_error(steps, order, dtype=torch.float64):
    """Final max-abs error of the restated solver (logSNR grid, no lower-order final steps) against the exact
    probability-flow solution x_0 = a_0 mu + sqrt(a_0^2 s^2 + s_0^2) / sqrt(a_T^2 s^2 + s_T^2) (x_T - a_T mu)."""
    ns = NoiseScheduleOracle(AC, dtype)

    def eps(x, t_input, c):
        t = t_input / 1000. + 1. / ns.total_N
        a, s = ns.marginal_alpha(t).view(-1, 1, 1, 1), ns.marginal_std(t).view(-1, 1, 1, 1)
        return s * (x - a * MU) / (a * a * SD * SD + s * s)

    orc = DPMSolverOracle(eps, AC, dtype)
    x_T = torch.randn((2, 3, 4, 4), generator=torch.Generator().manual_seed(0), dtype=dtype)
    x_0 = orc.sample(x_T, steps=steps, order=order, skip_type="logSNR", lower_order_final=False)
    assert len(orc.record) == steps
    tT, t0 = torch.tensor([1.], dtype=dtype), torch.tensor([1e-3], dtype=dtype)
    aT, sT, a0, s0 = ns.marginal_alpha(tT), ns.marginal_std(tT), ns.marginal_alpha(t0), ns.marginal_std(t0)
    exact = a0 * MU + torch.sqrt(a0 ** 2 * SD ** 2 + s0 ** 2) / torch.sqrt(aT ** 2 * SD ** 2 + sT ** 2) * (x_T - aT * MU)
    return float((x_0 - exact).abs().max())


def test_observed_order_on_gaussian_data():
    errs = {o: [_gaussian_error(S, o) for S in (10, 20, 40)] for o in (1, 2, 3)}
    rate = lambda e: [math.log2(e[i] / e[i + 1]) for i in range(2)]
    print({o: (["%.2f" % r for r in rate(e)], "%.2e" % e[-1]) for o, e in errs.items()})
    assert all(abs(r - 1.) <= 0.5 for r in rate(errs[1])), errs[1]
    assert all(abs(r - 2.) <= 0.5 for r in rate(errs[2])), errs[2]
    # the first-order start can cap the global order at 2, so order 3 is asked for at least 1.5
    assert all(r >= 1.5 for r in rate(errs[3])) and errs[3][-1] <= errs[2][-1], errs[3]


# ---- the host scalars, applied with the kernel's fp32 formulas, give the restatement's bits -------------------------------
def _toy_eps(x, t_input, c):
    return 0.3 * x * torch.sin(t_input.float() * 0.01).view(-1, 1, 1, 1) + 0.1 * torch.cos(x) + c.mean(dim=(1, 2)).view(-1, 1, 1, 1)


def _kernel_formula(x, e, order, coef, m1, m2):
    """sdb_dpm_solver_step as include/sdb200.h states it, in eager fp32 (python floats enter as fp32 scalars)."""
    sigma_s, alpha_s, c_x, c_0, c_1, c_2, inv_r0, inv_r1, c_r, c_d2 = coef
    m0 = (x - sigma_s * e) / alpha_s
    xn = c_x * x - c_0 * m0
    if order == 2:
        xn = xn - c_1 * (inv_r0 * (m0 - m1))
    elif order == 3:
        d10, d11 = inv_r0 * (m0 - m1), inv_r1 * (m1 - m2)
        xn = xn + c_1 * (d10 + c_r * (d10 - d11)) - c_2 * (c_d2 * (d10 - d11))
    return xn, m0


@pytest.mark.parametrize("steps,order,skip_type", [(2, 2, "time_uniform"), (3, 3, "time_uniform"), (5, 3, "logSNR"),
                                                   (14, 2, "time_quadratic"), (15, 3, "time_uniform"), (20, 2, "logSNR"),
                                                   (20, 1, "time_uniform")])
def test_host_scalars_reproduce_the_restatement(steps, order, skip_type):
    from sdb200.dpm_solver import DPM_Solver
    c = torch.randn((2, 7, 16), generator=torch.Generator().manual_seed(1))
    x_T = torch.randn((2, 4, 8, 8), generator=torch.Generator().manual_seed(2))
    orc = DPMSolverOracle(_toy_eps, AC, torch.float32, condition=c)
    want = orc.sample(x_T, steps=steps, order=order, skip_type=skip_type)
    solver = _solver()
    ts = solver.get_time_steps(skip_type, 1., 1e-3, steps)
    orders = DPM_Solver.step_orders(steps, order)
    x, hist = x_T, []
    for k in range(1, steps + 1):
        p = orders[k - 1]
        t_prev = [ts[i].reshape(1) for i in range(max(k - order, 0), k)]
        coef = solver.update_coefficients(t_prev, ts[k].reshape(1), p)
        t_in = torch.full((2,), float((ts[k - 1] - 1. / 1000) * 1000.))
        assert float(t_in[0]) == orc.record[k - 1][1]
        x, m0 = _kernel_formula(x, _toy_eps(x, t_in, c), p, coef, hist[-1] if p >= 2 else None, hist[-2] if p >= 3 else None)
        hist = (hist + [m0])[-2:]
    assert torch.equal(x, want)


# ---- interface --------------------------------------------------------------------------------------------------------------
def test_reference_signatures_and_no_ddim_methods():
    from sdb200.ddim import DDIMSampler
    from sdb200.dpm_solver import DPM_Solver, DPMSolverSampler
    names = lambda f: list(inspect.signature(f).parameters)
    assert names(DPMSolverSampler.sample) == names(DDIMSampler.sample)
    assert names(DPM_Solver.sample)[:9] == ["self", "x", "steps", "t_start", "t_end", "order", "skip_type", "method",
                                            "lower_order_final"]
    s = DPMSolverSampler(R.ModelShim(lambda x, t, c: x, AC))
    for name in ("ddim_sampling", "p_sample_ddim", "make_schedule", "stochastic_encode", "decode", "plms_sampling"):
        assert not hasattr(s, name), name
    assert s.alphas_cumprod.device.type == "cpu" and s.alphas_cumprod.dtype == torch.float32


def test_txt2img_signature():
    from sdb200.pipeline import LatentDiffusion
    p = inspect.signature(LatentDiffusion.txt2img).parameters
    assert "dpm_solver" in p and p["dpm_solver"].default is False and p["plms"].default is False


def test_unsupported_options_raise():
    from sdb200.dpm_solver import DPM_Solver, model_wrapper
    ns = _ns()
    for kw in (dict(model_type="x_start"), dict(model_type="v"), dict(model_type="score"), dict(guidance_type="classifier")):
        with pytest.raises(NotImplementedError):
            model_wrapper(None, ns, **kw)
    with pytest.raises(ValueError):
        model_wrapper(None, ns, guidance_type="cfg")
    with pytest.raises(NotImplementedError, match="predict_x0"):
        DPM_Solver(None, ns, predict_x0=False)
    with pytest.raises(NotImplementedError, match="thresholding"):
        DPM_Solver(None, ns, thresholding=True)
    solver, x = _solver(), torch.zeros(1, 4, 8, 8)
    for kw in (dict(method="singlestep"), dict(method="singlestep_fixed"), dict(method="adaptive"),
               dict(solver_type="taylor")):
        with pytest.raises(NotImplementedError):
            solver.sample(x, steps=10, **kw)
    with pytest.raises(ValueError):
        solver.sample(x, steps=10, solver_type="heun")
    with pytest.raises(ValueError):
        solver.sample(x, steps=10, skip_type="karras")
    with pytest.raises(AssertionError):                  # the reference's `assert steps >= order`
        solver.sample(x, steps=2, order=3)


# ---- sdb_dpm_solver_step host checks ----------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from sdb200 import _lib
    return _lib.load()


def test_dpm_solver_step_no_cpu_fallback(lib):
    from sdb200 import _lib, ops
    z = torch.zeros(4)
    with pytest.raises(_lib.SdbError):
        ops.dpm_solver_step(z, z, 1, [1.0] * 10)


# fake device addresses, 4 KB apart: never dereferenced, the checks reject the call first
X, E, U, M1, M2, XN, M0 = (0x100000 + 0x1000 * k for k in range(7))
N = 16


def _call(lib, x=X, e=E, u=None, m1=M1, m2=M2, order=3, xn=XN, m0=M0, n=N):
    return lib.sdb_dpm_solver_step(x, e, u, 7.5, 0.5, 0.8, m1, m2, order, 0.9, 0.1, 0.05, 0.02, 1.1, 0.9, 0.4, 0.6, xn, m0, n,
                                   None)


@pytest.mark.parametrize("case", [
    dict(x=None), dict(e=None), dict(n=0), dict(n=-4),                                # null inputs, empty problem
    dict(order=0), dict(order=4),                                                    # order outside 1..3
    dict(order=2, m1=None), dict(order=3, m1=None), dict(order=3, m2=None),          # history the order reads
    dict(xn=None, m0=None),                                                          # no output
    dict(xn=X), dict(m0=E), dict(xn=U, u=U), dict(m0=M1), dict(xn=M2),               # output == input
    dict(order=2, xn=M1),
    dict(xn=X + 4 * (N - 1)), dict(m0=E - 4 * (N - 1)),                              # output overlaps an input
    dict(m0=XN), dict(m0=XN + 8),                                                    # the two outputs overlap
])
def test_dpm_solver_step_host_checks(lib, case):
    assert _call(lib, **case) == -1, case
    assert lib.sdb_last_error_string().startswith(b"dpm_solver_step: "), case   # rejected by a check, not by a failed launch

