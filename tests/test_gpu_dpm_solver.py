"""GPU: the multistep DPM-Solver++ sampler (CompVis ldm/models/diffusion/dpm_solver/) and its fused update kernel
sdb_dpm_solver_step, against the eager fp32 CPU restatement in tests/dpm_oracle.py fed the same model outputs; and the
UNet at the fractional timesteps the solver feeds it."""
import pytest
import torch

from dpm_oracle import DPMSolverOracle
from gpu_util import randn, rel
from oracle import restate as R
from oracle import weights as W
from oracle.golden import load_golden
from test_gpu_plms import _count_calls, _GpuStub, _to, _toy_hybrid, _toy_ld

pytestmark = pytest.mark.gpu

EPS_TOL = {"fp32": 1e-5, "bf16": 1e-2}           # tests/test_gpu_models.py


def _toy_fn(hybrid):
    from oracle.make_golden import toy_model_fn
    if hybrid:
        return lambda x, t, c: _toy_hybrid(torch.cat([x] + c["c_concat"], 1), t, torch.cat(c["c_crossattn"], 1))
    return toy_model_fn


def _conds(B, hybrid):
    if hybrid:
        cc = torch.cat([(W.seeded_randn((B, 1, 8, 8), 62) > 0).float(), W.seeded_randn((B, 4, 8, 8), 63)], 1)
        return ({"c_concat": [cc], "c_crossattn": [W.seeded_randn((B, 7, 64), 64)]},
                {"c_concat": [cc], "c_crossattn": [W.seeded_randn((B, 7, 64), 65)]})
    return W.seeded_randn((B, 7, 64), 64), W.seeded_randn((B, 7, 64), 65)


class _CountSteps:
    def __init__(self, monkeypatch):
        from sdb200 import ops
        self.n, real = 0, ops.dpm_solver_step

        def spy(*a, **k):
            self.n += 1
            return real(*a, **k)
        monkeypatch.setattr(ops, "dpm_solver_step", spy)


# ---- 1. the kernel --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("per_sample", [(4, 8, 8), (3, 7, 5)])       # VEC = 4 and VEC = 1
def test_dpm_solver_step_kernel_bit_exact(cuda, per_sample):
    from sdb200 import ops
    from sdb200.dpm_solver import DPM_Solver, NoiseScheduleVP
    B = 3
    x, e, eu = randn(B, *per_sample, seed=1), randn(B, *per_sample, seed=2, scale=1.5), randn(B, *per_sample, seed=3)
    m1, m2 = randn(B, *per_sample, seed=4, scale=1.2), randn(B, *per_sample, seed=5, scale=1.2)
    xc, ec, uc, m1c, m2c = x.cpu(), e.cpu(), eu.cpu(), m1.cpu(), m2.cpu()
    solver = DPM_Solver(None, NoiseScheduleVP('discrete', alphas_cumprod=torch.tensor(R.sd_alphas_cumprod())))
    ts = solver.get_time_steps("time_uniform", 1., 1e-3, 20)
    full = lambda v: torch.full((1, 1, 1, 1), v)
    n_cases = 0
    for order in (1, 2, 3):
        # a real update of DPM-Solver-20: from t_9 to t_10 with the history at t_8, t_7
        coef = solver.update_coefficients([ts[i].reshape(1) for i in range(10 - order, 10)], ts[10].reshape(1), order)
        sigma_s, alpha_s, c_x, c_0, c_1, c_2, inv_r0, inv_r1, c_r, c_d2 = (full(v) for v in coef)
        for cfg in (None, 7.5):
            e_comb = ec if cfg is None else uc + cfg * (ec - uc)
            m0 = (xc - sigma_s * e_comb) / alpha_s
            if order == 1:
                want = c_x * xc - c_0 * m0
            elif order == 2:
                D1_0 = inv_r0 * (m0 - m1c)
                want = c_x * xc - c_0 * m0 - c_1 * D1_0
            else:
                D1_0, D1_1 = inv_r0 * (m0 - m1c), inv_r1 * (m1c - m2c)
                D1 = D1_0 + c_r * (D1_0 - D1_1)
                D2 = c_d2 * (D1_0 - D1_1)
                want = c_x * xc - c_0 * m0 + c_1 * D1 - c_2 * D2
            for want_m0 in (False, True):
                xn, m0_out = ops.dpm_solver_step(x, e, order, coef, e_uncond=None if cfg is None else eu, cfg_scale=cfg or 1.0,
                                                 m1=m1 if order >= 2 else None, m2=m2 if order >= 3 else None, want_m0=want_m0)
                assert torch.equal(xn.cpu(), want), (order, cfg, want_m0)
                assert (m0_out is None) != want_m0 and (not want_m0 or torch.equal(m0_out.cpu(), m0)), (order, cfg)
                n_cases += 1
    assert n_cases == 12
    # m0 alone; and history pointers the order does not read may be passed
    xn, m0_only = ops.dpm_solver_step(x, e, 1, coef, m1=m1, m2=m2, want_x_next=False)
    assert xn is None and torch.equal(m0_only.cpu(), (xc - full(coef[0]) * ec) / full(coef[1]))


# ---- 2. the loop with a stub eps-model --------------------------------------------------------------------------------------
LOOP_CASES = {"S%d_o%d" % (S, o): dict(S=S, order=o) for S in (2, 3, 5, 14, 15, 20) for o in (1, 2, 3) if S >= o}
LOOP_CASES.update({
    "logSNR_S5_o3": dict(S=5, order=3, skip_type="logSNR"), "logSNR_S20_o2": dict(S=20, order=2, skip_type="logSNR"),
    "quadratic_S5_o3": dict(S=5, order=3, skip_type="time_quadratic"),
    "quadratic_S20_o2": dict(S=20, order=2, skip_type="time_quadratic"),
    "no_lower_order_final_S10_o3": dict(S=10, order=3, lower_order_final=False),
    "cfg_tensor_S14_o3": dict(S=14, order=3, cfg=True), "cfg_hybrid_S6_o2": dict(S=6, order=2, cfg=True, hybrid=True),
})


@pytest.mark.parametrize("case", list(LOOP_CASES))
def test_dpm_solver_loop_bit_exact(cuda, case, monkeypatch):
    from sdb200.dpm_solver import DPM_Solver, DPMSolverSampler, model_wrapper
    kw = dict(LOOP_CASES[case])
    S, hybrid, cfg = kw.pop("S"), kw.pop("hybrid", False), kw.pop("cfg", False)
    ld = _toy_ld(hybrid)
    B = 2
    x_T = W.seeded_randn((B, 4, 8, 8), 61)
    c, uc = _conds(B, hybrid)
    scale = 7.5 if cfg else 1.
    ns = DPMSolverSampler(ld).noise_schedule
    model_fn = model_wrapper(ld, ns, model_type="noise", guidance_type="classifier-free", condition=_to(c, "cuda"),
                             unconditional_condition=_to(uc, "cuda") if cfg else None, guidance_scale=scale)
    calls, steps = _count_calls(ld), _CountSteps(monkeypatch)
    z = DPM_Solver(model_fn, ns).sample(x_T.cuda(), steps=S, **kw)
    orc = DPMSolverOracle(_toy_fn(hybrid), ld.alphas_cumprod.cpu(), condition=c, unconditional_condition=uc if cfg else None,
                          guidance_scale=scale)
    with torch.no_grad():
        zo = orc.sample(x_T, steps=S, **kw)
    assert calls == [2 * B if cfg else B] * S and steps.n == S, case          # S evaluations, one update kernel each
    assert [r[2] for r in orc.record] == calls
    assert torch.equal(z.cpu(), zo), (case, float((z.cpu() - zo).abs().max()))


@pytest.mark.parametrize("cfg,hybrid,given", [(False, False, True), (False, False, False), (True, False, False),
                                              (True, True, True)])
def test_dpm_solver_sampler_bit_exact(cuda, cfg, hybrid, given, monkeypatch):
    """DPMSolverSampler.sample: DPM-Solver++(2M), time_uniform, lower_order_final; x_T given or drawn on the device."""
    from sdb200.dpm_solver import DPMSolverSampler
    ld = _toy_ld(hybrid)
    B, S = 2, 10
    c, uc = _conds(B, hybrid)
    scale = 7.5 if cfg else 1.
    calls, steps = _count_calls(ld), _CountSteps(monkeypatch)
    torch.manual_seed(80)
    x_T = W.seeded_randn((B, 4, 8, 8), 61) if given else torch.randn((B, 4, 8, 8), device="cuda").cpu()
    torch.manual_seed(80)
    z, none = DPMSolverSampler(ld).sample(S, B, (4, 8, 8), conditioning=_to(c, "cuda"), x_T=x_T.cuda() if given else None,
                                          unconditional_guidance_scale=scale, unconditional_conditioning=_to(uc, "cuda"),
                                          eta=0.3, temperature=0.5, verbose=False)
    assert none is None and z.device.type == "cuda"
    orc = DPMSolverOracle(_toy_fn(hybrid), ld.alphas_cumprod.cpu(), condition=c, unconditional_condition=uc,
                          guidance_scale=scale)
    with torch.no_grad():
        zo = orc.sample(x_T, steps=S, order=2, skip_type="time_uniform", lower_order_final=True)
    assert calls == [2 * B if cfg else B] * S and steps.n == S
    assert torch.equal(z.cpu(), zo)


# ---- 3. no host synchronisation inside the loop -----------------------------------------------------------------------------
@pytest.mark.parametrize("cfg", [False, True])
def test_dpm_solver_loop_has_no_host_sync(cuda, cfg):
    from sdb200.dpm_solver import DPMSolverSampler
    from sdb200.pipeline import LatentDiffusion
    ld = LatentDiffusion(first_stage_config=False, unet=_GpuStub()).cuda()
    x_T, c, uc = randn(2, 4, 8, 8, seed=9), randn(2, 7, 64, seed=10), randn(2, 7, 64, seed=11)
    kw = dict(unconditional_guidance_scale=7.5, unconditional_conditioning=uc) if cfg else {}
    smp = DPMSolverSampler(ld)                     # the host copy of the schedule is made here
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        z, _ = smp.sample(20, 2, (4, 8, 8), conditioning=c, x_T=x_T, **kw)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert torch.isfinite(z).all()


# ---- 4. the UNet at fractional timesteps ----------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_unet_fractional_timesteps(cuda, mode):
    from sdb200.dpm_solver import DPM_Solver, NoiseScheduleVP
    from sdb200.openai_model import UNetModel
    g = load_golden("unet_tiny.pt")
    sd = W.make_state_dict(g["key_shapes"], g["seed"])
    net = UNetModel(**g["cfg"])
    net.load_state_dict(sd)
    net = net.cuda()
    net.compute_mode = mode
    ns = NoiseScheduleVP('discrete', alphas_cumprod=torch.tensor(R.sd_alphas_cumprod()))
    ts = DPM_Solver(None, ns).get_time_steps("time_uniform", 1., 1e-3, 20)
    t_in = (ts - 1e-3) * 1000.                                    # the sampler's model input times: 999, 949.05, ...
    picks = [float(t_in[i]) for i in (1, 2, 7, 19)]
    assert all(v != round(v) for v in picks)
    B = 2
    x = W.seeded_randn((B, 4, 8, 8), 90)
    ctx = W.seeded_randn((B, 7, 64), 91)
    for v in picks:
        t = torch.full((B,), v)
        want = R.unet_forward(sd, g["cfg"], x, t, ctx)
        net.use_cuda_graph = False
        eager = net(x.cuda(), t.cuda(), ctx.cuda())
        assert rel(eager, want) <= EPS_TOL[mode], (v, rel(eager, want))
        net.use_cuda_graph = True
        for _ in range(2):
            assert torch.equal(net(x.cuda(), t.cuda(), ctx.cuda()), eager), v
    # the fraction reaches the embedding: a timestep 0.25 away gives another output
    net.use_cuda_graph = False
    assert not torch.equal(net(x.cuda(), torch.full((B,), picks[0] + 0.25, device="cuda"), ctx.cuda()),
                           net(x.cuda(), torch.full((B,), picks[0], device="cuda"), ctx.cuda()))


# ---- 5. tiny nets end to end -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_tiny_dpm_solver_pipeline(cuda, mode):
    from sdb200.dpm_solver import DPMSolverSampler
    from sdb200.pipeline import LatentDiffusion
    gu, gv, ge = load_golden("unet_tiny.pt"), load_golden("vae_tiny.pt"), load_golden("vae_enc_tiny.pt")
    sdu = W.make_state_dict(gu["key_shapes"], gu["seed"])
    sdv = W.make_state_dict(gv["key_shapes"], gv["seed"])
    sdv.update(W.make_state_dict(ge["key_shapes"], ge["seed"]))
    ld = LatentDiffusion(unet_config=gu["cfg"], first_stage_config=gv["ddconfig"], compute_mode=mode)
    ld.model.diffusion_model.load_state_dict(sdu)
    ld.first_stage_model.load_state_dict(sdv, strict=True)
    ld = ld.cuda()
    B, S = 2, 10
    x_T = W.seeded_randn((B, 4, 8, 8), 75)
    ctx, uctx = W.seeded_randn((B, 7, 64), 76), W.seeded_randn((B, 7, 64), 77)
    z, _ = DPMSolverSampler(ld).sample(S, B, (4, 8, 8), conditioning=ctx.cuda(), x_T=x_T.cuda(), verbose=False,
                                       unconditional_guidance_scale=3.0, unconditional_conditioning=uctx.cuda())
    orc = DPMSolverOracle(lambda x, t, c: R.unet_forward(sdu, gu["cfg"], x, t, c), ld.alphas_cumprod.cpu(), condition=ctx,
                          unconditional_condition=uctx, guidance_scale=3.0)
    with torch.no_grad():
        z_ref = orc.sample(x_T, steps=S, order=2)
        img_ref = R.autoencoder_decode(sdv, gv["ddconfig"], z_ref / 0.18215)
    img = ld.decode_first_stage(z)
    assert len(orc.record) == S
    per_step = []
    for x_t, t_in, _ in orc.record:
        x2, t2 = torch.cat([x_t] * 2).cuda(), torch.full((2 * B,), t_in, device="cuda")
        e_u, e_c = ld.apply_model(x2, t2, torch.cat([uctx, ctx]).cuda()).chunk(2)
        want_u, want_c = R.unet_forward(sdu, gu["cfg"], torch.cat([x_t] * 2), t2.cpu(), torch.cat([uctx, ctx])).chunk(2)
        per_step += [rel(e_u, want_u), rel(e_c, want_c)]
    worst, median = max(per_step), sorted(per_step)[len(per_step) // 2]
    e_z = rel(z, z_ref)
    psnr = R.psnr_255(img.cpu(), img_ref)
    print("tiny DPM-Solver-%d %s: latent rel-L2 %.3e, PSNR %.1f dB, teacher-forced eps rel-L2 worst %.3e median %.3e" % (
        S, mode, e_z, psnr, worst, median))
    if mode == "fp32":
        assert worst <= EPS_TOL[mode]
    else:
        assert median <= EPS_TOL[mode]
    assert e_z <= (1e-4 if mode == "fp32" else 3e-2)
    assert psnr >= 40.0
    # txt2img(dpm_solver=True) is DPMSolverSampler.sample followed by decode_first_stage, bit for bit; dpm_solver wins over plms
    for plms in (False, True):
        z2, img2 = ld.txt2img(ctx.cuda(), B, ddim_steps=S, shape=(4, 8, 8), x_T=x_T.cuda(), unconditional_guidance_scale=3.0,
                              unconditional_conditioning=uctx.cuda(), dpm_solver=True, plms=plms)
        assert torch.equal(z2, z) and torch.equal(img2, img)


# ---- 6. SD size: a first-order and a second-order update ----------------------------------------------------------------------
def test_sd_unet_dpm_solver_steps_bit_exact(cuda):
    from sdb200.dpm_solver import DPM_Solver, DPMSolverSampler, model_wrapper
    from sdb200.pipeline import LatentDiffusion
    g = load_golden("unet_sd.pt")
    ld = LatentDiffusion(unet_config=g["cfg"], first_stage_config=False, compute_mode="bf16")
    ld.model.diffusion_model.load_state_dict(W.make_state_dict(g["key_shapes"], g["seed"]))
    ld = ld.cuda()
    B = 2
    x = W.seeded_randn((B, 4, 64, 64), 77)
    ctx, uctx = W.seeded_randn((B, 77, 768), 78), W.seeded_randn((B, 77, 768), 79)
    seen = []
    apply = ld.apply_model
    ld.apply_model = lambda x_, t_, c_, return_ids=False: seen.append((x_.cpu(), t_.cpu(), apply(x_, t_, c_))) or seen[-1][2]
    ns = DPMSolverSampler(ld).noise_schedule
    model_fn = model_wrapper(ld, ns, guidance_type="classifier-free", condition=ctx.cuda(), unconditional_condition=uctx.cuda(),
                             guidance_scale=7.5)
    # steps=2, order=2 without lower-order final steps: a first-order update, then a second-order one
    z = DPM_Solver(model_fn, ns).sample(x.cuda(), steps=2, order=2, lower_order_final=False)
    assert len(seen) == 2 and all(s[0].shape[0] == 2 * B for s in seen)
    outs = iter(seen)

    def replay(x_in, t_in, c_in):
        sx, st, e = next(outs)
        assert torch.equal(x_in, sx) and torch.equal(t_in, st)            # the restatement reached the same inputs
        return e.float().cpu()

    orc = DPMSolverOracle(replay, ld.alphas_cumprod.cpu(), condition=ctx, unconditional_condition=uctx, guidance_scale=7.5)
    e0 = seen[0][2].float().cpu()
    assert torch.isfinite(e0).all() and float(e0.abs().max()) > 0.1
    with torch.no_grad():
        zo = orc.sample(x, steps=2, order=2, lower_order_final=False)
    assert torch.equal(z.cpu(), zo)
