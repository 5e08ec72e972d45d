"""GPU: PLMSSampler (CompVis ldm/models/diffusion/plms.py) and its fused update kernel sdb_plms_step, against an eager fp32
CPU restatement of the reference's p_sample_plms / plms_sampling run on the same eps and the same random draws."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from gpu_util import randn, rel
from oracle import restate as R
from oracle import weights as W
from oracle.golden import load_golden

pytestmark = pytest.mark.gpu

EPS_TOL = {"fp32": 1e-5, "bf16": 1e-2}           # tests/test_gpu_models.py


def _gpu_randn(shape, repeat=False):
    """noise_like (ldm/modules/diffusionmodules/util.py) drawn on the GPU, copied to the host."""
    if repeat:
        return torch.randn((1, *shape[1:]), device="cuda").repeat(shape[0], *((1,) * (len(shape) - 1))).cpu()
    return torch.randn(shape, device="cuda").cpu()


def plms_combine(e_t, old_eps, e_t_next=None):
    """The multistep eps of p_sample_plms, as the reference writes each expression."""
    if len(old_eps) == 0:
        return (e_t + e_t_next) / 2
    if len(old_eps) == 1:
        return (3 * e_t - old_eps[-1]) / 2
    if len(old_eps) == 2:
        return (23 * e_t - 16 * old_eps[-1] + 5 * old_eps[-2]) / 12
    return (55 * e_t - 59 * old_eps[-1] + 37 * old_eps[-2] - 9 * old_eps[-3]) / 24


class PLMSOracle(R.DDIMOracle):
    """Eager fp32 restatement of PLMSSampler (plms.py: make_schedule's eta check, plms_sampling, p_sample_plms with
    get_model_output and get_x_prev_and_pred_x0), on R.DDIMOracle's schedule and coefficients.  CPU tensors; every random
    draw (noise_like on every get_x_prev_and_pred_x0 call, the dropout masks, q_sample's rand_like for the inpainting blend)
    is made on the GPU in the reference's order and copied over, so the sampler under test sees the same draws.
    It is written from the reference's formulas and is not pinned to a checkout of plms.py: none is available to
    oracle/make_golden.py.  `record` receives (x, t, eps) of every model evaluation without guidance."""

    def __init__(self, model, quantize=None):
        super().__init__(model)
        self.quantize = quantize
        self.record = []
        self.pred_x0s = []

    def make_schedule(self, ddim_num_steps, ddim_discretize="uniform", ddim_eta=0.):
        if ddim_eta != 0:
            raise ValueError('ddim_eta must be 0 for PLMS')
        super().make_schedule(ddim_num_steps, ddim_discretize, ddim_eta)

    def coefficients(self, index, b=1, use_original_steps=False):
        if not use_original_steps:
            return super().coefficients(index, b)
        m = self.model
        return tuple(torch.full((b, 1, 1, 1), tab[index]) for tab in (
            m.alphas_cumprod, m.alphas_cumprod_prev, m.ddim_sigmas_for_original_num_steps, m.sqrt_one_minus_alphas_cumprod))

    def model_output(self, x, t, c, scale=1., uc=None, score_corrector=None, corrector_kwargs=None):
        if uc is None or scale == 1.:
            e = self.model.apply_model(x, t, c)
            self.record.append((x, int(t[0]), e))
        else:
            x_in, t_in = torch.cat([x] * 2), torch.cat([t] * 2)
            if isinstance(c, dict):
                c_in = {k: [torch.cat([uc[k][i], c[k][i]]) for i in range(len(c[k]))] for k in c}
            else:
                c_in = torch.cat([uc, c])
            e_u, e_c = self.model.apply_model(x_in, t_in, c_in).chunk(2)
            e = e_u + scale * (e_c - e_u)
        if score_corrector is not None:
            e = score_corrector.modify_score(self.model, e, x, t, c, **corrector_kwargs)
        return e

    def x_prev_and_pred_x0(self, x, e_t, index, use_original_steps=False, quantize_denoised=False, temperature=1.,
                           noise_dropout=0., repeat_noise=False):
        a_t, a_prev, sigma_t, s1m = self.coefficients(index, x.shape[0], use_original_steps)
        pred_x0 = (x - s1m * e_t) / a_t.sqrt()
        if quantize_denoised:
            pred_x0 = self.quantize(pred_x0)[0]
        dir_xt = (1. - a_prev - sigma_t ** 2).sqrt() * e_t
        noise = sigma_t * _gpu_randn(x.shape, repeat_noise) * temperature
        if noise_dropout > 0.:
            noise = F.dropout(noise.cuda(), p=noise_dropout).cpu()
        return a_prev.sqrt() * pred_x0 + dir_xt + noise, pred_x0

    def p_sample_plms(self, x, c, t, index, old_eps, t_next, use_original_steps=False, quantize_denoised=False,
                      temperature=1., noise_dropout=0., repeat_noise=False, score_corrector=None, corrector_kwargs=None,
                      unconditional_guidance_scale=1., unconditional_conditioning=None):
        out = lambda x_, t_: self.model_output(x_, t_, c, unconditional_guidance_scale, unconditional_conditioning,
                                               score_corrector, corrector_kwargs)
        upd = lambda e: self.x_prev_and_pred_x0(x, e, index, use_original_steps, quantize_denoised, temperature, noise_dropout,
                                                repeat_noise)
        e_t = out(x, t)
        e_t_next = None
        if len(old_eps) == 0:
            x_prev, _ = upd(e_t)
            e_t_next = out(x_prev, t_next)
        x_prev, pred_x0 = upd(plms_combine(e_t, old_eps, e_t_next))
        return x_prev, pred_x0, e_t

    def _blend(self, x0, ts, mask, img):
        u = torch.rand(x0.shape, device="cuda").cpu()          # q_sample's torch.rand_like, as the reference writes it
        return self.model.q_sample(x0, ts, noise=u) * mask + (1. - mask) * img

    def plms_sampling(self, cond, x_T, ddim_use_original_steps=False, timesteps=None, log_every_t=100, mask=None, x0=None,
                      callback=None, img_callback=None, **kw):
        b = x_T.shape[0]
        if timesteps is None:
            timesteps = self.ddpm_num_timesteps if ddim_use_original_steps else self.ddim_timesteps
        elif not ddim_use_original_steps:
            subset_end = int(min(timesteps / self.ddim_timesteps.shape[0], 1) * self.ddim_timesteps.shape[0]) - 1
            timesteps = self.ddim_timesteps[:subset_end]
        img = x_T
        inter = {'x_inter': [img], 'pred_x0': [img]}
        time_range = list(reversed(range(0, timesteps))) if ddim_use_original_steps else np.flip(timesteps)
        total_steps = timesteps if ddim_use_original_steps else timesteps.shape[0]
        old_eps = []
        for i, step in enumerate(time_range):
            index = total_steps - i - 1
            ts = torch.full((b,), int(step), dtype=torch.long)
            ts_next = torch.full((b,), int(time_range[min(i + 1, len(time_range) - 1)]), dtype=torch.long)
            if mask is not None:
                img = self._blend(x0, ts, mask, img)
            img, pred_x0, e_t = self.p_sample_plms(img, cond, ts, index, old_eps, ts_next,
                                                   use_original_steps=ddim_use_original_steps, **kw)
            old_eps.append(e_t)
            if len(old_eps) >= 4:
                old_eps.pop(0)
            self.pred_x0s.append(pred_x0)
            if callback:
                callback(i)
            if img_callback:
                img_callback(pred_x0, i)
            if index % log_every_t == 0 or index == total_steps - 1:
                inter['x_inter'].append(img)
                inter['pred_x0'].append(pred_x0)
        return img, inter

    def sample(self, S, x_T, conditioning=None, quantize_x0=False, **kw):
        self.make_schedule(S)
        return self.plms_sampling(conditioning, x_T, quantize_denoised=quantize_x0, **kw)


# ---- toy models -----------------------------------------------------------------------------------------------------------
def _toy_hybrid(xc, t, ctx):
    from oracle.make_golden import toy_model_fn
    return toy_model_fn(xc[:, :4], t, ctx) + 0.05 * xc[:, 4:].mean(dim=1, keepdim=True)


class _ToyUNet(torch.nn.Module):
    """oracle.make_golden.toy_model_fn (hybrid: plus the mean of the concatenated channels) evaluated on the host, as the
    oracle evaluates it, result copied to the GPU."""

    def __init__(self, hybrid=False):
        super().__init__()
        self.hybrid = hybrid

    def forward(self, x, t, context=None):
        from oracle.make_golden import toy_model_fn
        fn = _toy_hybrid if self.hybrid else toy_model_fn
        return fn(x.cpu(), t.cpu(), None if context is None else context.cpu()).cuda()


class _Quantizer:
    @staticmethod
    def quantize(p):
        return torch.round(p * 4) / 4, None, None


class _Corrector:
    @staticmethod
    def modify_score(model, e, x, t, c, k=1.0):
        return e * k + 0.01 * x


def _toy_ld(hybrid=False):
    from sdb200.pipeline import LatentDiffusion
    ld = LatentDiffusion(first_stage_config=False, unet=_ToyUNet(hybrid), conditioning_key="hybrid" if hybrid else "crossattn").cuda()
    ld.first_stage_model = _Quantizer()
    # read by the use_original_steps branch, which takes sigma from the model as the reference does (eta = 0: zeros)
    ld.ddim_sigmas_for_original_num_steps = torch.zeros(1000, device="cuda")
    return ld


def _toy_oracle(hybrid=False):
    from oracle.make_golden import toy_model_fn
    if hybrid:
        fn = lambda x, t, c: _toy_hybrid(torch.cat([x] + c["c_concat"], 1), t, torch.cat(c["c_crossattn"], 1))
    else:
        fn = toy_model_fn
    shim = R.ModelShim(fn, R.sd_alphas_cumprod())
    shim.sqrt_one_minus_alphas_cumprod = torch.tensor(np.sqrt(1. - shim._ac64), dtype=torch.float32)
    shim.ddim_sigmas_for_original_num_steps = torch.zeros(1000)
    return PLMSOracle(shim, quantize=_Quantizer.quantize)


def _count_calls(ld):
    calls = []
    apply = ld.apply_model
    ld.apply_model = lambda x_, t_, c_, return_ids=False: calls.append(x_.shape[0]) or apply(x_, t_, c_)
    return calls


def _to(c, dev):
    if c is None:
        return None
    if isinstance(c, dict):
        return {k: [v.to(dev) for v in vs] for k, vs in c.items()}
    return c.to(dev)


# ---- 1. the kernel --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("per_sample", [(4, 8, 8), (3, 7, 5)])       # VEC = 4 and VEC = 1
def test_plms_step_kernel_bit_exact(cuda, per_sample):
    from sdb200 import ops
    B = 3
    x, e, eu = randn(B, *per_sample, seed=1), randn(B, *per_sample, seed=2, scale=1.5), randn(B, *per_sample, seed=3)
    olds = [randn(B, *per_sample, seed=4 + k, scale=1.2) for k in range(3)]
    noise = randn(B, *per_sample, seed=8)
    xc, ec, uc, nc = x.cpu(), e.cpu(), eu.cpu(), noise.cpu()
    oc = [o.cpu() for o in olds]
    # the derived coefficients of a real step (index 30 of PLMS-50), and a nonzero sigma for the noise cases
    from sdb200.plms import PLMSSampler
    smp = PLMSSampler(R.ModelShim(lambda *a: None, R.sd_alphas_cumprod()))
    smp.make_schedule(50, verbose=False)
    sqrt_at, sqrt_aprev, dir_coef, _, s1m = smp.derived_coefficients(30)
    full = lambda v: torch.full((1, 1, 1, 1), v)
    n_cases = 0
    for order in range(5):
        e_old = (oc[0],) if order == 0 else tuple(oc[:max(order - 1, 0)])
        for cfg in (None, 7.5):
            for nz in (None, noise):
                for temp in (1.0, 0.7):
                    sigma = 0.0 if nz is None else 0.25
                    e_comb = ec if cfg is None else uc + cfg * (ec - uc)
                    if order == 0:
                        e_p = (e_old[0] + e_comb) / 2
                    elif order == 1:
                        e_p = e_comb
                    else:
                        e_p = plms_combine(e_comb, list(reversed(e_old)))
                    p0 = (xc - full(s1m) * e_p) / full(sqrt_at)
                    xp = full(sqrt_aprev) * p0 + full(dir_coef) * e_p
                    if nz is not None:
                        xp = xp + full(sigma) * nc * temp
                    got = ops.plms_step(x, e, order, sqrt_at, sqrt_aprev, dir_coef, sigma, s1m,
                                        e_uncond=None if cfg is None else eu, cfg_scale=cfg or 1.0,
                                        e_old=[o.cuda() for o in e_old], noise=nz, temperature=temp,
                                        want_e=True, want_e_prime=True)
                    for name, g, w in zip(("e", "e'", "pred_x0", "x_prev"), got, (e_comb, e_p, p0, xp)):
                        assert torch.equal(g.cpu(), w), (order, cfg, nz is None, temp, name)
                    n_cases += 1
    assert n_cases == 40
    # outputs are optional; the ones returned do not depend on which others are requested
    e_c, e_p, p0, xp = ops.plms_step(x, e, 4, sqrt_at, sqrt_aprev, dir_coef, 0.0, s1m, e_uncond=eu, cfg_scale=7.5, e_old=olds,
                                     want_e=True, want_pred_x0=False)
    assert e_p is None and p0 is None
    full_out = ops.plms_step(x, e, 4, sqrt_at, sqrt_aprev, dir_coef, 0.0, s1m, e_uncond=eu, cfg_scale=7.5, e_old=olds,
                             want_e=True, want_e_prime=True)
    assert torch.equal(e_c, full_out[0]) and torch.equal(xp, full_out[3])


# ---- 2. the loop with a stub eps-model -------------------------------------------------------------------------------------
# S = 3 takes the 'quad' discretization: 'uniform' makes the step values 1, 334, 667, 1000, and 1000 is out of range (the
# reference's make_ddim_timesteps fails there too)
LOOP_CASES = {
    "S1": dict(S=1), "S2": dict(S=2), "S3": dict(S=3, discretize="quad"), "S4": dict(S=4), "S5": dict(S=5), "S20": dict(S=20),
    "log_every_t": dict(S=20, log_every_t=3),
    "cfg_tensor": dict(S=6, cfg=True),
    "cfg_hybrid": dict(S=6, cfg=True, hybrid=True),
    "mask": dict(S=6, mask=True),
    "quantize": dict(S=6, quantize_x0=True),
    "quantize_cfg": dict(S=5, quantize_x0=True, cfg=True),
    "noise_dropout": dict(S=6, noise_dropout=0.25, temperature=0.8),
    "score_corrector": dict(S=6, score_corrector=True, cfg=True),
    "timesteps_subset": dict(S=20, timesteps=9),
    "original_steps": dict(S=10, original=True, timesteps=30),
}


@pytest.mark.parametrize("case", list(LOOP_CASES))
def test_plms_loop_bit_exact(cuda, case):
    from sdb200.plms import PLMSSampler
    kw = dict(LOOP_CASES[case])
    S, hybrid, cfg = kw.pop("S"), kw.pop("hybrid", False), kw.pop("cfg", False)
    ld, orc = _toy_ld(hybrid), _toy_oracle(hybrid)
    B = 2
    x_T = W.seeded_randn((B, 4, 8, 8), 61)
    if hybrid:
        cc = torch.cat([(W.seeded_randn((B, 1, 8, 8), 62) > 0).float(), W.seeded_randn((B, 4, 8, 8), 63)], 1)
        c = {"c_concat": [cc], "c_crossattn": [W.seeded_randn((B, 7, 64), 64)]}
        uc = {"c_concat": [cc], "c_crossattn": [W.seeded_randn((B, 7, 64), 65)]}
    else:
        c, uc = W.seeded_randn((B, 7, 64), 64), W.seeded_randn((B, 7, 64), 65)
    common = {}
    if cfg:
        common.update(unconditional_guidance_scale=7.5)
    if kw.pop("score_corrector", False):
        common.update(score_corrector=_Corrector(), corrector_kwargs=dict(k=0.9))
    for k in ("temperature", "noise_dropout", "log_every_t"):
        if k in kw:
            common[k] = kw.pop(k)
    mask = x0 = None
    if kw.pop("mask", False):
        x0 = W.seeded_randn((B, 4, 8, 8), 66) * 0.5
        mask = (W.seeded_randn((B, 1, 8, 8), 67) > 0).float()
    quantize = kw.pop("quantize_x0", False)
    original, timesteps = kw.pop("original", False), kw.pop("timesteps", None)
    discretize = kw.pop("discretize", None)
    assert not kw
    seq, seq_o = [], []
    cbs = lambda s: dict(callback=lambda i: s.append(("cb", i)), img_callback=lambda p, i: s.append(("img", i, p.cpu())))

    smp = PLMSSampler(ld)
    calls = _count_calls(ld)
    torch.manual_seed(70)
    if timesteps is None and discretize is None:
        z, inter = smp.sample(S, B, (4, 8, 8), conditioning=_to(c, "cuda"), x_T=x_T.cuda(), verbose=False,
                              unconditional_conditioning=_to(uc, "cuda") if cfg else None, quantize_x0=quantize,
                              mask=_to(mask, "cuda"), x0=_to(x0, "cuda"), **common, **cbs(seq))
    else:
        smp.make_schedule(S, ddim_discretize=discretize or "uniform", verbose=False)
        z, inter = smp.plms_sampling(_to(c, "cuda"), (B, 4, 8, 8), x_T=x_T.cuda(), ddim_use_original_steps=original,
                                     timesteps=timesteps, unconditional_conditioning=_to(uc, "cuda") if cfg else None,
                                     quantize_denoised=quantize, mask=_to(mask, "cuda"), x0=_to(x0, "cuda"), **common,
                                     **cbs(seq))
    after = torch.randn(3, device="cuda")
    torch.manual_seed(70)
    with torch.no_grad():
        orc.make_schedule(S, ddim_discretize=discretize or "uniform")
        zo, inter_o = orc.plms_sampling(c, x_T, ddim_use_original_steps=original, timesteps=timesteps,
                                        unconditional_conditioning=uc if cfg else None, quantize_denoised=quantize,
                                        mask=mask, x0=x0, **common, **cbs(seq_o))
    assert torch.equal(after, torch.randn(3, device="cuda")), case               # same draws, same order
    n_steps = len(orc.pred_x0s)
    assert calls == [2 * B if cfg else B] * (n_steps + 1), case                  # S + 1 model evaluations
    assert torch.equal(z.cpu(), zo), case
    for key in ("x_inter", "pred_x0"):
        assert len(inter[key]) == len(inter_o[key]), (case, key)
        for a, b in zip(inter[key], inter_o[key]):
            assert torch.equal(a.cpu(), b), (case, key)
    assert [s[:2] for s in seq] == [s[:2] for s in seq_o] == [(k, i) for i in range(n_steps) for k in ("cb", "img")]
    assert all(torch.equal(a[2], b[2]) for a, b in zip(seq, seq_o) if a[0] == "img"), case
    if case == "original_steps":
        assert n_steps == 30
    if case == "timesteps_subset":
        assert n_steps == 8
    if case.startswith("S"):
        assert n_steps == S


def test_plms_rng_consumption(cuda):
    """S + 1 noise draws (two in the first step), and none with consume_rng_like_reference = False (same latent)."""
    from sdb200.plms import PLMSSampler
    ld = _toy_ld()
    B, S, shape = 2, 5, (2, 4, 8, 8)             # DDIM-5 on 1000 steps: exactly 5 step values
    x_T, c = W.seeded_randn(shape, 71).cuda(), W.seeded_randn((B, 7, 64), 72).cuda()
    torch.manual_seed(5)
    z, _ = PLMSSampler(ld).sample(S, B, shape[1:], conditioning=c, x_T=x_T, verbose=False)
    after = torch.randn(4, device="cuda")
    torch.manual_seed(5)
    for _ in range(S + 1):
        torch.randn(shape, device="cuda")
    assert torch.equal(after, torch.randn(4, device="cuda"))
    smp = PLMSSampler(ld)
    smp.consume_rng_like_reference = False
    torch.manual_seed(5)
    z2, _ = smp.sample(S, B, shape[1:], conditioning=c, x_T=x_T, verbose=False)
    after2 = torch.randn(4, device="cuda")
    torch.manual_seed(5)
    assert torch.equal(after2, torch.randn(4, device="cuda")) and torch.equal(z, z2)


# ---- 3. no host synchronisation inside the loop -----------------------------------------------------------------------------
class _GpuStub(torch.nn.Module):
    def forward(self, x, t, context=None):
        return 0.3 * x + 0.05 * context.mean(dim=(1, 2)).view(-1, 1, 1, 1)


@pytest.mark.parametrize("cfg", [False, True])
def test_plms_loop_has_no_host_sync(cuda, cfg):
    from sdb200.pipeline import LatentDiffusion
    from sdb200.plms import PLMSSampler
    ld = LatentDiffusion(first_stage_config=False, unet=_GpuStub()).cuda()
    x_T, c, uc = randn(2, 4, 8, 8, seed=9), randn(2, 7, 64, seed=10), randn(2, 7, 64, seed=11)
    kw = dict(unconditional_guidance_scale=7.5, unconditional_conditioning=uc) if cfg else {}
    smp = PLMSSampler(ld)
    smp.make_schedule(20, verbose=False)                             # host-side schedule tables (reads the model's buffers)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        z, _ = smp.plms_sampling(c, (2, 4, 8, 8), x_T=x_T, **kw)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert torch.isfinite(z).all()


# ---- 4. tiny nets end to end ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_tiny_plms_pipeline(cuda, mode):
    from sdb200.pipeline import LatentDiffusion
    from sdb200.plms import PLMSSampler
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
    ctx = W.seeded_randn((B, 7, 64), 76)
    z, inter = PLMSSampler(ld).sample(S, B, (4, 8, 8), conditioning=ctx.cuda(), x_T=x_T.cuda(), verbose=False)
    orc = PLMSOracle(R.ModelShim(lambda x, t, c: R.unet_forward(sdu, gu["cfg"], x, t, c), R.sd_alphas_cumprod()))
    with torch.no_grad():
        z_ref, inter_ref = orc.sample(S, x_T, conditioning=ctx)
        img_ref = R.autoencoder_decode(sdv, gv["ddconfig"], z_ref / 0.18215)
    img = ld.decode_first_stage(z)
    assert len(orc.record) == S + 1 and len(inter["x_inter"]) == len(inter_ref["x_inter"])
    per_step = [rel(ld.apply_model(x_t.cuda(), torch.full((B,), t, device="cuda"), ctx.cuda()), e_t) for x_t, t, e_t in orc.record]
    worst, median = max(per_step), sorted(per_step)[len(per_step) // 2]
    e_z = rel(z, z_ref)
    psnr = R.psnr_255(img.cpu(), img_ref)
    print("tiny PLMS-%d %s: latent rel-L2 %.3e, PSNR %.1f dB, teacher-forced eps rel-L2 worst %.3e median %.3e" % (
        S, mode, e_z, psnr, worst, median))
    if mode == "fp32":
        assert worst <= EPS_TOL[mode]
    else:
        assert median <= EPS_TOL[mode]
    assert e_z <= (1e-4 if mode == "fp32" else 3e-2)
    assert psnr >= 40.0
    # txt2img(plms=True) is PLMSSampler.sample followed by decode_first_stage, bit for bit
    z2, img2 = ld.txt2img(ctx.cuda(), B, ddim_steps=S, shape=(4, 8, 8), x_T=x_T.cuda(), plms=True)
    assert torch.equal(z2, z) and torch.equal(img2, img)
    with pytest.raises(ValueError):
        ld.txt2img(ctx.cuda(), B, ddim_steps=S, shape=(4, 8, 8), x_T=x_T.cuda(), eta=0.5, plms=True)


# ---- 5. SD size: the first step and a fourth-order step ---------------------------------------------------------------------
def test_sd_unet_plms_steps_bit_exact(cuda):
    from sdb200.pipeline import LatentDiffusion
    from sdb200.plms import PLMSSampler
    g = load_golden("unet_sd.pt")
    ld = LatentDiffusion(unet_config=g["cfg"], first_stage_config=False, compute_mode="bf16")
    ld.model.diffusion_model.load_state_dict(W.make_state_dict(g["key_shapes"], g["seed"]))
    ld = ld.cuda()
    B, S = 2, 50
    x = W.seeded_randn((B, 4, 64, 64), 77).cuda()
    ctx = W.seeded_randn((B, 77, 768), 78).cuda()
    seen = []
    apply = ld.apply_model
    ld.apply_model = lambda x_, t_, c_, return_ids=False: seen.append((x_.clone(), apply(x_, t_, c_))) or seen[-1][1]
    smp = PLMSSampler(ld)
    smp.make_schedule(S, verbose=False)
    orc = PLMSOracle(R.ModelShim(None, R.sd_alphas_cumprod()))
    orc.make_schedule(S)
    ts = torch.full((B,), int(smp.ddim_timesteps[-1]), device="cuda", dtype=torch.long)
    ts_next = torch.full((B,), int(smp.ddim_timesteps[-2]), device="cuda", dtype=torch.long)
    # first step: DDIM with e_t, the second evaluation at that x_prev and t_next, the update with (e_t + e_t_next) / 2
    xp, p0, e_t = smp.p_sample_plms(x, ctx, ts, S - 1, old_eps=[], t_next=ts_next)
    assert len(seen) == 2
    (x1, e1), (x2, e2) = seen
    e1c, e2c = e1.float().cpu(), e2.float().cpu()
    assert torch.isfinite(e1c).all() and float(e1c.abs().max()) > 0.1
    want_mid, _ = orc.x_prev_and_pred_x0(x.cpu(), e1c, S - 1)
    assert torch.equal(x2.cpu(), want_mid)                                   # the second call saw the restated x_prev
    want_xp, want_p0 = orc.x_prev_and_pred_x0(x.cpu(), plms_combine(e1c, [], e2c), S - 1)
    assert torch.equal(xp.cpu(), want_xp) and torch.equal(p0.cpu(), want_p0) and torch.equal(e_t.cpu(), e1c)
    # a fourth-order step with a seeded history
    old = [W.seeded_randn((B, 4, 64, 64), 79 + k).cuda() for k in range(3)]
    seen.clear()
    xp, p0, e_t = smp.p_sample_plms(x, ctx, ts_next, S - 2, old_eps=old, t_next=ts_next)
    (_, e3), = seen
    e3c = e3.float().cpu()
    want_xp, want_p0 = orc.x_prev_and_pred_x0(x.cpu(), plms_combine(e3c, [o.cpu() for o in old]), S - 2)
    assert torch.equal(xp.cpu(), want_xp) and torch.equal(p0.cpu(), want_p0) and torch.equal(e_t.cpu(), e3c)
