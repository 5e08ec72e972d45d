"""Drop-in `PLMSSampler` (reference: CompVis ldm/models/diffusion/plms.py, `scripts/txt2img.py --plms`): pseudo linear
multistep sampling whose per-step arithmetic (guidance combine, the multistep combine of the eps history and the DDIM
update) runs as ONE fused sm_100a kernel (sdb_plms_step).

Same constructor / method signatures, return values and duck-typed `model` interface as the reference.  The schedule,
its per-step coefficients, the model evaluation (2B classifier-free guidance calls, score corrector), the noise draws and
the inpainting blend are DDIMSampler's: PLMS is DDIM's update applied to a multistep eps.
"""
import torch

from . import ops
from .ddim import DDIMSampler, _f32_contiguous


class _NotInPLMS:
    """An inherited DDIMSampler method that CompVis's PLMSSampler does not have.  Reading it raises AttributeError, so it is
    hidden (`hasattr` is False) and a call says where to go instead."""

    def __set_name__(self, owner, name):
        self.name = name

    def __get__(self, obj, objtype=None):
        raise AttributeError("PLMSSampler has no %r (the reference's PLMS sampler offers only text-to-image sampling); "
                             "use DDIMSampler for it" % self.name)


class PLMSSampler(DDIMSampler):
    # img2img entry points and DDIM's own loop: not part of the reference's PLMSSampler
    stochastic_encode = _NotInPLMS()
    decode = _NotInPLMS()
    ddim_sampling = _NotInPLMS()
    p_sample_ddim = _NotInPLMS()

    def __init__(self, model, schedule="linear", **kwargs):
        super().__init__(model, schedule=schedule, **kwargs)

    def make_schedule(self, ddim_num_steps, ddim_discretize="uniform", ddim_eta=0., verbose=True):
        if ddim_eta != 0:
            raise ValueError('ddim_eta must be 0 for PLMS')
        super().make_schedule(ddim_num_steps, ddim_discretize=ddim_discretize, ddim_eta=ddim_eta, verbose=verbose)

    @torch.no_grad()
    def sample(self, S, batch_size, shape, conditioning=None, callback=None, normals_sequence=None, img_callback=None,
               quantize_x0=False, eta=0., mask=None, x0=None, temperature=1., noise_dropout=0., score_corrector=None,
               corrector_kwargs=None, verbose=True, x_T=None, log_every_t=100, unconditional_guidance_scale=1.,
               unconditional_conditioning=None, **kwargs):
        self._warn_conditioning_batch(conditioning, batch_size)
        self.make_schedule(ddim_num_steps=S, ddim_eta=eta, verbose=verbose)
        C, H, W = shape
        size = (batch_size, C, H, W)
        if verbose:
            print(f'Data shape for PLMS sampling is {size}')
        return self.plms_sampling(conditioning, size, callback=callback, img_callback=img_callback,
                                  quantize_denoised=quantize_x0, mask=mask, x0=x0, ddim_use_original_steps=False,
                                  noise_dropout=noise_dropout, temperature=temperature, score_corrector=score_corrector,
                                  corrector_kwargs=corrector_kwargs, x_T=x_T, log_every_t=log_every_t,
                                  unconditional_guidance_scale=unconditional_guidance_scale,
                                  unconditional_conditioning=unconditional_conditioning)

    @torch.no_grad()
    def plms_sampling(self, cond, shape, x_T=None, ddim_use_original_steps=False, callback=None, timesteps=None,
                      quantize_denoised=False, mask=None, x0=None, img_callback=None, log_every_t=100, temperature=1.,
                      noise_dropout=0., score_corrector=None, corrector_kwargs=None, unconditional_guidance_scale=1.,
                      unconditional_conditioning=None):
        device = self.model.betas.device
        b = shape[0]
        img = torch.randn(shape, device=device) if x_T is None else x_T
        time_range, total_steps = self._time_range(timesteps, ddim_use_original_steps)
        intermediates = {'x_inter': [img], 'pred_x0': [img]}
        # The eps history: device tensors the update kernel wrote (e_out) or the model's own outputs.  The latter are safe to
        # keep across later UNet calls because UNetModel._graph_forward returns `out.clone()`, never its static graph output.
        old_eps = []
        for i, step in enumerate(time_range):
            index = total_steps - i - 1
            ts = torch.full((b,), int(step), device=device, dtype=torch.long)
            ts_next = torch.full((b,), int(time_range[min(i + 1, len(time_range) - 1)]), device=device, dtype=torch.long)
            if mask is not None:
                assert x0 is not None
                img = self._inpaint_blend(x0, ts, mask, img)
            img, pred_x0, e_t = self.p_sample_plms(img, cond, ts, index=index, use_original_steps=ddim_use_original_steps,
                                                   quantize_denoised=quantize_denoised, temperature=temperature,
                                                   noise_dropout=noise_dropout, score_corrector=score_corrector,
                                                   corrector_kwargs=corrector_kwargs,
                                                   unconditional_guidance_scale=unconditional_guidance_scale,
                                                   unconditional_conditioning=unconditional_conditioning,
                                                   old_eps=old_eps, t_next=ts_next)
            old_eps.append(e_t)
            if len(old_eps) >= 4:
                old_eps.pop(0)
            if callback:
                callback(i)
            if img_callback:
                img_callback(pred_x0, i)
            if index % log_every_t == 0 or index == total_steps - 1:
                intermediates['x_inter'].append(img)
                intermediates['pred_x0'].append(pred_x0)
        return img, intermediates

    @torch.no_grad()
    def p_sample_plms(self, x, c, t, index, repeat_noise=False, use_original_steps=False, quantize_denoised=False,
                      temperature=1., noise_dropout=0., score_corrector=None, corrector_kwargs=None,
                      unconditional_guidance_scale=1., unconditional_conditioning=None, old_eps=None, t_next=None):
        """(x_prev, pred_x0, e_t); e_t is the guidance-combined eps of this step's first evaluation, what the history keeps.
        With an empty history the step is pseudo improved Euler: a DDIM update with e_t, a second model evaluation at that
        x_prev and t_next, then the update from x with (e_t + e_t_next) / 2."""
        old_eps = [] if old_eps is None else old_eps
        coef = self.derived_coefficients(index, use_original_steps)

        def model_eps(x_, t_):
            return self._model_eps(x_, c, t_, score_corrector, corrector_kwargs, unconditional_guidance_scale,
                                   unconditional_conditioning)

        def update(e, e_uncond, order, e_old, keep_e):
            """get_x_prev_and_pred_x0 of the multistep eps: (combined e if keep_e, pred_x0, x_prev)."""
            sqrt_at, sqrt_aprev, dir_coef, sigma_t, s1m = coef
            noise, k_sigma, k_temp = self._step_noise(x, sigma_t, temperature, noise_dropout, repeat_noise)
            f = _f32_contiguous
            ef, uf, nf = f(e), f(e_uncond), f(noise)
            e_c, e_p, pred_x0, x_prev = ops.plms_step(
                f(x), ef, order, sqrt_at, sqrt_aprev, dir_coef, k_sigma, s1m, e_uncond=uf, cfg_scale=unconditional_guidance_scale,
                e_old=e_old, noise=nf, temperature=k_temp, want_e=keep_e and uf is not None, want_e_prime=quantize_denoised,
                want_x_prev=not quantize_denoised)
            if keep_e and e_c is None:
                e_c = ef
            if quantize_denoised:
                # pred_x0 is replaced by the first stage's codebook projection before x_prev is formed from it and e'
                pred_x0 = f(self.model.first_stage_model.quantize(pred_x0)[0])
                x_prev = ops.ddim_xprev(pred_x0, e_p, sqrt_aprev, dir_coef, k_sigma, noise=nf, temperature=k_temp)
            return e_c, pred_x0, x_prev

        e_t, e_uncond = model_eps(x, t)
        if len(old_eps) == 0:
            e_t, _, x_prev = update(e_t, e_uncond, 1, (), keep_e=True)
            e_next, e_next_uncond = model_eps(x_prev, t_next)
            _, pred_x0, x_prev = update(e_next, e_next_uncond, 0, (e_t,), keep_e=False)
        else:
            e_old = tuple(reversed(old_eps[-3:]))            # old_eps[-1], old_eps[-2], old_eps[-3]
            e_t, pred_x0, x_prev = update(e_t, e_uncond, len(e_old) + 1, e_old, keep_e=True)
        return x_prev, pred_x0, e_t
