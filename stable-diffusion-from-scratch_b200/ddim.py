"""Drop-in `DDIMSampler` (reference: ldm/diffusion/ddim.py:12-243 == DDIM/ddim.py) whose update step
runs as ONE fused sm_100a kernel (sdb_ddim_step) instead of ~20 eager elementwise launches.

Same constructor / method signatures and the same duck-typed `model` interface as the reference
(`.num_timesteps`, `.betas`, `.alphas_cumprod`, `.alphas_cumprod_prev`, `.device`, `.apply_model`).
Schedule tables are built on the host with the reference's own mixed torch/numpy arithmetic so the
four per-step coefficients are bit-identical fp32 values.
"""
import numpy as np
import torch

from . import engine, ops


def make_ddim_timesteps(ddim_discr_method, num_ddim_timesteps, num_ddpm_timesteps, verbose=True):
    """ldm/modules/diffusionmodules/util.py:46-60."""
    if ddim_discr_method == 'uniform':
        c = num_ddpm_timesteps // num_ddim_timesteps
        ddim_timesteps = np.asarray(list(range(0, num_ddpm_timesteps, c)))
    elif ddim_discr_method == 'quad':
        ddim_timesteps = ((np.linspace(0, np.sqrt(num_ddpm_timesteps * .8), num_ddim_timesteps)) ** 2).astype(int)
    else:
        raise NotImplementedError(f'There is no ddim discretization method called "{ddim_discr_method}"')
    steps_out = ddim_timesteps + 1
    if verbose:
        print(f'Selected timesteps for ddim sampler: {steps_out}')
    return steps_out


def make_ddim_sampling_parameters(alphacums, ddim_timesteps, eta, verbose=True):
    """ldm/modules/diffusionmodules/util.py:63-74 (alphacums: CPU fp32 tensor)."""
    alphas = alphacums[ddim_timesteps]
    alphas_prev = np.asarray([alphacums[0]] + alphacums[ddim_timesteps[:-1]].tolist())
    sigmas = eta * np.sqrt((1 - alphas_prev) / (1 - alphas) * (1 - alphas / alphas_prev))
    if verbose:
        print(f'Selected alphas for ddim sampler: a_t: {alphas}; a_(t-1): {alphas_prev}')
        print(f'For the chosen value of eta, which is {eta}, '
              f'this results in the following sigma_t schedule for ddim sampler {sigmas}')
    return sigmas, alphas, alphas_prev


def _f32(v):
    """The fp32 value `torch.full((b,1,1,1), v)` would hold (ddim.py:191-194)."""
    return float(torch.full((1,), v).float().item()) if not torch.is_tensor(v) else float(v.float().item())


def _f32_contiguous(t):
    """t as the contiguous fp32 tensor the update kernels read (None passes through)."""
    return t if (t is None or (t.dtype == torch.float32 and t.is_contiguous())) else t.float().contiguous()


class DDIMSampler(object):
    def __init__(self, model, schedule="linear", **kwargs):
        super().__init__()
        self.model = model
        self._cfg_ctx = engine.TensorMemo(1)      # the CFG conditioning of one 2B call, built once per (uc, c) pair
        self.ddpm_num_timesteps = model.num_timesteps
        self.schedule = schedule
        # The reference always draws torch.randn in p_sample_ddim, even when sigma == 0 (util.py:264-267).  The draw cannot
        # change the result when sigma == 0, but it advances the global RNG: anything seeded before `sample()` and drawn
        # after it sees the reference's stream only if the draw is made here too.  Set False to skip the idle draws.
        self.consume_rng_like_reference = True

    def register_buffer(self, name, attr):
        if type(attr) == torch.Tensor:
            dev = getattr(self.model, "device", torch.device("cuda"))
            if attr.device != torch.device(dev):
                attr = attr.to(torch.device(dev))
        setattr(self, name, attr)

    def make_schedule(self, ddim_num_steps, ddim_discretize="uniform", ddim_eta=0., verbose=True):
        """ddim.py:25-54. Host-side, once per `sample`."""
        self.__dict__.pop("_coef_cache", None)      # derived per-step coefficients belong to ONE schedule
        self.ddim_timesteps = make_ddim_timesteps(ddim_discr_method=ddim_discretize, num_ddim_timesteps=ddim_num_steps,
                                                  num_ddpm_timesteps=self.ddpm_num_timesteps, verbose=verbose)
        alphas_cumprod = self.model.alphas_cumprod
        assert alphas_cumprod.shape[0] == self.ddpm_num_timesteps, 'alphas have to be defined for each timestep'
        to_torch = lambda x: x.clone().detach().to(torch.float32).to(self.model.device)

        self.register_buffer('betas', to_torch(self.model.betas))
        self.register_buffer('alphas_cumprod', to_torch(alphas_cumprod))
        self.register_buffer('alphas_cumprod_prev', to_torch(self.model.alphas_cumprod_prev))
        ac = alphas_cumprod.cpu()
        self.register_buffer('sqrt_alphas_cumprod', to_torch(np.sqrt(ac)))
        self.register_buffer('sqrt_one_minus_alphas_cumprod', to_torch(np.sqrt(1. - ac)))
        self.register_buffer('log_one_minus_alphas_cumprod', to_torch(np.log(1. - ac)))
        self.register_buffer('sqrt_recip_alphas_cumprod', to_torch(np.sqrt(1. / ac)))
        self.register_buffer('sqrt_recipm1_alphas_cumprod', to_torch(np.sqrt(1. / ac - 1)))

        ddim_sigmas, ddim_alphas, ddim_alphas_prev = make_ddim_sampling_parameters(
            alphacums=ac, ddim_timesteps=self.ddim_timesteps, eta=ddim_eta, verbose=verbose)
        # kept on the host: they are only ever read one scalar at a time
        self.ddim_sigmas = ddim_sigmas
        self.ddim_alphas = ddim_alphas
        self.ddim_alphas_prev = ddim_alphas_prev
        self.ddim_sqrt_one_minus_alphas = np.sqrt(1. - ddim_alphas)
        sigmas_for_original_sampling_steps = ddim_eta * torch.sqrt(
            (1 - self.alphas_cumprod_prev) / (1 - self.alphas_cumprod) * (1 - self.alphas_cumprod / self.alphas_cumprod_prev))
        self.register_buffer('ddim_sigmas_for_original_num_steps', sigmas_for_original_sampling_steps)

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
            print(f'Data shape for DDIM sampling is {size}, eta {eta}')
        return self.ddim_sampling(conditioning, size, callback=callback, img_callback=img_callback,
                                  quantize_denoised=quantize_x0, mask=mask, x0=x0, ddim_use_original_steps=False,
                                  noise_dropout=noise_dropout, temperature=temperature, score_corrector=score_corrector,
                                  corrector_kwargs=corrector_kwargs, x_T=x_T, log_every_t=log_every_t,
                                  unconditional_guidance_scale=unconditional_guidance_scale,
                                  unconditional_conditioning=unconditional_conditioning)

    @staticmethod
    def _warn_conditioning_batch(conditioning, batch_size):
        """ddim.py:80-87: a warning, not an error, when the conditioning's batch differs from batch_size."""
        if conditioning is not None:
            if isinstance(conditioning, dict):
                ctmp = conditioning[list(conditioning.keys())[0]]
                while isinstance(ctmp, list):         # {"c_concat": [..], "c_crossattn": [..]} of a hybrid model
                    ctmp = ctmp[0]
                cbs = ctmp.shape[0]
                if cbs != batch_size:
                    print(f"Warning: Got {cbs} conditionings but batch-size is {batch_size}")
            else:
                if conditioning.shape[0] != batch_size:
                    print(f"Warning: Got {conditioning.shape[0]} conditionings but batch-size is {batch_size}")

    def _time_range(self, timesteps, ddim_use_original_steps):
        """ddim.py:120-141: (the step values to visit, in order, as a list or array; their count)."""
        if timesteps is None:
            timesteps = self.ddpm_num_timesteps if ddim_use_original_steps else self.ddim_timesteps
        elif timesteps is not None and not ddim_use_original_steps:
            subset_end = int(min(timesteps / self.ddim_timesteps.shape[0], 1) * self.ddim_timesteps.shape[0]) - 1
            timesteps = self.ddim_timesteps[:subset_end]
        time_range = list(reversed(range(0, timesteps))) if ddim_use_original_steps else np.flip(timesteps)
        total_steps = timesteps if ddim_use_original_steps else timesteps.shape[0]
        return time_range, total_steps

    @torch.no_grad()
    def ddim_sampling(self, cond, shape, x_T=None, ddim_use_original_steps=False, callback=None, timesteps=None,
                      quantize_denoised=False, mask=None, x0=None, img_callback=None, log_every_t=100, temperature=1.,
                      noise_dropout=0., score_corrector=None, corrector_kwargs=None, unconditional_guidance_scale=1.,
                      unconditional_conditioning=None):
        """ddim.py:113-165."""
        device = self.model.betas.device
        b = shape[0]
        img = torch.randn(shape, device=device) if x_T is None else x_T
        time_range, total_steps = self._time_range(timesteps, ddim_use_original_steps)
        intermediates = {'x_inter': [img], 'pred_x0': [img]}
        # one device tensor of timesteps per step value (tiny H2D, outside the kernels' critical path)
        for i, step in enumerate(time_range):
            index = total_steps - i - 1
            ts = torch.full((b,), int(step), device=device, dtype=torch.long)
            if mask is not None:
                assert x0 is not None
                img = self._inpaint_blend(x0, ts, mask, img)
            img, pred_x0 = self.p_sample_ddim(img, cond, ts, index=index, use_original_steps=ddim_use_original_steps,
                                              quantize_denoised=quantize_denoised, temperature=temperature,
                                              noise_dropout=noise_dropout, score_corrector=score_corrector,
                                              corrector_kwargs=corrector_kwargs,
                                              unconditional_guidance_scale=unconditional_guidance_scale,
                                              unconditional_conditioning=unconditional_conditioning)
            if callback:
                callback(i)
            if img_callback:
                img_callback(pred_x0, i)
            if index % log_every_t == 0 or index == total_steps - 1:
                intermediates['x_inter'].append(img)
                intermediates['pred_x0'].append(pred_x0)
        return img, intermediates

    def _inpaint_blend(self, x0, ts, mask, img):
        """ddim.py:144-149: img_orig = model.q_sample(x0, ts); img = img_orig * mask + (1 - mask) * img.  When the model is
        a LatentDiffusion-like object with the schedule buffers q_sample reads (ldm/diffusion/ddpm.py:407-412), q_sample and
        the blend run as ONE kernel; q_sample's draw is torch.rand_like, exactly as the reference makes it.  Any other
        `model.q_sample` is honoured as given and only the blend is fused."""
        fused = getattr(self.model, "q_sample_coefficients", None)
        if fused is not None:
            a, c = fused(ts)
            noise = torch.rand_like(x0)                      # ddpm.py:409 (uniform, as written)
        else:
            a = torch.ones((x0.shape[0],), device=x0.device)
            c = torch.zeros((x0.shape[0],), device=x0.device)
            noise = x0
            x0 = self.model.q_sample(x0, ts)
        f = lambda t: t.float().contiguous()
        m = mask.to(x0.device)
        if m.dim() == x0.dim() and m.shape[1] not in (1, x0.shape[1]):
            raise ValueError("mask %s does not broadcast over x0 %s" % (tuple(m.shape), tuple(x0.shape)))
        m = f(m.expand(x0.shape[0], m.shape[1], *x0.shape[2:])) if m.dim() == x0.dim() else f(m.expand_as(x0))
        return ops.inpaint_blend(f(x0), f(noise), f(a), f(c), m, f(img))

    def coefficients(self, index, use_original_steps=False):
        """The fp32 scalars a_t, a_prev, sigma_t, sqrt(1-a_t) that ddim.py:191-194 broadcast to [b,1,1,1]."""
        alphas = self.model.alphas_cumprod if use_original_steps else self.ddim_alphas
        alphas_prev = self.model.alphas_cumprod_prev if use_original_steps else self.ddim_alphas_prev
        sqrt_one_minus_alphas = self.model.sqrt_one_minus_alphas_cumprod if use_original_steps else self.ddim_sqrt_one_minus_alphas
        sigmas = self.model.ddim_sigmas_for_original_num_steps if use_original_steps else self.ddim_sigmas
        return (_f32(alphas[index]), _f32(alphas_prev[index]), _f32(sigmas[index]), _f32(sqrt_one_minus_alphas[index]))

    def derived_coefficients(self, index, use_original_steps=False):
        """sqrt(a_t), sqrt(a_prev), sqrt(1 - a_prev - sigma^2), sigma_t, sqrt(1-a_t) as the fp32 values the
        reference's [b,1,1,1] tensors hold (ddim.py:191-205), evaluated with the reference's own torch
        expressions on host tensors.  (torch's CPU sqrt is not correctly rounded for every input — e.g. 4 of
        the 50 SD DDIM-50 alphas land 1 ulp off IEEE — so calling the same routine is what keeps the update
        bit-identical to the CPU-executed reference; cached per (index, schedule).)"""
        key = (index, use_original_steps)
        cache = self.__dict__.setdefault("_coef_cache", {})      # dropped by make_schedule
        if key not in cache:
            a_t, a_prev, sigma_t, s1m = self.coefficients(index, use_original_steps)
            ta, tp, ts = torch.full((1, 1, 1, 1), a_t), torch.full((1, 1, 1, 1), a_prev), torch.full((1, 1, 1, 1), sigma_t)
            cache[key] = (float(ta.sqrt()), float(tp.sqrt()), float((1. - tp - ts ** 2).sqrt()), sigma_t, s1m)
        return cache[key]

    @torch.no_grad()
    def p_sample_ddim(self, x, c, t, index, repeat_noise=False, use_original_steps=False, quantize_denoised=False,
                      temperature=1., noise_dropout=0., score_corrector=None, corrector_kwargs=None,
                      unconditional_guidance_scale=1., unconditional_conditioning=None):
        """ddim.py:167-206.  CFG runs the model on the unconditional and conditional halves separately
        (same per-sample arithmetic as the reference's concatenated 2B batch) and the combine
        e_uc + s*(e_c - e_uc) is fused into the update kernel."""
        e_t, e_uncond = self._model_eps(x, c, t, score_corrector, corrector_kwargs, unconditional_guidance_scale,
                                        unconditional_conditioning)
        sqrt_at, sqrt_aprev, dir_coef, sigma_t, s1m = self.derived_coefficients(index, use_original_steps)
        noise, k_sigma, k_temp = self._step_noise(x, sigma_t, temperature, noise_dropout, repeat_noise)
        f = _f32_contiguous
        xf, ef, uf, nf = f(x), f(e_t), f(e_uncond), f(noise)
        x_prev, pred_x0 = ops.ddim_step(xf, ef, sqrt_at, sqrt_aprev, dir_coef, k_sigma, s1m, e_uncond=uf,
                                        cfg_scale=unconditional_guidance_scale, noise=nf, temperature=k_temp)
        if quantize_denoised:
            # ddim.py:198-199: pred_x0 is replaced by the first stage's codebook projection before x_prev is formed
            pred_x0, _, *_ = self.model.first_stage_model.quantize(pred_x0)
            pred_x0 = f(pred_x0)
            x_prev = ops.ddim_xprev(pred_x0, ef, sqrt_aprev, dir_coef, k_sigma, e_uncond=uf, cfg_scale=unconditional_guidance_scale,
                                    noise=nf, temperature=k_temp)
        return x_prev, pred_x0

    def _model_eps(self, x, c, t, score_corrector, corrector_kwargs, unconditional_guidance_scale, unconditional_conditioning):
        """The model-evaluation half of p_sample_ddim (ddim.py:174-186; PLMS's get_model_output is the same code):
        (e_t, e_uncond).  With CFG and no score corrector, e_uncond is the unconditional half and the combine is left to the
        update kernel; otherwise e_uncond is None and e_t is the final eps."""
        e_uncond = None
        if unconditional_conditioning is None or unconditional_guidance_scale == 1.:
            e_t = self.model.apply_model(x, t, c)
        elif isinstance(c, torch.Tensor) and isinstance(unconditional_conditioning, torch.Tensor):
            # one 2B call like the reference (ddim.py:176-179).  The concatenated conditioning is built once per (uc, c)
            # pair and reused for every step, so a UNet that caches the context K/V projections keeps hitting its cache.
            uc = unconditional_conditioning
            c_in = self._cfg_ctx.get((c, uc), "tensor", lambda: torch.cat([uc, c]))
            e_uncond, e_t = self.model.apply_model(torch.cat([x] * 2), torch.cat([t] * 2), c_in).chunk(2)
            e_uncond, e_t = e_uncond.contiguous(), e_t.contiguous()
        elif self._cfg_dict_pairable(c, unconditional_conditioning):
            # image-conditioned ("concat" / "hybrid") models: one 2B call as well, every entry of the two dicts joined along the
            # batch as the reference's dict branch does.  Per-sample results are batch-invariant, so this gives the bits of the
            # two separate calls below; it also keeps ONE context tensor for all steps (the two calls alternate uc and c, which
            # makes a CUDA-graph UNet re-project the context K/V on every call).
            c_in = self._cfg_dict_in(c, unconditional_conditioning)
            e_uncond, e_t = self.model.apply_model(torch.cat([x] * 2), torch.cat([t] * 2), c_in).chunk(2)
            e_uncond, e_t = e_uncond.contiguous(), e_t.contiguous()
        else:
            e_uncond = self.model.apply_model(x, t, unconditional_conditioning)
            e_t = self.model.apply_model(x, t, c)
        if score_corrector is not None:
            assert self.model.parameterization == "eps"
            if e_uncond is not None:
                e_t = e_uncond + unconditional_guidance_scale * (e_t - e_uncond)
                e_uncond = None
            e_t = score_corrector.modify_score(self.model, e_t, x, t, c, **corrector_kwargs)
        return e_t, e_uncond

    def _step_noise(self, x, sigma_t, temperature, noise_dropout, repeat_noise):
        """The noise term of one update (ddim.py:200-204): (noise or None, sigma and temperature to pass to the kernel).  The
        draws follow the reference's: randn on every call unless consume_rng_like_reference is off and sigma_t == 0, and the
        dropout mask when noise_dropout > 0."""
        noise = None
        if sigma_t != 0.0 or self.consume_rng_like_reference or noise_dropout > 0.:
            if repeat_noise:
                noise = torch.randn((1, *x.shape[1:]), device=x.device).repeat(x.shape[0], *((1,) * (len(x.shape) - 1)))
            else:
                noise = torch.randn(x.shape, device=x.device)
        k_sigma, k_temp = sigma_t, temperature
        if noise_dropout > 0.:
            # ddim.py:202-204: dropout acts on the PRODUCT sigma_t * noise * temperature; the mask draw is torch's own RNG
            # (host-library plumbing like randn), so the product is formed here and enters the kernel with unit coefficients
            noise = torch.nn.functional.dropout(torch.full((1, 1, 1, 1), sigma_t, device=x.device) * noise * temperature, p=noise_dropout)
            k_sigma, k_temp = 1.0, 1.0
        elif sigma_t == 0.0:
            noise = None
        return noise, k_sigma, k_temp

    @staticmethod
    def _cfg_dict_pairable(c, uc):
        """Dict conditionings with a c_concat entry whose uc / c entries pair up one to one (same keys, same list lengths)."""
        if not (isinstance(c, dict) and isinstance(uc, dict)) or "c_concat" not in c or set(c) != set(uc):
            return False
        for k in c:
            a, b = c[k], uc[k]
            if isinstance(a, list) != isinstance(b, list):
                return False
            if isinstance(a, list):
                if len(a) != len(b) or not all(torch.is_tensor(v) for v in a + b):
                    return False
            elif not (torch.is_tensor(a) and torch.is_tensor(b)):
                return False
        return True

    def _cfg_dict_in(self, c, uc):
        """{k: [cat([uc[k][i], c[k][i]]) ...]} (tensor entries: cat([uc[k], c[k]])), built once per (uc, c) pair of live,
        unwritten tensors."""
        leaves = [(k, i, uc[k][i] if isinstance(uc[k], list) else uc[k], v)
                  for k in sorted(c) for i, v in (enumerate(c[k]) if isinstance(c[k], list) else [(None, c[k])])]
        build = lambda: {k: ([torch.cat([uc[k][i], c[k][i]]) for i in range(len(c[k]))] if isinstance(c[k], list)
                             else torch.cat([uc[k], c[k]])) for k in c}
        tensors = [t for _, _, u, v in leaves for t in (u, v)]
        return self._cfg_ctx.get(tensors, ("dict",) + tuple((k, i) for k, i, _, _ in leaves), build)

    @torch.no_grad()
    def stochastic_encode(self, x0, t, use_original_steps=False, noise=None):
        """ddim.py:208-222 (img2img entry, SURVEY.md §8 f3): x_t = sqrt(a_t) x0 + sqrt(1 - a_t) noise with the per-sample
        coefficients gathered at t, one fused kernel (individually rounded fp32 ops: bit-exact vs the eager reference)."""
        if use_original_steps:
            sqrt_alphas_cumprod = self.sqrt_alphas_cumprod
            sqrt_one_minus_alphas_cumprod = self.sqrt_one_minus_alphas_cumprod
        else:
            sqrt_alphas_cumprod = torch.sqrt(torch.as_tensor(self.ddim_alphas))
            sqrt_one_minus_alphas_cumprod = torch.as_tensor(self.ddim_sqrt_one_minus_alphas)
        if noise is None:
            noise = torch.randn_like(x0)
        dev = x0.device
        t = t.to(dev)
        sa = sqrt_alphas_cumprod.to(dev).gather(-1, t).float().contiguous()
        sb = sqrt_one_minus_alphas_cumprod.to(dev).gather(-1, t).float().contiguous()
        return ops.q_sample(x0.float().contiguous(), noise.float().contiguous(), sa, sb)

    @torch.no_grad()
    def decode(self, x_latent, cond, t_start, unconditional_guidance_scale=1.0, unconditional_conditioning=None,
               use_original_steps=False):
        """ddim.py:224-243."""
        timesteps = np.arange(self.ddpm_num_timesteps) if use_original_steps else self.ddim_timesteps
        timesteps = timesteps[:t_start]
        time_range = np.flip(timesteps)
        total_steps = timesteps.shape[0]
        x_dec = x_latent
        for i, step in enumerate(time_range):
            index = total_steps - i - 1
            ts = torch.full((x_latent.shape[0],), int(step), device=x_latent.device, dtype=torch.long)
            x_dec, _ = self.p_sample_ddim(x_dec, cond, ts, index=index, use_original_steps=use_original_steps,
                                          unconditional_guidance_scale=unconditional_guidance_scale,
                                          unconditional_conditioning=unconditional_conditioning)
        return x_dec
