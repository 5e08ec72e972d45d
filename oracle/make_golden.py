"""TEST INFRASTRUCTURE — generates tests/golden/*.pt by executing the UNMODIFIED reference.

Run in the build container only (needs /root/reference):
    python oracle/make_golden.py            # everything (spawns a subprocess for the DDPM UNet)
    python oracle/make_golden.py --part ddpm

Each fixture holds: the seeds, the (key, shape) list of the reference module's state dict (weights
are regenerated procedurally by oracle/weights.py), the seeded inputs' seeds, and the reference's
outputs.  While generating, the restatement in oracle/restate.py is checked against the reference
output (assert), so a committed fixture certifies "restate.py == reference" on that case.
"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ref_harness as RH  # noqa: E402
from oracle import restate as R  # noqa: E402
from oracle import weights as W  # noqa: E402
from oracle.golden import sample_flat  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")

TINY_UNET_CFG = dict(image_size=16, in_channels=4, out_channels=4, model_channels=64, attention_resolutions=[1, 2],
                     num_res_blocks=1, channel_mult=(1, 2), num_heads=2, use_spatial_transformer=True,
                     transformer_depth=1, context_dim=64, use_checkpoint=False, legacy=False)
TINY_VAE_DDCONFIG = dict(double_z=True, z_channels=4, resolution=32, in_channels=3, out_ch=3, ch=64, ch_mult=(1, 2),
                         num_res_blocks=1, attn_resolutions=[], dropout=0.0)


def save(name, obj):
    os.makedirs(GOLD, exist_ok=True)
    path = os.path.join(GOLD, name)
    torch.save(obj, path)
    print("wrote %s (%.1f KB)" % (path, os.path.getsize(path) / 1024))


def gen_unet(name, cfg, B, HW, S_ctx, seed, t_values, with_f64):
    net = RH.build_unet(cfg)
    ks = W.key_shapes_of(net)
    sd = W.make_state_dict(ks, seed)
    net.load_state_dict(sd, strict=True)
    x = W.seeded_randn((B, cfg["in_channels"], HW, HW), seed + 1)
    ctx = W.seeded_randn((B, S_ctx, cfg["context_dim"]), seed + 2)
    t = torch.tensor(t_values, dtype=torch.long)
    eps_ref = RH.run_unet(net, x, t, ctx)
    taps = {}
    with torch.no_grad():
        eps_or = R.unet_forward(sd, cfg, x, t, ctx, taps=taps)
    err = R.rel_l2(eps_or, eps_ref)
    print("%s: restatement vs reference rel-L2 = %.3e (eps std %.3f)" % (name, err, float(eps_ref.std())))
    assert err < 2e-5, err
    out = dict(cfg=cfg, seed=seed, key_shapes=ks, x_shape=tuple(x.shape), ctx_shape=tuple(ctx.shape),
               t=t, eps_ref=eps_ref.clone(), restate_err=err)
    # a few intermediate activations from the restatement (for layer-level debugging of the CUDA path)
    for k in ("input_blocks.1", "middle_block"):
        if taps[k].numel() <= 1 << 16:
            out["tap." + k] = taps[k].clone()
    if with_f64:
        sd64 = {k: v.double() for k, v in sd.items()}
        with torch.no_grad():
            eps64 = R.unet_forward(sd64, cfg, x.double(), t, ctx.double())
        out["eps_f64"] = eps64.clone()
        print("   fp32 reference vs f64 restatement rel-L2 = %.3e" % R.rel_l2(eps_ref, eps64))
    save(name + ".pt", out)


VARIANT_UNET_CFGS = {   # 'next' row f4: the non-transformer UNetModel variants (cf. the __main__ demo, openai_model/model.py:604-622)
    "unet_var_legacy": dict(image_size=16, in_channels=4, out_channels=4, model_channels=64, attention_resolutions=[1, 2],
                            num_res_blocks=1, channel_mult=(1, 2), num_head_channels=32, use_spatial_transformer=False,
                            use_scale_shift_norm=True, resblock_updown=True, num_classes=10, use_new_attention_order=False,
                            use_checkpoint=False, legacy=True),
    "unet_var_neworder": dict(image_size=16, in_channels=4, out_channels=4, model_channels=64, attention_resolutions=[2],
                              num_res_blocks=1, channel_mult=(1, 2), num_heads=2, use_spatial_transformer=False,
                              use_scale_shift_norm=False, resblock_updown=False, num_classes=None, use_new_attention_order=True,
                              use_checkpoint=False, legacy=True),
}


def gen_unet_variant(name, cfg, seed):
    net = RH.build_unet(cfg)
    ks = W.key_shapes_of(net)
    sd = W.make_state_dict(ks, seed)
    net.load_state_dict(sd, strict=True)
    B = 2
    x = W.seeded_randn((B, cfg["in_channels"], 16, 16), seed + 1)
    t = torch.tensor([981, 1], dtype=torch.long)
    y = torch.tensor([3, 7], dtype=torch.long) if cfg.get("num_classes") is not None else None
    eps_ref = RH.run_unet(net, x, t, None, y)
    with torch.no_grad():
        eps_or = R.unet_forward(sd, cfg, x, t, None, y=y)
        eps64 = R.unet_forward({k: v.double() for k, v in sd.items()}, cfg, x.double(), t, None, y=y)
    err = R.rel_l2(eps_or, eps_ref)
    print("%s: restatement vs reference rel-L2 = %.3e (eps std %.3f); fp32 reference vs f64 %.3e"
          % (name, err, float(eps_ref.std()), R.rel_l2(eps_ref, eps64)))
    assert err < 2e-5, err
    save(name + ".pt", dict(cfg=cfg, seed=seed, key_shapes=ks, x_shape=tuple(x.shape), t=t, y=y, eps_ref=eps_ref.clone(),
                            eps_f64=eps64.clone(), restate_err=err))


def gen_vae(name, ddconfig, B, zres, seed, with_f64):
    dec = RH.build_decoder(ddconfig)
    ks_dec = W.key_shapes_of(dec)
    ks = [("decoder." + k, s) for k, s in ks_dec] + [("post_quant_conv.weight", (ddconfig["z_channels"], 4, 1, 1)),
                                                      ("post_quant_conv.bias", (ddconfig["z_channels"],))]
    sd = W.make_state_dict(ks, seed)
    dec.load_state_dict({k[len("decoder."):]: v for k, v in sd.items() if k.startswith("decoder.")}, strict=True)
    z = W.seeded_randn((B, 4, zres, zres), seed + 1)
    with torch.no_grad(), RH.quiet():
        pq = torch.nn.functional.conv2d(z, sd["post_quant_conv.weight"], sd["post_quant_conv.bias"])   # autoencoder.py:310,338
        img_ref = dec(pq)
        img_or = R.autoencoder_decode(sd, ddconfig, z)
    err = R.rel_l2(img_or, img_ref)
    print("%s: restatement vs reference rel-L2 = %.3e (img std %.3f)" % (name, err, float(img_ref.std())))
    assert err < 2e-5, err
    out = dict(ddconfig=ddconfig, seed=seed, key_shapes=ks, z_shape=tuple(z.shape), img_ref=img_ref.clone(), restate_err=err)
    if with_f64:
        with torch.no_grad():
            img64 = R.autoencoder_decode({k: v.double() for k, v in sd.items()}, ddconfig, z.double())
        out["img_f64"] = img64.clone()
        print("   fp32 reference vs f64 restatement rel-L2 = %.3e" % R.rel_l2(img_ref, img64))
    save(name + ".pt", out)


def gen_vae_enc(name, ddconfig, B, res, seed):
    """Encoder + quant_conv + DiagonalGaussianDistribution of the reference, and the img2img entry
    DDIMSampler.stochastic_encode / decode on the resulting latent ('next' row f3)."""
    enc = RH.build_encoder(ddconfig)
    ks_enc = W.key_shapes_of(enc)
    zc = ddconfig["z_channels"]
    ks = [("encoder." + k, s) for k, s in ks_enc] + [("quant_conv.weight", (2 * zc, 2 * zc, 1, 1)), ("quant_conv.bias", (2 * zc,))]
    sd = W.make_state_dict(ks, seed)
    enc.load_state_dict({k[len("encoder."):]: v for k, v in sd.items() if k.startswith("encoder.")}, strict=True)
    x = W.seeded_randn((B, ddconfig["in_channels"], res, res), seed + 1)
    DG = RH.gaussian_distribution_class()
    with torch.no_grad(), RH.quiet():
        moments = torch.nn.functional.conv2d(enc(x), sd["quant_conv.weight"], sd["quant_conv.bias"])   # autoencoder.py:331-334
        post = DG(moments)
        torch.manual_seed(seed + 2)
        z_ref = post.sample()
        mean_or, logvar_or, std_or = R.autoencoder_encode(sd, ddconfig, x)
    torch.manual_seed(seed + 2)
    noise = torch.randn(post.mean.shape)                 # the draw sample() makes (distributions.py:36)
    assert torch.equal(z_ref, post.mean + post.std * noise)
    err = R.rel_l2(torch.cat([mean_or, logvar_or], 1), torch.cat([post.mean, post.logvar], 1))
    print("%s: encoder restatement vs reference rel-L2 = %.3e (moments std %.3f)" % (name, err, float(moments.std())))
    assert err < 2e-5, err
    assert R.rel_l2(std_or, post.std) < 2e-5
    with torch.no_grad():
        m64, lv64, _ = R.autoencoder_encode({k: v.double() for k, v in sd.items()}, ddconfig, x.double())
    print("   fp32 reference vs f64 restatement rel-L2 = %.3e" % R.rel_l2(torch.cat([post.mean, post.logvar], 1), torch.cat([m64, lv64], 1)))
    out = dict(ddconfig=ddconfig, seed=seed, key_shapes=ks, x_shape=tuple(x.shape), mean_ref=post.mean.clone(),
               logvar_ref=post.logvar.clone(), std_ref=post.std.clone(), noise=noise, z_ref=z_ref.clone(),
               mean_f64=m64.clone(), logvar_f64=lv64.clone(), kl_ref=post.kl().clone(), restate_err=err)
    # img2img entry on that latent: stochastic_encode with the reference sampler (toy eps-model, SD schedule)
    shim = R.ModelShim(toy_model_fn, R.sd_alphas_cumprod())
    ref = RH.make_cpu_sampler(shim)
    with RH.quiet():
        ref.make_schedule(ddim_num_steps=20, ddim_eta=0.0, verbose=False)
    t_enc = 12
    n2 = W.seeded_randn(tuple(z_ref.shape), seed + 3)
    ts = torch.full((B,), t_enc, dtype=torch.long)
    with RH.quiet():
        zt_ref = ref.stochastic_encode(z_ref, ts, noise=n2)
        zdec_ref = ref.decode(zt_ref, None, t_enc)
    zt_or = R.q_sample_ddim(z_ref, n2, ref.ddim_alphas, ref.ddim_sqrt_one_minus_alphas, ts)
    assert torch.equal(zt_or, zt_ref), "stochastic_encode restatement is not bit-exact"
    out.update(t_enc=t_enc, enc_noise=n2, zt_ref=zt_ref.clone(), zdec_ref=zdec_ref.clone())
    save(name + ".pt", out)


def gen_sd_traj(name="sd_traj", steps_kept=(0, 12, 25, 37, 49), img_samples=32768):
    """BASELINE config C2 at its own size: the UNMODIFIED reference UNetModel (SD-1.x kwargs) driven by the reference
    DDIMSampler (DDIM/ddim.py) for a full DDIM-50 run at B=1, 64x64x4 latent, 77x768 context, then the reference ldm
    Decoder on z / 0.18215 (ldm/diffusion/ddpm.py:1095) -> 3x512x512.  Stored: (x_t, t, e_t) at five steps of the
    reference trajectory (teacher-forced eps checks), the final latent and the decoded image (PSNR check) as its values
    at `img_samples` fixed positions (oracle/golden.py sample_index), which keeps the fixture under 1 MB.
    UNet weights = seed 31 (same as unet_sd.pt), VAE weights = seed 51 (same as vae_sd_z16.pt)."""
    import contextlib
    import io
    import time
    cfg = R.SD_UNET_CFG
    net = RH.build_unet(cfg)
    ks_u = W.key_shapes_of(net)
    sdu = W.make_state_dict(ks_u, 31)
    net.load_state_dict(sdu, strict=True)
    dec = RH.build_decoder(R.SD_VAE_DDCONFIG)
    ks_v = [("decoder." + k, s) for k, s in W.key_shapes_of(dec)] + [("post_quant_conv.weight", (4, 4, 1, 1)), ("post_quant_conv.bias", (4,))]
    sdv = W.make_state_dict(ks_v, 51)
    dec.load_state_dict({k[len("decoder."):]: v for k, v in sdv.items() if k.startswith("decoder.")}, strict=True)
    x_T = W.seeded_randn((1, 4, 64, 64), 2)       # SURVEY.md 8d: C2 seeds
    ctx = W.seeded_randn((1, 77, 768), 3)
    rec = []

    def fn(x, t, c):
        e = RH.run_unet(net, x, t, c)
        rec.append((x.clone(), int(t[0]), e.clone()))
        return e

    ref = RH.make_cpu_sampler(R.ModelShim(fn, R.sd_alphas_cumprod()))
    t0 = time.perf_counter()
    with torch.no_grad(), RH.quiet(), contextlib.redirect_stderr(io.StringIO()):
        z_ref, _ = ref.sample(S=50, batch_size=1, shape=(4, 64, 64), conditioning=ctx, verbose=False, x_T=x_T, eta=0.)
    t_traj = time.perf_counter() - t0
    assert len(rec) == 50
    with torch.no_grad(), RH.quiet():
        pq = torch.nn.functional.conv2d(z_ref / 0.18215, sdv["post_quant_conv.weight"], sdv["post_quant_conv.bias"])
        img_ref = dec(pq)
    print("%s: reference DDIM-50 %.1f s; z std %.3f max %.2f; img mean %.3f std %.3f, %.1f%% inside [-1,1]"
          % (name, t_traj, float(z_ref.std()), float(z_ref.abs().max()), float(img_ref.mean()), float(img_ref.std()),
             100 * float((img_ref.abs() <= 1).float().mean())))
    kept = []
    worst = 0.0
    for i in steps_kept:
        x_t, t, e_t = rec[i]
        with torch.no_grad():
            e_or = R.unet_forward(sdu, cfg, x_t, torch.tensor([t]), ctx)
        err = R.rel_l2(e_or, e_t)
        worst = max(worst, err)
        print("   step %2d (t=%d): restatement vs reference eps rel-L2 = %.3e, x_t std %.3f, eps std %.3f"
              % (i, t, err, float(x_t.std()), float(e_t.std())))
        assert err < 2e-5, err
        kept.append(dict(i=i, t=t, x_t=x_t, e_t=e_t))
    with torch.no_grad():
        img_or = R.autoencoder_decode(sdv, R.SD_VAE_DDCONFIG, z_ref / 0.18215)
    err_img = R.rel_l2(img_or, img_ref)
    print("   decode restatement vs reference rel-L2 = %.3e" % err_img)
    assert err_img < 2e-5, err_img
    save(name + ".pt", dict(cfg=cfg, ddconfig=R.SD_VAE_DDCONFIG, unet_seed=31, vae_seed=51, unet_key_shapes=ks_u, vae_key_shapes=ks_v,
                            x_T_seed=2, ctx_seed=3, steps=kept, all_t=[r[1] for r in rec], z_ref=z_ref.clone(),
                            img_shape=tuple(img_ref.shape), img_ref_s=sample_flat(img_ref, img_samples),
                            restate_err=worst, restate_err_img=err_img, ref_seconds=t_traj))


def gen_vae_full(name="vae_sd_z64", img_samples=65536):
    """BASELINE config C3 at its own size (B=1): the reference ldm Decoder on a 64x64x4 latent -> 3x512x512.
    `img_f64` is the float64 restatement rounded to fp32 for storage (3e-8 relative, against a 1e-5 bound).  Both images
    are stored as their values at `img_samples` fixed positions (oracle/golden.py sample_index: `img_ref_s`, `img_f64_s`)."""
    ddconfig = R.SD_VAE_DDCONFIG
    dec = RH.build_decoder(ddconfig)
    ks = [("decoder." + k, s) for k, s in W.key_shapes_of(dec)] + [("post_quant_conv.weight", (4, 4, 1, 1)), ("post_quant_conv.bias", (4,))]
    sd = W.make_state_dict(ks, 51)
    dec.load_state_dict({k[len("decoder."):]: v for k, v in sd.items() if k.startswith("decoder.")}, strict=True)
    z = W.seeded_randn((1, 4, 64, 64), 4)         # SURVEY.md 8d: C3 seed
    with torch.no_grad(), RH.quiet():
        pq = torch.nn.functional.conv2d(z, sd["post_quant_conv.weight"], sd["post_quant_conv.bias"])
        img_ref = dec(pq)
        img_or = R.autoencoder_decode(sd, ddconfig, z)
        img64 = R.autoencoder_decode({k: v.double() for k, v in sd.items()}, ddconfig, z.double())
    err = R.rel_l2(img_or, img_ref)
    print("%s: restatement vs reference rel-L2 = %.3e (img std %.3f); fp32 reference vs f64 %.3e"
          % (name, err, float(img_ref.std()), R.rel_l2(img_ref, img64)))
    assert err < 2e-5, err
    save(name + ".pt", dict(ddconfig=ddconfig, seed=51, z_seed=4, key_shapes=ks, z_shape=(1, 4, 64, 64), img_shape=tuple(img_ref.shape),
                            img_ref_s=sample_flat(img_ref, img_samples), img_f64_s=sample_flat(img64.float(), img_samples),
                            restate_err=err))


def gen_unet_96(name="unet_sd_96"):
    """BASELINE config C5 at its own size (B=1): one reference UNetModel step on a 96x96x4 latent (S = 9216 tokens)."""
    cfg = R.SD_UNET_CFG
    net = RH.build_unet(cfg)
    ks = W.key_shapes_of(net)
    sd = W.make_state_dict(ks, 31)
    net.load_state_dict(sd, strict=True)
    x = W.seeded_randn((1, 4, 96, 96), 5)         # SURVEY.md 8d: C5 seed
    ctx = W.seeded_randn((1, 77, 768), 3)
    t = torch.tensor([500], dtype=torch.long)
    eps_ref = RH.run_unet(net, x, t, ctx)
    with torch.no_grad():
        eps_or = R.unet_forward(sd, cfg, x, t, ctx)
        eps64 = R.unet_forward({k: v.double() for k, v in sd.items()}, cfg, x.double(), t, ctx.double())
    err = R.rel_l2(eps_or, eps_ref)
    print("%s: restatement vs reference rel-L2 = %.3e (eps std %.3f); fp32 reference vs f64 %.3e"
          % (name, err, float(eps_ref.std()), R.rel_l2(eps_ref, eps64)))
    assert err < 2e-5, err
    save(name + ".pt", dict(cfg=cfg, seed=31, key_shapes=ks, x_shape=(1, 4, 96, 96), x_seed=5, ctx_shape=(1, 77, 768), ctx_seed=3,
                            t=t, eps_ref=eps_ref.clone(), eps_f64=eps64.clone(), restate_err=err))


def toy_model_fn(x, t, c):
    """A cheap analytic eps-model so that sampler goldens do not depend on any network."""
    s = torch.sin(t.float() * 0.01).view(-1, 1, 1, 1)
    bias = 0.0 if c is None else c.mean(dim=(1, 2)).view(-1, 1, 1, 1)
    return 0.3 * x * s + 0.1 * torch.cos(x) + bias


def gen_ddim():
    ddim = RH.ddim_module()
    out = {}
    for sched_name, ac in (("sd", R.sd_alphas_cumprod()), ("ddpm", R.ddpm_alphas_cumprod())):
        for S, eta in ((50, 0.0), (50, 0.5), (10, 0.0), (20, 1.0)):
            shim = R.ModelShim(toy_model_fn, ac)
            ref = RH.make_cpu_sampler(shim)
            with RH.quiet():
                ref.make_schedule(ddim_num_steps=S, ddim_eta=eta, verbose=False)
            orc = R.DDIMOracle(shim)
            orc.make_schedule(S, ddim_eta=eta)
            tag = "%s.S%d.eta%g" % (sched_name, S, eta)
            out[tag + ".timesteps"] = torch.as_tensor(np.ascontiguousarray(ref.ddim_timesteps))
            coefs = []
            for index in range(S):
                b = 1
                # exactly the reference's four lines (ddim.py:191-194)
                a_t = torch.full((b, 1, 1, 1), ref.ddim_alphas[index])
                a_prev = torch.full((b, 1, 1, 1), ref.ddim_alphas_prev[index])
                sigma_t = torch.full((b, 1, 1, 1), ref.ddim_sigmas[index])
                s1m = torch.full((b, 1, 1, 1), ref.ddim_sqrt_one_minus_alphas[index])
                assert a_t.dtype == a_prev.dtype == sigma_t.dtype == s1m.dtype == torch.float32
                o = orc.coefficients(index)
                for u, v in zip((a_t, a_prev, sigma_t, s1m), o):
                    assert u.dtype == v.dtype and torch.equal(u, v)
                coefs.append(torch.stack([a_t.flatten(), a_prev.flatten(), sigma_t.flatten(), s1m.flatten()], 1))
            out[tag + ".coefs"] = torch.cat(coefs, 0)   # [S, 4] fp32: a_t, a_prev, sigma_t, sqrt(1-a_t)
            assert np.array_equal(ref.ddim_timesteps, orc.ddim_timesteps)
    # single steps (eta > 0 exercises the noise term; CFG exercises the combine)
    ac = R.sd_alphas_cumprod()
    shim = R.ModelShim(toy_model_fn, ac)
    for S, eta, cfg_scale in ((50, 0.0, 1.0), (50, 0.5, 1.0), (50, 0.0, 7.5), (20, 1.0, 3.0)):
        ref = RH.make_cpu_sampler(shim)
        with RH.quiet():
            ref.make_schedule(ddim_num_steps=S, ddim_eta=eta, verbose=False)
        orc = R.DDIMOracle(shim)
        orc.make_schedule(S, ddim_eta=eta)
        x = W.seeded_randn((2, 4, 8, 8), 77)
        c = W.seeded_randn((2, 5, 6), 78)
        uc = W.seeded_randn((2, 5, 6), 79) if cfg_scale != 1.0 else None
        for index in (S - 1, S // 2, 0):
            step = int(ref.ddim_timesteps[index])
            ts = torch.full((2,), step, dtype=torch.long)
            torch.manual_seed(4321 + index)
            with RH.quiet():
                xp_ref, p0_ref = ref.p_sample_ddim(x, c, ts, index=index, unconditional_guidance_scale=cfg_scale,
                                                   unconditional_conditioning=uc)
            torch.manual_seed(4321 + index)
            noise = torch.randn(x.shape)       # the draw noise_like() makes (diffusion_modules.py:264-267)
            xp, p0, e_t = orc.p_sample_ddim(x, c, ts, index, unconditional_guidance_scale=cfg_scale,
                                            unconditional_conditioning=uc, noise=noise)
            assert torch.equal(xp, xp_ref) and torch.equal(p0, p0_ref), "DDIM step restatement is not bit-exact"
            tag = "step.S%d.eta%g.cfg%g.i%d" % (S, eta, cfg_scale, index)
            out[tag] = dict(x=x, c=c, uc=uc, index=index, step=step, noise=noise, e_t=e_t, x_prev=xp_ref, pred_x0=p0_ref)
    # full trajectories with the toy model
    for S, cfg_scale in ((10, 1.0), (50, 1.0), (10, 5.0)):
        ref = RH.make_cpu_sampler(shim)
        x_T = W.seeded_randn((3, 4, 8, 8), 91)
        c = W.seeded_randn((3, 5, 6), 92)
        uc = W.seeded_randn((3, 5, 6), 93) if cfg_scale != 1.0 else None
        import contextlib
        import io
        with RH.quiet(), contextlib.redirect_stderr(io.StringIO()):
            z_ref, inter = ref.sample(S=S, batch_size=3, shape=(4, 8, 8), conditioning=c, verbose=False, x_T=x_T, eta=0.,
                                      unconditional_guidance_scale=cfg_scale, unconditional_conditioning=uc)
        orc = R.DDIMOracle(shim)
        z, inter_o = orc.sample(S, 3, (4, 8, 8), conditioning=c, eta=0., x_T=x_T,
                                unconditional_guidance_scale=cfg_scale, unconditional_conditioning=uc)
        assert torch.equal(z, z_ref), "DDIM trajectory restatement is not bit-exact"
        assert len(inter["x_inter"]) == len(inter_o["x_inter"])
        out["traj.S%d.cfg%g" % (S, cfg_scale)] = dict(x_T=x_T, c=c, uc=uc, z=z_ref, n_inter=len(inter["x_inter"]),
                                                      last_pred_x0=inter["pred_x0"][-1])
    save("ddim.pt", out)


def gen_ddim_mask():
    """Inpainting branch of ddim_sampling (ldm/diffusion/ddim.py:144-149): the reference sampler driven with mask / x0 and a
    model shim whose q_sample restates LatentDiffusion.q_sample (ldm/diffusion/ddpm.py:407-412; the class itself needs
    pytorch_lightning and cannot be imported) with a FIXED noise tensor, so the trajectory is reproducible on any device."""
    import contextlib
    import io
    out = {}
    ac = R.sd_alphas_cumprod()
    for S, cm in ((10, 1), (20, 4)):
        x_T = W.seeded_randn((2, 4, 8, 8), 101)
        x0 = W.seeded_randn((2, 4, 8, 8), 102)
        fixed = torch.from_numpy(np.random.Generator(np.random.PCG64(103)).random(size=(2, 4, 8, 8)).astype(np.float32))
        mask = (W.seeded_randn((2, cm, 8, 8), 104) > 0).float()
        c = W.seeded_randn((2, 5, 6), 105)

        def make_shim():
            sh = R.ModelShim(toy_model_fn, ac)
            base = sh.q_sample
            sh.q_sample = lambda xs, t, noise=None: base(xs, t, noise=fixed)
            return sh
        ref = RH.make_cpu_sampler(make_shim())
        with RH.quiet(), contextlib.redirect_stderr(io.StringIO()):
            z_ref, _ = ref.sample(S=S, batch_size=2, shape=(4, 8, 8), conditioning=c, verbose=False, x_T=x_T, eta=0., mask=mask, x0=x0)
        orc = R.DDIMOracle(make_shim())
        z, _ = orc.sample(S, 2, (4, 8, 8), conditioning=c, eta=0., x_T=x_T, mask=mask, x0=x0)
        assert torch.equal(z, z_ref), "inpainting trajectory restatement is not bit-exact"
        out["traj_mask.S%d.cm%d" % (S, cm)] = dict(x_T=x_T, x0=x0, q_noise=fixed, mask=mask, c=c, z=z_ref)
    save("ddim_mask.pt", out)


CLIP_TINY_CFG = dict(vocab_size=1000, hidden_size=128, intermediate_size=256, num_hidden_layers=2, num_attention_heads=2,
                     max_position_embeddings=77, layer_norm_eps=1e-5, hidden_act="quick_gelu")
CLIP_L14_CFG = dict(vocab_size=49408, hidden_size=768, intermediate_size=3072, num_hidden_layers=12, num_attention_heads=12,
                    max_position_embeddings=77, layer_norm_eps=1e-5, hidden_act="quick_gelu")


def gen_clip(name, cfg, B, seed):
    """'next' row f2: the text tower FrozenCLIPEmbedder calls (clip_encoder/modules.py:246-252) = HuggingFace CLIPTextModel, run
    here from the installed transformers package with procedurally generated weights; the restatement is asserted equal."""
    import transformers
    from transformers import CLIPTextConfig, CLIPTextModel
    hf = CLIPTextModel(CLIPTextConfig(**cfg)).eval()
    ks = W.key_shapes_of(hf)
    sd = W.make_state_dict(ks, seed)
    missing = hf.load_state_dict(sd, strict=False)
    assert not missing.unexpected_keys and all("position_ids" in k for k in missing.missing_keys), missing
    rng = np.random.Generator(np.random.PCG64(seed + 1))
    ids = torch.from_numpy(rng.integers(0, cfg["vocab_size"], size=(B, 77), dtype=np.int64))
    ids[:, 0] = cfg["vocab_size"] - 2            # BOS / EOS ids of the CLIP vocabulary layout
    ids[:, -1] = cfg["vocab_size"] - 1
    with torch.no_grad():
        z_ref = hf(input_ids=ids).last_hidden_state
        z_or = R.clip_text_forward(sd, cfg, ids)
        z64 = R.clip_text_forward({k: v.double() for k, v in sd.items()}, cfg, ids)
    err = R.rel_l2(z_or, z_ref)
    print("%s: restatement vs transformers %s CLIPTextModel rel-L2 = %.3e (z std %.3f); fp32 library vs f64 %.3e"
          % (name, transformers.__version__, err, float(z_ref.std()), R.rel_l2(z_ref, z64)))
    assert err < 2e-5, err
    save(name + ".pt", dict(cfg=cfg, seed=seed, key_shapes=ks, ids=ids, z_ref=z_ref.clone(), z_f64=z64.float().clone(), restate_err=err,
                            transformers_version=transformers.__version__))


def gen_ddpm():
    net = RH.build_ddpm_unet()
    ks = W.key_shapes_of(net)
    sd = W.make_state_dict(ks, 11)
    net.load_state_dict(sd, strict=True)
    x = W.seeded_randn((2, 3, 32, 32), 12)
    t = torch.tensor([500, 3], dtype=torch.long)
    with torch.no_grad():
        y_ref = net(x, t)
        y_or = R.ddpm_unet_forward(sd, x, t)
    err = R.rel_l2(y_or, y_ref)
    print("ddpm_unet: restatement vs reference rel-L2 = %.3e (out std %.3f)" % (err, float(y_ref.std())))
    assert err < 2e-5, err
    out = dict(seed=11, key_shapes=ks, x_shape=tuple(x.shape), t=t, y_ref=y_ref.clone(), restate_err=err)
    # config C1: DDIM-50, B=4, eta=0, reference sampler + reference UNet, end to end
    import contextlib
    import io
    sys.path.insert(0, os.path.join(RH.REF, "DDPM"))
    shim = R.ModelShim(lambda xx, tt, cc: net(xx, tt), R.ddpm_alphas_cumprod())
    ref = RH.make_cpu_sampler(shim)
    x_T = W.seeded_randn((4, 3, 32, 32), 13)
    with torch.no_grad(), RH.quiet(), contextlib.redirect_stderr(io.StringIO()):
        z_ref, _ = ref.sample(S=50, batch_size=4, shape=(3, 32, 32), conditioning=None, verbose=False, x_T=x_T, eta=0.)
    rec = []
    orc = R.DDIMOracle(R.ModelShim(lambda xx, tt, cc: R.ddpm_unet_forward(sd, xx, tt), R.ddpm_alphas_cumprod()))
    with torch.no_grad():
        z_or, _ = orc.sample(50, 4, (3, 32, 32), eta=0., x_T=x_T, record=rec)
    err = R.rel_l2(z_or, z_ref)
    print("C1 DDIM-50 B=4: restatement vs reference rel-L2 = %.3e" % err)
    assert err < 1e-4, err
    out["c1_x_T_seed"] = 13
    out["c1_z_ref"] = z_ref.clone()
    # teacher-forced per-step eps for three steps of the reference trajectory
    out["c1_steps"] = [dict(x_t=rec[i][0].clone(), t=rec[i][1], e_t=rec[i][2].clone()) for i in (0, 25, 49)]
    save("ddpm_unet.pt", out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--part", default="all")
    a = ap.parse_args()
    assert RH.available(), "reference tree not found at %s" % RH.REF
    torch.set_num_threads(os.cpu_count() or 1)
    if a.part in ("all", "ddim"):
        gen_ddim()
    if a.part in ("all", "unet"):
        gen_unet("unet_tiny", TINY_UNET_CFG, B=2, HW=16, S_ctx=7, seed=21, t_values=[981, 1], with_f64=True)
        gen_unet("unet_sd", R.SD_UNET_CFG, B=1, HW=64, S_ctx=77, seed=31, t_values=[500], with_f64=True)
    if a.part in ("all", "vae"):
        gen_vae("vae_tiny", TINY_VAE_DDCONFIG, B=2, zres=8, seed=41, with_f64=True)
        gen_vae("vae_sd_z16", R.SD_VAE_DDCONFIG, B=1, zres=16, seed=51, with_f64=True)
    if a.part in ("all", "unet_var"):
        for i, (name, cfg) in enumerate(VARIANT_UNET_CFGS.items()):
            gen_unet_variant(name, cfg, seed=81 + 10 * i)
    if a.part in ("all", "vae_enc"):
        gen_vae_enc("vae_enc_tiny", TINY_VAE_DDCONFIG, B=2, res=32, seed=61)
    if a.part in ("all", "clip"):
        gen_clip("clip_text_tiny", CLIP_TINY_CFG, B=2, seed=111)
        gen_clip("clip_text_l14", CLIP_L14_CFG, B=2, seed=121)
    if a.part in ("all", "ddim_mask"):
        gen_ddim_mask()
    if a.part in ("all", "sd_full", "sd_traj"):
        gen_sd_traj()
    if a.part in ("all", "sd_full", "vae_full"):
        gen_vae_full()
    if a.part in ("all", "sd_full", "unet_96"):
        gen_unet_96()
    if a.part == "ddpm":
        gen_ddpm()
    if a.part == "all":   # the DDPM tree's top-level `models` package clashes with ldm's aliases
        subprocess.check_call([sys.executable, os.path.abspath(__file__), "--part", "ddpm"])


if __name__ == "__main__":
    main()
