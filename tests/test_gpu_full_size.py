"""GPU: the parity claims of BASELINE.json at the FULL Stable-Diffusion-1.x shapes (configs[1] and configs[2]).

The fp32 (SIMT) mode is pinned to the reference at these shapes by test_gpu_models.py (unet_sd / vae_sd_z16 fixtures,
<= 1e-5).  Here the bf16 tensor-core mode runs the whole free-running pipeline — DDIM-50 on a 64x64x4 latent with a
77x768 context, then the 512x512x3 decode — next to the fp32 mode on the same weights, noise and conditioning:
per-step eps (teacher-forced on the fp32 trajectory) <= 1e-2, decoded image PSNR >= 40 dB.
"""
import pytest
import torch

from gpu_util import rel
from oracle import restate as R
from oracle import weights as W
from oracle.golden import load_golden, sample_flat

pytestmark = pytest.mark.gpu


def test_sd_ddim50_decode_bf16_vs_fp32(cuda):
    from sdb200.pipeline import LatentDiffusion
    gu, gv = load_golden("unet_sd.pt"), load_golden("vae_sd_z16.pt")
    ld = LatentDiffusion(unet_config=gu["cfg"], first_stage_config=gv["ddconfig"], compute_mode="fp32")
    ld.model.diffusion_model.load_state_dict(W.make_state_dict(gu["key_shapes"], gu["seed"]))
    r = ld.first_stage_model.load_state_dict(W.make_state_dict(gv["key_shapes"], gv["seed"]), strict=False)
    assert not r.unexpected_keys
    ld = ld.cuda()
    unet, vae = ld.model.diffusion_model, ld.first_stage_model
    B, S = 1, 50
    x_T = W.seeded_randn((B, 4, 64, 64), 2).cuda()
    ctx = W.seeded_randn((B, 77, 768), 3).cuda()

    # fp32 mode: free-running trajectory, recording (x_t, t, eps) of every step
    rec = []
    apply = ld.apply_model

    def recording(x, t, c):
        e = apply(x, t, c)
        rec.append((x.clone(), t.clone(), e.clone()))
        return e
    ld.apply_model = recording
    z32, img32 = ld.txt2img(ctx, B, ddim_steps=S, shape=(4, 64, 64), x_T=x_T)
    ld.apply_model = apply
    assert len(rec) == S and torch.isfinite(img32).all() and img32.shape == (B, 3, 512, 512)

    unet.compute_mode = "bf16"
    vae.compute_mode = "bf16"
    unet.use_cuda_graph = True
    worst = max(rel(ld.apply_model(x, t, ctx), e) for x, t, e in rec[::7] + [rec[-1]])      # teacher-forced per-step eps
    z16, img16 = ld.txt2img(ctx, B, ddim_steps=S, shape=(4, 64, 64), x_T=x_T)
    psnr = R.psnr_255(img16.cpu(), img32.cpu())
    print("SD-1.x DDIM-50 + decode, bf16 vs fp32 mode: worst teacher-forced eps rel-L2 %.3e, final latent rel-L2 %.3e, "
          "image PSNR %.1f dB" % (worst, rel(z16, z32), psnr))
    assert worst <= 1e-2
    assert psnr >= 40.0


def test_sd_vae_decode_full_size(cuda):
    """configs[2] shape: 64x64x4 -> 512x512x3, bf16 against the fp32 mode, and micro-batch invariance at full size."""
    from sdb200.autoencoder import AutoencoderKL
    g = load_golden("vae_sd_z16.pt")
    vae = AutoencoderKL(ddconfig=g["ddconfig"], embed_dim=4, compute_mode="fp32")
    vae.load_state_dict(W.make_state_dict(g["key_shapes"], g["seed"]), strict=False)
    vae = vae.cuda()
    z = W.seeded_randn((3, 4, 64, 64), 4).cuda()
    ref = vae.decode(z[:1])
    vae.compute_mode = "bf16"
    img = vae.decode(z)
    assert img.shape == (3, 3, 512, 512) and torch.isfinite(img).all()
    psnr = R.psnr_255(img[:1].cpu(), ref.cpu())
    print("SD VAE decode 512x512: bf16 vs fp32 mode rel-L2 %.3e, PSNR %.1f dB" % (rel(img[:1], ref), psnr))
    assert psnr >= 40.0
    vae.micro_batch = 2
    assert torch.equal(vae.decode(z), img)


# ---- pinned to the UNMODIFIED reference at the configs' own sizes (fixtures: oracle/make_golden.py --part sd_full) -------------
def _sd_pipeline(mode):
    from sdb200.pipeline import LatentDiffusion
    g = load_golden("sd_traj.pt")
    ld = LatentDiffusion(unet_config=g["cfg"], first_stage_config=g["ddconfig"], compute_mode=mode)
    ld.model.diffusion_model.load_state_dict(W.make_state_dict(g["unet_key_shapes"], g["unet_seed"]))
    r = ld.first_stage_model.load_state_dict(W.make_state_dict(g["vae_key_shapes"], g["vae_seed"]), strict=False)
    assert not r.unexpected_keys
    return g, ld.cuda()


def test_c2_teacher_forced_eps_vs_reference(cuda):
    """BASELINE configs[1] (C2): per-step eps at five steps of the REFERENCE's own DDIM-50 trajectory (reference x_t in,
    reference e_t as the truth): <= 1e-5 in the fp32 mode, <= 1e-2 in the bf16 mode — the north-star's stated tolerances."""
    g, ld = _sd_pipeline("fp32")
    unet = ld.model.diffusion_model
    ctx = W.seeded_randn((1, 77, 768), g["ctx_seed"]).cuda()
    for mode, tol in (("fp32", 1e-5), ("bf16", 1e-2)):
        unet.compute_mode = mode
        errs = []
        for st in g["steps"]:
            e = ld.apply_model(st["x_t"].cuda(), torch.tensor([st["t"]], device="cuda"), ctx)
            errs.append(rel(e, st["e_t"]))
        print("C2 teacher-forced eps vs reference, %s mode, steps %s: %s" % (mode, [s["i"] for s in g["steps"]], ["%.2e" % v for v in errs]))
        assert max(errs) <= tol, (mode, errs)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_c2_free_running_ddim50_image_psnr_vs_reference(cuda, mode):
    """C2 end to end: DDIM-50 from the reference's x_T and context, then the 512x512 decode, free-running, against the
    latent and the IMAGE the unmodified reference produced (PSNR >= 40 dB on the clamp-255 scale, BASELINE.md section 5)."""
    g, ld = _sd_pipeline(mode)
    ld.model.diffusion_model.use_cuda_graph = (mode == "bf16")
    x_T = W.seeded_randn((1, 4, 64, 64), g["x_T_seed"]).cuda()
    ctx = W.seeded_randn((1, 77, 768), g["ctx_seed"]).cuda()
    z, img = ld.txt2img(ctx, 1, ddim_steps=50, shape=(4, 64, 64), x_T=x_T)
    assert tuple(img.shape) == tuple(g["img_shape"])
    img = sample_flat(img, g["img_ref_s"].numel())          # the fixture stores the reference image at these positions
    psnr = R.psnr_255(img, g["img_ref_s"])
    ez, ei = rel(z, g["z_ref"]), rel(img, g["img_ref_s"])
    print("C2 free-running DDIM-50 + decode vs reference, %s mode: latent rel-L2 %.3e, image rel-L2 %.3e, PSNR %.1f dB" % (mode, ez, ei, psnr))
    assert psnr >= 40.0
    if mode == "fp32":
        assert ez <= 1e-4 and ei <= 1e-4          # 50 chained steps of a <= 1e-5 per-step error


def test_c3_vae_decode_512_vs_reference(cuda):
    """BASELINE configs[2] (C3) at its own size: 64x64x4 -> 512x512x3 against the reference Decoder's output.
    fp32 mode <= 1e-5 (vs the float64 restatement and vs the fp32 reference), bf16 mode PSNR >= 40 dB; a batch of 16
    (the config's batch) reproduces the single image bit for bit in every slot."""
    from sdb200.autoencoder import AutoencoderKL
    g = load_golden("vae_sd_z64.pt")
    vae = AutoencoderKL(ddconfig=g["ddconfig"], embed_dim=4, compute_mode="fp32")
    vae.load_state_dict(W.make_state_dict(g["key_shapes"], g["seed"]), strict=False)
    vae = vae.cuda()
    z = W.seeded_randn(g["z_shape"], g["z_seed"]).cuda()
    img32 = vae.decode(z)
    assert tuple(img32.shape) == tuple(g["img_shape"])
    n = g["img_ref_s"].numel()                              # the fixture stores both images at these positions
    e64, eref = rel(sample_flat(img32, n), g["img_f64_s"]), rel(sample_flat(img32, n), g["img_ref_s"])
    vae.compute_mode = "bf16"
    img16 = vae.decode(z)
    psnr = R.psnr_255(sample_flat(img16, n), g["img_ref_s"])
    print("C3 decode 512x512 vs reference: fp32 mode rel-L2 %.3e (vs f64 %.3e), bf16 mode rel-L2 %.3e, PSNR %.1f dB"
          % (eref, e64, rel(sample_flat(img16, n), g["img_ref_s"]), psnr))
    assert e64 <= 1e-5 and eref <= 1e-5
    assert psnr >= 40.0
    img_b = vae.decode(z.repeat(16, 1, 1, 1))
    assert img_b.shape == (16, 3, 512, 512)
    assert all(torch.equal(img_b[i], img16[0]) for i in range(16))


def test_c5_unet_96_vs_reference(cuda):
    """BASELINE configs[4] (C5) at its own size: one UNet step on a 96x96x4 latent (9216 tokens at the top level) against the
    unmodified reference's eps; fp32 <= 1e-5, bf16 <= 1e-2; CUDA-graph replay and a batch of 4 reproduce it."""
    from sdb200.openai_model import UNetModel
    g = load_golden("unet_sd_96.pt")
    net = UNetModel(**g["cfg"], compute_mode="fp32")
    net.load_state_dict(W.make_state_dict(g["key_shapes"], g["seed"]))
    net = net.cuda()
    x = W.seeded_randn(g["x_shape"], g["x_seed"]).cuda()
    ctx = W.seeded_randn(g["ctx_shape"], g["ctx_seed"]).cuda()
    t = g["t"].cuda()
    e32 = net(x, t, ctx)
    net.compute_mode = "bf16"
    e16 = net(x, t, ctx)
    print("C5 96x96 UNet step vs reference: fp32 mode %.3e (vs f64 %.3e), bf16 mode %.3e"
          % (rel(e32, g["eps_ref"]), rel(e32, g["eps_f64"]), rel(e16, g["eps_ref"])))
    assert rel(e32, g["eps_ref"]) <= 1e-5 and rel(e32, g["eps_f64"]) <= 1e-5
    assert rel(e16, g["eps_ref"]) <= 1e-2
    net.use_cuda_graph = True
    assert torch.equal(net(x, t, ctx), e16)
    eb = net(x.repeat(4, 1, 1, 1), t.repeat(4), ctx.repeat(4, 1, 1))
    assert all(torch.equal(eb[i], e16[0]) for i in range(4))
