"""CPU: the oracle restatement (oracle/restate.py) against the golden fixtures produced by the
UNMODIFIED reference (oracle/make_golden.py).  This is what pins the oracle."""
import numpy as np
import pytest
import torch

from oracle import restate as R
from oracle import weights as W
from oracle.golden import load_golden


def _sd(g):
    return W.make_state_dict(g["key_shapes"], g["seed"])


@pytest.mark.parametrize("name", ["unet_tiny", "unet_sd"])
def test_unet_restatement_matches_reference(name):
    g = load_golden(name + ".pt")
    sd = _sd(g)
    x = W.seeded_randn(g["x_shape"], g["seed"] + 1)
    ctx = W.seeded_randn(g["ctx_shape"], g["seed"] + 2)
    with torch.no_grad():
        eps = R.unet_forward(sd, g["cfg"], x, g["t"], ctx)
    assert R.rel_l2(eps, g["eps_ref"]) < 1e-5          # fp32 restatement vs fp32 reference
    assert R.rel_l2(g["eps_ref"], g["eps_f64"]) < 1e-5  # reference's own fp32 noise floor vs float64
    assert float(g["eps_ref"].abs().max()) > 0.1        # zero_module layers really were re-initialised


@pytest.mark.parametrize("name", ["vae_tiny", "vae_sd_z16"])
def test_vae_restatement_matches_reference(name):
    g = load_golden(name + ".pt")
    sd = _sd(g)
    z = W.seeded_randn(g["z_shape"], g["seed"] + 1)
    with torch.no_grad():
        img = R.autoencoder_decode(sd, g["ddconfig"], z)
    assert R.rel_l2(img, g["img_ref"]) < 1e-5
    assert R.rel_l2(g["img_ref"], g["img_f64"]) < 1e-5


def test_full_size_fixtures_match_reference():
    """The fixtures of BASELINE configs C2 / C3 / C5 AT THEIR OWN SIZE (oracle/make_golden.py --part sd_full ran the unmodified
    reference: DDIM-50 trajectory + 512x512 decode, a 64x64-latent decode, a 96x96-latent UNet step): the restatement
    reproduces one stored trajectory step, and the recorded restatement-vs-reference errors are at the fp32 noise floor."""
    g = load_golden("sd_traj.pt")
    assert g["restate_err"] < 1e-5 and g["restate_err_img"] < 1e-5
    assert [s["i"] for s in g["steps"]] == [0, 12, 25, 37, 49] and len(g["all_t"]) == 50 and g["all_t"][0] == 981 and g["all_t"][-1] == 1
    assert tuple(g["img_shape"]) == (1, 3, 512, 512) and tuple(g["z_ref"].shape) == (1, 4, 64, 64)
    assert float((g["img_ref_s"].abs() <= 1).float().mean()) > 0.9        # PSNR on the clamp-255 scale is not saturated
    st = g["steps"][2]
    sd = W.make_state_dict(g["unet_key_shapes"], g["unet_seed"])
    ctx = W.seeded_randn((1, 77, 768), g["ctx_seed"])
    with torch.no_grad():
        e = R.unet_forward(sd, g["cfg"], st["x_t"], torch.tensor([st["t"]]), ctx)
    assert R.rel_l2(e, st["e_t"]) < 1e-5
    # the trajectory's first input is the seeded x_T, and DDIM's update links consecutive stored quantities
    assert torch.equal(g["steps"][0]["x_t"], W.seeded_randn((1, 4, 64, 64), g["x_T_seed"]))
    gv = load_golden("vae_sd_z64.pt")
    assert gv["restate_err"] < 1e-5 and R.rel_l2(gv["img_ref_s"], gv["img_f64_s"]) < 1e-5 and tuple(gv["img_shape"]) == (1, 3, 512, 512)
    g9 = load_golden("unet_sd_96.pt")
    assert g9["restate_err"] < 1e-5 and R.rel_l2(g9["eps_ref"], g9["eps_f64"]) < 1e-5 and tuple(g9["eps_ref"].shape) == (1, 4, 96, 96)


@pytest.mark.parametrize("name", ["unet_var_legacy", "unet_var_neworder"])
def test_unet_variant_restatement_matches_reference(name):
    """'next' row f4: AttentionBlock (both attention orders), scale-shift norm, resblock_updown, class conditioning."""
    g = load_golden(name + ".pt")
    sd = _sd(g)
    x = W.seeded_randn(g["x_shape"], g["seed"] + 1)
    with torch.no_grad():
        eps = R.unet_forward(sd, g["cfg"], x, g["t"], None, y=g["y"])
    assert R.rel_l2(eps, g["eps_ref"]) < 1e-5
    assert R.rel_l2(g["eps_ref"], g["eps_f64"]) < 1e-5
    assert float(g["eps_ref"].abs().max()) > 0.1


def test_vae_encoder_restatement_matches_reference():
    """'next' row f3: Encoder + quant_conv + posterior moments, and stochastic_encode, against the reference's outputs."""
    g = load_golden("vae_enc_tiny.pt")
    sd = _sd(g)
    x = W.seeded_randn(g["x_shape"], g["seed"] + 1)
    with torch.no_grad():
        mean, logvar, std = R.autoencoder_encode(sd, g["ddconfig"], x)
    assert R.rel_l2(mean, g["mean_ref"]) < 1e-5 and R.rel_l2(logvar, g["logvar_ref"]) < 1e-5 and R.rel_l2(std, g["std_ref"]) < 1e-5
    assert R.rel_l2(g["mean_ref"], g["mean_f64"]) < 1e-5
    assert torch.allclose(mean + std * g["noise"], g["z_ref"], rtol=1e-5, atol=1e-6)
    o = R.DDIMOracle(R.ModelShim(lambda x, t, c: x, R.sd_alphas_cumprod()))
    o.make_schedule(20, ddim_eta=0.0)
    ts = torch.full((x.shape[0],), g["t_enc"], dtype=torch.long)
    zt = R.q_sample_ddim(g["z_ref"], g["enc_noise"], o.ddim_alphas, o.ddim_sqrt_one_minus_alphas, ts)
    assert torch.equal(zt, g["zt_ref"])


def test_ddpm_unet_restatement_matches_reference():
    g = load_golden("ddpm_unet.pt")
    sd = _sd(g)
    x = W.seeded_randn(g["x_shape"], 12)
    with torch.no_grad():
        y = R.ddpm_unet_forward(sd, x, g["t"])
    assert R.rel_l2(y, g["y_ref"]) < 1e-5
    st = g["c1_steps"][1]
    with torch.no_grad():
        e = R.ddpm_unet_forward(sd, st["x_t"], torch.full((4,), st["t"], dtype=torch.long))
    assert R.rel_l2(e, st["e_t"]) < 1e-5


def test_ddim_tables_and_steps_bit_exact():
    g = load_golden("ddim.pt")
    for sched, ac in (("sd", R.sd_alphas_cumprod()), ("ddpm", R.ddpm_alphas_cumprod())):
        for S, eta in ((50, 0.0), (50, 0.5), (10, 0.0), (20, 1.0)):
            o = R.DDIMOracle(R.ModelShim(lambda x, t, c: x, ac))
            o.make_schedule(S, ddim_eta=eta)
            tag = "%s.S%d.eta%g" % (sched, S, eta)
            assert np.array_equal(o.ddim_timesteps, g[tag + ".timesteps"].numpy())
            coefs = torch.cat([torch.stack([c.flatten() for c in o.coefficients(i)], 1) for i in range(S)], 0)
            assert torch.equal(coefs, g[tag + ".coefs"])
    assert list(g["sd.S50.eta0.timesteps"][:3].numpy()) == [1, 21, 41] and int(g["sd.S50.eta0.timesteps"][-1]) == 981


def test_ddim_trajectory_bit_exact():
    from oracle.make_golden import toy_model_fn
    g = load_golden("ddim.pt")
    shim = R.ModelShim(toy_model_fn, R.sd_alphas_cumprod())
    for S, cfg in ((10, 1.0), (50, 1.0), (10, 5.0)):
        t = g["traj.S%d.cfg%g" % (S, cfg)]
        z, inter = R.DDIMOracle(shim).sample(S, 3, (4, 8, 8), conditioning=t["c"], eta=0., x_T=t["x_T"],
                                             unconditional_guidance_scale=cfg, unconditional_conditioning=t["uc"])
        assert torch.equal(z, t["z"])
        assert len(inter["x_inter"]) == t["n_inter"]


@pytest.mark.parametrize("name", ["clip_text_tiny"])
def test_clip_text_restatement_matches_library(name):
    """'next' row f2: the CLIP text tower restatement against HuggingFace CLIPTextModel's output (the fixture), and — when the
    transformers package is importable — against the library run here on the same procedurally generated weights."""
    g = load_golden(name + ".pt")
    sd = _sd(g)
    with torch.no_grad():
        z = R.clip_text_forward(sd, g["cfg"], g["ids"])
    assert R.rel_l2(z, g["z_ref"]) < 1e-5 and R.rel_l2(g["z_ref"], g["z_f64"]) < 1e-5
    # causality: changing a later token never changes an earlier position
    ids2 = g["ids"].clone()
    ids2[:, 40:] = (ids2[:, 40:] + 7) % g["cfg"]["vocab_size"]
    with torch.no_grad():
        z2 = R.clip_text_forward(sd, g["cfg"], ids2)
    assert torch.equal(z2[:, :40], z[:, :40]) and not torch.equal(z2[:, 40:], z[:, 40:])
    try:
        from transformers import CLIPTextConfig, CLIPTextModel
    except Exception:
        return
    hf = CLIPTextModel(CLIPTextConfig(**g["cfg"])).eval()
    hf.load_state_dict(sd, strict=False)
    with torch.no_grad():
        assert R.rel_l2(hf(input_ids=g["ids"]).last_hidden_state, g["z_ref"]) < 1e-5
