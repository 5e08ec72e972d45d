"""CPU: host-side logic of the drop-in modules (no kernels are launched here)."""
import numpy as np
import pytest
import torch
from torch import nn

from oracle import restate as R
from oracle import weights as W
from oracle.golden import load_golden


def _keys(m):
    return [(k, tuple(v.shape)) for k, v in m.state_dict().items()]


def test_unet_state_dict_keys_match_reference():
    from sdb200.openai_model import UNetModel
    for name in ("unet_tiny", "unet_sd"):
        g = load_golden(name + ".pt")
        with torch.device("meta"):
            m = UNetModel(**g["cfg"])
        assert _keys(m) == [(k, tuple(s)) for k, s in g["key_shapes"]]


def test_vae_state_dict_keys_match_reference():
    from sdb200.autoencoder import AutoencoderKL
    ge = load_golden("vae_enc_tiny.pt")
    for name in ("vae_tiny", "vae_sd_z16"):
        g = load_golden(name + ".pt")
        with torch.device("meta"):
            m = AutoencoderKL(ddconfig=g["ddconfig"], embed_dim=4)
        dec_side = sorted(k for k in _keys(m) if k[0].startswith(("decoder.", "post_quant_conv.")))
        assert dec_side == sorted((k, tuple(s)) for k, s in g["key_shapes"])
        if name == "vae_tiny":       # same ddconfig as the encoder fixture: the union is the reference AutoencoderKL's key set
            assert sorted(_keys(m)) == sorted([(k, tuple(s)) for k, s in g["key_shapes"]] + [(k, tuple(s)) for k, s in ge["key_shapes"]])


def test_ddpm_unet_state_dict_keys_match_reference():
    from sdb200.ddpm_unet import UNet
    g = load_golden("ddpm_unet.pt")
    with torch.device("meta"):
        m = UNet(image_size=32, input_channels=3)
    assert _keys(m) == [(k, tuple(s)) for k, s in g["key_shapes"]]


def test_unsupported_options_raise():
    from sdb200.openai_model import UNetModel
    base = dict(image_size=8, in_channels=4, model_channels=32, out_channels=4, num_res_blocks=1, attention_resolutions=[1],
                num_heads=2)
    with pytest.raises(NotImplementedError):
        UNetModel(**base, use_spatial_transformer=True, context_dim=8, n_embed=16)      # codebook head
    with pytest.raises(NotImplementedError):
        UNetModel(**base, use_spatial_transformer=True, context_dim=8, dims=3)
    with pytest.raises(AssertionError):
        UNetModel(**base, use_spatial_transformer=True)                # context_dim missing (reference assert, model.py:317-318)
    with pytest.raises(AssertionError):
        UNetModel(**base, context_dim=8)                               # context without the spatial transformer (model.py:320-321)


def test_unet_variant_state_dict_keys_match_reference():
    """'next' row f4: AttentionBlock / scale-shift / resblock_updown / class-conditional variants keep the reference's keys."""
    from sdb200.openai_model import UNetModel
    for name in ("unet_var_legacy", "unet_var_neworder"):
        g = load_golden(name + ".pt")
        with torch.device("meta"):
            m = UNetModel(**g["cfg"])
        assert _keys(m) == [(k, tuple(s)) for k, s in g["key_shapes"]]


def test_sampler_schedule_bit_exact_vs_reference_tables():
    from sdb200.ddim import DDIMSampler
    g = load_golden("ddim.pt")
    for sched, ac in (("sd", R.sd_alphas_cumprod()), ("ddpm", R.ddpm_alphas_cumprod())):
        shim = R.ModelShim(lambda x, t, c: x, ac)
        for S, eta in ((50, 0.0), (50, 0.5), (10, 0.0), (20, 1.0)):
            s = DDIMSampler(shim)
            s.make_schedule(S, ddim_eta=eta, verbose=False)
            tag = "%s.S%d.eta%g" % (sched, S, eta)
            assert np.array_equal(s.ddim_timesteps, g[tag + ".timesteps"].numpy())
            got = torch.tensor([s.coefficients(i) for i in range(S)], dtype=torch.float64)
            assert torch.equal(got, g[tag + ".coefs"].double())        # the four fp32 scalars, bit for bit
    with pytest.raises(NotImplementedError):
        DDIMSampler(shim).make_schedule(10, ddim_discretize="nope", verbose=False)


def test_pipeline_schedule_matches_oracle():
    from sdb200.pipeline import LatentDiffusion, make_beta_schedule
    ac = np.cumprod(1. - make_beta_schedule("linear", 1000, 0.00085, 0.0120), axis=0)
    assert np.array_equal(ac, R.sd_alphas_cumprod())


def test_geglu_packing_roundtrip():
    from sdb200 import ops
    inner, K, bn = 256, 64, 128
    torch.manual_seed(0)
    w = torch.randn(2 * inner, K)
    b = torch.randn(2 * inner)
    wp, bp = ops.pack_geglu_weight(w, b, bn)
    h = bn // 2
    x = torch.randn(5, K)
    ref = (x @ w[:inner].T + b[:inner]) * torch.nn.functional.gelu(x @ w[inner:].T + b[inner:])
    y = x @ wp.T + bp
    tiles = y.reshape(5, -1, 2, h)
    got = (tiles[:, :, 0] * torch.nn.functional.gelu(tiles[:, :, 1])).reshape(5, inner)
    assert torch.allclose(got, ref, atol=1e-4, rtol=1e-5)


def test_conv_weight_packing():
    from sdb200 import ops
    w = torch.randn(6, 4, 3, 3)
    p = ops.pack_conv_weight(w, torch.float32)
    assert p.shape == (9, 6, 4)
    assert torch.equal(p[1 * 3 + 2], w[:, :, 1, 2])


def test_shard_range_and_per_sample_seeds():
    from sdb200.distributed import per_sample_randn, shard_range
    for B, Wd in ((64, 8), (10, 4), (3, 8), (0, 2)):
        spans = [shard_range(B, r, Wd) for r in range(Wd)]
        assert spans[0][0] == 0 and spans[-1][1] == B
        assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
        assert max(h - l for l, h in spans) - min(h - l for l, h in spans) <= 1
    full = per_sample_randn(range(6), (2, 3), 1000)
    parts = torch.cat([per_sample_randn(range(*shard_range(6, r, 4)), (2, 3), 1000) for r in range(4)], 0)
    assert torch.equal(full, parts)


def test_upsample_weight_folding_is_exact():
    """nearest-2x upsample + conv3x3(pad 1) == four 2x2 phase convs with the folded taps (ops.fold_upsample_weights);
    checked in float64 on the CPU (no kernels involved: this is the host-side weight transform)."""
    import torch.nn.functional as F
    from sdb200 import ops
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2, 5, 6, 7, generator=g, dtype=torch.float64)
    w = torch.randn(4, 5, 3, 3, generator=g, dtype=torch.float64)
    ref = F.conv2d(F.interpolate(x, scale_factor=2, mode="nearest"), w, padding=1)
    wf = ops.fold_upsample_weights(w, torch.float64)
    out = torch.zeros_like(ref)
    xp = F.pad(x, (1, 1, 1, 1))
    H, W = x.shape[2:]
    for p_, (py, px) in enumerate(ops.UP2_PHASES):
        k = wf[p_].reshape(2, 2, 4, 5).permute(2, 3, 0, 1)
        out[:, :, py::2, px::2] = F.conv2d(xp[:, :, py:py + H + 1, px:px + W + 1], k)
    assert float((out - ref).abs().max()) < 1e-5      # the fold itself runs in fp32


def test_launch_plan_table_is_well_formed():
    from sdb200.tc_plans import PLANS
    assert len(PLANS) > 10
    for key, (variant, bn, sk, best_us, auto_us) in PLANS.items():
        assert key[0] in ("conv", "gemm") and len(key) == 10
        assert variant in (1, 2) and bn in (32, 64, 128, 160, 256) and 1 <= sk <= 16
        assert not (variant == 2 and bn < 128)
        assert best_us <= auto_us


def test_next_row_modules_have_no_cpu_fallback():
    """'next' rows f3 / f4 run on the same kernels: CPU tensors raise instead of silently computing in PyTorch."""
    from sdb200 import _lib, ops
    from sdb200.autoencoder import DiagonalGaussianDistribution
    with pytest.raises(_lib.SdbError):
        DiagonalGaussianDistribution(torch.zeros(1, 8, 2, 2))
    with pytest.raises(_lib.SdbError):
        ops.q_sample(torch.zeros(2, 4), torch.zeros(2, 4), torch.ones(2), torch.ones(2))
    with pytest.raises(_lib.SdbError):
        ops.avgpool2x2(torch.zeros(1, 2, 2, 4))
    with pytest.raises(_lib.SdbError):
        ops.scale_shift_affine(torch.ones(4), torch.zeros(4), torch.zeros(2, 8))


def test_bench_reference_arm_line(monkeypatch, capsys):
    """bench.py --impl reference: one JSON line with the sdb200 arm's metric / unit / workload, steps and warm-up honoured,
    e2e == value with zero copy bytes, cpu_baseline describing the run (the timed sample itself is stubbed here)."""
    import json
    import sys
    import bench
    calls = []

    def fake(ddim_steps, repeats=1):
        calls.append(ddim_steps)
        return 1.0 / (ddim_steps * 2.0 + 4.0), 16, 2.0, 4.0
    monkeypatch.setattr(bench, "cpu_reference_images_per_s", fake)
    monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--gpus", "2", "--steps", "3", "--warmup", "2"])
    monkeypatch.setenv("RANK", "0")
    bench.main()
    out = [l for l in capsys.readouterr().out.splitlines() if l.startswith("{")]
    assert len(out) == 1 and len(calls) == 5
    d = json.loads(out[0])
    assert d["impl"] == "reference" and d["metric"] == "512px DDIM-50 images/sec" and d["unit"] == "images/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 2 and d["steps"] == 3 and d["warmup"] == 2
    assert d["config"]["workload"] == "SD-1.x UNet DDIM-50 + VAE decode, 64x64x4 latent -> 512x512x3, ctx 77x768, batch 8 per GPU"
    assert abs(d["value"] - 1.0 / 104.0) < 1e-12 and abs(d["ms_per_step"] - 8 * 104.0 * 1000.0) < 1e-6
    assert d["e2e"] == {"value": d["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == 16 and d["cpu_baseline"]["value"] == d["value"]
    # every other rank exits without work
    monkeypatch.setenv("RANK", "1")
    bench.main()
    assert capsys.readouterr().out.strip() == ""


def test_bench_dump_outputs(tmp_path, monkeypatch):
    """bench.py --dump-outputs: one float32 .npy per output, whole while they fit the size limit; above it, each output is
    replaced by the same share of its values at fixed, distinct positions."""
    import sys
    import bench
    from oracle.golden import sample_flat, sample_index
    z, img = torch.randn(2, 4, 8, 8), torch.randn(2, 3, 16, 16, dtype=torch.float64)
    bench.dump_outputs(str(tmp_path / "whole"), {"latents": z, "images": img})
    got = np.load(tmp_path / "whole" / "images.npy")
    assert got.dtype == np.float32 and np.array_equal(got, img.float().numpy())
    assert np.array_equal(np.load(tmp_path / "whole" / "latents.npy"), z.numpy())
    monkeypatch.setattr(bench, "DUMP_BYTES", 1024)          # 8 KB of outputs -> an eighth of each
    bench.dump_outputs(str(tmp_path / "sampled"), {"latents": z, "images": img})
    lat, ims = np.load(tmp_path / "sampled" / "latents.npy"), np.load(tmp_path / "sampled" / "images.npy")
    assert lat.shape == (64,) and ims.shape == (192,) and (lat.nbytes + ims.nbytes) <= 1024
    assert np.array_equal(lat, sample_flat(z, 64).numpy()) and np.array_equal(ims, sample_flat(img.float(), 192).numpy())
    assert sample_index(3 * 512 * 512, 65536).unique().numel() == 65536
    for argv in (["--config", "c3"], ["--impl", "reference"], ["--steps", "0"]):
        monkeypatch.setattr(sys, "argv", ["bench.py", "--dump-outputs", str(tmp_path / "x")] + argv)
        with pytest.raises(SystemExit):
            bench.parse()


def _tiny_unet():
    from sdb200.openai_model import UNetModel
    return UNetModel(image_size=8, in_channels=4, model_channels=32, out_channels=4, num_res_blocks=1, attention_resolutions=[1],
                     num_heads=2, use_spatial_transformer=True, context_dim=8, channel_mult=(1,))


def test_tensor_memo_is_keyed_on_the_live_tensor():
    """The cross-attention K/V cache (an engine.TensorMemo) must not confuse a new conditioning tensor with a freed one that
    had the same address, shape and version (ADVICE r1: data_ptr()-keyed entries collided after the allocator recycled the
    block), nor keep a projection of a tensor written in place or moved."""
    memo = _tiny_unet()._ctx_cache
    built = []

    def get(t, key):
        return memo.get((t,), key, lambda: built.append(key) or "kv-%d" % len(built))

    a = torch.zeros(2, 7, 8)
    key = ("bf16", 1234, id(a))
    assert get(a, key) == "kv-1" and get(a, key) == "kv-1"     # built once, then a hit
    b = torch.zeros(2, 7, 8)
    assert get(b, key) == "kv-2"                               # same shape / version, different object
    a.add_(1)
    assert get(a, key) == "kv-3"                               # modified in place since it was projected
    del a
    import gc
    gc.collect()
    c = torch.zeros(2, 7, 8)
    assert get(c, key) == "kv-4"                               # even if id() / the address is recycled, the weakref is dead
    lin = nn.Linear(8, 8)
    w = lin.weight
    assert get(w, "w") == "kv-5"
    v0, p0 = w._version, w.data_ptr()
    lin.to(torch.float64)                                      # same Parameter object, same _version, new storage
    assert lin.weight is w and w._version == v0 and w.data_ptr() != p0
    assert get(w, "w") == "kv-6"
    for i in range(400):                                       # bounded: dead entries are dropped, then the memo is cleared
        get(torch.zeros(1), ("k", i))
        assert len(memo._entries) <= 256


def test_weight_packs_are_invalidated_through_a_parent_module():
    """Packed copies / graphs must be dropped when a checkpoint is loaded through a PARENT (nn.Module.load_state_dict recurses
    via _load_from_state_dict and never calls the child's override), when .to() is applied to the parent, and when a
    parameter is written in place (EMA copy_to)."""
    from sdb200.autoencoder import AutoencoderKL
    from sdb200.ddpm_unet import UNet
    from sdb200.engine import PackedConv
    from sdb200.pipeline import LatentDiffusion
    vae_cfg = dict(double_z=True, z_channels=4, resolution=16, in_channels=3, out_ch=3, ch=32, ch_mult=(1,), num_res_blocks=1,
                   attn_resolutions=[], dropout=0.0)
    ld = LatentDiffusion(unet=_tiny_unet(), first_stage_model=AutoencoderKL(ddconfig=vae_cfg, embed_dim=4))
    unet, vae = ld.model.diffusion_model, ld.first_stage_model
    ddpm = UNet(image_size=32)
    ddpm_parent = nn.Sequential(ddpm)

    def poison():
        unet._packed = {"bf16": "stale"}
        unet._graphs = {"k": "stale"}
        vae.decoder._packed = {"bf16": "stale"}
        vae.encoder._packed = {"bf16": "stale"}
        ddpm._packed = {"bf16": "stale"}

    def clean():
        return (unet._packed == {} and unet._graphs == {} and vae.decoder._packed == {} and vae.encoder._packed == {}
                and ddpm._packed == {})

    poison()
    ld.load_state_dict(ld.state_dict())
    ddpm_parent.load_state_dict(ddpm_parent.state_dict())
    assert clean()
    poison()
    ld.to(torch.float32)                                       # _apply on the parent
    ddpm_parent.to(torch.float32)
    assert clean()
    # in-place parameter update: the fingerprint changes, the next forward re-packs
    unet._check_weights()
    unet._packed = {"bf16": "stale"}
    unet._check_weights()
    assert unet._packed == {"bf16": "stale"}                    # nothing changed: kept
    with torch.no_grad():
        unet.out[2].weight.mul_(0.5)
    unet._check_weights()
    assert unet._packed == {}
    vae.decoder._check_weights()
    vae.decoder._packed = {"bf16": "stale"}
    with torch.no_grad():
        vae.decoder.conv_in.weight.add_(1.0)
    vae.decoder._check_weights()
    assert vae.decoder._packed == {}
    ddpm._check_weights()
    ddpm._packed = {"bf16": "stale"}
    with torch.no_grad():
        ddpm.initial_conv.weight.mul_(0.5)
    ddpm._check_weights()
    assert ddpm._packed == {}
    # quant_conv / post_quant_conv are packed per call as views of their parameters: an in-place write reaches the next call
    conv = vae.post_quant_conv
    with torch.no_grad():
        conv.weight.add_(1.0)
    pc = PackedConv(conv.weight, conv.bias, "fp32")
    assert pc.w.untyped_storage().data_ptr() == conv.weight.untyped_storage().data_ptr()
    assert pc.bias.untyped_storage().data_ptr() == conv.bias.untyped_storage().data_ptr()
    assert torch.equal(pc.w.reshape(conv.weight.shape[:2]), conv.weight.detach().reshape(conv.weight.shape[:2]))


def test_sampler_defaults_and_coefficient_cache():
    """consume_rng_like_reference defaults to the reference's behaviour; the derived-coefficient cache belongs to one
    schedule (make_schedule drops it) instead of being tagged by recyclable id()s."""
    from oracle import restate as R
    from sdb200.ddim import DDIMSampler
    shim = R.ModelShim(None, R.sd_alphas_cumprod())
    s = DDIMSampler(shim)
    assert s.consume_rng_like_reference is True
    s.make_schedule(50, ddim_eta=0.0, verbose=False)
    c0 = s.derived_coefficients(10)
    assert c0[3] == 0.0
    s.make_schedule(50, ddim_eta=1.0, verbose=False)
    c1 = s.derived_coefficients(10)
    assert c1[3] > 0.0 and c1[2] != c0[2]                      # sigma and the direction coefficient follow the new eta
    s.make_schedule(20, ddim_eta=0.0, verbose=False)
    assert s.derived_coefficients(10)[0] != c0[0]


def test_ops_reject_foreign_devices():
    """require_cuda: CPU tensors are refused (no fallback) — the device-binding checks need two GPUs and live in the gpu tests."""
    from sdb200 import _lib
    with pytest.raises(_lib.SdbError):
        _lib.require_cuda(torch.zeros(1))


def test_clip_text_state_dict_keys_match_fixture():
    """FrozenCLIPEmbedder.transformer has HuggingFace CLIPTextModel's parameter names and shapes (ViT-L/14 text tower)."""
    from oracle.golden import load_golden
    from sdb200.clip_text import CLIPTextModel, FrozenCLIPEmbedder
    g = load_golden("clip_text_l14.pt")
    with torch.device("meta"):
        m = CLIPTextModel(g["cfg"])
    mine = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    want = {k: tuple(s) for k, s in g["key_shapes"]}
    assert mine == want
    with torch.device("meta"):
        e = FrozenCLIPEmbedder(config=load_golden("clip_text_tiny.pt")["cfg"])
    assert all(not p.requires_grad for p in e.parameters()) and e.max_length == 77
    with pytest.raises(Exception):
        e.transformer(input_ids=torch.zeros(2, 77, dtype=torch.long))       # CPU tensors: no fallback
