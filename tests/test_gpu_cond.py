"""GPU: the conditioning stages of sdb200.encoders — sdb_embed_rows, sdb_interpolate_nchw, the x-transformers encoder of
TransformerEmbedder / BERTEmbedder, ClassEmbedder (a one-key context, Sk = 1, in the UNet), SpatialRescaler, and four tiny
LDMs sampled end to end with them (text, class, semantic synthesis, inpainting on a VQ first stage).

The encoder restatement below is written from CompVis latent-diffusion (ldm/modules/x_transformer.py: TransformerWrapper,
Encoder, Attention, FeedForward; ldm/modules/encoders/modules.py) and is not pinned to a reference checkout, none being
available to this repository's fixtures.  It runs in fp64 on the GPU (the 1280 x 32 tower is too slow in fp64 on a CPU)."""
import pytest
import torch
import torch.nn.functional as F

from gpu_util import rel
from oracle import restate as R
from oracle import weights as W
from oracle.golden import load_golden

pytestmark = pytest.mark.gpu

NAN = float("nan")


def _same(a, b):
    a, b = a.cpu(), b.cpu()
    return a.shape == b.shape and bool(((a == b) | (a.isnan() & b.isnan())).all())


# ---- restatements --------------------------------------------------------------------------------------------------------
def xtransformer_ref(sd, depth, ids, p="transformer."):
    """TransformerWrapper(ids, return_embeddings=True) with attn_layers=Encoder(dim, depth), eval, in sd's dtype."""
    D = sd[p + "token_emb.weight"].shape[1]
    B, S = ids.shape
    x = sd[p + "token_emb.weight"][ids] + sd[p + "pos_emb.emb.weight"][:S][None]
    for i in range(2 * depth):
        q_ = "%sattn_layers.layers.%d." % (p, i)
        h = F.layer_norm(x, (D,), sd[q_ + "0.weight"], sd[q_ + "0.bias"], 1e-5)
        if i % 2 == 0:
            q, k, v = (F.linear(h, sd[q_ + "1.to_%s.weight" % n]).view(B, S, 8, 64).transpose(1, 2) for n in "qkv")
            a = torch.softmax((q @ k.transpose(-1, -2)) * 64 ** -0.5, dim=-1) @ v
            out = F.linear(a.transpose(1, 2).reshape(B, S, 512), sd[q_ + "1.to_out.weight"], sd[q_ + "1.to_out.bias"])
        else:
            h = F.gelu(F.linear(h, sd[q_ + "1.net.0.0.weight"], sd[q_ + "1.net.0.0.bias"]))
            out = F.linear(h, sd[q_ + "1.net.2.weight"], sd[q_ + "1.net.2.bias"])
        x = out + x
    return F.layer_norm(x, (D,), sd[p + "norm.weight"], sd[p + "norm.bias"], 1e-5)


# ---- 1. sdb_embed_rows ----------------------------------------------------------------------------------------------------
def test_embed_rows_bits_and_bad_ids(cuda):
    from sdb200 import ops
    table = W.seeded_randn((1000, 96), 1).cuda()
    pos = W.seeded_randn((77, 96), 2).cuda()
    for B, S in ((1, 77), (8, 77), (3, 20)):
        ids = torch.randint(0, 1000, (B, S), generator=torch.Generator().manual_seed(B * S)).cuda()
        out = ops.embed_rows(table, ids.reshape(-1), pos=pos, seq_len=S)
        assert torch.equal(out, (table[ids] + pos[:S][None]).reshape(B * S, 96))
        assert torch.equal(ops.embed_rows(table, ids.reshape(-1)), table[ids.reshape(-1)])
    ids = torch.tensor([5, -1, 7, 1000, 2 ** 40, 999], device="cuda")
    for p in (pos, None):
        out = ops.embed_rows(table, ids, pos=p, seq_len=6 if p is not None else 0)
        torch.cuda.synchronize()
        ref = table[ids.clamp(0, 999)] + (pos[:6] if p is not None else 0)
        ref[[1, 3, 4]] = NAN
        assert _same(out, ref)


# ---- 2. the x-transformers encoder ----------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def big_state():
    from sdb200 import encoders as E
    m = E.BERTEmbedder(1280, 32, use_tokenizer=False)
    sd = W.make_state_dict(W.key_shapes_of(m), 301)
    return sd


@pytest.mark.parametrize("size", ["tiny", "1280x32"])
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_encoder_against_restatement(cuda, size, mode, request):
    from sdb200 import encoders as E
    if size == "tiny":
        n_embed, n_layer, vocab = 64, 2, 100
        bert = E.BERTEmbedder(n_embed, n_layer, vocab, use_tokenizer=False, compute_mode=mode)
        sd = W.make_state_dict(W.key_shapes_of(bert), 302)
    else:
        n_embed, n_layer, vocab = 1280, 32, 30522
        bert = E.BERTEmbedder(n_embed, n_layer, use_tokenizer=False, compute_mode=mode)
        sd = request.getfixturevalue("big_state")
    bert.load_state_dict(sd, strict=True)
    bert = bert.cuda()
    tr = E.TransformerEmbedder(n_embed, n_layer, vocab, compute_mode=mode)
    tr.load_state_dict(sd, strict=True)
    tr = tr.cuda()
    sd64 = {k: v.double().cuda() for k, v in sd.items() if "to_logits" not in k}
    for B in (1, 8):
        for S in (77, 20):
            ids = torch.randint(0, vocab, (B, S), generator=torch.Generator().manual_seed(1000 * B + S)).cuda()
            z = bert(ids)
            with torch.no_grad():
                ref = xtransformer_ref(sd64, n_layer, ids)
            e = rel(z, ref)
            print("encoder %s %s B=%d S=%d: rel-L2 %.3e" % (size, mode, B, S, e))
            assert z.shape == (B, S, n_embed) and z.dtype == torch.float32
            assert e <= (1e-5 if mode == "fp32" else 1e-2)
            assert torch.equal(bert.encode(ids), z) and torch.equal(tr(ids), z) and torch.equal(tr.encode(ids), z)
            if S == 77:             # no mask: a late token changes the first position
                ids2 = ids.clone()
                ids2[:, 60] = (ids2[:, 60] + 1) % vocab
                z2 = bert(ids2)
                assert not torch.equal(z2[:, 0], z[:, 0])
    # a warmed call makes no host sync
    ids = torch.randint(0, vocab, (8, 77), generator=torch.Generator().manual_seed(5)).cuda()
    bert(ids)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        z = bert(ids)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert torch.isfinite(z).all()


# ---- 3. ClassEmbedder and a one-key context in the UNet -------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("graph", [False, True])
def test_class_embedder_sk1_unet(cuda, mode, graph):
    from sdb200 import encoders as E
    from sdb200.openai_model import UNetModel
    ce = E.ClassEmbedder(64, n_classes=10)
    sdc = W.make_state_dict(W.key_shapes_of(ce), 311)
    ce.load_state_dict(sdc, strict=True)
    ce = ce.cuda()
    cls = torch.tensor([3, 9], device="cuda")
    c = ce({"class": cls})
    assert c.shape == (2, 1, 64) and torch.equal(c, sdc["embedding.weight"].cuda()[cls][:, None])
    assert torch.equal(ce({"label": cls}, key="label"), c)
    bad = ce({"class": torch.tensor([3, 10, -1], device="cuda")})
    assert torch.equal(bad[0], c[0]) and bad[1:].isnan().all()
    g = load_golden("unet_tiny.pt")
    cfg = dict(g["cfg"])
    net = UNetModel(**cfg, compute_mode=mode)
    sd = W.make_state_dict(W.key_shapes_of(net), g["seed"])
    net.load_state_dict(sd)
    net = net.cuda()
    net.use_cuda_graph = graph
    x = W.seeded_randn((2, 4, 16, 16), 312)
    t = torch.tensor([10, 700])
    for _ in range(2 if graph else 1):
        eps = net(x.cuda(), t.cuda(), context=c)
    with torch.no_grad():
        ref = R.unet_forward({k: v.double() for k, v in sd.items()}, cfg, x.double(), t, c.double().cpu())
    e = rel(eps, ref)
    print("UNet with a [2, 1, 64] ClassEmbedder context %s graph=%s: rel-L2 %.3e" % (mode, graph, e))
    assert e <= (1e-5 if mode == "fp32" else 1e-2)


# ---- 4. sdb_interpolate_nchw ----------------------------------------------------------------------------------------------
def _ulps(a, b):
    """max |a - b| in units of b's last place (fp32)."""
    a, b = a.float(), b.float()
    ulp = (torch.nextafter(b.abs(), torch.full_like(b, float("inf"))) - b.abs()).clamp_min(torch.finfo(torch.float32).tiny)
    return float(((a - b).abs() / ulp).max())


def _check_interp(out, ref, mode, what, worst):
    assert out.shape == ref.shape, what
    if mode in ("nearest", "area"):
        assert torch.equal(out, ref), what
    else:
        u = _ulps(out, ref)
        worst[mode] = max(worst.get(mode, 0.0), u)
        assert u <= 2.0, "%s: %.1f ulp" % (what, u)


def test_interpolate_against_torch(cuda):
    from sdb200 import encoders as E
    from sdb200 import ops
    worst, worst_map = {}, 0.0
    for shape in ((2, 182, 64, 64), (3, 3, 37, 53)):
        x = W.seeded_randn(shape, sum(shape)).cuda()
        C = shape[1]
        for method in ("nearest", "bilinear", "bicubic", "area"):
            # size=: one stage, with and without the map
            for size in ((23, 41), (shape[2] * 2 - 3, shape[3] + 5)):
                ref = F.interpolate(x, size=size, mode=method)
                _check_interp(ops.interpolate(x, size=size, mode=method), ref, method, "%s size=%s %s" % (method, size, shape),
                              worst)
            for mult in (0.5, 0.25, 2, 0.75):
                for n_stages in (0, 1, 2):
                    for remap in (False, True):
                        m = E.SpatialRescaler(n_stages, method, mult, in_channels=C, out_channels=3 if remap else None,
                                              bias=remap and mult == 2)
                        if remap:
                            m.load_state_dict(W.make_state_dict(W.key_shapes_of(m), 321))
                        m = m.cuda()
                        out = m(x)
                        ref = x
                        for _ in range(n_stages):
                            ref = F.interpolate(ref, scale_factor=mult, mode=method)
                        what = "%s x%s stages=%d map=%s %s" % (method, mult, n_stages, remap, shape)
                        if not remap:
                            _check_interp(out, ref, method, what, worst)
                            continue
                        w = m.channel_mapper.weight.double().reshape(3, C)
                        ref64 = torch.einsum("oc,nchw->nohw", w, ref.double())
                        if m.channel_mapper.bias is not None:
                            ref64 = ref64 + m.channel_mapper.bias.double()[None, :, None, None]
                        e = rel(out, ref64)
                        worst_map = max(worst_map, e)
                        assert out.shape == ref64.shape and e <= 1e-6, "%s: rel-L2 %.3e" % (what, e)
    print("interpolate vs torch CUDA: max ulp %s; with the channel map max rel-L2 vs fp64 %.3e" % (worst, worst_map))


# ---- 5. end to end ---------------------------------------------------------------------------------------------------------
def _ldm(cfg_name, key, mode, first_stage_model=None, ld_kw=None, **over):
    from sdb200.pipeline import LatentDiffusion
    g = load_golden(cfg_name + ".pt")
    cfg = dict(g["cfg"], **over)
    ld = LatentDiffusion(unet_config=cfg, first_stage_config=False, first_stage_model=first_stage_model, conditioning_key=key,
                         compute_mode=mode, **(ld_kw or {}))
    sd = W.make_state_dict(W.key_shapes_of(ld.model.diffusion_model), g["seed"])
    ld.model.diffusion_model.load_state_dict(sd)
    return ld, sd, cfg


def _sample_and_check(ld, sd, cfg, key, c, uc, c_ref, uc_ref, shape, mode, what, x_seed):
    from test_gpu_conditioning import DictDDIMOracle, _anc_oracle, _restated_wrapper
    k = "c_concat" if key == "concat" else "c_crossattn"
    x_T = W.seeded_randn((2,) + shape, x_seed)
    fn = _restated_wrapper(sd, cfg, key)
    cd, ucd = {k: [c]}, (None if uc is None else {k: [uc]})
    crd, ucrd = {k: [c_ref.float().cpu()]}, (None if uc_ref is None else {k: [uc_ref.float().cpu()]})
    scale = 1.0 if uc is None else 4.0
    torch.manual_seed(41)
    z, _ = ld.sample_log(cd, 2, ddim=True, ddim_steps=10, shape=shape, x_T=x_T.cuda(), eta=0.0,
                         unconditional_guidance_scale=scale, unconditional_conditioning=ucd)
    torch.manual_seed(41)
    orc = DictDDIMOracle(R.ModelShim(fn, R.sd_alphas_cumprod()))
    with torch.no_grad():
        z_ref, _ = orc.sample(10, 2, shape, conditioning=crd, eta=0.0, x_T=x_T, unconditional_guidance_scale=scale,
                              unconditional_conditioning=ucrd)
    e = rel(z, z_ref)
    msg = "%s %s: DDIM-10 CFG %.1f latent rel-L2 %.3e" % (what, mode, scale, e)
    assert e <= (1e-5 if mode == "fp32" else 2e-2), msg
    if mode == "fp32":
        torch.manual_seed(42)
        za = ld.p_sample_loop(cd, (2,) + shape, x_T=x_T.cuda(), timesteps=8)
        torch.manual_seed(42)
        with torch.no_grad():
            za_ref, _ = _anc_oracle(fn).p_sample_loop(crd, x_T, 8)
        ea = rel(za, za_ref)
        msg += ", p_sample_loop latent rel-L2 %.3e" % ea
        assert ea <= 1e-4, msg
    print(msg)
    return z


def _kl_first_stage(mode):
    from sdb200.autoencoder import AutoencoderKL
    g = load_golden("vae_tiny.pt")
    fs = AutoencoderKL(ddconfig=g["ddconfig"], embed_dim=4, compute_mode=mode)
    sd = W.make_state_dict(W.key_shapes_of(fs), g["seed"])
    fs.load_state_dict(sd)
    return fs.cuda(), g, {k: v.double() for k, v in sd.items()}


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_text_ldm(cuda, mode):
    from sdb200 import encoders as E
    from test_gpu_vq import _image_check
    fs, g, sdv = _kl_first_stage(mode)
    te = E.TransformerEmbedder(64, 2, 100, compute_mode=mode)
    sdt = W.make_state_dict(W.key_shapes_of(te), 331)
    te.load_state_dict(sdt, strict=True)
    ld, sd, cfg = _ldm("unet_tiny", "crossattn", mode, first_stage_model=fs)
    ld.cond_stage_model = te
    ld = ld.cuda()
    ids = torch.randint(1, 100, (2, 77), generator=torch.Generator().manual_seed(332))
    pad = torch.zeros_like(ids)
    c, uc = ld.get_learned_conditioning(ids.cuda()), ld.get_learned_conditioning(pad.cuda())
    sd64 = {k: v.double().cuda() for k, v in sdt.items()}
    c_ref, uc_ref = xtransformer_ref(sd64, 2, ids.cuda()), xtransformer_ref(sd64, 2, pad.cuda())
    z = _sample_and_check(ld, sd, cfg, "crossattn", c, uc, c_ref, uc_ref, (4, 8, 8), mode, "text LDM", 333)
    img = ld.decode_first_stage(z)
    with torch.no_grad():
        _image_check(img, R.autoencoder_decode(sdv, g["ddconfig"], (1. / ld.scale_factor * z).double().cpu()), mode,
                     "text LDM KL decode")


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_class_ldm(cuda, mode):
    from sdb200 import encoders as E
    ce = E.ClassEmbedder(64, n_classes=10)
    sdc = W.make_state_dict(W.key_shapes_of(ce), 341)
    ce.load_state_dict(sdc, strict=True)
    ld, sd, cfg = _ldm("unet_tiny", "crossattn", mode)
    ld.cond_stage_model = ce
    ld = ld.cuda()
    cls = torch.tensor([2, 7])
    c = ld.get_learned_conditioning({"class": cls.cuda()})
    uc = ld.get_learned_conditioning({"class": torch.tensor([9, 9], device="cuda")})
    tab = sdc["embedding.weight"]
    _sample_and_check(ld, sd, cfg, "crossattn", c, uc, tab[cls][:, None], tab[[9, 9]][:, None], (4, 8, 8), mode,
                      "class LDM (Sk = 1)", 342)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_semantic_synthesis_ldm(cuda, mode):
    from sdb200 import encoders as E
    sr = E.SpatialRescaler(n_stages=2, method="bilinear", multiplier=0.5, in_channels=182, out_channels=3)
    sr.load_state_dict(W.make_state_dict(W.key_shapes_of(sr), 351), strict=True)
    ld, sd, cfg = _ldm("unet_var_neworder", "concat", mode, in_channels=7)
    ld.cond_stage_model = sr
    ld = ld.cuda()
    seg = F.one_hot(torch.randint(0, 182, (2, 64, 64), generator=torch.Generator().manual_seed(352)), 182)
    seg = seg.permute(0, 3, 1, 2).float().contiguous()
    c = ld.get_learned_conditioning(seg.cuda())
    h = F.interpolate(F.interpolate(seg.cuda(), scale_factor=0.5, mode="bilinear"), scale_factor=0.5, mode="bilinear")
    c_ref = torch.einsum("oc,nchw->nohw", sr.channel_mapper.weight.double().reshape(3, 182), h.double())
    assert rel(c, c_ref) <= 1e-6
    _sample_and_check(ld, sd, cfg, "concat", c, None, c_ref, None, (4, 16, 16), mode, "semantic-synthesis LDM", 353)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_inpainting_ldm_first_stage_as_cond_stage(cuda, mode):
    from sdb200 import ops
    from test_gpu_vq import _dd, _first_stage, encoder_ref
    fs, sdv = _first_stage("VQModelInterface", _dd("none"), mode)
    ld, sd, cfg = _ldm("unet_var_neworder", "concat", mode, first_stage_model=fs, in_channels=7, out_channels=3,
                       ld_kw=dict(cond_stage_config="__is_first_stage__", scale_factor=1.0, channels=3, image_size=16))
    assert ld.cond_stage_model is fs
    ld = ld.cuda()
    image = W.seeded_randn((2, 3, 64, 64), 361)
    mask = (W.seeded_randn((2, 1, 64, 64), 362) > 0).float()
    masked = (1 - mask) * image
    c = ld.get_learned_conditioning(masked.cuda())
    cm = ops.interpolate(mask.cuda(), size=c.shape[-2:], mode="nearest")
    assert torch.equal(cm, F.interpolate(mask.cuda(), size=c.shape[-2:], mode="nearest"))
    c = torch.cat([c, cm], 1)
    with torch.no_grad():
        h_ref = R._conv(sdv, "quant_conv", encoder_ref(sdv, _dd("none"), masked.double()))
    c_ref = torch.cat([h_ref, cm.double().cpu()], 1)
    _sample_and_check(ld, sd, cfg, "concat", c, None, c_ref, None, (3, 16, 16), mode, "inpainting LDM", 363)
