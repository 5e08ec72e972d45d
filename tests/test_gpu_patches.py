"""GPU: LatentDiffusion's split_input_params branch — sdb_patch_unfold / sdb_patch_fold, apply_model, decode_first_stage and
encode_first_stage on crops run as one batch — bit for bit against the reference's per-crop loop.

The restatement below is written from CompVis latent-diffusion's LatentDiffusion (ldm/diffusion/ddpm.py: get_fold_unfold,
apply_model's split branch, decode_first_stage / encode_first_stage with patch_distributed_vq); it is not pinned to a
reference checkout, none being available to this repository's fixtures.  It runs with torch on the same GPU: F.unfold, one
call of the SAME sdb200 module per crop, torch.stack, * weighting, F.fold, / normalization.  The weighting is the
reference's expression restated in tests/test_patches_host.py."""
import pytest
import torch
import torch.nn.functional as F

from oracle import weights as W
from oracle.golden import load_golden
from test_patches_host import SPLIT, _bits, ref_get_weighting

pytestmark = pytest.mark.gpu

IMAGE_KEYS = ("image", "LR_image", "segmentation", "bbox_img")


# ---- the reference's branches, restated ---------------------------------------------------------------------------------
def ref_get_fold_unfold(sp, x, kernel_size, stride, uf=1, df=1):
    bs, nc, h, w = x.shape
    Ly = (h - kernel_size[0]) // stride[0] + 1
    Lx = (w - kernel_size[1]) // stride[1] + 1
    unfold = lambda t: F.unfold(t, kernel_size, dilation=1, padding=0, stride=stride)
    if uf == 1 and df == 1:
        fks, fst, out = kernel_size, stride, (h, w)
    elif uf > 1:
        fks, fst, out = (kernel_size[0] * uf, kernel_size[0] * uf), (stride[0] * uf, stride[1] * uf), (h * uf, w * uf)
    else:
        fks, fst, out = (kernel_size[0] // df, kernel_size[0] // df), (stride[0] // df, stride[1] // df), (h // df, w // df)
    fold = lambda t: F.fold(t, out, fks, dilation=1, padding=0, stride=fst)
    f = uf if uf > 1 else 1
    kh, kw = (kernel_size[0] * f, kernel_size[1] * f) if df == 1 else (kernel_size[0] // df, kernel_size[1] // df)
    weighting = ref_get_weighting(sp, kh, kw, Ly, Lx).to(x.device).to(x.dtype)
    normalization = fold(weighting).view(1, 1, *out)
    weighting = weighting.view((1, 1, kh, kw, Ly * Lx))
    return fold, unfold, normalization, weighting


def ref_apply_model(ld, x_noisy, t, cond):
    if not isinstance(cond, dict):
        if not isinstance(cond, list):
            cond = [cond]
        cond = {("c_concat" if ld.model.conditioning_key == "concat" else "c_crossattn"): cond}
    sp = ld.split_input_params
    assert len(cond) == 1
    ks, stride = sp["ks"], sp["stride"]
    fold, unfold, normalization, weighting = ref_get_fold_unfold(sp, x_noisy, ks, stride)
    z = unfold(x_noisy)
    z = z.view((z.shape[0], -1, ks[0], ks[1], z.shape[-1]))
    z_list = [z[:, :, :, :, i] for i in range(z.shape[-1])]
    if ld.cond_stage_key in IMAGE_KEYS and ld.model.conditioning_key:
        c_key = next(iter(cond.keys()))
        c = next(iter(cond.values()))
        assert len(c) == 1
        c = unfold(c[0])
        c = c.view((c.shape[0], -1, ks[0], ks[1], c.shape[-1]))
        cond_list = [{c_key: [c[:, :, :, :, i]]} for i in range(c.shape[-1])]
    else:
        cond_list = [cond for i in range(z.shape[-1])]
    output_list = [ld.model(z_list[i], t, **cond_list[i]) for i in range(z.shape[-1])]
    o = torch.stack(output_list, axis=-1)
    o = o * weighting
    o = o.view((o.shape[0], -1, o.shape[-1]))
    return fold(o) / normalization


def ref_first_stage(ld, x, fn, uf=1, df=1):
    sp = ld.split_input_params
    ks, stride = sp["ks"], sp["stride"]
    bs, nc, h, w = x.shape
    if ks[0] > h or ks[1] > w:
        ks = (min(ks[0], h), min(ks[1], w))
    if stride[0] > h or stride[1] > w:
        stride = (min(stride[0], h), min(stride[1], w))
    fold, unfold, normalization, weighting = ref_get_fold_unfold(sp, x, ks, stride, uf=uf, df=df)
    z = unfold(x)
    z = z.view((z.shape[0], -1, ks[0], ks[1], z.shape[-1]))
    o = torch.stack([fn(z[:, :, :, :, i]) for i in range(z.shape[-1])], axis=-1)
    o = o * weighting
    o = o.view((o.shape[0], -1, o.shape[-1]))
    return fold(o) / normalization


def ref_decode(ld, z, force_not_quantize=False):
    from sdb200.autoencoder import VQModelInterface
    z = 1. / ld.scale_factor * z
    fs = ld.first_stage_model
    fn = (lambda v: fs.decode(v, force_not_quantize=force_not_quantize)) if isinstance(fs, VQModelInterface) else fs.decode
    return ref_first_stage(ld, z, fn, uf=ld.split_input_params["vqf"])


def _sp(**kw):
    return dict(SPLIT, **kw)


# ---- 1. kernels ----------------------------------------------------------------------------------------------------------
GRIDS = [  # (H, W, ks, stride): stride < ks, = ks, > ks, ragged edges, non-square, a single crop
    (16, 16, (8, 8), (4, 4)), (16, 16, (8, 8), (8, 8)), (17, 19, (5, 5), (7, 6)), (18, 15, (6, 4), (3, 5)),
    (12, 12, (12, 12), (4, 4)), (40, 24, (16, 8), (8, 4)), (10, 13, (4, 4), (3, 3))]


@pytest.mark.parametrize("H,W,ks,stride", GRIDS)
@pytest.mark.parametrize("B,C", [(1, 1), (2, 3), (3, 6)])
def test_patch_unfold_bit_exact(cuda, H, W, ks, stride, B, C):
    from sdb200 import ops
    x = torch.randn(B, C, H, W, device="cuda")
    got = ops.patch_unfold(x, ks, stride)
    u = F.unfold(x, ks, stride=stride)
    L = u.shape[-1]
    u = u.view(B, C, ks[0], ks[1], L)
    assert got.shape == (L * B, C, ks[0], ks[1])
    for l in range(L):
        assert torch.equal(got[l * B:(l + 1) * B], u[..., l])


def _fold_case(B, C, H, W, ks, stride, uf=1, df=1, tie=False, seed=0):
    """(crops o in the kernel's layout, the restated reference's fold(o * weighting) / normalization, fold args)."""
    from sdb200.pipeline import LatentDiffusion
    sp = _sp(tie_braker=tie)
    x = torch.zeros(B, C, H, W, device="cuda")
    fold, _, normalization, weighting = ref_get_fold_unfold(sp, x, ks, stride, uf=uf, df=df)
    kh, kw = weighting.shape[2:4]
    L = weighting.shape[-1]
    g = torch.Generator(device="cuda").manual_seed(seed)
    o5 = torch.randn(B, C, kh, kw, L, device="cuda", generator=g)
    ref = fold((o5 * weighting).view(B, -1, L)) / normalization
    o = o5.permute(4, 0, 1, 2, 3).contiguous().view(L * B, C, kh, kw)
    ld = LatentDiffusion(first_stage_config=False, unet=torch.nn.Identity())
    ld.split_input_params = sp
    geo = ld._split_geometry(H, W, ks, stride, uf=uf, df=df)
    wpix, wcrop = ld._patch_weights(kh, kw, geo[0][0], geo[0][1], "cuda")
    return o, ref, (B, geo[0], geo[2], geo[3], wpix, wcrop), o5, weighting, fold, normalization


@pytest.mark.parametrize("H,W,ks,stride", GRIDS)
@pytest.mark.parametrize("B,C", [(1, 1), (2, 3), (3, 6)])
@pytest.mark.parametrize("tie", [False, True])
def test_patch_fold_bit_exact(cuda, H, W, ks, stride, B, C, tie):
    from sdb200 import ops
    o, ref, args, *_ = _fold_case(B, C, H, W, ks, stride, tie=tie, seed=H * W + B)
    got = ops.patch_fold(o, *args)
    assert _bits(got, ref)
    if not tie:                                                   # (a 1-crop-wide grid has 0/0 tie weights: NaN throughout)
        uncovered = stride[0] > ks[0] or stride[1] > ks[1] or (H - ks[0]) % stride[0] or (W - ks[1]) % stride[1]
        assert bool(got.isnan().any()) == bool(uncovered)         # pixels no crop covers are 0/0


@pytest.mark.parametrize("mode", [dict(uf=4, H=16, W=16, ks=(8, 8), stride=(4, 4)), dict(uf=4, H=64, W=64, ks=(32, 32), stride=(16, 16)),
                                  dict(df=4, H=64, W=64, ks=(32, 32), stride=(16, 16)), dict(df=4, H=128, W=96, ks=(32, 32), stride=(32, 16))])
@pytest.mark.parametrize("tie", [False, True])
def test_patch_fold_vqf_sizes(cuda, mode, tie):
    from sdb200 import ops
    m = dict(mode)
    o, ref, args, *_ = _fold_case(2, 3, m.pop("H"), m.pop("W"), m.pop("ks"), m.pop("stride"), tie=tie, **m)
    assert _bits(ops.patch_fold(o, *args), ref)


def test_patch_fold_nan_crop_and_graph(cuda):
    from sdb200 import ops
    o, ref, args, o5, weighting, fold, normalization = _fold_case(2, 3, 16, 16, (8, 8), (4, 4))
    o5 = o5.clone()
    o5[1, 2, 0, 0, 4] = float("nan")                             # crop l = 4 (centre), its top-left pixel (4, 4)
    o = o5.permute(4, 0, 1, 2, 3).contiguous().view(-1, 3, 8, 8)
    got = ops.patch_fold(o, *args)
    ref = fold((o5 * weighting).view(2, -1, 9)) / normalization
    assert _bits(got, ref)
    nan = got.isnan()
    assert int(nan.sum()) == 1 and bool(nan[1, 2, 4, 4])        # only where that crop covers that pixel
    # CUDA graph capture and replay with new crops
    static = o.clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ops.patch_fold(static, *args)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = ops.patch_fold(static, *args)
    o2 = torch.randn_like(o)
    static.copy_(o2)
    g.replay()
    assert _bits(out, ops.patch_fold(o2, *args))


# ---- 2. apply_model --------------------------------------------------------------------------------------------------------
def _concat_ld(mode, cond_stage_key="LR_image"):
    from sdb200.pipeline import LatentDiffusion
    g = load_golden("unet_var_neworder.pt")
    cfg = dict(g["cfg"], in_channels=6, out_channels=3)
    ld = LatentDiffusion(unet_config=cfg, first_stage_config=False, conditioning_key="concat", compute_mode=mode,
                         scale_factor=1.0, channels=3, image_size=16, cond_stage_key=cond_stage_key)
    ld.model.diffusion_model.load_state_dict(W.make_state_dict(W.key_shapes_of(ld.model.diffusion_model), g["seed"]))
    ld.split_input_params = _sp(ks=(8, 8), stride=(4, 4), vqf=4)
    return ld.cuda()


def _xattn_ld(mode, graph):
    from sdb200.pipeline import LatentDiffusion
    g = load_golden("unet_tiny.pt")
    ld = LatentDiffusion(unet_config=dict(g["cfg"]), first_stage_config=False, conditioning_key="crossattn", compute_mode=mode,
                         cond_stage_key="txt")
    ld.model.diffusion_model.load_state_dict(W.make_state_dict(W.key_shapes_of(ld.model.diffusion_model), g["seed"]))
    ld.model.diffusion_model.use_cuda_graph = graph
    ld.split_input_params = _sp(ks=(8, 8), stride=(4, 4), tie_braker=True)
    return ld.cuda()


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("pb", [None, 1, 5])
def test_apply_model_concat_bit_exact(cuda, mode, pb):
    ld = _concat_ld(mode)
    ld.patch_batch = pb
    x = W.seeded_randn((2, 3, 16, 16), 91).cuda()
    c = W.seeded_randn((2, 3, 16, 16), 92).cuda()
    t = torch.tensor([999, 17], device="cuda")
    got = ld.apply_model(x, t, c)
    ref = ref_apply_model(ld, x, t, c)
    assert torch.isfinite(got).all() and _bits(got, ref)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("pb", [None, 1, 5])
def test_apply_model_crossattn_bit_exact(cuda, mode, graph, pb):
    ld = _xattn_ld(mode, graph)
    ld.patch_batch = pb
    x = W.seeded_randn((2, 4, 16, 16), 93).cuda()
    ctx = W.seeded_randn((2, 7, 64), 94).cuda()
    t = torch.tensor([500, 3], device="cuda")
    got = ld.apply_model(x, t, ctx)
    got2 = ld.apply_model(x, t, ctx)
    ref = ref_apply_model(ld, x, t, ctx)
    assert torch.isfinite(got).all() and _bits(got, ref) and _bits(got2, ref)


@pytest.mark.parametrize("pb", [None, 5])
def test_context_projection_once_per_conditioning(cuda, pb):
    ld = _xattn_ld("bf16", True)
    ld.patch_batch = pb
    x = W.seeded_randn((2, 4, 16, 16), 95).cuda()
    ctx = W.seeded_randn((2, 7, 64), 96).cuda()
    t = torch.tensor([700, 300], device="cuda")
    ld.apply_model(x, t, ctx)                                    # captures the graphs
    replays = []
    orig = torch.cuda.CUDAGraph.replay
    torch.cuda.CUDAGraph.replay = lambda self: replays.append(1) or orig(self)
    try:
        ctx2 = ctx + 1                                            # a new conditioning: one projection per chunk shape
        for _ in range(4):
            ld.apply_model(x, t, ctx2)
    finally:
        torch.cuda.CUDAGraph.replay = orig
    chunks = 1 if pb is None else 2
    print("patch_batch=%s: %d replays over 4 steps" % (pb, len(replays)))
    assert len(replays) == 4 * chunks + chunks


# ---- 3. first stage --------------------------------------------------------------------------------------------------------
def _vq(mode="fp32"):
    from sdb200.autoencoder import VQModelInterface
    from test_gpu_vq import VQ_DD
    m = VQModelInterface(3, ddconfig=dict(VQ_DD, attn_type="none"), lossconfig=None, n_embed=8192, compute_mode=mode)
    m.load_state_dict(W.make_state_dict(W.key_shapes_of(m), 41))
    return m.cuda()


def _ld_with(fs, vqf, scale_factor=1.0, **sp):
    from sdb200.pipeline import LatentDiffusion
    ld = LatentDiffusion(first_stage_config=False, first_stage_model=fs, unet=torch.nn.Identity(), scale_factor=scale_factor)
    ld.split_input_params = _sp(vqf=vqf, **sp)
    return ld.cuda()


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_decode_first_stage_vq_bit_exact(cuda, mode):
    ld = _ld_with(_vq(mode), 4, scale_factor=0.5, ks=(8, 8), stride=(4, 4))
    z = W.seeded_randn((2, 3, 16, 16), 97).cuda()
    for fnq in (False, True):
        got = ld.decode_first_stage(z, force_not_quantize=fnq)
        assert got.shape == (2, 3, 64, 64) and torch.isfinite(got).all()
        assert _bits(got, ref_decode(ld, z, force_not_quantize=fnq))
    ld.first_stage_model.micro_batch = 5
    assert _bits(ld.decode_first_stage(z), ref_decode(ld, z))


def test_decode_first_stage_kl_and_identity_bit_exact(cuda):
    from sdb200.autoencoder import AutoencoderKL, IdentityFirstStage
    gv = load_golden("vae_tiny.pt")
    vae = AutoencoderKL(ddconfig=gv["ddconfig"], embed_dim=4, compute_mode="bf16")
    vae.load_state_dict(W.make_state_dict(gv["key_shapes"], gv["seed"]), strict=False)
    ld = _ld_with(vae.cuda(), 2, scale_factor=0.18215, ks=(8, 8), stride=(4, 4), tie_braker=True)
    z = W.seeded_randn((2, 4, 16, 16), 98).cuda()
    got = ld.decode_first_stage(z)
    assert got.shape == (2, 3, 32, 32) and _bits(got, ref_decode(ld, z))
    ld = _ld_with(IdentityFirstStage(), 1, ks=(6, 6), stride=(3, 3))
    got = ld.decode_first_stage(z)
    assert _bits(got, ref_decode(ld, z))
    assert _bits(ld.encode_first_stage(z), got)                    # vqf = 1: encode folds the same crops


def test_encode_first_stage_vq_bit_exact(cuda):
    ld = _ld_with(_vq("bf16"), 4, ks=(32, 32), stride=(16, 16))
    x = W.seeded_randn((2, 3, 64, 64), 99).cuda()
    got = ld.encode_first_stage(x)
    assert ld.split_input_params["original_image_size"] == (64, 64)
    ref = ref_first_stage(ld, x, ld.first_stage_model.encode, df=4)
    assert got.shape == (2, 3, 16, 16) and torch.isfinite(got).all() and _bits(got, ref)


# ---- 4. end to end: a tiny SR-style LDM (concat, VQ first stage, 3 x 3 crops) ---------------------------------------------
def _sr_ldm():
    ld = _concat_ld("bf16")
    ld.first_stage_model = _vq("bf16")
    return ld


class _Restated:
    """Runs `fn` with ld.apply_model replaced by the restated per-crop loop (the sampler code is the same)."""

    def __init__(self, ld):
        self.ld = ld

    def __enter__(self):
        self.ld.apply_model = lambda x, t, c, return_ids=False: ref_apply_model(self.ld, x, t, c)

    def __exit__(self, *a):
        del self.ld.apply_model


def test_sr_ldm_ddim_cfg_p_sample_loop_and_decode(cuda):
    ld = _sr_ldm()
    B = 2
    lr = W.seeded_randn((B, 3, 16, 16), 101).cuda()
    ulr = torch.zeros_like(lr)
    x_T = W.seeded_randn((B, 3, 16, 16), 102).cuda()
    calls = []
    model_fwd = ld.model.forward
    ld.model.forward = lambda x, t, **kw: calls.append(x.shape[0]) or model_fwd(x, t, **kw)
    res = {}
    for name in ("batched", "restated"):
        ctx = _Restated(ld) if name == "restated" else None
        if ctx:
            ctx.__enter__()
        try:
            calls.clear()
            torch.manual_seed(5)
            z, _ = ld.sample_log(lr, B, ddim=True, ddim_steps=10, shape=(3, 16, 16), x_T=x_T, eta=0.5,
                                 unconditional_guidance_scale=2.0, unconditional_conditioning=ulr)
            n_ddim = list(calls)
            za = ld.p_sample_loop(lr, (B, 3, 16, 16), x_T=z, timesteps=5, verbose=False)
            after = torch.randn(4, device="cuda")
            res[name] = (z, za, after, n_ddim)
        finally:
            if ctx:
                ctx.__exit__()
    zb, zab, ab, nb = res["batched"]
    zr, zar, ar, nr = res["restated"]
    assert nb == [2 * B * 9] * 10 and nr == [2 * B] * 90           # one 2B call over 9 crops per step, against 9 calls
    assert _bits(zb, zr) and _bits(zab, zar) and torch.equal(ab, ar)
    img = ld.decode_first_stage(zab)
    assert img.shape == (B, 3, 64, 64) and torch.isfinite(img).all() and _bits(img, ref_decode(ld, zab))


def test_split_step_and_decode_make_no_host_sync(cuda):
    from sdb200.ddim import DDIMSampler
    ld = _sr_ldm()
    lr = W.seeded_randn((2, 3, 16, 16), 103).cuda()
    ulr = torch.zeros_like(lr)
    x = W.seeded_randn((2, 3, 16, 16), 104).cuda()
    smp = DDIMSampler(ld)
    smp.make_schedule(5, ddim_eta=0.5, verbose=False)
    ts = torch.full((2,), 333, device="cuda", dtype=torch.long)
    smp.derived_coefficients(2)
    smp.p_sample_ddim(x, lr, ts, index=2, unconditional_guidance_scale=2.0, unconditional_conditioning=ulr)
    ld.decode_first_stage(x)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        x1, _ = smp.p_sample_ddim(x, lr, ts, index=2, unconditional_guidance_scale=2.0, unconditional_conditioning=ulr)
        img = ld.decode_first_stage(x1)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert torch.isfinite(img).all()
