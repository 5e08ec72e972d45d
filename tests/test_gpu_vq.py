"""GPU: the VQ-regularised first stage — sdb_vq_quantize / sdb_vq_codebook_gather, VectorQuantizer2, VQModel /
VQModelInterface, and a VQ latent-diffusion model end to end.

The quantizer restatement below is written from taming's VectorQuantizer2.forward (ldm/tamming/quantize.py:213-311,
eval, legacy=True); it is not pinned to a reference checkout, none being available to this repository's fixtures.
Index rule: distances are recomputed in fp64; a row whose two best codes are within 1e-5 * (|z|^2 + |e_best|^2) is a
near tie and may take either code, every other row must take the fp64 argmin.  Images are then restated from the
kernel's own indices, so a legitimate near tie cannot fail an image comparison."""
import pytest
import torch
import torch.nn.functional as F

from gpu_util import rel
from oracle import restate as R
from oracle import weights as W
from oracle.golden import load_golden

pytestmark = pytest.mark.gpu

VQ_DD = dict(double_z=False, z_channels=3, resolution=64, in_channels=3, out_ch=3, ch=64, ch_mult=(1, 2, 4),
             num_res_blocks=1, attn_resolutions=[], dropout=0.0)


def _same(a, b):
    a, b = a.cpu(), b.cpu()
    return a.shape == b.shape and bool(((a == b) | (a.isnan() & b.isnan())).all())


def _rows(z, layout):
    """[M, D] rows in (n, h, w) order."""
    return (z.permute(0, 2, 3, 1) if layout == "nchw" else z).reshape(-1, z.shape[1 if layout == "nchw" else 3])


def index_rule(zf, Wc, idx, chunk=4096):
    """(rows breaking the index rule, near-tie rows): fp64 distances on the device, checker side."""
    z64, w64, idx = zf.double().cuda(), Wc.double().cuda(), idx.reshape(-1).cuda()
    ee = (w64 ** 2).sum(1)
    bad = ties = 0
    for r0 in range(0, z64.shape[0], chunk):
        zc = z64[r0:r0 + chunk]
        zz = (zc ** 2).sum(1)
        d = zz[:, None] + ee[None] - 2 * zc @ w64.T
        dmin, amin = d.min(1)
        tol = 1e-5 * (zz + ee[amin])
        got = d.gather(1, idx[r0:r0 + chunk, None]).squeeze(1)
        bad += int((~((got - dmin) <= tol)).sum())
        ties += int(((d <= (dmin + tol)[:, None]).sum(1) > 1).sum())
    return bad, ties


def quantize_ref(z, Wc, beta=0.25, idx=None):
    """VectorQuantizer2.forward (legacy) on the host, NCHW fp32 z: indices from fp64 distances unless the kernel's `idx` is
    given; returns (z_q = z + (W[idx] - z) in fp32, fp64 loss, idx)."""
    z, Wc = z.cpu(), Wc.cpu()
    zf = _rows(z, "nchw")
    if idx is None:
        z64, w64 = zf.double(), Wc.double()
        idx = ((z64 ** 2).sum(1, keepdim=True) + (w64 ** 2).sum(1) - 2 * z64 @ w64.T).argmin(1)
    idx = idx.reshape(-1).cpu()
    e = Wc[idx]
    zq = (zf + (e - zf)).reshape(z.shape[0], z.shape[2], z.shape[3], -1).permute(0, 3, 1, 2).contiguous()
    loss = ((e.double() - zf.double()) ** 2).mean() * (1 + beta)
    return zq, float(loss), idx


# ---- 1. the kernel ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [1, 8])
@pytest.mark.parametrize("n_e", [1, 17, 8192, 16384])
@pytest.mark.parametrize("D", [1, 3, 4, 16])
def test_vq_quantize_index_rule_zq_bits_and_loss(cuda, D, n_e, N):
    from sdb200 import ops
    g = torch.Generator().manual_seed(1000 * D + n_e + N)
    z = torch.randn(N, D, 64, 64, generator=g)
    Wc = torch.randn(n_e, D, generator=g) * 0.7
    zf = _rows(z, "nchw")
    zg, Wg = z.cuda(), Wc.cuda()
    inputs = {"nchw": zg, "nhwc": zg.permute(0, 2, 3, 1).contiguous()}
    idx0 = None
    for zl, zin in inputs.items():
        for ql in ("nchw", "nhwc"):
            zq, idx, loss = ops.vq_quantize(zin, Wg, beta=0.25, z_layout=zl, zq_layout=ql)
            if idx0 is None:
                idx0 = idx
                bad, ties = index_rule(zf, Wc, idx)
                print("D=%d n_e=%d M=%d: %d rows, %d near ties, %d off the index rule" % (D, n_e, zf.shape[0], zf.shape[0], ties, bad))
                assert bad == 0
            assert torch.equal(idx, idx0), "indices depend on the layouts"
            zq_ref, loss_ref, _ = quantize_ref(z, Wc, idx=idx)
            assert _same(zq if ql == "nchw" else zq.permute(0, 3, 1, 2), zq_ref)
            assert abs(float(loss) - loss_ref) <= 1e-5 * loss_ref
    _, idx_only, _ = ops.vq_quantize(zg, Wg, want_zq=False, want_loss=False)
    assert torch.equal(idx_only, idx0)


def test_vq_exact_cases(cuda):
    from sdb200 import ops
    g = torch.Generator().manual_seed(7)
    z = torch.randn(1, 3, 64, 64, generator=g)
    base = torch.randn(4096, 3, generator=g)
    # duplicated rows, one copy in each half of the codebook (so in different slices): the lower index wins
    Wd = torch.cat([base, base]).cuda()
    zq, idx, _ = ops.vq_quantize(z.cuda(), Wd)
    assert int(idx.max()) < 4096 and index_rule(_rows(z, "nchw"), Wd, idx)[0] == 0
    # NaN in z: that row takes index 0, its z_q carries the NaN, the loss is NaN
    zn = z.clone()
    zn[0, 1, 5, 7] = float("nan")
    zq, idx, loss = ops.vq_quantize(zn.cuda(), Wd)
    row = 5 * 64 + 7
    assert int(idx[row]) == 0 and bool(zq[0, 1, 5, 7].isnan()) and bool(loss.isnan())
    assert _same(zq, quantize_ref(zn, Wd, idx=idx)[0])
    # NaN codes: the first one wins every row, as torch.argmin does
    Wn = Wd.clone()
    Wn[5000, 2] = float("nan")
    Wn[123, 0] = float("nan")
    _, idx, _ = ops.vq_quantize(z.cuda(), Wn)
    assert bool((idx == 123).all())


def test_vq_split_matches_single_slice(cuda):
    """One 64x64 image is split over codebook slices; the same image inside an 80-image batch is not (80 * 4096 rows fill
    the GPU on their own).  Same indices, same z_q bits."""
    from sdb200 import _lib, ops
    lib = _lib.load()
    M1, Mb, n_e = 4096, 80 * 4096, 8192
    assert lib.sdb_vq_ws_bytes(M1, n_e) > 16 * M1 and lib.sdb_vq_ws_bytes(Mb, n_e) < 16 * Mb     # split / one slice
    g = torch.Generator().manual_seed(8)
    z = torch.randn(1, 3, 64, 64, generator=g).cuda()
    Wc = torch.randn(n_e, 3, generator=g).cuda()
    zq1, idx1, _ = ops.vq_quantize(z, Wc)
    zqb, idxb, _ = ops.vq_quantize(z.repeat(80, 1, 1, 1).contiguous(), Wc)
    assert torch.equal(idx1, idxb[:M1]) and torch.equal(idxb[:M1], idxb[-M1:])
    assert torch.equal(zq1, zqb[:1])


def test_codebook_gather(cuda):
    from sdb200.quantize import VectorQuantizer2
    q = VectorQuantizer2(8192, 3, 0.25).cuda()
    q.embedding.weight.data.copy_(torch.randn(8192, 3))
    Wc = q.embedding.weight.detach()
    idx = torch.randint(0, 8192, (2 * 16 * 16,), device="cuda")
    out = q.get_codebook_entry(idx, (2, 16, 16, 3))
    assert torch.equal(out, Wc[idx].reshape(2, 16, 16, 3).permute(0, 3, 1, 2))
    flat = q.get_codebook_entry(idx.reshape(2, 16, 16), None)
    assert torch.equal(flat, Wc[idx].reshape(2, 16, 16, 3))
    bad = idx.clone()
    bad[3], bad[10] = -1, 8192
    out = q.get_codebook_entry(bad, (2, 16, 16, 3)).permute(0, 2, 3, 1).reshape(-1, 3)
    assert bool(out[3].isnan().all()) and bool(out[10].isnan().all())
    keep = torch.ones(512, dtype=torch.bool)
    keep[3] = keep[10] = False
    assert torch.equal(out[keep.cuda()], Wc[idx][keep.cuda()])


def test_vector_quantizer_module(cuda):
    from sdb200.quantize import VectorQuantizer2
    q = VectorQuantizer2(512, 3, 0.25, sane_index_shape=True).cuda()
    z = torch.randn(2, 3, 16, 16, device="cuda") * 0.01
    zq, loss, (p, e, idx) = q(z)
    assert p is None and e is None and idx.shape == (2, 16, 16)
    zq_ref, loss_ref, _ = quantize_ref(z, q.embedding.weight.detach(), idx=idx)
    assert _same(zq, zq_ref) and abs(float(loss) - loss_ref) <= 1e-5 * loss_ref
    # the weight is read on every call: an in-place update is seen by the next one
    with torch.no_grad():
        q.embedding.weight.mul_(0.5)
    zq2, _, _ = q(z)
    assert _same(zq2, quantize_ref(z, q.embedding.weight.detach(), idx=q(z)[2][2])[0])


def test_vq_quantize_cuda_graph(cuda):
    from sdb200 import ops
    g = torch.Generator().manual_seed(9)
    Wc = torch.randn(8192, 3, generator=g).cuda()
    static = torch.randn(8, 3, 64, 64, generator=g).cuda()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ops.vq_quantize(static, Wc, zq_layout="nhwc")
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        outs = ops.vq_quantize(static, Wc, zq_layout="nhwc")
    for seed in (10, 11):
        z2 = torch.randn(8, 3, 64, 64, generator=torch.Generator().manual_seed(seed)).cuda()
        static.copy_(z2)
        graph.replay()
        ref = ops.vq_quantize(z2, Wc, zq_layout="nhwc")
        torch.cuda.synchronize()
        assert all(torch.equal(a, b) for a, b in zip(outs, ref))


# ---- 2. the first stage against the restatement -------------------------------------------------------------------------
def _attn_on(dd):
    return dd.get("attn_type", "vanilla") != "none"


def encoder_ref(sd, dd, x, p="encoder."):
    """Encoder.forward (ldm/modules/diffusionmodules/model.py:434-465) as oracle.restate.encoder_forward, with
    attn_type "none" (make_attn -> Identity) honoured."""
    ch_mult = tuple(dd["ch_mult"])
    nres, nrb, attn = len(ch_mult), dd["num_res_blocks"], _attn_on(dd)
    curr_res = dd["resolution"]
    h = R._conv(sd, p + "conv_in", x, padding=1)
    for i_level in range(nres):
        for i_block in range(nrb):
            h = R.vae_resnet_block(sd, "%sdown.%d.block.%d" % (p, i_level, i_block), h)
            if attn and curr_res in dd["attn_resolutions"]:
                h = R.vae_attn_block(sd, "%sdown.%d.attn.%d" % (p, i_level, i_block), h)
        if i_level != nres - 1:
            h = R._conv(sd, "%sdown.%d.downsample.conv" % (p, i_level), F.pad(h, (0, 1, 0, 1)), stride=2, padding=0)
            curr_res //= 2
    h = R.vae_resnet_block(sd, p + "mid.block_1", h)
    if attn:
        h = R.vae_attn_block(sd, p + "mid.attn_1", h)
    h = R.vae_resnet_block(sd, p + "mid.block_2", h)
    return R._conv(sd, p + "conv_out", R._swish(R._gn(sd, p + "norm_out", h, 1e-6)), padding=1)


def decoder_ref(sd, dd, z, p="decoder."):
    """Decoder.forward (model.py:541-574) as oracle.restate.decoder_forward, with attn_type "none" honoured."""
    ch_mult = tuple(dd["ch_mult"])
    nres, nrb, attn = len(ch_mult), dd["num_res_blocks"], _attn_on(dd)
    curr_res = dd["resolution"] // 2 ** (nres - 1)
    h = R._conv(sd, p + "conv_in", z, padding=1)
    h = R.vae_resnet_block(sd, p + "mid.block_1", h)
    if attn:
        h = R.vae_attn_block(sd, p + "mid.attn_1", h)
    h = R.vae_resnet_block(sd, p + "mid.block_2", h)
    for i_level in reversed(range(nres)):
        for i_block in range(nrb + 1):
            h = R.vae_resnet_block(sd, "%sup.%d.block.%d" % (p, i_level, i_block), h)
            if attn and curr_res in dd["attn_resolutions"]:
                h = R.vae_attn_block(sd, "%sup.%d.attn.%d" % (p, i_level, i_block), h)
        if i_level != 0:
            h = R._conv(sd, "%sup.%d.upsample.conv" % (p, i_level), F.interpolate(h, scale_factor=2.0, mode="nearest"), padding=1)
            curr_res *= 2
    return R._conv(sd, p + "conv_out", R._swish(R._gn(sd, p + "norm_out", h, 1e-6)), padding=1)


def vq_decode_ref(sd, dd, quant):
    return decoder_ref(sd, dd, R._conv(sd, "post_quant_conv", quant))


def _dd(attn):
    return dict(VQ_DD, attn_type="none") if attn == "none" else dict(VQ_DD, attn_type="vanilla")


def _first_stage(cls, dd, mode, n_embed=8192, seed=41):
    from sdb200 import autoencoder as A
    if cls == "VQModelInterface":
        m = A.VQModelInterface(3, ddconfig=dd, lossconfig=None, n_embed=n_embed, compute_mode=mode)
    else:
        m = A.VQModel(ddconfig=dd, lossconfig=None, n_embed=n_embed, embed_dim=3, compute_mode=mode)
    sd = W.make_state_dict(W.key_shapes_of(m), seed)
    m.load_state_dict(sd)
    return m.cuda(), {k: v.double() for k, v in sd.items()}


def _image_check(img, ref, mode, what):
    e, psnr = rel(img, ref), R.psnr_255(img.cpu(), ref.float())
    print("%s %s: rel-L2 %.3e, PSNR %.1f dB" % (what, mode, e, psnr))
    assert img.shape == ref.shape
    if mode == "fp32":
        assert e <= 1e-5
    else:
        assert psnr >= 40.0


@pytest.mark.parametrize("attn", ["none", "mid"])
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_vq_first_stage_against_restatement(cuda, attn, mode):
    dd = _dd(attn)
    m, sd = _first_stage("VQModelInterface", dd, mode)
    Wc = m.quantize.embedding.weight.detach()
    x = W.seeded_randn((2, 3, 64, 64), 51)
    h = m.encode(x.cuda())
    with torch.no_grad():
        h_ref = R._conv(sd, "quant_conv", encoder_ref(sd, dd, x.double()))
    eh = rel(h, h_ref)
    print("VQModelInterface.encode %s attn=%s: rel-L2 %.3e" % (mode, attn, eh))
    assert eh <= (1e-5 if mode == "fp32" else 2e-2)
    _, _, (_, _, idx) = m.quantize(h)
    bad, ties = index_rule(_rows(h, "nchw"), Wc, idx)
    assert bad == 0
    img = m.decode(h)
    with torch.no_grad():
        _image_check(img, vq_decode_ref(sd, dd, Wc.double().cpu()[idx.cpu()].reshape(2, 16, 16, 3).permute(0, 3, 1, 2)), mode,
                     "VQModelInterface.decode attn=%s" % attn)
        _image_check(m.decode(h, force_not_quantize=True), vq_decode_ref(sd, dd, h.double().cpu()), mode,
                     "VQModelInterface.decode(force_not_quantize) attn=%s" % attn)
    m.micro_batch = 1
    assert torch.equal(m.decode(h), img)
    # VQModel.forward: encode -> quantize -> decode, with the indices and the commitment loss
    vm, _ = _first_stage("VQModel", dd, mode)
    dec, diff, ind = vm(x.cuda(), return_pred_indices=True)
    hp = vm.encode_to_prequant(x.cuda())
    assert index_rule(_rows(hp, "nchw"), Wc, ind)[0] == 0
    _, loss_ref, _ = quantize_ref(hp, Wc, idx=ind)
    assert abs(float(diff) - loss_ref) <= 1e-5 * loss_ref
    with torch.no_grad():
        _image_check(dec, vq_decode_ref(sd, dd, Wc.double().cpu()[ind.cpu()].reshape(2, 16, 16, 3).permute(0, 3, 1, 2)), mode,
                     "VQModel.forward attn=%s" % attn)


def test_attn_type_none_with_attn_resolutions(cuda):
    """Encoder / Decoder with attn_type="none" and a non-empty attn_resolutions: the Identity blocks are skipped."""
    from sdb200.autoencoder import Decoder, Encoder
    dd = dict(VQ_DD, attn_type="none", attn_resolutions=[16])
    for cls, inp, ref_fn in ((Encoder, (2, 3, 64, 64), encoder_ref), (Decoder, (2, 3, 16, 16), decoder_ref)):
        net = cls(**dd, compute_mode="fp32")
        sd = W.make_state_dict(W.key_shapes_of(net), 61)
        net.load_state_dict(sd)
        x = W.seeded_randn(inp, 62)
        y = net.cuda()(x.cuda())
        with torch.no_grad():
            y_ref = ref_fn({k: v.double() for k, v in sd.items()}, dd, x.double(), p="")
        e = rel(y, y_ref)
        print("%s attn_type=none attn_resolutions=[16] fp32: rel-L2 %.3e" % (cls.__name__, e))
        assert e <= 1e-5


def test_vq_decode_has_no_host_sync(cuda):
    m, _ = _first_stage("VQModelInterface", _dd("none"), "bf16")
    h = W.seeded_randn((8, 3, 16, 16), 71).cuda()
    m.decode(h)
    m.decode(h, force_not_quantize=True)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        img = m.decode(h)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert torch.isfinite(img).all()


# ---- 3. a VQ latent-diffusion model (VQ-f4 inpainting layout: 3 latent + 1 mask + 3 masked-image channels) ---------------
def _vq_ldm(mode):
    from sdb200.pipeline import LatentDiffusion
    g = load_golden("unet_var_neworder.pt")
    cfg = dict(g["cfg"], in_channels=7, out_channels=3)
    fs, sdv = _first_stage("VQModelInterface", _dd("none"), mode)
    ld = LatentDiffusion(unet_config=cfg, first_stage_config=False, first_stage_model=fs, conditioning_key="concat",
                         compute_mode=mode, scale_factor=1.0, channels=3, image_size=16)
    sdu = W.make_state_dict(W.key_shapes_of(ld.model.diffusion_model), g["seed"])
    ld.model.diffusion_model.load_state_dict(sdu)
    cond = torch.cat([(W.seeded_randn((2, 1, 16, 16), 81) > 0).float(), W.seeded_randn((2, 3, 16, 16), 82)], 1)
    return ld.cuda(), sdu, cfg, sdv, cond, W.seeded_randn((2, 3, 16, 16), 83)


def _quantizer_ref(Wc):
    return lambda p: quantize_ref(p, Wc)[0]


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_vq_ldm_ddim_and_decode(cuda, mode):
    from test_gpu_conditioning import DictDDIMOracle, _restated_wrapper
    ld, sdu, cfg, sdv, cond, x_T = _vq_ldm(mode)
    fs = ld.first_stage_model
    Wc = fs.quantize.embedding.weight.detach()
    torch.manual_seed(31)
    z, _ = ld.sample_log(cond.cuda(), 2, ddim=True, ddim_steps=10, shape=(3, 16, 16), x_T=x_T.cuda(), eta=0.0)
    torch.manual_seed(31)
    orc = DictDDIMOracle(R.ModelShim(_restated_wrapper(sdu, cfg, "concat"), R.sd_alphas_cumprod()))
    with torch.no_grad():
        z_ref, _ = orc.sample(10, 2, (3, 16, 16), conditioning=cond, eta=0.0, x_T=x_T)
    e = rel(z, z_ref)
    print("VQ LDM DDIM-10 %s: latent rel-L2 %.3e" % (mode, e))
    assert e <= (1e-5 if mode == "fp32" else 2e-2)
    img = ld.decode_first_stage(z)
    img_nq = ld.decode_first_stage(z, force_not_quantize=True)
    _, _, (_, _, idx) = fs.quantize(z)
    assert index_rule(_rows(z, "nchw"), Wc, idx)[0] == 0
    with torch.no_grad():
        _image_check(img, vq_decode_ref(sdv, _dd("none"), Wc.double().cpu()[idx.cpu()].reshape(2, 16, 16, 3).permute(0, 3, 1, 2)),
                     mode, "VQ LDM decode_first_stage")
        _image_check(img_nq, vq_decode_ref(sdv, _dd("none"), z.double().cpu()), mode, "VQ LDM decode_first_stage(force_not_quantize)")


class QuantizedDDIMOracle:
    """p_sample_ddim of ldm/diffusion/ddim.py with quantize_denoised: pred_x0 goes through the first stage's quantizer
    before x_prev is formed; every noise draw is made on the GPU in the reference's order."""

    def __init__(self, base, quantize):
        self.base, self.quantize = base, quantize
        base.p_sample_ddim = self.p_sample_ddim

    def p_sample_ddim(self, x, c, t, index, temperature=1., unconditional_guidance_scale=1., unconditional_conditioning=None,
                      noise=None):
        e_t = self.base.model.apply_model(x, t, c)
        a_t, a_prev, sigma_t, s1m = self.base.coefficients(index, x.shape[0])
        pred_x0 = self.quantize((x - s1m * e_t) / a_t.sqrt())
        dir_xt = (1. - a_prev - sigma_t ** 2).sqrt() * e_t
        noise = torch.randn(x.shape, device="cuda").cpu()
        return a_prev.sqrt() * pred_x0 + dir_xt + sigma_t * noise * temperature, pred_x0, e_t


def test_real_quantizer_in_the_samplers(cuda):
    from test_gpu_ancestral import AncestralOracle
    from test_gpu_conditioning import DictDDIMOracle, _restated_wrapper
    ld, sdu, cfg, sdv, cond, x_T = _vq_ldm("fp32")
    qref = _quantizer_ref(ld.first_stage_model.quantize.embedding.weight.detach())
    fn = _restated_wrapper(sdu, cfg, "concat")
    torch.manual_seed(41)
    z, _ = ld.sample_log(cond.cuda(), 2, ddim=True, ddim_steps=8, shape=(3, 16, 16), x_T=x_T.cuda(), eta=0.5, quantize_x0=True)
    torch.manual_seed(41)
    orc = DictDDIMOracle(R.ModelShim(fn, R.sd_alphas_cumprod()))
    QuantizedDDIMOracle(orc, qref)
    with torch.no_grad():
        z_ref, _ = orc.sample(8, 2, (3, 16, 16), conditioning=cond, eta=0.5, x_T=x_T)
    e = rel(z, z_ref)
    torch.manual_seed(42)
    za = ld.p_sample_loop(cond.cuda(), (2, 3, 16, 16), x_T=x_T.cuda(), timesteps=8, quantize_denoised=True)
    torch.manual_seed(42)
    with torch.no_grad():
        za_ref, _ = AncestralOracle(R.ModelShim(fn, R.sd_alphas_cumprod()), quantize=lambda p: (qref(p), None, None)).p_sample_loop(
            cond, x_T, 8, quantize_denoised=True)
    ea = rel(za, za_ref)
    print("real VectorQuantizer2: DDIM-8 quantize_x0 latent rel-L2 %.3e, p_sample_loop quantize_denoised %.3e" % (e, ea))
    assert e <= 1e-4 and ea <= 1e-4
