"""GPU: image-conditioned LatentDiffusion ("concat", "hybrid" and "adm" conditioning keys, ldm/diffusion/ddpm.py:1992-2034).

- the two-source layout kernel (sdb_nchw_concat_to_nhwc) against cat + permute + pad / bf16 / split on the host, exactly;
- UNetModel.forward_concat against forward(torch.cat(...)), bit for bit, eager and CUDA graph;
- a 9-channel SD-size UNet against oracle.restate.unet_forward on the concatenated input;
- DDIM with classifier-free guidance on a tiny hybrid model (one 2B call == two calls, bit for bit; trajectory and RNG position
  against the restated sampler), the ancestral loop, and tiny adm / concat models.
The restatement oracle.restate.unet_forward is pinned to the reference's fixtures for in_channels=4 only; for other channel
counts it is the same code on a wider first conv, so the parity below checks this repository against its own restatement."""
import contextlib

import pytest
import torch

from gpu_util import nhwc, rel
from oracle import restate as R
from oracle import weights as W
from oracle.golden import load_golden

pytestmark = pytest.mark.gpu

EPS_TOL = {"fp32": 1e-5, "bf16": 1e-2}           # tests/test_gpu_models.py


# ---- helpers ------------------------------------------------------------------------------------------------------------
def _cfg(name, **over):
    g = load_golden(name + ".pt")
    cfg = dict(g["cfg"])
    cfg.update(over)
    return cfg, g["seed"]


def _unet(cfg, seed, mode, graph=False):
    from sdb200.openai_model import UNetModel
    net = UNetModel(**cfg, compute_mode=mode)
    sd = W.make_state_dict(W.key_shapes_of(net), seed)
    net.load_state_dict(sd)
    net = net.cuda()
    net.use_cuda_graph = graph
    return net, sd


def _ld(cfg, seed, key, mode="fp32"):
    from sdb200.pipeline import LatentDiffusion
    ld = LatentDiffusion(unet_config=cfg, first_stage_config=False, conditioning_key=key, compute_mode=mode)
    sd = W.make_state_dict(W.key_shapes_of(ld.model.diffusion_model), seed)
    ld.model.diffusion_model.load_state_dict(sd)
    return ld.cuda(), sd


def _restated_wrapper(sd, cfg, key):
    """DiffusionWrapper.forward of the reference on restate.unet_forward (CPU)."""
    def fn(x, t, cond):
        if not isinstance(cond, dict):
            cond = {("c_concat" if key == "concat" else "c_crossattn"): [cond]}
        cc, ca = cond.get("c_concat"), cond.get("c_crossattn")
        if key == "concat":
            return R.unet_forward(sd, cfg, torch.cat([x] + cc, 1), t, None)
        if key == "hybrid":
            return R.unet_forward(sd, cfg, torch.cat([x] + cc, 1), t, torch.cat(ca, 1))
        if key == "adm":
            return R.unet_forward(sd, cfg, x, t, None, y=ca[0])
        return R.unet_forward(sd, cfg, x, t, torch.cat(ca, 1))
    return fn


class DictDDIMOracle(R.DDIMOracle):
    """R.DDIMOracle with the reference's dict branch of the CFG batch (c_in[k] = [cat([uc[k][i], c[k][i]])]) and every
    noise draw made on the GPU in the reference's order, so the sampler under test sees the same draws."""

    def p_sample_ddim(self, x, c, t, index, temperature=1., unconditional_guidance_scale=1.,
                      unconditional_conditioning=None, noise=None):
        b = x.shape[0]
        uc = unconditional_conditioning
        if uc is None or unconditional_guidance_scale == 1.:
            e_t = self.model.apply_model(x, t, c)
        else:
            c_in = {k: [torch.cat([uc[k][i], c[k][i]]) for i in range(len(c[k]))] for k in c}
            e_t_uncond, e_t = self.model.apply_model(torch.cat([x] * 2), torch.cat([t] * 2), c_in).chunk(2)
            e_t = e_t_uncond + unconditional_guidance_scale * (e_t - e_t_uncond)
        a_t, a_prev, sigma_t, s1m = self.coefficients(index, b)
        pred_x0 = (x - s1m * e_t) / a_t.sqrt()
        dir_xt = (1. - a_prev - sigma_t ** 2).sqrt() * e_t
        noise = torch.randn(x.shape, device="cuda").cpu()
        x_prev = a_prev.sqrt() * pred_x0 + dir_xt + sigma_t * noise * temperature
        return x_prev, pred_x0, e_t


# ---- 1. the layout kernel -----------------------------------------------------------------------------------------------
def _expect_layout(x0, x1, out_dtype, pad_to, split):
    x = torch.cat([x0, x1], 1) if x1 is not None else x0
    h = nhwc(x.cpu())
    Cc = h.shape[-1]
    if split:
        hi = h.to(torch.bfloat16)
        lo = (h - hi.float()).to(torch.bfloat16)
        parts = [hi, lo]
        used = 2 * Cc
    else:
        parts, used = [h.to(out_dtype)], Cc
    Cd = max(used, pad_to)
    if Cd > used:
        parts.append(torch.zeros(*h.shape[:-1], Cd - used, dtype=out_dtype))
    return torch.cat(parts, -1)


def _raw_concat(x0, x1, out, split):
    """sdb_nchw_concat_to_nhwc called directly (x1 may be None: the C1 = 0 case)."""
    from sdb200 import _lib
    N, C0, H, W_ = x0.shape
    C1 = 0 if x1 is None else x1.shape[1]
    rc = _lib.load().sdb_nchw_concat_to_nhwc(_lib.ptr(x0), C0, None if x1 is None else _lib.ptr(x1), C1, _lib.ptr(out),
                                             _lib.dtype_code(out.dtype), out.shape[-1], int(split), N, H * W_, _lib.stream_ptr())
    _lib.check(rc, "nchw_concat_to_nhwc")
    return out


LAYOUT_CASES = [(4, 1, "split"), (4, 1, "bf16"), (4, 1, "f32"), (4, 5, "split"), (4, 5, "bf16"), (4, 5, "f32"),
                (9, 7, "split"), (9, 7, "bf16"), (9, 7, "f32"), (3, 30, "bf16"), (3, 30, "f32")]


@pytest.mark.parametrize("C0,C1,kind", LAYOUT_CASES)
def test_layout_kernel_two_sources(cuda, C0, C1, kind):
    from sdb200 import ops
    g = torch.Generator().manual_seed(C0 * 100 + C1)
    N, H, W_ = 3, 5, 13                                       # HW = 65: partial 32-pixel tiles
    x0 = (torch.randn(N, C0, H, W_, generator=g) * 3).cuda()
    x1 = (torch.randn(N, C1, H, W_, generator=g) * 3).cuda()
    dt = torch.float32 if kind == "f32" else torch.bfloat16
    split = kind == "split"
    for pad_to in ((32,) if split else (0, 32, 40)):
        got = ops.nchw_to_nhwc(x0, out_dtype=dt, pad_to=pad_to, split=split, x1=x1)
        want = _expect_layout(x0, x1, dt, pad_to, split)
        assert got.dtype == want.dtype and got.shape == want.shape, (got.shape, want.shape)
        assert torch.equal(got.cpu(), want), (C0, C1, kind, pad_to)
    assert torch.equal(ops.nchw_to_nhwc(x0, out_dtype=dt, pad_to=32 if split else 0, split=split, x1=x1).cpu(),
                       ops.nchw_to_nhwc(torch.cat([x0, x1], 1).contiguous(), out_dtype=dt, pad_to=32 if split else 0,
                                        split=split).cpu())


@pytest.mark.parametrize("kind", ["split", "bf16", "f32"])
@pytest.mark.parametrize("C", [4, 9, 33])
def test_layout_kernel_c1_zero_matches_old_entry_points(cuda, kind, C):
    from sdb200 import ops
    if kind == "split" and 2 * C > 32:
        pytest.skip("split operand is 32 channels wide here")
    x = (torch.randn(2, C, 7, 9, generator=torch.Generator().manual_seed(C)) * 3).cuda()
    dt = torch.float32 if kind == "f32" else torch.bfloat16
    pad = 32 if kind == "split" else (0 if kind == "f32" else 40)
    old = ops.nchw_to_nhwc(x, out_dtype=dt, pad_to=pad, split=kind == "split")     # sdb_nchw_to_nhwc[_split]
    new = _raw_concat(x, None, torch.full_like(old, float("nan")), kind == "split")
    assert torch.equal(old.view(torch.int16 if dt == torch.bfloat16 else torch.int32).cpu(),
                       new.view(torch.int16 if dt == torch.bfloat16 else torch.int32).cpu())
    assert torch.equal(old.cpu(), _expect_layout(x, None, dt, pad, kind == "split"))


def test_layout_kernel_argument_checks(cuda):
    from sdb200 import _lib
    x = torch.zeros(1, 4, 4, 4, device="cuda")
    out = torch.zeros(1, 4, 4, 32, device="cuda", dtype=torch.bfloat16)
    L = _lib.load()
    p, s = _lib.ptr, _lib.stream_ptr()
    assert L.sdb_nchw_concat_to_nhwc(p(x), 4, None, 5, p(out), 1, 32, 0, 1, 16, s) == -1       # C1 > 0 needs src1
    assert L.sdb_nchw_concat_to_nhwc(p(x), 4, p(x), 0, p(out), 1, 32, 0, 1, 16, s) == -1       # src1 given with C1 = 0
    assert L.sdb_nchw_concat_to_nhwc(p(x), 4, p(x), 4, p(out), 1, 15, 1, 1, 16, s) == -1       # split: dst_C < 2C
    assert L.sdb_nchw_concat_to_nhwc(p(x), 4, p(x), 4, p(out), 0, 32, 1, 1, 16, s) == -1       # split: fp32 destination


# ---- 2. forward_concat == forward(cat) ---------------------------------------------------------------------------------
def _concat_inputs(B, HW, ctx_shape, seed):
    x = W.seeded_randn((B, 4, HW, HW), seed).cuda()
    m = (W.seeded_randn((B, 1, HW, HW), seed + 1) > 0).float().cuda()
    z = W.seeded_randn((B, 4, HW, HW), seed + 2).cuda()
    ctx = W.seeded_randn((B, *ctx_shape), seed + 3).cuda()
    t = torch.tensor([981, 500, 21, 1][:B], device="cuda")
    return x, m, z, ctx, t


@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_forward_concat_tiny_bit_exact(cuda, mode, graph):
    cfg, seed = _cfg("unet_tiny", in_channels=9)
    net, _ = _unet(cfg, seed, mode, graph)
    x, m, z, ctx, t = _concat_inputs(2, 8, (7, 64), 40)
    want = net(torch.cat([x, m, z], 1), t, ctx)
    for cc in ([m, z], torch.cat([m, z], 1)):
        got = net.forward_concat(x, cc, t, context=ctx)
        assert torch.equal(got, want)
    assert torch.isfinite(want).all() and float(want.abs().max()) > 0.1
    # a changed c_concat between replays: a new tensor, then the same tensor written in place
    z2 = W.seeded_randn(tuple(z.shape), 49).cuda()
    want2 = net(torch.cat([x, m, z2], 1), t, ctx)
    assert not torch.equal(want2, want)
    assert torch.equal(net.forward_concat(x, [m, z2], t, context=ctx), want2)
    assert torch.equal(net.forward_concat(x, [m, z], t, context=ctx), want)
    zz = z.clone()
    assert torch.equal(net.forward_concat(x, [m, zz], t, context=ctx), want)
    zz.copy_(z2)
    assert torch.equal(net.forward_concat(x, [m, zz], t, context=ctx), want2)
    # bf16 inputs come back in bf16, as forward's do
    xb = x.to(torch.bfloat16)
    assert torch.equal(net.forward_concat(xb, [m.to(torch.bfloat16), z.to(torch.bfloat16)], t, context=ctx),
                       net(torch.cat([xb, m.to(torch.bfloat16), z.to(torch.bfloat16)], 1), t, ctx))


def test_forward_and_forward_concat_interleaved_graphs(cuda):
    """On one model, graphs captured for forward (9-channel input) and forward_concat (4 + 5 channels) are kept apart."""
    cfg, seed = _cfg("unet_tiny", in_channels=9)
    net, _ = _unet(cfg, seed, "bf16", graph=False)
    x, m, z, ctx, t = _concat_inputs(2, 8, (7, 64), 50)
    xs = [x, W.seeded_randn(tuple(x.shape), 58).cuda()]
    cs = [torch.cat([m, z], 1), torch.cat([1 - m, z * 0.5], 1)]
    eager = {(i, j): net(torch.cat([xs[i], cs[j]], 1), t, ctx) for i in range(2) for j in range(2)}
    net.use_cuda_graph = True
    for i, j in [(0, 0), (1, 1), (0, 1), (1, 0), (0, 0)]:
        assert torch.equal(net(torch.cat([xs[i], cs[j]], 1), t, ctx), eager[i, j])
        assert torch.equal(net.forward_concat(xs[i], cs[j], t, context=ctx), eager[i, j])
        assert torch.equal(net.forward_concat(xs[i], [cs[j][:, :1], cs[j][:, 1:]], t, context=ctx), eager[i, j])
    assert len(net._graphs) == 2


def test_forward_concat_sd_size(cuda):
    """SD-size 9-channel UNet: forward_concat == forward(cat) bit for bit (bf16 eager and graph, fp32 eager), and eps against
    the restatement on the concatenated input for three timesteps."""
    cfg, seed = _cfg("unet_sd", in_channels=9)
    net, sd = _unet(cfg, seed, "bf16")
    B = 1
    x, m, z, ctx, _ = _concat_inputs(B, 64, (77, 768), 60)
    ts = [torch.tensor([v], device="cuda") for v in (981, 500, 21)]
    bf = []
    for t in ts:
        want = net(torch.cat([x, m, z], 1), t, ctx)
        assert torch.equal(net.forward_concat(x, [m, z], t, context=ctx), want)
        bf.append(want)
    net.use_cuda_graph = True
    for t, want in zip(ts, bf):
        assert torch.equal(net.forward_concat(x, [m, z], t, context=ctx), want)
    net.use_cuda_graph = False
    net.compute_mode = "fp32"
    f32 = []
    for t in ts:
        want = net(torch.cat([x, m, z], 1), t, ctx)
        assert torch.equal(net.forward_concat(x, [m, z], t, context=ctx), want)
        f32.append(want)
    sd64 = {k: v.double() for k, v in sd.items()}
    xin = torch.cat([x, m, z], 1).cpu().double()
    for t, e_bf, e_32 in zip(ts, bf, f32):
        with torch.no_grad():
            ref = R.unet_forward(sd64, cfg, xin, t.cpu(), ctx.cpu().double())
        eb, ef = rel(e_bf, ref), rel(e_32, ref)
        print("SD 9-channel t=%d: eps rel-L2 fp32 %.3e, bf16 %.3e" % (int(t), ef, eb))
        assert ef <= EPS_TOL["fp32"] and eb <= EPS_TOL["bf16"]


# ---- 3. DDIM with CFG on a tiny hybrid model ---------------------------------------------------------------------------
def _hybrid_setup(mode="fp32", graph=False):
    cfg, seed = _cfg("unet_tiny", in_channels=9)
    ld, sd = _ld(cfg, seed, "hybrid", mode)
    ld.model.diffusion_model.use_cuda_graph = graph
    B = 2
    m = (W.seeded_randn((B, 1, 8, 8), 81) > 0).float()
    zc = W.seeded_randn((B, 4, 8, 8), 82)
    cc = torch.cat([m, zc], 1)
    c = {"c_concat": [cc], "c_crossattn": [W.seeded_randn((B, 7, 64), 83)]}
    uc = {"c_concat": [cc], "c_crossattn": [W.seeded_randn((B, 7, 64), 84)]}
    x_T = W.seeded_randn((B, 4, 8, 8), 85)
    return ld, sd, cfg, c, uc, x_T


def _cuda(d):
    return {k: [v.cuda() for v in vs] for k, vs in d.items()}


@contextlib.contextmanager
def _two_call_path():
    """DDIMSampler with the 2B dict path switched off: CFG on dict conditionings takes two calls per step."""
    from sdb200.ddim import DDIMSampler
    saved = DDIMSampler.__dict__["_cfg_dict_pairable"]
    DDIMSampler._cfg_dict_pairable = staticmethod(lambda c, uc: False)
    try:
        yield
    finally:
        DDIMSampler._cfg_dict_pairable = saved


@pytest.mark.parametrize("eta", [0.0, 0.5])
def test_hybrid_ddim_cfg(cuda, eta):
    ld, sd, cfg, c, uc, x_T = _hybrid_setup()
    B, S, scale = 2, 10, 3.0
    cg, ucg = _cuda(c), _cuda(uc)
    calls = []
    apply = ld.apply_model
    ld.apply_model = lambda x_, t_, c_, return_ids=False: calls.append(x_.shape[0]) or apply(x_, t_, c_)
    torch.manual_seed(11)
    z, inter = ld.sample_log(cg, B, ddim=True, ddim_steps=S, shape=(4, 8, 8), x_T=x_T.cuda(), eta=eta,
                             unconditional_guidance_scale=scale, unconditional_conditioning=ucg)
    after = torch.randn(4, device="cuda")
    assert calls == [2 * B] * S                                       # one 2B call per step
    # the two-call path on the same draws gives the same bits
    calls.clear()
    torch.manual_seed(11)
    with _two_call_path():
        z2, _ = ld.sample_log(cg, B, ddim=True, ddim_steps=S, shape=(4, 8, 8), x_T=x_T.cuda(), eta=eta,
                              unconditional_guidance_scale=scale, unconditional_conditioning=ucg)
    assert calls == [B] * (2 * S)
    assert torch.equal(z, z2)
    # against the restated sampler on the same draws; the RNG ends where the reference's does
    torch.manual_seed(11)
    orc = DictDDIMOracle(R.ModelShim(_restated_wrapper(sd, cfg, "hybrid"), R.sd_alphas_cumprod()))
    with torch.no_grad():
        z_ref, inter_ref = orc.sample(S, B, (4, 8, 8), conditioning=c, eta=eta, x_T=x_T, unconditional_guidance_scale=scale,
                                      unconditional_conditioning=uc)
    assert torch.equal(after, torch.randn(4, device="cuda"))
    e = rel(z, z_ref)
    print("hybrid DDIM-%d CFG %.1f eta %.1f fp32: latent rel-L2 %.3e" % (S, scale, eta, e))
    assert e <= 1e-4
    assert len(inter["x_inter"]) == len(inter_ref["x_inter"])


def test_hybrid_cfg_2b_graph_keeps_context_projection(cuda):
    """bf16 + CUDA graph: the 2B dict path gives the two-call path's bits, and the context K/V projection graph is replayed
    once for the whole loop (the two calls alternate uc and c, so they re-project on every call)."""
    ld, sd, cfg, c, uc, x_T = _hybrid_setup("bf16", graph=True)
    cg, ucg = _cuda(c), _cuda(uc)
    S = 6
    n = len(range(0, 1000, 1000 // S))       # DDIM-6 on 1000 steps takes 7 (make_ddim_timesteps, 'uniform')
    kw = dict(ddim=True, ddim_steps=S, shape=(4, 8, 8), x_T=x_T.cuda(), eta=0.5, unconditional_guidance_scale=7.5,
              unconditional_conditioning=ucg)
    replays = []
    orig = torch.cuda.CUDAGraph.replay
    torch.cuda.CUDAGraph.replay = lambda self: replays.append(1) or orig(self)
    try:
        torch.manual_seed(3)
        z, _ = ld.sample_log(cg, 2, **kw)
        n2b = len(replays)
        replays.clear()
        torch.manual_seed(3)
        with _two_call_path():
            z2, _ = ld.sample_log(cg, 2, **kw)
        n2 = len(replays)
    finally:
        torch.cuda.CUDAGraph.replay = orig
    assert torch.equal(z, z2)
    print("graph replays over %d CFG steps: 2B path %d, two-call path %d" % (n, n2b, n2))
    assert n2b == n + 1                      # n UNet bodies + one K/V projection
    assert n2 == 2 * n + 2 * n               # 2n bodies + a K/V projection before each of them


def test_hybrid_ddim_has_no_host_sync(cuda):
    ld, sd, cfg, c, uc, x_T = _hybrid_setup("bf16", graph=True)
    cg, ucg = _cuda(c), _cuda(uc)
    kw = dict(ddim=True, ddim_steps=5, shape=(4, 8, 8), x_T=x_T.cuda(), eta=0.5, unconditional_guidance_scale=7.5,
              unconditional_conditioning=ucg)
    from sdb200.ddim import DDIMSampler
    smp = DDIMSampler(ld)
    smp.make_schedule(5, ddim_eta=0.5, verbose=False)
    for i in range(3):
        smp.derived_coefficients(i)
    ld.sample_log(cg, 2, **kw)                                       # captures the 2B graph
    ts = torch.full((2,), 333, device="cuda", dtype=torch.long)
    ld.p_sample(x_T.cuda(), cg, ts)                                 # the B graph and the ancestral schedule table
    torch.cuda.synchronize()
    img = x_T.cuda()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for i in (2, 1, 0):
            img, _ = smp.p_sample_ddim(img, cg, ts, index=i, unconditional_guidance_scale=7.5, unconditional_conditioning=ucg)
        img = ld.p_sample(img, cg, ts)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert torch.isfinite(img).all()


# ---- 4. ancestral loop, adm and concat models ---------------------------------------------------------------------------
def _anc_oracle(fn):
    from test_gpu_ancestral import AncestralOracle
    return AncestralOracle(R.ModelShim(fn, R.sd_alphas_cumprod()))


def test_hybrid_p_sample_loop(cuda):
    ld, sd, cfg, c, uc, x_T = _hybrid_setup()
    T = 12
    torch.manual_seed(21)
    z, inter = ld.p_sample_loop(_cuda(c), (2, 4, 8, 8), x_T=x_T.cuda(), timesteps=T, return_intermediates=True)
    after = torch.randn(4, device="cuda")
    torch.manual_seed(21)
    orc = _anc_oracle(_restated_wrapper(sd, cfg, "hybrid"))
    with torch.no_grad():
        z_ref, inter_ref = orc.p_sample_loop(c, x_T, T)
    assert torch.equal(after, torch.randn(4, device="cuda"))
    e = rel(z, z_ref)
    print("hybrid p_sample_loop T=%d fp32: latent rel-L2 %.3e" % (T, e))
    assert e <= 1e-4 and len(inter) == len(inter_ref)


@pytest.mark.parametrize("key", ["adm", "concat"])
def test_adm_and_concat_models(cuda, key):
    if key == "adm":
        cfg, seed = _cfg("unet_var_legacy")                      # num_classes=10, AttentionBlock, scale-shift norm
        cond = torch.tensor([3, 7])
    else:
        cfg, seed = _cfg("unet_var_neworder", in_channels=9)     # no cross-attention: conv_in takes 4 + 5 channels
        cond = torch.cat([(W.seeded_randn((2, 1, 16, 16), 91) > 0).float(), W.seeded_randn((2, 4, 16, 16), 92)], 1)
    ld, sd = _ld(cfg, seed, key)
    x_T = W.seeded_randn((2, 4, 16, 16), 93)
    fn = _restated_wrapper(sd, cfg, key)
    torch.manual_seed(31)
    z, _ = ld.sample_log(cond.cuda(), 2, ddim=True, ddim_steps=8, shape=(4, 16, 16), x_T=x_T.cuda(), eta=0.5)
    torch.manual_seed(31)
    orc = DictDDIMOracle(R.ModelShim(fn, R.sd_alphas_cumprod()))
    with torch.no_grad():
        z_ref, _ = orc.sample(8, 2, (4, 16, 16), conditioning=cond, eta=0.5, x_T=x_T)
    e = rel(z, z_ref)
    torch.manual_seed(32)
    za = ld.p_sample_loop(cond.cuda(), (2, 4, 16, 16), x_T=x_T.cuda(), timesteps=8)
    torch.manual_seed(32)
    with torch.no_grad():
        za_ref, _ = _anc_oracle(fn).p_sample_loop(cond, x_T, 8)
    ea = rel(za, za_ref)
    print("%s: DDIM-8 latent rel-L2 %.3e, p_sample_loop latent rel-L2 %.3e" % (key, e, ea))
    assert e <= 1e-4 and ea <= 1e-4
