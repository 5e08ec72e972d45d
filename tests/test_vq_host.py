"""CPU: the VQ first stage's Python surface (VQModel / VQModelInterface / VectorQuantizer2 / IdentityFirstStage: kwargs,
state-dict keys, the cases that are not built, taming's asserts), LatentDiffusion.decode_first_stage routing, and the
host-side argument checks of the sdb_vq_* entry points."""
import pytest
import torch
from torch import nn

from oracle import weights as W

DDCONFIG = dict(double_z=False, z_channels=3, resolution=32, in_channels=3, out_ch=3, ch=32, ch_mult=(1, 2, 4),
                num_res_blocks=1, attn_resolutions=[], dropout=0.0)


def _vq(cls_name="VQModelInterface", **kw):
    from sdb200 import autoencoder as A
    args = dict(ddconfig=DDCONFIG, lossconfig={"target": "torch.nn.Identity"}, n_embed=64, embed_dim=3)
    args.update(kw)
    if cls_name == "VQModelInterface":
        return A.VQModelInterface(args.pop("embed_dim"), **args)
    return getattr(A, cls_name)(**args)


def test_constructor_kwargs_and_state_dict_keys():
    m = _vq("VQModel", ckpt_path=None, ignore_keys=[], image_key="image", colorize_nlabels=None, monitor="val/rec_loss",
            batch_resize_range=None, scheduler_config=None, lr_g_factor=1.0, remap=None, sane_index_shape=True,
            use_ema=False, compute_mode="fp32", micro_batch=4)
    assert m.monitor == "val/rec_loss" and m.quantize.sane_index_shape and m.micro_batch == 4
    sd = m.state_dict()
    assert tuple(sd["quantize.embedding.weight"].shape) == (64, 3)
    assert tuple(sd["quant_conv.weight"].shape) == (3, 3, 1, 1)                  # z_channels -> embed_dim
    assert tuple(sd["post_quant_conv.weight"].shape) == (3, 3, 1, 1)             # embed_dim -> z_channels
    assert tuple(sd["encoder.conv_out.weight"].shape) == (3, 128, 3, 3)          # double_z=False: z_channels outputs
    assert tuple(sd["decoder.conv_in.weight"].shape) == (128, 3, 3, 3)
    vqi = _vq(embed_dim=3, n_embed=64)
    assert vqi.embed_dim == 3 and vqi.n_embed == 64
    assert set(vqi.state_dict()) == set(sd)
    # a CompVis-style checkpoint: the model's keys plus the training loss's; only loss.* comes back, as unexpected
    ck = W.make_state_dict(W.key_shapes_of(vqi), 5)
    ck["loss.discriminator.main.0.weight"] = torch.zeros(64, 3, 4, 4)
    ck["loss.logvar"] = torch.zeros(())
    r = vqi.load_state_dict(ck, strict=False)
    assert r.missing_keys == [] and sorted(r.unexpected_keys) == ["loss.discriminator.main.0.weight", "loss.logvar"]
    assert torch.equal(vqi.quantize.embedding.weight, ck["quantize.embedding.weight"])


def test_vector_quantizer_kwargs_and_init():
    from sdb200.quantize import VectorQuantizer2
    q = VectorQuantizer2(8192, 3, 0.25, remap=None, unknown_index="random", sane_index_shape=False, legacy=False)
    assert (q.n_e, q.e_dim, q.beta, q.legacy, q.re_embed) == (8192, 3, 0.25, False, 8192)
    assert list(q.state_dict()) == ["embedding.weight"]
    w = q.embedding.weight
    assert tuple(w.shape) == (8192, 3) and float(w.detach().abs().max()) <= 1.0 / 8192


def test_not_built_cases_raise():
    from sdb200.pipeline import LatentDiffusion
    from sdb200.quantize import VectorQuantizer2
    with pytest.raises(NotImplementedError):
        VectorQuantizer2(16, 3, 0.25, remap="remap.npy")
    with pytest.raises(NotImplementedError):
        VectorQuantizer2(16, 17, 0.25)
    with pytest.raises(NotImplementedError):
        VectorQuantizer2(16, 0, 0.25)
    with pytest.raises(NotImplementedError):
        _vq("VQModel", remap="remap.npy")
    with pytest.raises(NotImplementedError):
        _vq("VQModel", use_ema=True)
    with pytest.raises(NotImplementedError):
        _vq("VQModel").decode_code(torch.zeros(1, 8, 8, dtype=torch.long))
    ld = LatentDiffusion(first_stage_config=False, unet=nn.Linear(1, 1), scale_factor=1.0, channels=3)
    ld.first_stage_model = _vq()
    with pytest.raises(NotImplementedError):
        ld.decode_first_stage(torch.zeros(1, 3, 8, 8), predict_cids=True)


def test_taming_asserts():
    from sdb200.quantize import VectorQuantizer2
    q = VectorQuantizer2(16, 3, 0.25)
    z = torch.zeros(1, 3, 4, 4)
    for kw in (dict(temp=0.5), dict(rescale_logits=True), dict(return_logits=True)):
        with pytest.raises(AssertionError, match="Gumbel"):
            q(z, **kw)


def test_no_cpu_fallback():
    import __graft_entry__ as ge
    ge.build()
    from sdb200 import _lib, ops
    from sdb200.quantize import VectorQuantizer2
    q = VectorQuantizer2(16, 3, 0.25)
    with pytest.raises(_lib.SdbError):
        q(torch.zeros(1, 3, 4, 4), temp=1.0)
    with pytest.raises(_lib.SdbError):
        ops.vq_quantize(torch.zeros(1, 3, 4, 4), torch.zeros(16, 3))
    with pytest.raises(_lib.SdbError):
        _vq().decode(torch.zeros(1, 3, 8, 8))


def test_identity_first_stage():
    from sdb200.autoencoder import IdentityFirstStage
    x = torch.randn(2, 3, 8, 8)
    f = IdentityFirstStage(1, 2, foo="bar")
    assert f.encode(x) is x and f.decode(x, 7) is x and f(x) is x and f.quantize(x) is x
    fv = IdentityFirstStage(vq_interface=True)
    q, loss, info = fv.quantize(x)
    assert q is x and loss is None and info == [None, None, None]


def test_decode_first_stage_routing():
    from sdb200.autoencoder import VQModelInterface
    from sdb200.pipeline import LatentDiffusion

    class FakeVQ(VQModelInterface):
        def __init__(self):
            nn.Module.__init__(self)
            self.calls = []

        def decode(self, h, force_not_quantize=False):
            self.calls.append((h.clone(), force_not_quantize))
            return h

    class FakeKL(nn.Module):
        def __init__(self):
            super().__init__()
            self.calls = []

        def decode(self, z):                     # one argument only: the KL first stage is called as before
            self.calls.append(z.clone())
            return z

    ld = LatentDiffusion(first_stage_config=False, unet=nn.Linear(1, 1), scale_factor=0.5, channels=3)
    z = torch.randn(1, 3, 4, 4)
    ld.first_stage_model = FakeVQ()
    ld.decode_first_stage(z)
    ld.decode_first_stage(z, force_not_quantize=True)
    calls = ld.first_stage_model.calls
    assert [f for _, f in calls] == [False, True]
    assert all(torch.equal(h, 1. / 0.5 * z) for h, _ in calls)
    ld.first_stage_model = FakeKL()
    ld.decode_first_stage(z)
    ld.decode_first_stage(z, force_not_quantize=True)
    assert len(ld.first_stage_model.calls) == 2 and torch.equal(ld.first_stage_model.calls[0], 2. * z)


def test_vq_entry_point_argument_checks():
    import __graft_entry__ as ge
    ge.build()
    from sdb200 import _lib
    lib = _lib.load()
    f = 256                                                   # never dereferenced: the checks run before any launch
    assert lib.sdb_vq_ws_bytes(0, 8) == -1 and lib.sdb_vq_ws_bytes(4096, 0) == -1
    assert lib.sdb_vq_ws_bytes(4096, 1) >= 8 * 4096 and lib.sdb_vq_ws_bytes(32768, 16384) > 0

    def q(z=f, zl=0, N=1, HW=64, D=3, cb=f, n_e=16, zq=f, zql=1, idx=f, loss=f, ws=f, ctr=f):
        return lib.sdb_vq_quantize(z, zl, N, HW, D, cb, n_e, 0.25, zq, zql, idx, loss, ws, ctr, None)

    assert q(z=None) == -1 and b"null" in lib.sdb_last_error_string()
    assert q(cb=None) == -1
    assert q(ws=None) == -1
    assert q(zq=None, idx=None, loss=None) == -1                                 # nothing to compute
    assert q(ctr=None) == -1                                                     # loss without its ticket counter
    assert q(D=0) == -1 and q(D=17) == -1 and b"D=17" in lib.sdb_last_error_string()
    assert q(n_e=0) == -1 and q(N=0) == -1 and q(HW=0) == -1
    assert q(zl=2) == -1 and q(zql=-1) == -1 and b"layout" in lib.sdb_last_error_string()

    def g(idx=f, M=64, cb=f, n_e=16, D=3, out=f, lay=0, HW=64):
        return lib.sdb_vq_codebook_gather(idx, M, cb, n_e, D, out, lay, HW, None)

    assert g(idx=None) == -1 and g(cb=None) == -1 and g(out=None) == -1
    assert g(D=0) == -1 and g(D=17) == -1 and g(n_e=0) == -1 and g(M=0) == -1 and g(M=65) == -1
    assert g(lay=2) == -1 and b"vq_codebook_gather" in lib.sdb_last_error_string()
