"""CPU: LatentDiffusion's split_input_params branch (ldm/diffusion/ddpm.py:1030-1139, 1344-1437) on the host — the weighting
helpers against the reference's expressions, the crop geometry, the conditioning rules, which first stages the branch takes,
and the host-side argument checks of sdb_patch_unfold / sdb_patch_fold.  The two kernels are replaced here by torch
restatements on the CPU (F.unfold / F.fold), so the routing can be checked without a GPU."""
import pytest
import torch
import torch.nn.functional as F
from torch import nn

from sdb200 import ops
from sdb200.pipeline import LatentDiffusion

SPLIT = dict(ks=(4, 4), stride=(2, 2), vqf=4, patch_distributed_vq=True, tie_braker=False, clip_max_weight=0.5,
             clip_min_weight=0.01, clip_max_tie_weight=0.5, clip_min_tie_weight=0.01)


# ---- the reference's expressions, restated -------------------------------------------------------------------------------
def ref_meshgrid(h, w):
    y = torch.arange(0, h).view(h, 1, 1).repeat(1, w, 1)
    x = torch.arange(0, w).view(1, w, 1).repeat(h, 1, 1)
    return torch.cat([y, x], dim=-1)


def ref_delta_border(h, w):
    arr = ref_meshgrid(h, w) / torch.tensor([h - 1, w - 1]).view(1, 1, 2)
    dist_left_up = torch.min(arr, dim=-1, keepdims=True)[0]
    dist_right_down = torch.min(1 - arr, dim=-1, keepdims=True)[0]
    return torch.min(torch.cat([dist_left_up, dist_right_down], dim=-1), dim=-1)[0]


def ref_get_weighting(sp, h, w, Ly, Lx):
    weighting = torch.clip(ref_delta_border(h, w), sp["clip_min_weight"], sp["clip_max_weight"])
    weighting = weighting.view(1, h * w, 1).repeat(1, 1, Ly * Lx)
    if sp["tie_braker"]:
        L_weighting = torch.clip(ref_delta_border(Ly, Lx), sp["clip_min_tie_weight"], sp["clip_max_tie_weight"])
        weighting = weighting * L_weighting.view(1, 1, Ly * Lx)
    return weighting


def _bits(a, b):
    return a.shape == b.shape and a.dtype == b.dtype and bool(((a == b) | (a.isnan() & b.isnan())).all())


# ---- CPU stand-ins for the two kernels (same contract as ops.patch_unfold / ops.patch_fold) -------------------------------
def cpu_unfold(x, ks, stride):
    B, C, H, W_ = x.shape
    Ly, Lx = ops.patch_grid(H, W_, ks, stride)
    if Ly < 1 or Lx < 1:
        raise ops._lib.SdbError("crop larger than the image")
    u = F.unfold(x.float(), ks, stride=stride)
    return u.view(B, C, ks[0], ks[1], -1).permute(4, 0, 1, 2, 3).reshape(-1, C, ks[0], ks[1])


def cpu_fold(o, B, grid, stride, out_hw, wpix, wcrop=None):
    L = grid[0] * grid[1]
    _, C, KH, KW = o.shape
    w = wpix.view(1, KH * KW, 1).repeat(1, 1, L)
    if wcrop is not None:
        w = w * wcrop.view(1, 1, L)
    oo = o.view(L, B, C, KH, KW).permute(1, 2, 3, 4, 0) * w.view(1, 1, KH, KW, L)
    return F.fold(oo.reshape(B, -1, L), out_hw, (KH, KW), stride=stride) / F.fold(w, out_hw, (KH, KW), stride=stride)


@pytest.fixture
def cpu_kernels(monkeypatch):
    calls = []
    monkeypatch.setattr(ops, "patch_unfold", lambda x, ks, st: calls.append(("unfold", tuple(x.shape), ks, st)) or cpu_unfold(x, ks, st))
    monkeypatch.setattr(ops, "patch_fold", lambda o, B, g, st, hw, wp, wc=None:
                        calls.append(("fold", tuple(o.shape), B, g, st, hw)) or cpu_fold(o, B, g, st, hw, wp, wc))
    return calls


class Recorder(nn.Module):
    """Batch-invariant eps-model stub: records its calls, returns 0.5 * x (+ the mean of a concat / context input)."""

    def __init__(self):
        super().__init__()
        self.calls = []

    def forward(self, x, t, context=None, y=None):
        self.calls.append((x.shape[0], t.clone(), context))
        return x * 0.5 + (0 if context is None else context.mean((1, 2)).view(-1, 1, 1, 1))


def _ld(key="concat", cond_stage_key="image", **sp):
    ld = LatentDiffusion(first_stage_config=False, unet=Recorder(), conditioning_key=key, cond_stage_key=cond_stage_key,
                         scale_factor=1.0, channels=3)
    if sp is not None:
        ld.split_input_params = dict(SPLIT, **sp)
    return ld


# ---- 1. weighting helpers -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("h,w", [(1, 1), (2, 3), (7, 7), (16, 12), (128, 128), (512, 512)])
def test_meshgrid_and_delta_border_bits(h, w):
    ld = _ld()
    m = ld.meshgrid(h, w)
    assert m.dtype == torch.int64 and torch.equal(m, ref_meshgrid(h, w))
    d = ld.delta_border(h, w)
    assert d.dtype == torch.float32 and _bits(d, ref_delta_border(h, w))


@pytest.mark.parametrize("tie", [False, True])
@pytest.mark.parametrize("h,w,Ly,Lx", [(4, 4, 3, 3), (16, 8, 2, 5), (128, 128, 3, 3), (512, 512, 3, 3), (8, 8, 1, 1)])
def test_get_weighting_bits_and_device_tables(h, w, Ly, Lx, tie):
    ld = _ld(tie_braker=tie, clip_min_weight=0.02, clip_max_weight=0.4, clip_min_tie_weight=0.05, clip_max_tie_weight=0.45)
    wt = ld.get_weighting(h, w, Ly, Lx, "cpu")
    assert _bits(wt, ref_get_weighting(ld.split_input_params, h, w, Ly, Lx))
    wpix, wcrop = ld._patch_weights(h, w, Ly, Lx, "cpu")
    assert wpix.shape == (h * w,) and (wcrop is None) == (not tie)
    table = wpix.view(h * w, 1).repeat(1, Ly * Lx) * (wcrop.view(1, -1) if tie else 1)
    assert _bits(table, wt[0])                                    # fl(wpix[p] * wcrop[l]) is the reference's element
    assert ld._patch_weights(h, w, Ly, Lx, "cpu")[0] is wpix      # cached per geometry
    ld.split_input_params["clip_max_weight"] = 0.3
    assert not torch.equal(ld._patch_weights(h, w, Ly, Lx, "cpu")[0], wpix) or h * w <= 4


# ---- 2. geometry ----------------------------------------------------------------------------------------------------------
def test_crop_grid_and_fold_geometry():
    assert ops.patch_grid(256, 256, (128, 128), (64, 64)) == (3, 3)
    assert ops.patch_grid(16, 12, (8, 4), (4, 4)) == (3, 3)
    assert ops.patch_grid(10, 10, (4, 4), (3, 3)) == (3, 3)          # (10 - 4) // 3 + 1
    assert ops.patch_grid(9, 9, (4, 4), (5, 5)) == (2, 2)            # stride > ks
    ld = _ld()
    assert ld._split_geometry(256, 256, (128, 128), (64, 64)) == ((3, 3), (128, 128), (64, 64), (256, 256))
    assert ld._split_geometry(16, 12, (8, 4), (4, 4)) == ((3, 3), (8, 4), (4, 4), (16, 12))
    assert ld._split_geometry(64, 64, (32, 32), (16, 16), uf=4) == ((3, 3), (128, 128), (64, 64), (256, 256))
    assert ld._split_geometry(256, 256, (128, 128), (64, 64), df=4) == ((3, 3), (32, 32), (16, 16), (64, 64))
    for kw in (dict(uf=4), dict(df=4)):
        with pytest.raises(NotImplementedError):
            ld._split_geometry(64, 64, (32, 16), (16, 16), **kw)


class FakeVQ(nn.Module):
    def __init__(self, f=4):
        super().__init__()
        self.f, self.calls = f, []

    def decode(self, h):
        self.calls.append(tuple(h.shape))
        return h.repeat_interleave(self.f, 2).repeat_interleave(self.f, 3)

    def encode(self, x):
        self.calls.append(tuple(x.shape))
        return x[:, :, ::self.f, ::self.f].contiguous()


def test_decode_and_encode_reduce_ks_and_stride(cpu_kernels, capsys):
    ld = _ld(ks=(128, 128), stride=(64, 64), vqf=4)
    ld.first_stage_model = FakeVQ()
    z = torch.randn(2, 3, 16, 16)
    img = ld.decode_first_stage(z)
    assert "reducing Kernel" in capsys.readouterr().out
    assert cpu_kernels[0] == ("unfold", (2, 3, 16, 16), (16, 16), (16, 16))
    assert ld.first_stage_model.calls == [(2, 3, 16, 16)]
    assert cpu_kernels[1] == ("fold", (2, 3, 64, 64), 2, (1, 1), (64, 64), (64, 64))
    assert img.shape == (2, 3, 64, 64) and torch.allclose(img, ld.first_stage_model.decode(z))
    cpu_kernels.clear()
    ld.split_input_params.update(ks=(8, 8), stride=(4, 4))
    ld.decode_first_stage(torch.randn(1, 3, 16, 16))
    assert cpu_kernels[0][2:] == ((8, 8), (4, 4)) and cpu_kernels[1][1:] == ((9, 3, 32, 32), 1, (3, 3), (16, 16), (64, 64))
    # encode: df = vqf, the image size is recorded
    cpu_kernels.clear()
    ld.split_input_params.update(ks=(32, 32), stride=(16, 16))
    x = torch.randn(1, 3, 64, 64)
    h = ld.encode_first_stage(x)
    assert ld.split_input_params["original_image_size"] == (64, 64)
    assert cpu_kernels[1][1:] == ((9, 3, 8, 8), 1, (3, 3), (4, 4), (16, 16)) and h.shape == (1, 3, 16, 16)
    # patch_distributed_vq False: the whole latent
    ld.split_input_params["patch_distributed_vq"] = False
    ld.first_stage_model.calls.clear()
    ld.decode_first_stage(z)
    assert ld.first_stage_model.calls == [(2, 3, 16, 16)]


def test_encode_rejects_kl_and_non_tensor_first_stages(cpu_kernels):
    from sdb200.autoencoder import AutoencoderKL
    ld = _ld(ks=(32, 32), stride=(16, 16))
    ld.first_stage_model = AutoencoderKL(ddconfig=dict(double_z=True, z_channels=4, resolution=32, in_channels=3, out_ch=3,
                                                       ch=32, ch_mult=(1, 2), num_res_blocks=1, attn_resolutions=[]), embed_dim=4)
    with pytest.raises(NotImplementedError):
        ld.encode_first_stage(torch.randn(1, 3, 64, 64))
    assert cpu_kernels == []                                      # rejected before any kernel

    class TupleEncoder(FakeVQ):
        def encode(self, x):
            return (x, None, None)
    ld.first_stage_model = TupleEncoder()
    with pytest.raises(NotImplementedError):
        ld.encode_first_stage(torch.randn(1, 3, 64, 64))


# ---- 3. apply_model ------------------------------------------------------------------------------------------------------
def test_image_keys_cut_the_conditioning(cpu_kernels):
    for csk in LatentDiffusion.SPLIT_IMAGE_KEYS:
        ld = _ld("concat", csk, ks=(4, 4), stride=(2, 2))
        fc = []
        ld.model.diffusion_model.forward_concat = lambda x, cc, t, **kw: fc.append((x, cc, t)) or x * 0.5 + cc[0][:, :3]
        x, c = torch.randn(2, 3, 8, 8), torch.randn(2, 3, 8, 8)
        t = torch.tensor([5, 7])
        out = ld.apply_model(x, t, c)
        assert len(fc) == 1 and fc[0][0].shape == (18, 3, 4, 4)  # 3 x 3 crops, one batch
        assert torch.equal(fc[0][1][0], cpu_unfold(c, (4, 4), (2, 2))) and torch.equal(fc[0][2], t.repeat(9))
        assert torch.allclose(out, 0.5 * x + c, atol=1e-6)
        # not 4-d or not the latent's size
        for bad in (torch.randn(2, 3, 8), torch.randn(2, 3, 8, 6)):
            with pytest.raises(ValueError):
                ld.apply_model(x, t, bad)


def test_other_keys_repeat_the_conditioning_and_cache_it(cpu_kernels):
    ld = _ld("crossattn", "caption", ks=(4, 4), stride=(2, 2))
    x, ctx = torch.randn(2, 3, 8, 8), torch.randn(2, 5, 6)
    t = torch.tensor([1, 2])
    out = ld.apply_model(x, t, ctx)
    ld.apply_model(x, t, ctx)
    calls = ld.model.diffusion_model.calls
    assert [n for n, _, _ in calls] == [18, 18]
    assert torch.equal(calls[0][2], ctx.repeat(9, 1, 1)) and calls[0][2] is calls[1][2]     # one repeated tensor
    assert torch.allclose(out, 0.5 * x + ctx.mean((1, 2)).view(-1, 1, 1, 1), atol=1e-6)
    ctx.add_(1.0)                                                 # written in place: a new repeat
    ld.apply_model(x, t, ctx)
    assert calls[2][2] is not calls[0][2] and torch.equal(calls[2][2], ctx.repeat(9, 1, 1))
    # conditioning_key None: the model is called without conditioning
    ld0 = _ld(None, "image", ks=(4, 4), stride=(2, 2))
    ld0.apply_model(x, t, None)
    assert ld0.model.diffusion_model.calls[0][0] == 18


@pytest.mark.parametrize("pb", [None, 1, 4, 9, 100])
def test_patch_batch_chunks(cpu_kernels, pb):
    ld = _ld("crossattn", "caption", ks=(4, 4), stride=(2, 2))
    ld.patch_batch = pb
    x, ctx = torch.randn(2, 3, 8, 8), torch.randn(2, 5, 6)
    out = ld.apply_model(x, torch.tensor([3, 4]), ctx)
    n = 9 if pb is None else min(pb, 9)
    sizes = [2 * min(n, 9 - l0) for l0 in range(0, 9, n)]
    assert [c[0] for c in ld.model.diffusion_model.calls] == sizes
    ld.patch_batch = None
    assert torch.equal(out, ld.apply_model(x, torch.tensor([3, 4]), ctx))


def test_split_asserts_and_unsupported_keys(cpu_kernels):
    ld = _ld("hybrid", "LR_image")
    x = torch.randn(1, 3, 8, 8)
    with pytest.raises(AssertionError):                           # hybrid: two conditioning entries
        ld.apply_model(x, torch.tensor([1]), {"c_concat": [x], "c_crossattn": [torch.randn(1, 5, 6)]})
    ld = _ld("concat", "LR_image")
    with pytest.raises(AssertionError):
        ld.apply_model(x, torch.tensor([1]), x, return_ids=True)
    with pytest.raises(AssertionError):                           # one tensor in the list
        ld.apply_model(x, torch.tensor([1]), {"c_concat": [x, x]})
    ld = _ld("crossattn", "coordinates_bbox")
    with pytest.raises(NotImplementedError):
        ld.apply_model(x, torch.tensor([1]), torch.randn(1, 5, 6))
    assert cpu_kernels == []


def test_hasattr_switches_the_branch():
    """With split_input_params the call goes to the crop kernels (which refuse CPU tensors); without it, the whole latent."""
    ld = _ld("crossattn", "caption")
    x, ctx = torch.randn(1, 3, 8, 8), torch.randn(1, 5, 6)
    with pytest.raises(ops._lib.SdbError):
        ld.apply_model(x, torch.tensor([1]), ctx)
    assert ld.model.diffusion_model.calls == []
    delattr(ld, "split_input_params")
    ld.apply_model(x, torch.tensor([1]), ctx)
    assert ld.model.diffusion_model.calls[0][0] == 1
    assert not hasattr(LatentDiffusion(first_stage_config=False, unet=Recorder()), "split_input_params")


def test_constructor_defaults():
    ld = LatentDiffusion(first_stage_config=False, unet=Recorder())
    assert ld.cond_stage_key == "image" and ld.patch_batch is None


# ---- 4. C-ABI argument checks (never dereferenced: the checks run before any launch) ---------------------------------------
def test_patch_entry_point_argument_checks():
    import __graft_entry__ as ge
    ge.build()
    from sdb200 import _lib
    lib = _lib.load()
    p = 256

    def u(x=p, B=1, C=3, H=8, W=8, kh=4, kw=4, sh=2, sw=2, out=p):
        return lib.sdb_patch_unfold(x, B, C, H, W, kh, kw, sh, sw, out, None)
    assert u(x=None) == -1 and b"null" in lib.sdb_last_error_string()
    assert u(out=None) == -1
    for bad in (dict(B=0), dict(C=0), dict(H=0), dict(W=-1), dict(kh=0), dict(kw=0), dict(sh=0), dict(sw=-2)):
        assert u(**bad) == -1, bad
    assert u(kh=9) == -1 and b"larger" in lib.sdb_last_error_string()

    def f(o=p, B=1, C=3, KH=4, KW=4, Ly=3, Lx=3, SH=2, SW=2, OH=8, OW=8, wpix=p, wcrop=None, L=9, out=p):
        return lib.sdb_patch_fold(o, B, C, KH, KW, Ly, Lx, SH, SW, OH, OW, wpix, wcrop, L, out, None)
    assert f(o=None) == -1 and f(wpix=None) == -1 and f(out=None) == -1
    for bad in (dict(B=0), dict(C=0), dict(KH=0), dict(KW=0), dict(Ly=0), dict(Lx=-1), dict(SH=0), dict(SW=0), dict(OH=0),
                dict(OW=0)):
        assert f(**bad) == -1, bad
    assert f(L=8) == -1 and b"L=8" in lib.sdb_last_error_string()
    assert f(OH=7) == -1 and b"outside" in lib.sdb_last_error_string()
    assert f(Lx=4, L=12) == -1 and f(KW=5) == -1
