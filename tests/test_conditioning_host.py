"""CPU: the conditioning keys of DiffusionWrapper (ldm/diffusion/ddpm.py:1992-2034), LatentDiffusion.apply_model's key rule,
DDIMSampler.sample with a dict of lists, and the argument checks UNetModel.forward_concat makes before any kernel runs."""
import pytest
import torch

from sdb200.ddim import DDIMSampler
from sdb200.openai_model import UNetModel
from sdb200.pipeline import DiffusionWrapper, LatentDiffusion

TINY = dict(image_size=8, in_channels=9, out_channels=4, model_channels=32, attention_resolutions=[1], num_res_blocks=1,
            channel_mult=(1,), num_heads=2, use_spatial_transformer=True, transformer_depth=1, context_dim=16, legacy=False)


class Recorder(torch.nn.Module):
    """Eps-model stub that records how it was called."""

    def __init__(self, with_concat=False):
        super().__init__()
        self.calls = []
        if with_concat:
            self.forward_concat = self._forward_concat

    def forward(self, x, t, context=None, y=None):
        self.calls.append(("forward", x, t, context, y))
        return x[:, :4] * 0.5

    def _forward_concat(self, x, c_concat, timesteps=None, context=None, y=None):
        self.calls.append(("forward_concat", x, list(c_concat), timesteps, context, y))
        return x * 0.5


def _inputs(B=2):
    g = torch.Generator().manual_seed(0)
    x = torch.randn(B, 4, 8, 8, generator=g)
    t = torch.tensor([5, 7][:B])
    m = torch.randn(B, 1, 8, 8, generator=g)
    z = torch.randn(B, 4, 8, 8, generator=g)
    ctx = torch.randn(B, 3, 16, generator=g)
    ctx2 = torch.randn(B, 2, 16, generator=g)
    return x, t, m, z, ctx, ctx2


def test_key_none():
    x, t, *_ = _inputs()
    r = Recorder()
    DiffusionWrapper(r, None)(x, t)
    (name, xx, tt, ctx, y), = r.calls
    assert name == "forward" and xx is x and tt is t and ctx is None and y is None


def test_key_crossattn_passes_one_context_unchanged():
    x, t, m, z, ctx, ctx2 = _inputs()
    r = Recorder()
    w = DiffusionWrapper(r, "crossattn")
    w(x, t, c_crossattn=[ctx])
    w(x, t, c_crossattn=[ctx, ctx2])
    assert r.calls[0][3] is ctx
    assert torch.equal(r.calls[1][3], torch.cat([ctx, ctx2], 1))


@pytest.mark.parametrize("has_fc", [True, False])
def test_key_concat(has_fc):
    x, t, m, z, ctx, _ = _inputs()
    r = Recorder(with_concat=has_fc)
    DiffusionWrapper(r, "concat")(x, t, c_concat=[m, z])
    (call,) = r.calls
    if has_fc:
        name, xx, cc, tt, c, y = call
        assert name == "forward_concat" and xx is x and cc[0] is m and cc[1] is z and tt is t and c is None and y is None
    else:
        name, xx, tt, c, y = call
        assert name == "forward" and torch.equal(xx, torch.cat([x, m, z], 1)) and tt is t and c is None and y is None


@pytest.mark.parametrize("has_fc", [True, False])
def test_key_hybrid(has_fc):
    x, t, m, z, ctx, ctx2 = _inputs()
    r = Recorder(with_concat=has_fc)
    w = DiffusionWrapper(r, "hybrid")
    w(x, t, c_concat=[m, z], c_crossattn=[ctx])
    w(x, t, c_concat=[torch.cat([m, z], 1)], c_crossattn=[ctx, ctx2])
    if has_fc:
        assert [c[0] for c in r.calls] == ["forward_concat"] * 2
        assert r.calls[0][1] is x and r.calls[0][2][0] is m and r.calls[0][4] is ctx
        assert torch.equal(r.calls[1][4], torch.cat([ctx, ctx2], 1))
    else:
        assert [c[0] for c in r.calls] == ["forward"] * 2
        assert torch.equal(r.calls[0][1], torch.cat([x, m, z], 1)) and r.calls[0][3] is ctx
        assert torch.equal(r.calls[1][3], torch.cat([ctx, ctx2], 1))


def test_key_adm():
    x, t, *_ = _inputs()
    y = torch.tensor([3, 1])
    r = Recorder(with_concat=True)
    DiffusionWrapper(r, "adm")(x, t, c_crossattn=[y])
    (name, xx, tt, ctx, yy), = r.calls
    assert name == "forward" and xx is x and tt is t and ctx is None and yy is y


@pytest.mark.parametrize("key", ["crossattn-adm", "hybrid-adm", "concatenate", ""])
def test_unknown_key_rejected(key):
    with pytest.raises(AssertionError):
        DiffusionWrapper(Recorder(), key)
    with pytest.raises(AssertionError):
        LatentDiffusion(first_stage_config=False, unet=Recorder(), conditioning_key=key)


@pytest.mark.parametrize("key,where", [("concat", "c_concat"), ("hybrid", "c_crossattn"), ("crossattn", "c_crossattn"),
                                       ("adm", "c_crossattn")])
def test_apply_model_key_rule(key, where):
    x, t, m, *_ = _inputs()
    ld = LatentDiffusion(first_stage_config=False, unet=Recorder(), conditioning_key=key)
    seen = {}
    ld.model.forward = lambda x_, t_, **cond: seen.update(cond) or x_
    ld.apply_model(x, t, m)
    assert list(seen) == [where] and seen[where][0] is m
    seen.clear()
    ld.apply_model(x, t, [m])
    assert list(seen) == [where] and seen[where][0] is m
    seen.clear()
    ld.apply_model(x, t, {"c_concat": [m], "c_crossattn": [x]})          # a dict goes through as given
    assert set(seen) == {"c_concat", "c_crossattn"}


def test_ddim_sample_accepts_dict_of_lists(capsys):
    x, t, m, z, ctx, _ = _inputs()
    s = DDIMSampler(LatentDiffusion(first_stage_config=False, unet=Recorder(), conditioning_key="hybrid"))
    got = {}

    def fake_sampling(cond, size, **kw):
        got["cond"], got["size"] = cond, size
        return "done", {}

    s.ddim_sampling = fake_sampling
    cond = {"c_concat": [torch.cat([m, z], 1)], "c_crossattn": [ctx]}
    assert s.sample(5, 2, (4, 8, 8), cond, verbose=False)[0] == "done"
    assert got["cond"] is cond and got["size"] == (2, 4, 8, 8)
    assert "Warning" not in capsys.readouterr().out
    s.sample(5, 3, (4, 8, 8), cond, verbose=False)
    assert "Got 2 conditionings but batch-size is 3" in capsys.readouterr().out
    s.sample(5, 2, (4, 8, 8), {"c_crossattn": [[ctx]]}, verbose=False)          # nested lists are descended too
    assert "Warning" not in capsys.readouterr().out


def test_ddim_cfg_dict_pairing_rule():
    x, t, m, z, ctx, ctx2 = _inputs()
    ok = DDIMSampler._cfg_dict_pairable
    c = {"c_concat": [m], "c_crossattn": [ctx]}
    assert ok(c, {"c_concat": [m], "c_crossattn": [ctx2]})
    assert ok({"c_concat": m}, {"c_concat": z[:, :1]})
    assert not ok({"c_crossattn": [ctx]}, {"c_crossattn": [ctx2]})              # crossattn-only: the two-call path as before
    assert not ok(c, {"c_crossattn": [ctx2]})
    assert not ok(c, {"c_concat": [m, m], "c_crossattn": [ctx2]})
    assert not ok(ctx, ctx2)


def test_ddim_cfg_dict_cache():
    x, t, m, z, ctx, _ = _inputs()
    ctx2 = torch.randn_like(ctx)
    s = DDIMSampler(LatentDiffusion(first_stage_config=False, unet=Recorder(), conditioning_key="hybrid"))
    c = {"c_concat": [m], "c_crossattn": [ctx]}
    uc = {"c_concat": [m], "c_crossattn": [ctx2]}
    a = s._cfg_dict_in(c, uc)
    assert torch.equal(a["c_concat"][0], torch.cat([m, m])) and torch.equal(a["c_crossattn"][0], torch.cat([ctx2, ctx]))
    b = s._cfg_dict_in(c, uc)
    assert b is a and b["c_crossattn"][0] is a["c_crossattn"][0]                 # same pair: the cached tensors
    ctx.mul_(2.0)                                                                 # written in place: rebuilt
    d = s._cfg_dict_in(c, uc)
    assert d is not a and torch.equal(d["c_crossattn"][0], torch.cat([ctx2, ctx]))
    e = s._cfg_dict_in({"c_concat": [m], "c_crossattn": [ctx.clone()]}, uc)      # a new tensor object: rebuilt
    assert e is not d


def test_forward_concat_checks_before_any_kernel():
    net = UNetModel(**TINY)
    x, t, m, z, ctx, _ = _inputs()
    with pytest.raises(ValueError, match="in_channels=9"):
        net.forward_concat(x, [m], t, context=ctx)                                    # 4 + 1 != 9
    with pytest.raises(ValueError, match="in_channels=9"):
        net.forward_concat(x, [m, z, m], t, context=ctx)
    with pytest.raises(ValueError, match="N, H, W"):
        net.forward_concat(x, [m, z[:1]], t, context=ctx)
    with pytest.raises(ValueError, match="N, H, W"):
        net.forward_concat(x, [m, z[..., :4]], t, context=ctx)
    with pytest.raises(ValueError, match="4-D"):
        net.forward_concat(x, [m, z.flatten(2)], t, context=ctx)
    with pytest.raises(ValueError, match="tensor"):
        net.forward_concat(x, [], t, context=ctx)
    with pytest.raises(ValueError, match="tensor"):
        net.forward_concat(x, None, t, context=ctx)
    with pytest.raises(ValueError, match="one device"):
        net.forward_concat(x, [m.to("meta"), z], t, context=ctx)
    with pytest.raises(ValueError, match="one device"):
        net.forward_concat(x, [m, z], t.to("meta"), context=ctx)
    with pytest.raises(ValueError, match="one device"):
        net.forward_concat(x, torch.cat([m, z], 1), t, context=ctx.to("meta"))

