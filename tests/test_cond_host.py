"""CPU: the conditioning stages of sdb200.encoders and LatentDiffusion's cond-stage rules (ldm/diffusion/ddpm.py
instantiate_cond_stage / get_learned_conditioning) on the host — constructor kwargs, the exact state-dict keys, strict
loading of CompVis-keyed state dicts, SpatialRescaler's asserts and output-size rule, the routing with stub models, and the
host-side argument checks of sdb_embed_rows / sdb_interpolate_nchw."""
import ctypes as C

import pytest
import torch
from torch import nn

from sdb200 import encoders as E
from sdb200 import ops
from sdb200.pipeline import LatentDiffusion


def _layer_keys(depth):
    keys = []
    for i in range(2 * depth):
        p = "transformer.attn_layers.layers.%d." % i
        keys += [p + "0.weight", p + "0.bias"]
        if i % 2 == 0:
            keys += [p + "1.to_q.weight", p + "1.to_k.weight", p + "1.to_v.weight", p + "1.to_out.weight", p + "1.to_out.bias"]
        else:
            keys += [p + "1.net.0.0.weight", p + "1.net.0.0.bias", p + "1.net.2.weight", p + "1.net.2.bias"]
    return (["transformer.token_emb.weight", "transformer.pos_emb.emb.weight"] + keys
            + ["transformer.norm.weight", "transformer.norm.bias", "transformer.to_logits.weight", "transformer.to_logits.bias"])


def test_text_embedders_kwargs_keys_and_shapes():
    b = E.BERTEmbedder(64, 2)
    assert b.use_tknz_fn and b.max_seq_len == 77 and b.device == "cuda" and b.tokenizer is None
    assert b.transformer.num_tokens == 30522 and b.transformer.max_seq_len == 77 and b.transformer.emb_dropout.p == 0.0
    assert E.BERTEmbedder(64, 2, embedding_dropout=0.1).transformer.emb_dropout.p == 0.1
    t = E.TransformerEmbedder(64, 3, 500)
    assert t.transformer.max_seq_len == 77 and t.device == "cuda"
    for m, depth in ((b, 2), (t, 3)):
        assert list(m.state_dict()) == _layer_keys(depth)
    sd = t.state_dict()
    assert sd["transformer.token_emb.weight"].shape == (500, 64) and sd["transformer.pos_emb.emb.weight"].shape == (77, 64)
    p = "transformer.attn_layers.layers."
    assert sd[p + "0.1.to_q.weight"].shape == (512, 64) and sd[p + "0.1.to_out.weight"].shape == (64, 512)
    assert sd[p + "1.1.net.0.0.weight"].shape == (256, 64) and sd[p + "1.1.net.2.weight"].shape == (64, 256)
    assert sd["transformer.to_logits.weight"].shape == (500, 64)


def test_strict_load_with_to_logits():
    t = E.TransformerEmbedder(64, 2, 100)
    sd = {k: torch.randn(v.shape) for k, v in t.state_dict().items()}
    E.TransformerEmbedder(64, 2, 100).load_state_dict(sd, strict=True)
    E.BERTEmbedder(64, 2, 100).load_state_dict(sd, strict=True)
    del sd["transformer.to_logits.bias"]
    with pytest.raises(RuntimeError):
        E.TransformerEmbedder(64, 2, 100).load_state_dict(sd, strict=True)


def test_class_embedder_and_rescaler_keys():
    c = E.ClassEmbedder(32)
    assert c.key == "class" and list(c.state_dict()) == ["embedding.weight"] and c.embedding.weight.shape == (1000, 32)
    assert E.ClassEmbedder(8, n_classes=10, key="class_label").key == "class_label"
    assert list(E.SpatialRescaler().state_dict()) == []
    r = E.SpatialRescaler(n_stages=2, in_channels=182, out_channels=3)
    assert list(r.state_dict()) == ["channel_mapper.weight"] and r.channel_mapper.weight.shape == (3, 182, 1, 1)
    assert list(E.SpatialRescaler(in_channels=4, out_channels=2, bias=True).state_dict()) == [
        "channel_mapper.weight", "channel_mapper.bias"]
    r = E.SpatialRescaler()
    assert r.n_stages == 1 and r.method == "bilinear" and r.multiplier == 0.5 and not r.remap_output
    assert E.FrozenCLIPEmbedder is __import__("sdb200.clip_text", fromlist=["x"]).FrozenCLIPEmbedder


def test_rescaler_asserts_and_4d_linear_rejected():
    with pytest.raises(AssertionError):
        E.SpatialRescaler(method="nearest-exact")
    with pytest.raises(AssertionError):
        E.SpatialRescaler(n_stages=-1)
    x = torch.zeros(1, 3, 8, 8)
    for m in ("linear", "trilinear"):
        E.SpatialRescaler(method=m)                    # accepted by the constructor, as in the reference
        with pytest.raises(NotImplementedError):
            ops.interpolate(x, scale_factor=0.5, mode=m)
    with pytest.raises(ValueError):
        ops.interpolate(x, scale_factor=0.5, mode="nearest-exact")
    x = torch.zeros(1, 3, 8, 8)
    assert E.SpatialRescaler(n_stages=0)(x) is x       # no stage and no map: the input itself


@pytest.mark.parametrize("hw", [(64, 64), (37, 53), (7, 5)])
@pytest.mark.parametrize("s", [0.5, 0.25, 2, 0.75, 1.5, 0.3])
def test_output_size_rule_matches_torch(hw, s):
    x = torch.zeros(1, 1, *hw)
    assert ops.interpolate_size(hw, scale_factor=s) == tuple(torch.nn.functional.interpolate(x, scale_factor=s).shape[-2:])
    assert ops.interpolate_size(hw, size=(5, 9)) == (5, 9) and ops.interpolate_size(hw, size=4) == (4, 4)
    with pytest.raises(ValueError):
        ops.interpolate_size(hw)
    with pytest.raises(ValueError):
        ops.interpolate_size(hw, scale_factor=s, size=4)


# ---- LatentDiffusion cond-stage rules ----------------------------------------------------------------------------------------
class Stub(nn.Module):
    def __init__(self, tag):
        super().__init__()
        self.tag = tag
        self.lin = nn.Linear(1, 1)

    def forward(self, c):
        return ("forward", self.tag, c)

    def encode(self, c):
        return ("encode", self.tag, c)

    def custom(self, c):
        return ("custom", self.tag, c)


class NoEncode(nn.Module):
    def forward(self, c):
        return ("forward", c)


class DistStage(nn.Module):
    """encode returns a DiagonalGaussianDistribution (AutoencoderKL); its kernel is replaced by a host stub."""

    def encode(self, c):
        from sdb200.autoencoder import DiagonalGaussianDistribution
        d = DiagonalGaussianDistribution.__new__(DiagonalGaussianDistribution)
        d.mean, d.deterministic = c * 2, False
        return d


def _ld(**kw):
    return LatentDiffusion(unet=nn.Identity(), first_stage_config=False, **kw)


def test_cond_stage_config_routing():
    fs = Stub("first")
    ld = LatentDiffusion(unet=nn.Identity(), first_stage_model=fs, cond_stage_config="__is_first_stage__")
    assert ld.cond_stage_model is fs and ld.model.conditioning_key == "crossattn"
    assert ld.get_learned_conditioning(3) == ("encode", "first", 3)
    ld = _ld(cond_stage_config="__is_unconditional__", conditioning_key="concat")
    assert ld.cond_stage_model is None and ld.model.conditioning_key is None
    ld = _ld(cond_stage_model=Stub("c"))
    assert ld.cond_stage_forward is None and not ld.cond_stage_trainable
    assert ld.get_learned_conditioning(1) == ("encode", "c", 1)
    assert _ld(cond_stage_model=NoEncode()).get_learned_conditioning(2) == ("forward", 2)
    ld = _ld(cond_stage_model=Stub("c"), cond_stage_forward="custom")
    assert ld.get_learned_conditioning(5) == ("custom", "c", 5)
    with pytest.raises(AssertionError):
        _ld(cond_stage_model=Stub("c"), cond_stage_forward="missing").get_learned_conditioning(5)
    assert _ld(cond_stage_model=Stub("c"), cond_stage_trainable=True).cond_stage_trainable
    with pytest.raises(NotImplementedError):
        _ld(cond_stage_config={"target": "ldm.modules.encoders.modules.ClassEmbedder"})
    with pytest.raises(AssertionError):
        _ld(cond_stage_config="__is_first_stage__", cond_stage_trainable=True)
    with pytest.raises(ValueError):
        _ld(cond_stage_config="__is_unconditional__", cond_stage_model=Stub("c"))


def test_distribution_conditioning_takes_the_mode():
    c = _ld(cond_stage_model=DistStage()).get_learned_conditioning(torch.ones(2))
    assert torch.equal(c, torch.full((2,), 2.0))


# ---- C-ABI argument checks (never dereferenced: the checks run before any launch) ---------------------------------------------
def test_cond_entry_point_argument_checks():
    import __graft_entry__ as ge
    ge.build()
    from sdb200 import _lib
    lib = _lib.load()
    p = 256

    def e(table=p, ids=p, n=4, dim=8, vocab=10, pos=None, S=0, out=p):
        return lib.sdb_embed_rows(table, ids, n, dim, vocab, pos, S, out, None)
    assert e(table=None) == -1 and b"null" in lib.sdb_last_error_string()
    assert e(ids=None) == -1 and e(out=None) == -1
    for bad in (dict(n=0), dict(dim=0), dict(vocab=0), dict(vocab=-3)):
        assert e(**bad) == -1, bad
    assert e(pos=p, S=0) == -1 and b"seq_len" in lib.sdb_last_error_string()

    def i(x=p, N=1, Cc=3, H=8, W=8, OH=4, OW=4, mode=1, sh=0.5, sw=0.5, w=None, b=None, Cout=0, out=p):
        return lib.sdb_interpolate_nchw(x, N, Cc, H, W, OH, OW, mode, C.c_double(sh), C.c_double(sw), w, b, Cout, out, None)
    assert i(x=None) == -1 and i(out=None) == -1
    for bad in (dict(N=0), dict(Cc=0), dict(H=0), dict(W=-1), dict(OH=0), dict(OW=0), dict(mode=4), dict(mode=-1),
                dict(sh=-1.0)):
        assert i(**bad) == -1, bad
    assert i(Cout=3) == -1 and b"Cout=3" in lib.sdb_last_error_string()
    assert i(b=p) == -1 and i(w=p, Cout=0) == -1
    assert i(OH=1 << 16, OW=1 << 16) == -1 and b"too large" in lib.sdb_last_error_string()
