"""Drop-in `FrozenCLIPEmbedder` (reference: clip_encoder/modules.py:212-256) — SURVEY.md §8 'next' row f2, the text
conditioner that produces the `context` [B, 77, 768] the UNet's cross-attention reads.

The reference class wraps two objects of a third-party dependency, HuggingFace `transformers` (`CLIPTokenizer`,
`CLIPTextModel`; `transformers==4.49.0` in req.txt, 5.5 in this image), and returns `outputs.last_hidden_state`.  The
tokenizer is host-side string processing and stays HF's; the text tower — token + position embedding, 12 pre-LayerNorm
transformer layers with CAUSAL self-attention (12 heads of 64) and a quick-GELU MLP, final LayerNorm — runs here on the
same sm_100a kernels as the UNet: `tc_attention_kernel` with its causal mask (one 128-key tile covers the 77 tokens),
tcgen05 GEMMs with fused bias / residual, `layernorm_kernel`.  Module and parameter names are HF's
(`text_model.encoder.layers.N.self_attn.q_proj.weight`, ...), so `load_state_dict(CLIPTextModel(...).state_dict())` works
unchanged.  torch.nn layers are parameter holders only; there is no CPU or PyTorch fallback.
"""
import torch
from torch import nn

from . import engine, ops
from .engine import PackedLinear

CLIP_VIT_L14_TEXT = dict(vocab_size=49408, hidden_size=768, intermediate_size=3072, num_hidden_layers=12,
                         num_attention_heads=12, max_position_embeddings=77, layer_norm_eps=1e-5, hidden_act="quick_gelu")


class CLIPTextEmbeddings(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        self.token_embedding = nn.Embedding(cfg["vocab_size"], cfg["hidden_size"])
        self.position_embedding = nn.Embedding(cfg["max_position_embeddings"], cfg["hidden_size"])


class CLIPAttention(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        D = cfg["hidden_size"]
        self.k_proj, self.v_proj, self.q_proj, self.out_proj = nn.Linear(D, D), nn.Linear(D, D), nn.Linear(D, D), nn.Linear(D, D)


class CLIPMLP(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        self.fc1 = nn.Linear(cfg["hidden_size"], cfg["intermediate_size"])
        self.fc2 = nn.Linear(cfg["intermediate_size"], cfg["hidden_size"])


class CLIPEncoderLayer(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        self.self_attn = CLIPAttention(cfg)
        self.layer_norm1 = nn.LayerNorm(cfg["hidden_size"], eps=cfg["layer_norm_eps"])
        self.mlp = CLIPMLP(cfg)
        self.layer_norm2 = nn.LayerNorm(cfg["hidden_size"], eps=cfg["layer_norm_eps"])


class CLIPEncoder(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        self.layers = nn.ModuleList([CLIPEncoderLayer(cfg) for _ in range(cfg["num_hidden_layers"])])


class CLIPTextTransformer(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        self.embeddings = CLIPTextEmbeddings(cfg)
        self.encoder = CLIPEncoder(cfg)
        self.final_layer_norm = nn.LayerNorm(cfg["hidden_size"], eps=cfg["layer_norm_eps"])


class TextModelOutput(object):
    """The one field of HF's BaseModelOutputWithPooling that FrozenCLIPEmbedder reads (clip_encoder/modules.py:251)."""

    def __init__(self, last_hidden_state):
        self.last_hidden_state = last_hidden_state

    def __getitem__(self, i):
        return (self.last_hidden_state,)[i]


class CLIPTextModel(engine.PackedWeights, nn.Module):
    """HF `CLIPTextModel` (text tower only, `last_hidden_state` only), same state-dict keys.  `config`: a dict with the keys of
    CLIP_VIT_L14_TEXT, or an HF CLIPTextConfig.  Extra keyword: compute_mode "bf16" (tensor cores) / "fp32" (SIMT parity mode)."""

    def __init__(self, config=None, compute_mode=None):
        super().__init__()
        cfg = dict(CLIP_VIT_L14_TEXT)
        if config is not None:
            src = config if isinstance(config, dict) else {k: getattr(config, k) for k in CLIP_VIT_L14_TEXT if hasattr(config, k)}
            cfg.update(src)
        if cfg["hidden_act"] not in ("quick_gelu", "gelu"):
            raise NotImplementedError("sdb200 CLIPTextModel: hidden_act %r is not built" % (cfg["hidden_act"],))
        D, H = cfg["hidden_size"], cfg["num_attention_heads"]
        if D % H or (D // H) % 8 or D // H > 192 or D % 8:
            raise NotImplementedError("sdb200 CLIPTextModel: head size %d unsupported" % (D // max(H, 1)))
        self.config = cfg
        self.compute_mode = compute_mode or engine.default_mode()
        self.text_model = CLIPTextTransformer(cfg)
        self._init_packing()

    def _build_pack(self, mode):
        tm = self.text_model
        P = {"tok": tm.embeddings.token_embedding.weight.detach().float().contiguous(),
             "pos": tm.embeddings.position_embedding.weight.detach().float().contiguous(), "pos_rep": {}}
        for i, L in enumerate(tm.encoder.layers):
            a = L.self_attn
            P[("qkv", i)] = PackedLinear(torch.cat([a.q_proj.weight, a.k_proj.weight, a.v_proj.weight], 0),
                                         torch.cat([a.q_proj.bias, a.k_proj.bias, a.v_proj.bias], 0), mode)
            P[("out", i)] = PackedLinear(a.out_proj.weight, a.out_proj.bias, mode)
            P[("fc1", i)] = PackedLinear(L.mlp.fc1.weight, L.mlp.fc1.bias, mode)
            P[("fc2", i)] = PackedLinear(L.mlp.fc2.weight, L.mlp.fc2.bias, mode)
        return P

    def _forward_tokens(self, ids, mode):
        cfg = self.config
        P = self.packed(mode)
        B, S = ids.shape
        D, H = cfg["hidden_size"], cfg["num_attention_heads"]
        d = D // H
        assert S <= cfg["max_position_embeddings"], "sequence longer than the position table"
        odt = engine.op_dtype(mode)
        scale = d ** -0.5
        act = 3 if cfg["hidden_act"] == "quick_gelu" else 2
        x = ops.gather_rows(P["tok"], ids.reshape(-1).contiguous())                              # [B*S, D] fp32
        pos = P["pos_rep"].get((B, S))
        if pos is None:
            pos = P["pos_rep"][(B, S)] = P["pos"][:S].repeat(B, 1).contiguous()
        x = ops.add(x, pos)
        W3 = 3 * D
        for i, L in enumerate(self.text_model.encoder.layers):
            a = ops.layernorm(x, L.layer_norm1.weight, L.layer_norm1.bias, L.layer_norm1.eps, out_dtype=odt)
            qkv = engine.linear(a, P[("qkv", i)], out_dtype=odt, rows_per_item=S)               # [B*S, 3D]: q | k | v
            if mode == "bf16":
                o = ops.attention_tc(qkv, qkv[:, D:], qkv[:, 2 * D:], B, H, S, S, d, engine.head_pad(d), scale,
                                     (S * W3, W3, d), (S * W3, W3, d), (S * W3, W3, d), dense=True, causal=True)
                o = o.reshape(B * S, D)
            else:
                o = engine.attention_fp32(qkv, qkv[:, D:], qkv[:, 2 * D:], B, H, S, S, d, scale, causal=True)
            x = engine.linear(o, P[("out", i)], residual=x, rows_per_item=S)
            a = ops.layernorm(x, L.layer_norm2.weight, L.layer_norm2.bias, L.layer_norm2.eps, out_dtype=odt)
            h = engine.linear(a, P[("fc1", i)], rows_per_item=S)                                # fp32 [B*S, 4D]
            h = ops.activation(h, act, out_dtype=odt)
            x = engine.linear(h, P[("fc2", i)], residual=x, rows_per_item=S)
        fl = self.text_model.final_layer_norm
        return ops.layernorm(x, fl.weight, fl.bias, fl.eps, out_dtype=torch.float32).reshape(B, S, D)

    @torch.no_grad()
    def forward(self, input_ids=None, **kwargs):
        from ._lib import require_cuda
        assert input_ids is not None and input_ids.dim() == 2, "input_ids [B, S] expected"
        with torch.cuda.device(input_ids.device):
            require_cuda(input_ids)
            self._check_weights()
            ids = input_ids.to(torch.int64).contiguous()
            return TextModelOutput(self._forward_tokens(ids, self.compute_mode))


class FrozenCLIPEmbedder(nn.Module):
    """Uses the CLIP transformer encoder for text (clip_encoder/modules.py:212-256): `forward(text)` -> [B, max_length, 768].

    Differences forced by the missing network: the architecture is built from `config` (ViT-L/14 text tower by default) with
    PyTorch's default initialisation instead of `from_pretrained(version)` — load HF weights with
    `self.transformer.load_state_dict(CLIPTextModel.from_pretrained(version).state_dict())` or `FrozenCLIPEmbedder.from_hf(...)`;
    the tokenizer is created on first use from the local HF cache.  `forward` also accepts an int tensor of token ids."""

    def __init__(self, version="openai/clip-vit-large-patch14", device="cuda", max_length=77, config=None, compute_mode=None):
        super().__init__()
        self.version = version
        self.tokenizer = None
        self.transformer = CLIPTextModel(config, compute_mode=compute_mode)
        self.device = device
        self.max_length = max_length
        self.freeze()

    @classmethod
    def from_hf(cls, version="openai/clip-vit-large-patch14", device="cuda", max_length=77, compute_mode=None):
        from transformers import CLIPTextModel as HFText
        hf = HFText.from_pretrained(version)
        self = cls(version, device, max_length, config=hf.config, compute_mode=compute_mode)
        self.transformer.load_state_dict(hf.state_dict(), strict=False)
        return self.to(device)

    def freeze(self):
        self.transformer = self.transformer.eval()
        for param in self.parameters():
            param.requires_grad = False

    def _tokens(self, text):
        if torch.is_tensor(text):
            return text
        if self.tokenizer is None:
            from transformers import CLIPTokenizer
            self.tokenizer = CLIPTokenizer.from_pretrained(self.version)       # raises when the vocabulary is not cached locally
        enc = self.tokenizer(text, truncation=True, max_length=self.max_length, return_length=True,
                             return_overflowing_tokens=False, padding="max_length", return_tensors="pt")
        return enc["input_ids"]

    def forward(self, text):
        tokens = self._tokens(text).to(self.device)
        outputs = self.transformer(input_ids=tokens)
        return outputs.last_hidden_state

    def encode(self, text):
        return self(text)
