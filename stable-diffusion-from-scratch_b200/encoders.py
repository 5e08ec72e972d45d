"""The conditioning stages of the latent-diffusion family (ldm/modules/encoders/modules.py, ldm/modules/x_transformer.py):
`BERTEmbedder`, `TransformerEmbedder`, `ClassEmbedder`, `SpatialRescaler`, and `FrozenCLIPEmbedder` re-exported from
clip_text.py, so that every conditioner of the reference's modules.py has one import path.

The two text embedders instantiate x-transformers' `TransformerWrapper(num_tokens, max_seq_len, attn_layers=Encoder(dim,
depth), emb_dropout)` and call it with `return_embeddings=True`.  Only what that reaches is built, in eval:
  x = token_emb(ids) + pos_emb.emb(arange(S))                      one sdb_embed_rows launch
  2 * depth pre-norm layers alternating 'a' and 'f', each x = block(LayerNorm(x)) + x
    'a'  8 heads of 64 (inner 512 whatever dim is), to_q / to_k / to_v without bias, to_out Linear(512, dim) with bias,
         scale 64 ** -0.5, fp32 softmax and NO mask: all S positions, padding included, attend to each other
    'f'  Linear(dim, 4 dim), exact-erf GELU, Linear(4 dim, dim)
  x = norm(x)                                                      the returned embeddings
The reference's semantics are restated here from CompVis latent-diffusion; this module is not pinned to a checkout of it.
Module and parameter names are x-transformers' (`transformer.attn_layers.layers.{i}.1.to_q.weight`, ...).  The unused
`transformer.to_logits` head exists so that CompVis checkpoints load strictly; it is never packed.  torch.nn layers are
parameter holders only; there is no CPU or PyTorch fallback.
"""
import torch
from torch import nn

from . import engine, ops
from .clip_text import FrozenCLIPEmbedder
from .engine import PackedLinear

__all__ = ["TransformerWrapper", "Encoder", "TransformerEmbedder", "BERTEmbedder", "ClassEmbedder", "SpatialRescaler",
           "FrozenCLIPEmbedder"]

DIM_HEAD, HEADS = 64, 8          # x-transformers' DEFAULT_DIM_HEAD and AttentionLayers' heads: what the embedders get


class AbsolutePositionalEmbedding(nn.Module):
    def __init__(self, dim, max_seq_len):
        super().__init__()
        self.emb = nn.Embedding(max_seq_len, dim)
        nn.init.normal_(self.emb.weight, std=0.02)


class Residual(nn.Module):
    pass


class Attention(nn.Module):
    def __init__(self, dim, dim_head=DIM_HEAD, heads=HEADS):
        super().__init__()
        inner = dim_head * heads
        self.scale = dim_head ** -0.5
        self.heads = heads
        self.to_q = nn.Linear(dim, inner, bias=False)
        self.to_k = nn.Linear(dim, inner, bias=False)
        self.to_v = nn.Linear(dim, inner, bias=False)
        self.dropout = nn.Dropout(0.0)
        self.to_out = nn.Linear(inner, dim)


class FeedForward(nn.Module):
    def __init__(self, dim, mult=4):
        super().__init__()
        inner = int(dim * mult)
        self.net = nn.Sequential(nn.Sequential(nn.Linear(dim, inner), nn.GELU()), nn.Dropout(0.0), nn.Linear(inner, dim))


class Encoder(nn.Module):
    """x-transformers `Encoder(dim, depth)` (AttentionLayers, causal=False, pre-norm, default block ('a', 'f'))."""

    def __init__(self, dim, depth):
        super().__init__()
        self.dim = dim
        self.depth = depth
        self.layer_types = ("a", "f") * depth
        self.layers = nn.ModuleList()
        for t in self.layer_types:
            block = Attention(dim) if t == "a" else FeedForward(dim)
            self.layers.append(nn.ModuleList([nn.LayerNorm(dim), block, Residual()]))


class TransformerWrapper(engine.PackedWeights, nn.Module):
    """x-transformers `TransformerWrapper(num_tokens, max_seq_len, attn_layers, emb_dropout)` as the embedders use it:
    `forward(ids, return_embeddings=True)` -> [B, S, dim] fp32.  Extra keyword: compute_mode "bf16" (tensor cores) /
    "fp32" (SIMT parity mode)."""

    def __init__(self, *, num_tokens, max_seq_len, attn_layers, emb_dropout=0.0, compute_mode=None):
        super().__init__()
        dim = attn_layers.dim
        if dim % 8:
            raise NotImplementedError("sdb200 TransformerWrapper: dim %d is not a multiple of 8" % dim)
        self.max_seq_len = max_seq_len
        self.num_tokens = num_tokens
        self.token_emb = nn.Embedding(num_tokens, dim)
        self.pos_emb = AbsolutePositionalEmbedding(dim, max_seq_len)
        self.emb_dropout = nn.Dropout(emb_dropout)      # the identity in eval
        self.project_emb = nn.Identity()                # emb_dim == dim
        self.attn_layers = attn_layers
        self.norm = nn.LayerNorm(dim)
        nn.init.normal_(self.token_emb.weight, std=0.02)
        self.to_logits = nn.Linear(dim, num_tokens)     # present in checkpoints, unused by return_embeddings=True
        self.compute_mode = compute_mode or engine.default_mode()
        self._init_packing()

    def _build_pack(self, mode):
        P = {"tok": self.token_emb.weight.detach().float().contiguous(),
             "pos": self.pos_emb.emb.weight.detach().float().contiguous()}
        layers = self.attn_layers.layers
        for i in range(self.attn_layers.depth):
            a, f = layers[2 * i][1], layers[2 * i + 1][1]
            P[("qkv", i)] = PackedLinear(torch.cat([a.to_q.weight, a.to_k.weight, a.to_v.weight], 0), None, mode)
            P[("out", i)] = PackedLinear(a.to_out.weight, a.to_out.bias, mode)
            P[("ff1", i)] = PackedLinear(f.net[0][0].weight, f.net[0][0].bias, mode)
            P[("ff2", i)] = PackedLinear(f.net[2].weight, f.net[2].bias, mode)
        return P

    def _forward_tokens(self, ids, mode):
        P = self.packed(mode)
        B, S = ids.shape
        D = self.attn_layers.dim
        inner, W3 = HEADS * DIM_HEAD, 3 * HEADS * DIM_HEAD
        odt = engine.op_dtype(mode)
        layers = self.attn_layers.layers
        x = ops.embed_rows(P["tok"], ids.reshape(-1), pos=P["pos"], seq_len=S)                   # [B*S, D] fp32
        for i in range(self.attn_layers.depth):
            na, a = layers[2 * i][0], layers[2 * i][1]
            nf = layers[2 * i + 1][0]
            h = ops.layernorm(x, na.weight, na.bias, na.eps, out_dtype=odt)
            qkv = engine.linear(h, P[("qkv", i)], out_dtype=odt, rows_per_item=S)                # [B*S, 3*512]: q | k | v
            if mode == "bf16":
                st = (S * W3, W3, DIM_HEAD)
                o = ops.attention_tc(qkv, qkv[:, inner:], qkv[:, 2 * inner:], B, HEADS, S, S, DIM_HEAD,
                                     engine.head_pad(DIM_HEAD), a.scale, st, st, st, dense=True, causal=False)
                o = o.reshape(B * S, inner)
            else:
                o = engine.attention_fp32(qkv, qkv[:, inner:], qkv[:, 2 * inner:], B, HEADS, S, S, DIM_HEAD, a.scale)
            x = engine.linear(o, P[("out", i)], residual=x, rows_per_item=S)
            h = ops.layernorm(x, nf.weight, nf.bias, nf.eps, out_dtype=odt)
            h = engine.linear(h, P[("ff1", i)], rows_per_item=S)                                 # fp32 [B*S, 4D]
            h = ops.activation(h, 2, out_dtype=odt)                                              # exact-erf GELU
            x = engine.linear(h, P[("ff2", i)], residual=x, rows_per_item=S)
        return ops.layernorm(x, self.norm.weight, self.norm.bias, self.norm.eps, out_dtype=torch.float32).reshape(B, S, D)

    @torch.no_grad()
    def forward(self, x, return_embeddings=False):
        from ._lib import require_cuda
        if not return_embeddings:
            raise NotImplementedError("sdb200 TransformerWrapper: only return_embeddings=True (the embedders' call) is built")
        if x.dim() != 2:
            raise ValueError("TransformerWrapper: token ids [B, S] expected (got %s)" % (tuple(x.shape),))
        if x.shape[1] > self.max_seq_len:
            raise ValueError("TransformerWrapper: %d tokens exceed max_seq_len=%d" % (x.shape[1], self.max_seq_len))
        with torch.cuda.device(x.device):
            require_cuda(x)
            self._check_weights()
            return self._forward_tokens(x.to(torch.int64).contiguous(), self.compute_mode)


class TransformerEmbedder(nn.Module):
    """Some transformer encoder layers (modules.py TransformerEmbedder): `forward(tokens)` -> [B, S, n_embed]."""

    def __init__(self, n_embed, n_layer, vocab_size, max_seq_len=77, device="cuda", compute_mode=None):
        super().__init__()
        self.device = device
        self.transformer = TransformerWrapper(num_tokens=vocab_size, max_seq_len=max_seq_len,
                                              attn_layers=Encoder(dim=n_embed, depth=n_layer), compute_mode=compute_mode)

    def forward(self, tokens):
        tokens = tokens.to(self.device)
        return self.transformer(tokens, return_embeddings=True)

    def encode(self, x):
        return self(x)


class BERTEmbedder(nn.Module):
    """Uses the BERT tokenizer and some transformer encoder layers (modules.py BERTEmbedder): `forward(text)` ->
    [B, max_seq_len, n_embed].  `text` is a list of strings or a [B, S] int tensor of token ids.  The tokenizer, HF
    `BertTokenizerFast("bert-base-uncased")`, is created on first use from the local HF cache (it raises when the vocabulary
    is not cached; nothing is downloaded) with padding="max_length", max_length=max_seq_len, truncation=True."""

    TOKENIZER = "bert-base-uncased"

    def __init__(self, n_embed, n_layer, vocab_size=30522, max_seq_len=77, device="cuda", use_tokenizer=True,
                 embedding_dropout=0.0, compute_mode=None):
        super().__init__()
        self.use_tknz_fn = use_tokenizer
        self.max_seq_len = max_seq_len
        self.tokenizer = None
        self.device = device
        self.transformer = TransformerWrapper(num_tokens=vocab_size, max_seq_len=max_seq_len,
                                              attn_layers=Encoder(dim=n_embed, depth=n_layer), emb_dropout=embedding_dropout,
                                              compute_mode=compute_mode)

    def _tokens(self, text):
        if torch.is_tensor(text):
            return text
        if not self.use_tknz_fn:
            raise ValueError("BERTEmbedder(use_tokenizer=False) takes token ids, not text")
        if self.tokenizer is None:
            from transformers import BertTokenizerFast
            self.tokenizer = BertTokenizerFast.from_pretrained(self.TOKENIZER, local_files_only=True)
        enc = self.tokenizer(text, truncation=True, max_length=self.max_seq_len, return_length=True,
                             return_overflowing_tokens=False, padding="max_length", return_tensors="pt")
        return enc["input_ids"]

    def forward(self, text):
        tokens = self._tokens(text).to(self.device)
        return self.transformer(tokens, return_embeddings=True)

    def encode(self, text):
        return self(text)


class ClassEmbedder(nn.Module):
    """modules.py ClassEmbedder: `forward(batch, key=None)` -> embedding(batch[key][:, None]) as [B, 1, embed_dim] fp32, one
    sdb_embed_rows launch.  A class id outside [0, n_classes) gives a NaN row."""

    def __init__(self, embed_dim, n_classes=1000, key="class"):
        super().__init__()
        self.key = key
        self.embedding = nn.Embedding(n_classes, embed_dim)

    @torch.no_grad()
    def forward(self, batch, key=None):
        from ._lib import require_cuda
        if key is None:
            key = self.key
        c = batch[key]
        w = self.embedding.weight
        with torch.cuda.device(w.device):
            require_cuda(c, w)
            ids = c.to(torch.int64).reshape(-1).contiguous()
            table = w.detach() if w.dtype == torch.float32 and w.is_contiguous() else w.detach().float().contiguous()
            return ops.embed_rows(table, ids).reshape(c.shape[0], 1, w.shape[1])


class SpatialRescaler(nn.Module):
    """modules.py SpatialRescaler: `n_stages` x F.interpolate(x, scale_factor=multiplier, mode=method), then the optional
    1x1 `channel_mapper` (in_channels -> out_channels).  Each stage is one sdb_interpolate_nchw launch and the channel map
    is fused into the last one; n_stages = 0 with a map is the map alone, still one launch."""

    METHODS = ["nearest", "linear", "bilinear", "trilinear", "bicubic", "area"]

    def __init__(self, n_stages=1, method="bilinear", multiplier=0.5, in_channels=3, out_channels=None, bias=False):
        super().__init__()
        self.n_stages = n_stages
        assert self.n_stages >= 0
        assert method in self.METHODS
        self.method = method
        self.multiplier = multiplier
        self.remap_output = out_channels is not None
        if self.remap_output:
            self.channel_mapper = nn.Conv2d(in_channels, out_channels, 1, bias=bias)

    @torch.no_grad()
    def forward(self, x):
        if self.n_stages == 0 and not self.remap_output:
            return x
        x = x.float().contiguous()
        w = b = None
        if self.remap_output:
            w = self.channel_mapper.weight.detach().float().reshape(self.channel_mapper.out_channels, -1).contiguous()
            b = None if self.channel_mapper.bias is None else self.channel_mapper.bias.detach().float().contiguous()
        with torch.cuda.device(x.device):
            if self.n_stages == 0:                  # nearest at the input's own size is the identity
                return ops.interpolate(x, size=tuple(x.shape[-2:]), mode="nearest", weight=w, bias=b)
            for stage in range(self.n_stages):
                last = stage == self.n_stages - 1
                x = ops.interpolate(x, scale_factor=self.multiplier, mode=self.method, weight=w if last else None,
                                    bias=b if last else None)
            return x

    def encode(self, x):
        return self(x)
