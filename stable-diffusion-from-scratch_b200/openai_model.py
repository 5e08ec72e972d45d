"""Drop-in `UNetModel` (reference: openai_model/model.py:259-595) running on libsdb200.so.

Same class names, constructor kwargs, state-dict keys and `forward(x, timesteps, context)` signature
as the reference, so `instantiate_from_config` with `target: sdb200.openai_model.UNetModel` and
`load_state_dict` of a reference checkpoint work unchanged.  The torch.nn layer objects below are
parameter HOLDERS only (they give the reference's key names / shapes); their `forward` is never
called — all arithmetic goes through hand-written sm_100a kernels (ops.py), channels-last.

Scope: SURVEY.md §8a — the SpatialTransformer variant used by Stable Diffusion v1 (`use_spatial_transformer=True`) is the
hot path — plus the 'next' row f4: the AttentionBlock variants (QKVAttentionLegacy / FlashAttention orders),
`use_scale_shift_norm`, `resblock_updown` and class conditioning (`num_classes`), built from the same kernels.
Still unsupported constructor options (dims != 2, conv_resample=False, n_embed) raise NotImplementedError instead of
silently computing something else.
"""
import math
import os
import weakref

import torch
from torch import nn

from . import _lib, engine, ops
from .engine import PackedConv, PackedLinear, head_pad


class GroupNorm32(nn.GroupNorm):
    """Holder for GroupNorm32 (openai_model/utils.py:15-22)."""


def normalization(channels):
    return GroupNorm32(32, channels)


def Normalize(in_channels):   # openai_model/attention.py:10-11
    return nn.GroupNorm(num_groups=32, num_channels=in_channels, eps=1e-6, affine=True)


def zero_module(module):
    for p in module.parameters():
        p.detach().zero_()
    return module


class TimestepBlock(nn.Module):
    pass


class TimestepEmbedSequential(nn.Sequential, TimestepBlock):
    """openai_model/model.py:37-67 (dispatch happens in UNetModel._run_block)."""


class Downsample(nn.Module):
    """openai_model/model.py:71-97: conv3x3 stride 2 pad 1."""

    def __init__(self, channels, use_conv, dims=2, out_channels=None, padding=1):
        super().__init__()
        if dims != 2 or not use_conv:
            raise NotImplementedError("sdb200 Downsample supports dims=2, use_conv=True")
        self.channels = channels
        self.out_channels = out_channels or channels
        self.op = nn.Conv2d(self.channels, self.out_channels, 3, stride=2, padding=padding)


class Upsample(nn.Module):
    """openai_model/model.py:100-131: nearest x2 then conv3x3."""

    def __init__(self, channels, use_conv, dims=2, out_channels=None, padding=1):
        super().__init__()
        if dims != 2 or not use_conv:
            raise NotImplementedError("sdb200 Upsample supports dims=2, use_conv=True")
        self.channels = channels
        self.out_channels = out_channels or channels
        self.conv = nn.Conv2d(self.channels, self.out_channels, 3, padding=padding)


class ResBlock(TimestepBlock):
    """openai_model/model.py:139-252."""

    def __init__(self, channels, emb_channels, dropout, out_channels=None, use_conv=False,
                 use_scale_shift_norm=False, dims=2, use_checkpoint=False, up=False, down=False):
        super().__init__()
        if dims != 2:
            raise NotImplementedError("sdb200 ResBlock supports dims=2")
        self.channels = channels
        self.emb_channels = emb_channels
        self.out_channels = out_channels or channels
        self.use_scale_shift_norm = use_scale_shift_norm
        # h_upd / x_upd (model.py:184-191) are parameter-free: nearest x2 or avg_pool2d(2)
        self.updown = "up" if up else ("down" if down else None)
        self.h_upd = self.x_upd = nn.Identity()
        self.in_layers = nn.Sequential(normalization(channels), nn.SiLU(), nn.Conv2d(channels, self.out_channels, 3, padding=1))
        self.emb_layers = nn.Sequential(nn.SiLU(), nn.Linear(emb_channels, 2 * self.out_channels if use_scale_shift_norm else self.out_channels))
        self.out_layers = nn.Sequential(normalization(self.out_channels), nn.SiLU(), nn.Dropout(p=dropout),
                                        zero_module(nn.Conv2d(self.out_channels, self.out_channels, 3, padding=1)))
        if self.out_channels == channels:
            self.skip_connection = nn.Identity()
        elif use_conv:
            self.skip_connection = nn.Conv2d(channels, self.out_channels, 3, padding=1)
        else:
            self.skip_connection = nn.Conv2d(channels, self.out_channels, 1)


class QKVAttentionLegacy(nn.Module):
    """openai_model/attention.py:485-523 (parameter-free): softmax_scale = ch ** -0.25 as the reference passes it."""

    def __init__(self, n_heads):
        super().__init__()
        self.n_heads = n_heads


class FlashAttention(nn.Module):
    """openai_model/attention.py:366-399 (parameter-free): softmax_scale = ch ** -0.5; the result is permuted to
    [N,H,T,ch] before being reshaped to [N,T,H*ch] (kept as executed)."""

    def __init__(self, n_heads):
        super().__init__()
        self.n_heads = n_heads


class AttentionBlock(nn.Module):
    """openai_model/attention.py:538-599: GroupNorm32 -> qkv conv1d -> attention -> proj_out conv1d -> + x."""

    def __init__(self, channels, num_heads=1, num_head_channels=-1, use_checkpoint=False, use_new_attention_order=False):
        super().__init__()
        self.channels = channels
        if num_head_channels == -1:
            self.num_heads = num_heads
        else:
            assert channels % num_head_channels == 0, \
                f"q, k, v channels {channels} is not divisible by num_head_channels {num_head_channels}"
            self.num_heads = channels // num_head_channels
        self.use_new_attention_order = use_new_attention_order
        self.norm = normalization(channels)
        self.qkv = nn.Conv1d(channels, channels * 3, 1)
        self.attention = FlashAttention(self.num_heads) if use_new_attention_order else QKVAttentionLegacy(self.num_heads)
        self.proj_out = zero_module(nn.Conv1d(channels, channels, 1))


class CrossAttention(nn.Module):
    """openai_model/attention.py:24-117."""

    def __init__(self, query_dim, context_dim=None, heads=8, dim_head=64, dropout=0.):
        super().__init__()
        inner_dim = dim_head * heads
        context_dim = query_dim if context_dim is None else context_dim
        self.scale = dim_head ** -0.5
        self.heads = heads
        self.dim_head = dim_head
        self.to_q = nn.Linear(query_dim, inner_dim, bias=False)
        self.to_k = nn.Linear(context_dim, inner_dim, bias=False)
        self.to_v = nn.Linear(context_dim, inner_dim, bias=False)
        self.to_out = nn.Sequential(nn.Linear(inner_dim, query_dim), nn.Dropout(dropout))


class GELU(nn.Module):
    """The reference's GEGLU, class named `GELU` (openai_model/attention.py:129-141)."""

    def __init__(self, dim_in, dim_out):
        super().__init__()
        self.proj = nn.Linear(dim_in, dim_out * 2)


class FeedForward(nn.Module):
    """openai_model/attention.py:146-172 (glu=True is what BasicTransformerBlock uses)."""

    def __init__(self, dim, dim_out=None, mult=4, glu=False, dropout=0.):
        super().__init__()
        if not glu:
            raise NotImplementedError("sdb200 FeedForward: only the gated (GEGLU) variant is on the hot path")
        inner_dim = int(dim * mult)
        dim_out = dim if dim_out is None else dim_out
        self.net = nn.Sequential(GELU(dim, inner_dim), nn.Dropout(dropout), nn.Linear(inner_dim, dim_out))


class BasicTransformerBlock(nn.Module):
    """openai_model/attention.py:187-257."""

    def __init__(self, dim, n_heads, d_head, dropout=0., context_dim=None, gated_ff=True, checkpoint=True):
        super().__init__()
        self.attn1 = CrossAttention(query_dim=dim, heads=n_heads, dim_head=d_head, dropout=dropout)
        self.ff = FeedForward(dim=dim, dropout=dropout, glu=gated_ff)
        self.attn2 = CrossAttention(query_dim=dim, context_dim=context_dim, heads=n_heads, dim_head=d_head, dropout=dropout)
        self.norm1 = nn.LayerNorm(dim)
        self.norm2 = nn.LayerNorm(dim)
        self.norm3 = nn.LayerNorm(dim)


class SpatialTransformer(nn.Module):
    """openai_model/attention.py:303-363."""

    def __init__(self, in_channels, n_heads, d_head, depth=1, dropout=0., context_dim=None):
        super().__init__()
        self.in_channels = in_channels
        self.n_heads, self.d_head = n_heads, d_head
        inner_dim = n_heads * d_head
        self.norm = Normalize(in_channels)
        self.proj_in = nn.Conv2d(in_channels, inner_dim, kernel_size=1, stride=1, padding=0)
        self.transformer_blocks = nn.ModuleList(
            [BasicTransformerBlock(inner_dim, n_heads, d_head, dropout=dropout, context_dim=context_dim) for _ in range(depth)])
        self.proj_out = zero_module(nn.Conv2d(inner_dim, in_channels, kernel_size=1, stride=1, padding=0))


class _SideResult:
    """A tensor produced on a side stream; get() makes the consuming stream wait for it (once) and hands it out."""

    def __init__(self, tensor, side, main):
        self.tensor, self.side, self.main = tensor, side, main

    def get(self):
        if self.side is not None:
            self.main.wait_stream(self.side)
            _lib.stream_fence()                           # the consumer's launch must honour the join
            if not torch.cuda.is_current_stream_capturing():
                self.tensor.record_stream(self.main)      # allocated on the side stream's pool, read on the main stream
            self.side = None
        return self.tensor


class UNetModel(nn.Module):
    """The full UNet with attention and timestep embedding (openai_model/model.py:259-595).

    Extra keyword (not in the reference): `compute_mode` = "bf16" (tcgen05 tensor cores, default) or
    "fp32" (SIMT, the <= 1e-5 parity mode); also settable later via `.compute_mode`.
    """

    def __init__(self, image_size, in_channels, model_channels, out_channels, num_res_blocks, attention_resolutions,
                 dropout=0, channel_mult=(1, 2, 4, 8), conv_resample=True, dims=2, num_classes=None,
                 use_checkpoint=False, use_fp16=False, num_heads=-1, num_head_channels=-1, num_heads_upsample=-1,
                 use_scale_shift_norm=False, resblock_updown=False, use_new_attention_order=False,
                 use_spatial_transformer=False, transformer_depth=1, context_dim=None, n_embed=None, legacy=True,
                 compute_mode=None):
        super().__init__()
        if use_spatial_transformer:
            assert context_dim is not None, 'Fool!! You forgot to include the dimension of your cross-attention conditioning...'
        if context_dim is not None:
            assert use_spatial_transformer, 'Fool!! You forgot to use the spatial transformer for your cross-attention conditioning...'
            if not isinstance(context_dim, int):
                context_dim = list(context_dim)
        if num_heads_upsample == -1:
            num_heads_upsample = num_heads
        if num_heads == -1:
            assert num_head_channels != -1, 'Either num_heads or num_head_channels has to be set'
        if num_head_channels == -1:
            assert num_heads != -1, 'Either num_heads or num_head_channels has to be set'
        if n_embed is not None or dims != 2 or not conv_resample:
            raise NotImplementedError("sdb200 UNetModel: codebook heads (n_embed), dims != 2 and conv_resample=False are not built")

        self.image_size = image_size
        self.in_channels = in_channels
        self.model_channels = model_channels
        self.out_channels = out_channels
        self.num_res_blocks = num_res_blocks
        self.attention_resolutions = attention_resolutions
        self.dropout = dropout
        self.channel_mult = channel_mult
        self.conv_resample = conv_resample
        self.num_classes = num_classes
        self.use_checkpoint = use_checkpoint
        self.dtype = torch.float16 if use_fp16 else torch.float32
        self.num_heads = num_heads
        self.num_head_channels = num_head_channels
        self.num_heads_upsample = num_heads_upsample
        self.predict_codebook_ids = False
        self.compute_mode = compute_mode or engine.default_mode()
        self.t_emb_fp16_round = True     # `t_emb.half()`, openai_model/model.py:566
        self.conv_in_tensor_cores = os.environ.get("SDB200_CONV_IN_TC", "1") != "0"   # bf16 mode: first conv on tcgen05 with a split (hi | lo) latent
        self.use_cuda_graph = False
        self.emb_side_stream = os.environ.get("SDB200_EMB_SIDE_STREAM", "1") != "0"   # time-embedding chain beside conv_in
        self.skip_side_stream = os.environ.get("SDB200_SKIP_SIDE_STREAM", "1") != "0"  # ResBlock 1x1 skip conv beside conv1
        self.dense_heads = os.environ.get("SDB200_DENSE_HEADS", "1") != "0"     # q/k/v layout, see _tblock (0 = zero-padded heads)

        time_embed_dim = model_channels * 4
        self.time_embed = nn.Sequential(nn.Linear(model_channels, time_embed_dim), nn.SiLU(), nn.Linear(time_embed_dim, time_embed_dim))
        if self.num_classes is not None:
            self.label_emb = nn.Embedding(num_classes, time_embed_dim)

        cur_heads = [num_heads]     # the reference reassigns `num_heads` inside its loops (model.py:388-395)

        def attn_for(ch, heads_arg=None):
            if num_head_channels == -1:
                dim_head = ch // cur_heads[0]
            else:
                cur_heads[0] = ch // num_head_channels
                dim_head = num_head_channels
            if legacy:
                dim_head = ch // cur_heads[0] if use_spatial_transformer else num_head_channels
            if use_spatial_transformer:
                return SpatialTransformer(ch, cur_heads[0], dim_head, depth=transformer_depth, context_dim=context_dim)
            return AttentionBlock(ch, num_heads=cur_heads[0] if heads_arg is None else heads_arg, num_head_channels=dim_head,
                                  use_new_attention_order=use_new_attention_order)

        def res(cin, cout=None, **kw):
            return ResBlock(cin, time_embed_dim, dropout, out_channels=cout, use_scale_shift_norm=use_scale_shift_norm, **kw)

        self.input_blocks = nn.ModuleList([TimestepEmbedSequential(nn.Conv2d(in_channels, model_channels, 3, padding=1))])
        input_block_chans = [model_channels]
        ch = model_channels
        ds = 1
        for level, mult in enumerate(channel_mult):
            for _ in range(num_res_blocks):
                layers = [res(ch, mult * model_channels)]
                ch = mult * model_channels
                if ds in attention_resolutions:
                    layers.append(attn_for(ch))
                self.input_blocks.append(TimestepEmbedSequential(*layers))
                input_block_chans.append(ch)
            if level != len(channel_mult) - 1:
                self.input_blocks.append(TimestepEmbedSequential(
                    res(ch, ch, down=True) if resblock_updown else Downsample(ch, conv_resample, out_channels=ch)))
                input_block_chans.append(ch)
                ds *= 2
        self.middle_block = TimestepEmbedSequential(res(ch), attn_for(ch), res(ch))
        self.output_blocks = nn.ModuleList([])
        for level, mult in list(enumerate(channel_mult))[::-1]:
            for i in range(num_res_blocks + 1):
                ich = input_block_chans.pop()
                layers = [res(ch + ich, model_channels * mult)]
                ch = model_channels * mult
                if ds in attention_resolutions:
                    layers.append(attn_for(ch, num_heads_upsample))
                if level and i == num_res_blocks:
                    layers.append(res(ch, ch, up=True) if resblock_updown else Upsample(ch, conv_resample, out_channels=ch))
                    ds //= 2
                self.output_blocks.append(TimestepEmbedSequential(*layers))
        self.out = nn.Sequential(normalization(ch), nn.SiLU(), zero_module(nn.Conv2d(model_channels, out_channels, 3, padding=1)))

        self._packed = {}        # mode -> packed weights
        self._ctx_cache = {}     # (mode, block, id(context)) -> (weakref(context), version, projected K/V)
        # a parent's load_state_dict (e.g. LatentDiffusion's) never calls the override below: drop the packed copies from a hook
        self.register_load_state_dict_post_hook(lambda module, incompatible_keys: module._invalidate())
        self._kv_pinned = None   # graph mode: {id(block): projected K/V of the static context buffer}
        self._graphs = {}
        self._padbufs = {}       # (rows, width, d, dp) -> zero-initialised padded-head projection buffer

    # ---- weight packing ---------------------------------------------------------------------------
    def _invalidate(self):
        self._packed = {}
        self._ctx_cache = {}
        self._graphs = {}
        self._padbufs = {}
        self.__dict__.pop("_param_list", None)
        self.__dict__.pop("_fp_seen", None)

    def _padbuf(self, rows, width, d, dp, dev):
        """Persistent [rows, width] bf16 buffer for q/k/v heads stored padded from d to dp channels.  The GEMM
        epilogue only ever writes the d real channels of each head, so the pad channels stay zero after the one
        initial fill; every layer with the same geometry shares the buffer (use is stream-ordered)."""
        key = (rows, width, d, dp, str(dev))
        buf = self._padbufs.get(key)
        if buf is None:
            buf = torch.zeros((rows, width), dtype=torch.bfloat16, device=dev)
            self._padbufs[key] = buf
        return buf

    def load_state_dict(self, *a, **k):
        r = super().load_state_dict(*a, **k)
        self._invalidate()
        return r

    def _apply(self, fn, *a, **k):
        r = super()._apply(fn, *a, **k)
        self._invalidate()
        return r

    def _weights_fingerprint(self):
        """Changes whenever a parameter is replaced or written in place (EMA `copy_to`, optimizer step, a parent module's
        load_state_dict — which recurses through `_load_from_state_dict` and never reaches the override above)."""
        ps = self.__dict__.get("_param_list")
        if ps is None:
            ps = self.__dict__["_param_list"] = list(self.parameters())
        return (ps[0].data_ptr(), ps[0].device, sum(p._version for p in ps))

    def _check_weights(self):
        fp = self._weights_fingerprint()
        if fp != self.__dict__.get("_fp_seen"):
            if self.__dict__.get("_fp_seen") is not None:
                self._invalidate()
            self.__dict__["_fp_seen"] = fp

    def _res_blocks(self):
        for m in self.modules():
            if isinstance(m, ResBlock):
                yield m

    def _pack(self, mode):
        if mode in self._packed:
            return self._packed[mode]
        if mode not in engine.MODES:
            raise ValueError("compute_mode must be one of %s" % (engine.MODES,))
        P = {}
        dev = self.time_embed[0].weight.device
        half = self.model_channels // 2
        # frequencies exactly as timestep_embedding builds them (openai_model/utils.py:235-238), on the host
        P["freqs"] = torch.exp(-math.log(10000) * torch.arange(start=0, end=half, dtype=torch.float32) / half).to(dev)
        P["te0"] = (self.time_embed[0].weight.detach().float().contiguous(), self.time_embed[0].bias.detach().float().contiguous())
        P["te2"] = (self.time_embed[2].weight.detach().float().contiguous(), self.time_embed[2].bias.detach().float().contiguous())
        if self.num_classes is not None:
            P["label_emb"] = self.label_emb.weight.detach().float().contiguous()
        # all ResBlock emb_layers as ONE skinny GEMM [sum(Cout), emb]; its 20160 x 1280 matrix is stored in bf16 in the bf16 mode
        # (like every other weight there): streaming it is the whole cost of the launch (103 MB in fp32)
        ws, bs, off = [], [], 0
        for rb in self._res_blocks():
            lin = rb.emb_layers[1]
            ws.append(lin.weight.detach().float())
            bs.append(lin.bias.detach().float())
            P[("emb_off", id(rb))] = (off, lin.out_features)
            off += lin.out_features
        P["emb_w"] = torch.cat(ws, 0).contiguous()
        if mode == "bf16" and P["emb_w"].shape[1] % 8 == 0:
            P["emb_w"] = P["emb_w"].to(torch.bfloat16)
        P["emb_b"] = torch.cat(bs, 0).contiguous()
        for m in self.modules():
            if isinstance(m, ResBlock):
                P[("c1", id(m))] = PackedConv(m.in_layers[2].weight, m.in_layers[2].bias, mode)
                P[("c2", id(m))] = PackedConv(m.out_layers[3].weight, m.out_layers[3].bias, mode)
                if isinstance(m.skip_connection, nn.Conv2d):
                    P[("skip", id(m))] = PackedConv(m.skip_connection.weight, m.skip_connection.bias, mode)
            elif isinstance(m, Downsample):
                P[("op", id(m))] = PackedConv(m.op.weight, m.op.bias, mode, stride=2, pad=1)
            elif isinstance(m, Upsample):
                P[("conv", id(m))] = PackedConv(m.conv.weight, m.conv.bias, mode, up2=True)
            elif isinstance(m, AttentionBlock):
                Cc = m.channels
                P[("qkv", id(m))] = PackedLinear(m.qkv.weight.reshape(3 * Cc, Cc), m.qkv.bias, mode)
                P[("aout", id(m))] = PackedLinear(m.proj_out.weight.reshape(Cc, Cc), m.proj_out.bias, mode)
            elif isinstance(m, SpatialTransformer):
                P[("pin", id(m))] = PackedConv(m.proj_in.weight, m.proj_in.bias, mode)
                P[("pout", id(m))] = PackedConv(m.proj_out.weight, m.proj_out.bias, mode)
            elif isinstance(m, BasicTransformerBlock):
                a1, a2 = m.attn1, m.attn2
                P[("qkv1", id(m))] = PackedLinear(torch.cat([a1.to_q.weight, a1.to_k.weight, a1.to_v.weight], 0), None, mode)
                P[("o1", id(m))] = PackedLinear(a1.to_out[0].weight, a1.to_out[0].bias, mode)
                P[("q2", id(m))] = PackedLinear(a2.to_q.weight, None, mode)
                P[("kv2", id(m))] = PackedLinear(torch.cat([a2.to_k.weight, a2.to_v.weight], 0), None, mode)
                P[("o2", id(m))] = PackedLinear(a2.to_out[0].weight, a2.to_out[0].bias, mode)
                P[("ff1", id(m))] = PackedLinear(m.ff.net[0].proj.weight, m.ff.net[0].proj.bias, mode, geglu=True)
                P[("ff2", id(m))] = PackedLinear(m.ff.net[2].weight, m.ff.net[2].bias, mode)
        cin_w = self.input_blocks[0][0].weight
        P["conv_in_split"] = False
        if mode == "bf16" and 2 * cin_w.shape[1] <= 32 and self.conv_in_tensor_cores:
            # conv_in on the tensor cores (the SIMT kernel needs 109 us for this 0.75 GFLOP layer at batch 8; tcgen05 ~15 us and
            # its epilogue hands the following GroupNorm its statistics).  The latent's C channels become a 32-channel operand
            # (a whole 64-byte TMA row): bf16(x) | bf16(x - bf16(x)) | zeros, with the weights repeated for the residual half, so
            # x_t itself is NOT rounded to bf16 — rounding it moved eps rel-L2 from 7.05e-3 to 7.64e-3 when this was first tried.
            c_in = cin_w.shape[1]
            w = cin_w.detach()
            cin_w = torch.cat([w, w, w.new_zeros(w.shape[0], 32 - 2 * c_in, w.shape[2], w.shape[3])], 1)
            P["conv_in_split"] = True
        P["conv_in"] = PackedConv(cin_w, self.input_blocks[0][0].bias, mode)
        P["conv_out"] = PackedConv(self.out[2].weight, self.out[2].bias, mode)
        self._packed[mode] = P
        return P

    # ---- building blocks (all tensors NHWC / [rows, C]) ---------------------------------------------
    @staticmethod
    def _gn(norm, x, mode, act, x1=None, out_dtype=None, want_raw=False):
        dt = out_dtype if out_dtype is not None else engine.op_dtype(mode)
        return ops.groupnorm(x, norm.weight, norm.bias, norm.eps, act=act, out_dtype=dt, x1=x1,
                             groups=norm.num_groups, exact=(mode == "fp32"), want_raw=want_raw)

    def _res(self, rb, P, mode, x, x1, emb_all):
        """ResBlock._forward (openai_model/model.py:232-252); x1 = skip tensor to be channel-concatenated."""
        c1, c2 = P[("c1", id(rb))], P[("c2", id(rb))]
        off, n = P[("emb_off", id(rb))]
        sk = P.get(("skip", id(rb)))
        ss = rb.use_scale_shift_norm
        raw = None
        if rb.updown is not None:
            # 'next' row f4 (resblock_updown): h_upd / x_upd between GroupNorm+SiLU and the conv (model.py:233-238)
            assert x1 is None
            h = self._gn(rb.in_layers[0], x, mode, 1, out_dtype=torch.float32)
            if rb.updown == "up":
                h = ops.cast_concat(h, None, up=2, out_dtype=c1.in_dtype)
                x = ops.cast_concat(x, None, up=2, out_dtype=torch.float32)
            else:
                h = ops.avgpool2x2(h, out_dtype=c1.in_dtype)
                x = ops.avgpool2x2(x)
        elif sk is not None and sk.in_dtype == torch.bfloat16:
            # the 1x1 skip conv's bf16 operand (the raw concat) comes out of the same pass as the normalised one
            h, raw = self._gn(rb.in_layers[0], x, mode, 1, x1=x1, out_dtype=c1.in_dtype, want_raw=True)
        else:
            h = self._gn(rb.in_layers[0], x, mode, 1, x1=x1, out_dtype=c1.in_dtype)
        rowvec = self._emb_rows(emb_all)[:, off:off + n]      # first use of the time embedding: joins its side stream (once)
        xs_side = None
        if sk is not None and self.skip_side_stream and mode == "bf16":
            # skip_connection(x) (a 1x1 conv, memory- / latency-bound) depends only on the block input: it runs on a side stream
            # beside conv1 + GroupNorm of the main branch and fills the SMs their last waves leave idle; joined before conv2
            main = torch.cuda.current_stream()
            side = self.__dict__.get("_side_stream2")
            if side is None or side.device != main.device:
                side = self.__dict__["_side_stream2"] = torch.cuda.Stream(device=main.device)
            side.wait_stream(main)
            with torch.cuda.stream(side):
                _lib.stream_fence()
                xs_side = _SideResult(self._skip_conv(sk, raw, x, x1), side, main)
        if ss:
            # out_norm(h) * (1 + scale) + shift (model.py:244-248): scale / shift folded into per-sample GroupNorm rows
            h = engine.conv(h, c1, want_stats=True)
            norm = rb.out_layers[0]
            g2, b2 = ops.scale_shift_affine(norm.weight, norm.bias, rowvec)
            h = ops.groupnorm(h, g2, b2, norm.eps, act=1, out_dtype=c2.in_dtype, groups=norm.num_groups, exact=(mode == "fp32"))
        else:
            h = engine.conv(h, c1, rowvec=rowvec, want_stats=True)      # conv + bias + emb_out[..., None, None]
            h = self._gn(rb.out_layers[0], h, mode, 1, out_dtype=c2.in_dtype)
        if sk is not None:
            xs = self._emb_rows(xs_side) if xs_side is not None else self._skip_conv(sk, raw, x, x1)
        else:
            assert x1 is None
            xs = x
        return engine.conv(h, c2, residual=xs, want_stats=True)     # conv + bias + skip_connection(x)

    @staticmethod
    def _skip_conv(sk, raw, x, x1):
        xs = raw if raw is not None else ops.cast_concat(x, x1, up=1, out_dtype=sk.in_dtype)
        return engine.conv(xs, sk)

    @staticmethod
    def _emb_rows(emb_all):
        return emb_all.get() if isinstance(emb_all, _SideResult) else emb_all

    def _attnblock(self, ab, P, mode, x):
        """AttentionBlock._forward (openai_model/attention.py:588-599), 'next' row f4.  The qkv conv's output channels are
        (q | k | v) x heads x ch in both attention orders (attention.py:381,509); the tcgen05 kernel writes its result
        straight into the layout the reference's reshape produces (head-major for FlashAttention's permute, :393-397)."""
        B, Hh, Ww, Cc = x.shape
        T = Hh * Ww
        H = ab.num_heads
        d = Cc // H
        new_order = ab.use_new_attention_order
        scale = d ** -0.5 if new_order else 1.0 / math.sqrt(math.sqrt(d))
        odt = engine.op_dtype(mode)
        xn = self._gn(ab.norm, x, mode, 0, out_dtype=odt).reshape(B * T, Cc)
        o_strides = (H * T * d, d, T * d) if new_order else (T * Cc, Cc, d)
        if mode == "bf16":
            dp = head_pad(d)
            qkv = engine.linear(xn, P[("qkv", id(ab))], out_dtype=odt, rows_per_item=T)                       # dense [B*T, 3C]
            W3 = 3 * Cc
            o = ops.attention_tc(qkv, qkv[:, Cc:], qkv[:, 2 * Cc:], B, H, T, T, d, dp, scale,
                                 (T * W3, W3, d), (T * W3, W3, d), (T * W3, W3, d), o_strides=o_strides, dense=True)
        else:
            qkv = engine.linear(xn, P[("qkv", id(ab))], rows_per_item=T)                                       # [B*T, 3C]
            o = self._attn_fp32(qkv, 3 * Cc, 0, qkv, 3 * Cc, Cc, qkv, 3 * Cc, 2 * Cc, B, H, T, T, d, scale, o_strides=o_strides)
        out = engine.linear(o.reshape(B * T, Cc), P[("aout", id(ab))], residual=x.reshape(B * T, Cc), rows_per_item=T)
        return out.reshape(B, Hh, Ww, Cc)

    def _ctx_lookup(self, key, src):
        """Cache entries are valid only for the SAME live tensor object, unmodified since: a data_ptr()/shape key alone
        collides when the allocator hands a freed conditioning's address to the next prompt's."""
        hit = self._ctx_cache.get(key)
        if hit is not None and hit[0]() is src and hit[1] == src._version:
            return hit[2]
        return None

    def _ctx_store(self, key, src, val):
        if len(self._ctx_cache) > 256:
            self._ctx_cache = {k: v for k, v in self._ctx_cache.items() if v[0]() is not None}
            if len(self._ctx_cache) > 256:
                self._ctx_cache.clear()
        self._ctx_cache[key] = (weakref.ref(src), src._version, val)

    def _kv_context(self, blk, P, mode, context, src=None):
        """to_k / to_v of the (step-invariant) context, cached per LIVE context tensor (`src` = the caller's own tensor
        object when `context` is a converted temporary of it)."""
        pinned = self._kv_pinned
        if pinned is not None:                       # CUDA-graph mode: projections live in their own graph (see _graph_forward)
            return pinned[id(blk)]
        src = context if src is None else src
        key = (mode, id(blk), id(src))
        hit = self._ctx_lookup(key, src)
        if hit is not None:
            return hit
        a2 = blk.attn2
        H, d = a2.heads, a2.dim_head
        B, Sk, Cc = context.shape
        if mode == "bf16":
            cb = self._ctx_lookup(("ctx_bf16", id(src)), src)
            if cb is None:
                cb = ops.cast_concat(context.reshape(1, 1, B * Sk, Cc).contiguous(), None, out_dtype=torch.bfloat16).reshape(B * Sk, Cc)
                self._ctx_store(("ctx_bf16", id(src)), src, cb)
            if self.dense_heads:
                kv = engine.linear(cb, P[("kv2", id(blk))], out_dtype=torch.bfloat16, rows_per_item=Sk)                                   # [B*Sk, 2*H*d]
            else:
                dp = head_pad(d)
                kv = engine.linear(cb, P[("kv2", id(blk))], out_dtype=torch.bfloat16, col_group=d, col_group_stride=dp, rows_per_item=Sk)   # [B*Sk, 2*H*dp]
        else:
            kv = engine.linear(context.reshape(B * Sk, Cc), P[("kv2", id(blk))], rows_per_item=Sk)                                      # [B*Sk, 2*H*d]
        self._ctx_store(key, src, kv)
        return kv

    def _tblock(self, blk, P, mode, t, B, S, context, final_dtype=torch.float32):
        """BasicTransformerBlock._forward (openai_model/attention.py:233-257) on tokens t [B*S, C] fp32."""
        a1, a2 = blk.attn1, blk.attn2
        H, d = a1.heads, a1.dim_head
        Cc = H * d
        odt = engine.op_dtype(mode)
        Sk = context.shape[1]
        kv = self._kv_context(blk, P, mode, context, src=self.__dict__.get("_ctx_src"))
        if mode == "bf16" and self.dense_heads:
            # q / k / v are the plain projection outputs ([rows, H*d], heads side by side); the attention kernel's tensor maps
            # are d channels wide and TMA zero-fills the pad channels of each 64-channel tile.  Against the zero-padded layout
            # (below, kept for A/B measurements) the projections write whole lines instead of 80 of every 128 bytes.
            dp = head_pad(d)
            W3 = 3 * Cc
            a = ops.layernorm(t, blk.norm1.weight, blk.norm1.bias, blk.norm1.eps, out_dtype=odt)
            qkv = engine.linear(a, P[("qkv1", id(blk))], out_dtype=odt, rows_per_item=S)                      # [B*S, 3C]
            o = ops.attention_tc(qkv, qkv[:, Cc:], qkv[:, 2 * Cc:], B, H, S, S, d, dp, a1.scale,
                                 (S * W3, W3, d), (S * W3, W3, d), (S * W3, W3, d), dense=True)
            t = engine.linear(o.reshape(B * S, Cc), P[("o1", id(blk))], residual=t, rows_per_item=S)
            a = ops.layernorm(t, blk.norm2.weight, blk.norm2.bias, blk.norm2.eps, out_dtype=odt)
            q = engine.linear(a, P[("q2", id(blk))], out_dtype=odt, rows_per_item=S)                          # [B*S, C]
            W2 = 2 * Cc
            o = ops.attention_tc(q, kv, kv[:, Cc:], B, H, S, Sk, d, dp, a2.scale,
                                 (S * Cc, Cc, d), (Sk * W2, W2, d), (Sk * W2, W2, d), dense=True)
            t = engine.linear(o.reshape(B * S, Cc), P[("o2", id(blk))], residual=t, rows_per_item=S)
        elif mode == "bf16":
            dp = head_pad(d)
            W3 = 3 * H * dp
            a = ops.layernorm(t, blk.norm1.weight, blk.norm1.bias, blk.norm1.eps, out_dtype=odt)
            qkv = engine.linear(a, P[("qkv1", id(blk))], out_dtype=odt, col_group=d, col_group_stride=dp, rows_per_item=S,
                                out=self._padbuf(B * S, W3, d, dp, t.device))                                  # [B*S, 3*H*dp]
            o = ops.attention_tc(qkv, qkv[:, H * dp:], qkv[:, 2 * H * dp:], B, H, S, S, d, dp, a1.scale,
                                 (S * W3, W3, dp), (S * W3, W3, dp), (S * W3, W3, dp))
            t = engine.linear(o.reshape(B * S, Cc), P[("o1", id(blk))], residual=t, rows_per_item=S)
            a = ops.layernorm(t, blk.norm2.weight, blk.norm2.bias, blk.norm2.eps, out_dtype=odt)
            q = engine.linear(a, P[("q2", id(blk))], out_dtype=odt, col_group=d, col_group_stride=dp, rows_per_item=S,
                              out=self._padbuf(B * S, H * dp, d, dp, t.device))                                # [B*S, H*dp]
            W2 = 2 * H * dp
            o = ops.attention_tc(q, kv, kv[:, H * dp:], B, H, S, Sk, d, dp, a2.scale,
                                 (S * H * dp, H * dp, dp), (Sk * W2, W2, dp), (Sk * W2, W2, dp))
            t = engine.linear(o.reshape(B * S, Cc), P[("o2", id(blk))], residual=t, rows_per_item=S)
        else:
            a = ops.layernorm(t, blk.norm1.weight, blk.norm1.bias, blk.norm1.eps, out_dtype=odt)
            qkv = engine.linear(a, P[("qkv1", id(blk))], rows_per_item=S)                                                     # [B*S, 3C]
            o = self._attn_fp32(qkv, 3 * Cc, 0, qkv, 3 * Cc, Cc, qkv, 3 * Cc, 2 * Cc, B, H, S, S, d, a1.scale)
            t = engine.linear(o, P[("o1", id(blk))], residual=t, rows_per_item=S)
            a = ops.layernorm(t, blk.norm2.weight, blk.norm2.bias, blk.norm2.eps, out_dtype=odt)
            q = engine.linear(a, P[("q2", id(blk))], rows_per_item=S)
            o = self._attn_fp32(q, Cc, 0, kv, 2 * Cc, 0, kv, 2 * Cc, Cc, B, H, S, Sk, d, a2.scale)
            t = engine.linear(o, P[("o2", id(blk))], residual=t, rows_per_item=S)
        a = ops.layernorm(t, blk.norm3.weight, blk.norm3.bias, blk.norm3.eps, out_dtype=odt)
        g = engine.linear(a, P[("ff1", id(blk))], out_dtype=odt, rows_per_item=S)          # GEGLU fused (bf16) or gemm + geglu kernel (fp32)
        # `final_dtype` bf16: the block's result only feeds proj_out's tensor-core operand, so it is rounded here
        t = engine.linear(g, P[("ff2", id(blk))], residual=t, rows_per_item=S, out_dtype=final_dtype)
        return t

    @staticmethod
    def _attn_fp32(q, ldq, qoff, k, ldk, koff, v, ldv, voff, B, H, Sq, Sk, d, scale, o_strides=None):
        """softmax(q k^T * scale) v per (batch, head) with strided fp32 SIMT GEMMs; returns [B*Sq, H*d]
        (o_strides = (batch, seq, head) element strides of another output layout)."""
        Cc = H * d
        dev = q.device
        scores = torch.empty((B, H, Sq, Sk), dtype=torch.float32, device=dev)
        qv = q.reshape(-1)[qoff:]
        kv_ = k.reshape(-1)[koff:]
        vv = v.reshape(-1)[voff:]
        ops.gemm_simt(qv, kv_, out=scores, M=Sq, N=Sk, K=d, lda=ldq, ldb=ldk, ldc=Sk, batch=(B, H),
                      sa=(Sq * ldq, d), sb=(Sk * ldk, d), sc=(H * Sq * Sk, Sq * Sk))
        Pm = ops.softmax_rows(scores, scale)
        out = torch.empty((B * Sq, Cc), dtype=torch.float32, device=dev)
        o_bs, o_ss, o_hs = o_strides if o_strides is not None else (Sq * Cc, Cc, d)
        ops.gemm_simt(Pm, vv, out=out, b_kn=True, M=Sq, N=d, K=Sk, lda=Sk, ldb=ldv, ldc=o_ss, batch=(B, H),
                      sa=(H * Sq * Sk, Sq * Sk), sb=(Sk * ldv, d), sc=(o_bs, o_hs))
        return out

    def _st(self, st, P, mode, x, context):
        """SpatialTransformer.forward (openai_model/attention.py:336-363); NHWC makes both rearranges free."""
        B, Hh, Ww, Cc = x.shape
        pin, pout = P[("pin", id(st))], P[("pout", id(st))]
        xn = self._gn(st.norm, x, mode, 0, out_dtype=pin.in_dtype)
        t = engine.conv(xn, pin).reshape(B * Hh * Ww, -1)
        nblk = len(st.transformer_blocks)
        for i, blk in enumerate(st.transformer_blocks):
            t = self._tblock(blk, P, mode, t, B, Hh * Ww, context,
                             final_dtype=pout.in_dtype if i == nblk - 1 else torch.float32)
        inner = t.shape[-1]
        tt = t.reshape(B, Hh, Ww, inner)
        if tt.dtype != pout.in_dtype:
            tt = ops.cast_concat(tt, None, out_dtype=pout.in_dtype)
        return engine.conv(tt, pout, residual=x, want_stats=True)

    def _run_block(self, seq, P, mode, h, x1, emb_all, context):
        for layer in seq:
            if isinstance(layer, ResBlock):
                h = self._res(layer, P, mode, h, x1, emb_all)
                x1 = None
            elif isinstance(layer, SpatialTransformer):
                h = self._st(layer, P, mode, h, context)
            elif isinstance(layer, AttentionBlock):
                h = self._attnblock(layer, P, mode, h)
            elif isinstance(layer, Downsample):
                pc = P[("op", id(layer))]
                hx = ops.cast_concat(h, None, out_dtype=pc.in_dtype) if pc.in_dtype == torch.bfloat16 else h
                h = engine.conv(hx, pc, want_stats=True)
            elif isinstance(layer, Upsample):
                pc = P[("conv", id(layer))]
                if pc.use_tc:      # sub-pixel form: four 2x2 convs on the low-resolution tensor, no 4x intermediate
                    h = engine.conv_up2(ops.cast_concat(h, None, out_dtype=torch.bfloat16), pc, want_stats=True)
                else:
                    h = engine.conv(h, pc, up=2)
            elif isinstance(layer, nn.Conv2d):
                h = engine.conv(h, P["conv_in"], want_stats=True)
            else:
                raise NotImplementedError(type(layer))
        assert x1 is None
        return h

    # ---- forward ----------------------------------------------------------------------------------
    def _time_embedding(self, P, t_f32, y):
        t_emb = ops.timestep_embedding(t_f32, P["freqs"], round_fp16=self.t_emb_fp16_round)
        e = ops.skinny_linear(t_emb, P["te0"][0], P["te0"][1], act_out=1)        # Linear -> SiLU
        # time_embed[2] then every ResBlock's SiLU -> Linear (openai_model/model.py:195-201), batched
        emb = ops.skinny_linear(e, P["te2"][0], P["te2"][1])
        if y is not None:                                                        # emb + label_emb(y), model.py:567-569
            emb = ops.add(emb, ops.gather_rows(P["label_emb"], y))
        return ops.skinny_linear(emb, P["emb_w"], P["emb_b"], act_in=1)

    def _forward_nhwc(self, x_nchw, t_f32, context, mode, y=None, x1_nchw=None):
        """x1_nchw: channels appended to x's for conv_in (forward_concat); the concat happens inside the layout kernel."""
        P = self._pack(mode)
        if self.emb_side_stream:
            # The time-embedding chain (4 launches that stream the 20160 x 1280 emb_layers matrix, ~0.1 ms) depends on t only and
            # is first needed by the first ResBlock's conv epilogue: it runs on a side stream beside the layout change, conv_in
            # and the first GroupNorm (a fork / join that CUDA-graph capture records as such).
            main = torch.cuda.current_stream()
            side = self.__dict__.get("_side_stream")
            if side is None or side.device != main.device:
                side = self.__dict__["_side_stream"] = torch.cuda.Stream(device=main.device)
            side.wait_stream(main)
            with torch.cuda.stream(side):
                _lib.stream_fence()
                emb_all = _SideResult(self._time_embedding(P, t_f32, y), side, main)
        else:
            emb_all = self._time_embedding(P, t_f32, y)
        h = ops.nchw_to_nhwc(x_nchw, out_dtype=P["conv_in"].in_dtype, pad_to=P["conv_in"].cin, split=P["conv_in_split"], x1=x1_nchw)
        hs = []
        for module in self.input_blocks:
            h = self._run_block(module, P, mode, h, None, emb_all, context)
            hs.append(h)
        h = self._run_block(self.middle_block, P, mode, h, None, emb_all, context)
        for module in self.output_blocks:
            h = self._run_block(module, P, mode, h, hs.pop(), emb_all, context)     # torch.cat folded into GN / cast
        self._emb_rows(emb_all)      # (a model without ResBlocks: still join the side stream)
        co = P["conv_out"]
        h = self._gn(self.out[0], h, mode, 1, out_dtype=co.in_dtype)
        h = engine.conv(h, co)
        return ops.nhwc_to_nchw(h)

    @torch.no_grad()
    def forward(self, x, timesteps=None, context=None, y=None, **kwargs):
        """Apply the model to an input batch (openai_model/model.py:550-595).
        x [N,C,H,W], timesteps [N] (int or float), context [N,S,context_dim] -> [N,out_channels,H,W] in x.dtype."""
        return self._forward_impl(x, None, timesteps, context, y)

    @torch.no_grad()
    def forward_concat(self, x, c_concat, timesteps=None, context=None, y=None):
        """forward(torch.cat([x, *c_concat], 1), timesteps, context, y), bit for bit, without the concatenated tensor: the
        channel concat of a "concat" / "hybrid" conditioned model (ldm/diffusion/ddpm.py:1992-2034, e.g. an inpainting UNet's
        4 latent + 1 mask + 4 masked-image channels) is done by the layout kernel that feeds conv_in.
        c_concat: a tensor [N,Cc,H,W] or a list of them (a list of several is joined once, here).  Shapes must agree with x
        and the channels add up to in_channels; a mismatch raises ValueError before any kernel runs."""
        if torch.is_tensor(c_concat):
            c_concat = [c_concat]
        if not isinstance(c_concat, (list, tuple)) or len(c_concat) == 0 or not all(torch.is_tensor(c) for c in c_concat):
            raise ValueError("c_concat must be a tensor or a non-empty list of tensors")
        if x.dim() != 4 or any(c.dim() != 4 for c in c_concat):
            raise ValueError("forward_concat needs 4-D [N,C,H,W] tensors, got x %s and c_concat %s" % (
                tuple(x.shape), [tuple(c.shape) for c in c_concat]))
        for c in c_concat:
            if c.shape[0] != x.shape[0] or c.shape[2:] != x.shape[2:]:
                raise ValueError("c_concat %s does not match x %s in N, H, W" % (tuple(c.shape), tuple(x.shape)))
            if c.device != x.device:
                raise ValueError("c_concat is on %s, x on %s: all inputs must be on one device" % (c.device, x.device))
        for name, v in (("timesteps", timesteps), ("context", context), ("y", y)):
            if v is not None and v.device != x.device:
                raise ValueError("%s is on %s, x on %s: all inputs must be on one device" % (name, v.device, x.device))
        total = x.shape[1] + sum(c.shape[1] for c in c_concat)
        if total != self.in_channels:
            raise ValueError("x has %d channels and c_concat %s: %d in all, the model takes in_channels=%d" % (
                x.shape[1], [c.shape[1] for c in c_concat], total, self.in_channels))
        cc = c_concat[0] if len(c_concat) == 1 else torch.cat(list(c_concat), 1)
        return self._forward_impl(x, cc, timesteps, context, y)

    def _forward_impl(self, x, x1, timesteps, context, y):
        assert (y is not None) == (self.num_classes is not None), "must specify y if and only if the model is class-conditional"
        from ._lib import require_cuda
        with torch.cuda.device(x.device):
            require_cuda(x, x1, timesteps, context, y)
            self._check_weights()
            mode = self.compute_mode
            xin = x.float().contiguous()
            x1in = x1.float().contiguous() if x1 is not None else None
            tin = timesteps.float().contiguous()
            cin = context.float().contiguous() if context is not None else None
            if y is not None:
                assert y.shape == (x.shape[0],)
                y = y.to(torch.int64).contiguous()
            if self.use_cuda_graph and y is None and cin is not None:
                out = self._graph_forward(xin, tin, cin, mode, ctx_src=context, x1=x1in)
            else:
                # K/V projections of the conditioning are cached against the CALLER's tensor object (cin may be a temporary)
                self.__dict__["_ctx_src"] = context if cin is not context else None
                try:
                    out = self._forward_nhwc(xin, tin, cin, mode, y=y, x1_nchw=x1in)
                finally:
                    self.__dict__["_ctx_src"] = None
        return out if x.dtype == torch.float32 else out.to(x.dtype)

    # ---- CUDA graph replay of one UNet call ------------------------------------------------------------
    def _project_context(self, P, mode, context):
        """to_k / to_v of `context` for every transformer block -> {id(block): kv}."""
        self._kv_pinned = None
        self._ctx_cache.clear()
        return {id(m): self._kv_context(m, P, mode, context) for m in self.modules() if isinstance(m, BasicTransformerBlock)}

    def _graph_forward(self, x, t, ctx, mode, ctx_src=None, x1=None):
        """Two graphs per (mode, shapes): the context projections (to_k / to_v of every cross-attention; they depend on the
        context only, which a sampler passes unchanged for all its steps — ldm/diffusion/ddim.py:174 calls apply_model with
        the same `c` 50 times) are replayed only when the caller's context tensor changed; the UNet body every call.
        x1 (forward_concat): the concatenated channels, a static input copied in on every replay like x.  Its shape is part of
        the key (None for forward), so a graph captured for one entry is never replayed for the other."""
        key = (mode, tuple(x.shape), tuple(ctx.shape), None if x1 is None else tuple(x1.shape))
        g = self._graphs.get(key)
        if g is None:
            sx, st_, sc = x.clone(), t.clone(), ctx.clone()
            sx1 = x1.clone() if x1 is not None else None
            P = self._pack(mode)
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                for _ in range(2):            # warm-up: pack weights, set kernel attributes
                    self._forward_nhwc(sx, st_, sc, mode, x1_nchw=sx1)
            torch.cuda.current_stream().wait_stream(s)
            kv_graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(kv_graph):
                pinned = self._project_context(P, mode, sc)
            self._kv_pinned = pinned
            graph = torch.cuda.CUDAGraph()
            try:
                with torch.cuda.graph(graph, pool=kv_graph.pool()):
                    out = self._forward_nhwc(sx, st_, sc, mode, x1_nchw=sx1)
            finally:
                self._kv_pinned = None
                self._ctx_cache.clear()
            g = [graph, kv_graph, sx, st_, sc, out, None, pinned, sx1]      # `pinned` keeps the projections' memory alive
            self._graphs[key] = g
        graph, kv_graph, sx, st_, sc, out, seen = g[:7]
        sx.copy_(x)
        if x1 is not None:
            g[8].copy_(x1)
        st_.copy_(t)
        # same live tensor object, not modified in place since the last call => same conditioning
        src = ctx_src if ctx_src is not None else ctx
        same = seen is not None and seen[0]() is src and seen[1] == src._version
        if not same:                          # new conditioning: copy it in and re-project K / V
            sc.copy_(ctx)
            kv_graph.replay()
            g[6] = (weakref.ref(src), src._version)
        graph.replay()
        return out.clone()
