"""Drop-in DDPM `UNet` (reference: DDPM/models/unet.py:11-81, DDPM/models/layers.py:6-339) — the
32x32x3 parity configuration (BASELINE.json configs[0]) — running on libsdb200.so.

Same class / attribute names and state-dict keys as the reference; torch.nn layers hold parameters
only.  `forward(input_tensor, time)` takes `time` as int64 timesteps like the reference.
"""
import torch
from torch import nn

from . import engine, ops
from .engine import PackedConv, PackedLinear, head_pad


class TransformerPositionalEmbedding(nn.Module):
    """layers.py:6-34: interleaved sin/cos table looked up by timestep (pe_matrix is a plain attribute, not a buffer)."""

    def __init__(self, dimension, max_timesteps=1000):
        super().__init__()
        assert dimension % 2 == 0, "Embedding dimension must be even"
        self.dimension = dimension
        self.pe_matrix = torch.zeros(max_timesteps, dimension)
        even_indices = torch.arange(0, self.dimension, 2)
        log_term = torch.log(torch.tensor(10000.0)) / self.dimension
        div_term = torch.exp(even_indices * -log_term)
        timesteps = torch.arange(max_timesteps).unsqueeze(1)
        self.pe_matrix[:, 0::2] = torch.sin(timesteps * div_term)
        self.pe_matrix[:, 1::2] = torch.cos(timesteps * div_term)


class ConvBlock(nn.Module):
    def __init__(self, in_channels, out_channels, groups=8):
        super().__init__()
        self.conv = nn.Conv2d(in_channels, out_channels, kernel_size=3, padding=1)
        self.norm = nn.GroupNorm(groups, out_channels)
        self.act = nn.SiLU()


class DownsampleBlock(nn.Module):
    def __init__(self, in_channels, out_channels, stride, padding):
        super().__init__()
        self.conv = nn.Conv2d(in_channels, out_channels, 3, stride=stride, padding=padding)


class UpsampleBlock(nn.Module):
    def __init__(self, in_channels, out_channels, scale_factor=2.0):
        super().__init__()
        self.scale = scale_factor
        self.conv = nn.Conv2d(in_channels, out_channels, 3, padding=1)


class ResNetBlock(nn.Module):
    def __init__(self, in_channels, out_channels, *, time_emb_channels=None, num_groups=8):
        super().__init__()
        self.time_embedding_projectile = (nn.Sequential(nn.SiLU(), nn.Linear(time_emb_channels, out_channels))
                                          if time_emb_channels else None)
        self.block1 = ConvBlock(in_channels, out_channels, groups=num_groups)
        self.block2 = ConvBlock(out_channels, out_channels, groups=num_groups)
        self.residual_conv = nn.Conv2d(in_channels, out_channels, 1) if in_channels != out_channels else nn.Identity()


class SelfAttentionBlock(nn.Module):
    def __init__(self, num_heads, in_channels, num_groups=32, embedding_dim=256):
        super().__init__()
        self.num_heads = num_heads
        self.d_model = embedding_dim
        self.d_keys = embedding_dim // num_heads
        self.d_values = embedding_dim // num_heads
        self.query_projection = nn.Linear(in_channels, embedding_dim)
        self.key_projection = nn.Linear(in_channels, embedding_dim)
        self.value_projection = nn.Linear(in_channels, embedding_dim)
        self.final_projection = nn.Linear(embedding_dim, embedding_dim)
        self.norm = nn.GroupNorm(num_channels=embedding_dim, num_groups=num_groups)


class _Block(nn.Module):
    def __init__(self, in_channels, out_channels, num_layers, time_emb_channels, num_groups, num_att_heads=None,
                 downsample=None, upsample=None):
        super().__init__()
        res, att = [], []
        for i in range(num_layers):
            ic = in_channels if i == 0 else out_channels
            res.append(ResNetBlock(in_channels=ic, out_channels=out_channels, time_emb_channels=time_emb_channels, num_groups=num_groups))
            if num_att_heads is not None:
                att.append(SelfAttentionBlock(in_channels=out_channels, embedding_dim=out_channels, num_heads=num_att_heads, num_groups=num_groups))
        self.resnet_blocks = nn.ModuleList(res)
        if num_att_heads is not None:
            self.attention_blocks = nn.ModuleList(att)
        if downsample is not None:
            self.downsample = DownsampleBlock(in_channels=out_channels, out_channels=out_channels, stride=2, padding=1) if downsample else None
        if upsample is not None:
            self.upsample = UpsampleBlock(in_channels=out_channels, out_channels=out_channels) if upsample else None


class ConvDownBlock(_Block):
    def __init__(self, in_channels, out_channels, num_layers, time_emb_channels, num_groups, downsample=True):
        super().__init__(in_channels, out_channels, num_layers, time_emb_channels, num_groups, downsample=downsample)


class ConvUpBlock(_Block):
    def __init__(self, in_channels, out_channels, num_layers, time_emb_channels, num_groups, upsample=True):
        super().__init__(in_channels, out_channels, num_layers, time_emb_channels, num_groups, upsample=upsample)


class AttentionDownBlock(_Block):
    def __init__(self, in_channels, out_channels, num_layers, time_emb_channels, num_groups, num_att_heads, downsample=True):
        super().__init__(in_channels, out_channels, num_layers, time_emb_channels, num_groups, num_att_heads, downsample=downsample)


class AttentionUpBlock(_Block):
    def __init__(self, in_channels, out_channels, num_layers, time_emb_channels, num_groups, num_att_heads, upsample=True):
        super().__init__(in_channels, out_channels, num_layers, time_emb_channels, num_groups, num_att_heads, upsample=upsample)


class UNet(engine.PackedWeights, nn.Module):
    """DDPM/models/unet.py:11-81."""

    def __init__(self, image_size=256, input_channels=3, compute_mode=None):
        super().__init__()
        self.compute_mode = compute_mode or engine.default_mode()
        self.initial_conv = nn.Conv2d(in_channels=input_channels, out_channels=128, kernel_size=3, stride=1, padding='same')
        self.positional_encoding = nn.Sequential(TransformerPositionalEmbedding(dimension=128), nn.Linear(128, 128 * 4),
                                                 nn.GELU(), nn.Linear(128 * 4, 128 * 4))
        T = 128 * 4
        self.downsample_blocks = nn.ModuleList([
            ConvDownBlock(128, 128, 2, T, 32), ConvDownBlock(128, 128, 2, T, 32), ConvDownBlock(128, 256, 2, T, 32),
            AttentionDownBlock(256, 256, 2, T, 32, 4), ConvDownBlock(256, 512, 2, T, 32)])
        self.bottleneck = AttentionDownBlock(512, 512, 2, T, 32, 4, downsample=False)
        self.upsample_blocks = nn.ModuleList([
            ConvUpBlock(512 + 512, 512, 2, T, 32), AttentionUpBlock(512 + 256, 256, 2, T, 32, 4),
            ConvUpBlock(256 + 256, 256, 2, T, 32), ConvUpBlock(256 + 128, 128, 2, T, 32), ConvUpBlock(128 + 128, 128, 2, T, 32)])
        self.output_conv = nn.Sequential(nn.GroupNorm(num_channels=256, num_groups=32), nn.SiLU(), nn.Conv2d(256, 3, 3, padding=1))
        self._init_packing()

    def _build_pack(self, mode):
        P = {}
        dev = self.initial_conv.weight.device
        P["pe"] = self.positional_encoding[0].pe_matrix.to(dev).float().contiguous()
        f = lambda t: t.detach().float().contiguous()
        P["pl1"] = (f(self.positional_encoding[1].weight), f(self.positional_encoding[1].bias))
        P["pl3"] = (f(self.positional_encoding[3].weight), f(self.positional_encoding[3].bias))
        ws, bs, off = [], [], 0
        for m in self.modules():
            if isinstance(m, ResNetBlock):
                lin = m.time_embedding_projectile[1]
                ws.append(f(lin.weight)); bs.append(f(lin.bias))
                P[("toff", id(m))] = (off, lin.out_features)
                off += lin.out_features
                P[("c1", id(m))] = PackedConv(m.block1.conv.weight, m.block1.conv.bias, mode)
                P[("c2", id(m))] = PackedConv(m.block2.conv.weight, m.block2.conv.bias, mode)
                if isinstance(m.residual_conv, nn.Conv2d):
                    P[("rc", id(m))] = PackedConv(m.residual_conv.weight, m.residual_conv.bias, mode)
            elif isinstance(m, SelfAttentionBlock):
                P[("qkv", id(m))] = PackedLinear(
                    torch.cat([m.query_projection.weight, m.key_projection.weight, m.value_projection.weight], 0),
                    torch.cat([m.query_projection.bias, m.key_projection.bias, m.value_projection.bias], 0), mode)
                P[("fp", id(m))] = PackedLinear(m.final_projection.weight, m.final_projection.bias, mode)
            elif isinstance(m, DownsampleBlock):
                P[("dc", id(m))] = PackedConv(m.conv.weight, m.conv.bias, mode, stride=2, pad=1)
            elif isinstance(m, UpsampleBlock):
                P[("uc", id(m))] = PackedConv(m.conv.weight, m.conv.bias, mode)
        P["tw"], P["tb"] = torch.cat(ws, 0).contiguous(), torch.cat(bs, 0).contiguous()
        P["ic"] = PackedConv(self.initial_conv.weight, self.initial_conv.bias, mode)
        P["oc"] = PackedConv(self.output_conv[2].weight, self.output_conv[2].bias, mode)
        return P

    @staticmethod
    def _to_op(x, pc):
        return ops.cast_concat(x, None, out_dtype=torch.bfloat16) if pc.in_dtype == torch.bfloat16 else x

    def _convblock(self, cb, pc, mode, x_op, rowvec=None, out_dtype=torch.float32):
        """ConvBlock (layers.py:37-48): conv -> GroupNorm -> SiLU."""
        h = engine.conv(x_op, pc)
        return ops.groupnorm(h, cb.norm.weight, cb.norm.bias, cb.norm.eps, act=1, out_dtype=out_dtype,
                             groups=cb.norm.num_groups, exact=(mode == "fp32"))

    def _resnet(self, rb, P, mode, x, x1, temb_all):
        """ResNetBlock.forward (layers.py:323-338); x1 = skip tensor to concatenate (UNet.forward torch.cat)."""
        c1, c2 = P[("c1", id(rb))], P[("c2", id(rb))]
        off, n = P[("toff", id(rb))]
        xin = ops.cast_concat(x, x1, out_dtype=c1.in_dtype) if (x1 is not None or c1.in_dtype == torch.bfloat16) else x
        h = self._convblock(rb.block1, c1, mode, xin)                               # fp32
        # x = time_emb[:, :, None, None] + h, emitted directly as block2's conv operand
        h = ops.add_rowvec(h, temb_all[:, off:off + n], out_dtype=c2.in_dtype)
        h = self._convblock(rb.block2, c2, mode, h)
        if ("rc", id(rb)) in P:
            rc = P[("rc", id(rb))]
            xr = xin if xin.dtype == rc.in_dtype else ops.cast_concat(x, x1, out_dtype=rc.in_dtype)
            return engine.conv(xr, rc, residual=h)
        assert x1 is None
        return ops.add(h, x)

    def _attn(self, ab, P, mode, x):
        """SelfAttentionBlock.forward (layers.py:160-200): post-norm MHA over h*w tokens."""
        B, Hh, Ww, Cc = x.shape
        S = Hh * Ww
        H, d = ab.num_heads, ab.d_keys
        t = x.reshape(B * S, Cc)
        scale = d ** -0.5
        if mode == "bf16":
            dp = head_pad(d)
            tb = ops.cast_concat(x, None, out_dtype=torch.bfloat16).reshape(B * S, Cc)
            qkv = engine.linear(tb, P[("qkv", id(ab))], out_dtype=torch.bfloat16, col_group=d, col_group_stride=dp)
            W3 = 3 * H * dp
            o = ops.attention_tc(qkv, qkv[:, H * dp:], qkv[:, 2 * H * dp:], B, H, S, S, d, dp, scale,
                                 (S * W3, W3, dp), (S * W3, W3, dp), (S * W3, W3, dp)).reshape(B * S, Cc)
        else:
            qkv = engine.linear(t, P[("qkv", id(ab))])
            o = engine.attention_fp32(qkv, qkv[:, Cc:], qkv[:, 2 * Cc:], B, H, S, S, d, scale)
        y = engine.linear(o, P[("fp", id(ab))], residual=t).reshape(B, Hh, Ww, Cc)      # final_projection + input
        return ops.groupnorm(y, ab.norm.weight, ab.norm.bias, ab.norm.eps, act=0, out_dtype=torch.float32,
                             groups=ab.norm.num_groups, exact=(mode == "fp32"))

    def _block(self, blk, P, mode, x, x1, temb_all):
        atts = getattr(blk, "attention_blocks", None)
        for j, rb in enumerate(blk.resnet_blocks):
            x = self._resnet(rb, P, mode, x, x1 if j == 0 else None, temb_all)
            if atts is not None:
                x = self._attn(atts[j], P, mode, x)
        if getattr(blk, "downsample", None) is not None:
            pc = P[("dc", id(blk.downsample))]
            x = engine.conv(self._to_op(x, pc), pc)
        if getattr(blk, "upsample", None) is not None:
            pc = P[("uc", id(blk.upsample))]
            x = engine.conv(ops.upsample_bilinear2x(x, out_dtype=pc.in_dtype), pc)
        return x

    @torch.no_grad()
    def forward(self, input_tensor, time):
        from ._lib import require_cuda
        require_cuda(input_tensor, time)
        self._check_weights()
        mode = self.compute_mode
        P = self.packed(mode)
        te = ops.gather_rows(P["pe"], time.long().contiguous())                      # pe_matrix[timestep]
        te = ops.skinny_linear(te, P["pl1"][0], P["pl1"][1], act_out=2)             # Linear -> GELU
        te = ops.skinny_linear(te, P["pl3"][0], P["pl3"][1])
        temb_all = ops.skinny_linear(te, P["tw"], P["tb"], act_in=1)                # every block's SiLU -> Linear
        x0 = engine.conv(ops.nchw_to_nhwc(input_tensor.float().contiguous()), P["ic"])
        skips = [x0]
        x = x0
        for blk in self.downsample_blocks:
            x = self._block(blk, P, mode, x, None, temb_all)
            skips.append(x)
        skips = list(reversed(skips))
        x = self._block(self.bottleneck, P, mode, x, None, temb_all)
        for blk, skip in zip(self.upsample_blocks, skips):
            x = self._block(blk, P, mode, x, skip, temb_all)
        oc = P["oc"]
        gn = self.output_conv[0]
        h = ops.groupnorm(x, gn.weight, gn.bias, gn.eps, act=1, out_dtype=oc.in_dtype, x1=skips[-1],
                          groups=gn.num_groups, exact=(mode == "fp32"))
        out = ops.nhwc_to_nchw(engine.conv(h, oc))
        return out if input_tensor.dtype == torch.float32 else out.to(input_tensor.dtype)
