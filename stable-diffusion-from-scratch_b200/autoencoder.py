"""Drop-in VAE `Decoder` / `AutoencoderKL.decode` (reference: ldm/modules/diffusionmodules/model.py:
468-574 and ldm/models/autoencoder.py:293-340) running on libsdb200.so, plus the 'next' row f3 of SURVEY.md §8:
`Encoder` (model.py:370-465), `AutoencoderKL.encode` (autoencoder.py:331-335) and `DiagonalGaussianDistribution`
(ldm/modules/distributions/distributions.py:24-65) built from the same kernels.

Same constructor kwargs and state-dict keys (`decoder.conv_in`, `decoder.mid.block_1.norm1`,
`decoder.up.L.block.K.conv1`, `decoder.up.L.upsample.conv`, `decoder.norm_out`, `decoder.conv_out`,
`post_quant_conv`) as the reference.  torch.nn layers are parameter holders only.
`VAE.autoencoder.AutoEncoderKL.decode` (VAE/autoencoder.py:126-132) is served by the same class
through the `AutoEncoderKL` alias; its fp16-only 8-head mid attention (Unet/attention.py:221-264)
is NOT replicated — the numerical oracle is the canonical `ldm` decoder (SURVEY.md §8a V2).

The VQ-regularised first stage of the reference's VQ latent-diffusion models (`VQModel`, `VQModelInterface`,
ldm/models/autoencoder.py; `IdentityFirstStage` for pixel-space models) is built from the same Encoder / Decoder
with `double_z=False`, and taming's `VectorQuantizer2` (sdb200.quantize) on the sdb_vq_quantize kernels.
"""
import torch
from torch import nn

from . import engine, ops
from .engine import PackedConv, PackedLinear


def Normalize(in_channels, num_groups=32):   # ldm/modules/diffusionmodules/model.py:40-41
    return nn.GroupNorm(num_groups=num_groups, num_channels=in_channels, eps=1e-6, affine=True)


class Upsample(nn.Module):
    def __init__(self, in_channels, with_conv):
        super().__init__()
        if not with_conv:
            raise NotImplementedError("sdb200 VAE Upsample: resamp_with_conv=False is outside the hot path")
        self.with_conv = with_conv
        self.conv = nn.Conv2d(in_channels, in_channels, kernel_size=3, stride=1, padding=1)


class Downsample(nn.Module):
    """ldm/modules/diffusionmodules/model.py:62-81: zero pad (0,1,0,1) then conv3x3 stride 2 without padding."""

    def __init__(self, in_channels, with_conv):
        super().__init__()
        if not with_conv:
            raise NotImplementedError("sdb200 VAE Downsample: resamp_with_conv=False (avg_pool2d) is not built")
        self.with_conv = with_conv
        self.conv = nn.Conv2d(in_channels, in_channels, kernel_size=3, stride=2, padding=0)


class ResnetBlock(nn.Module):
    def __init__(self, *, in_channels, out_channels=None, conv_shortcut=False, dropout, temb_channels=512):
        super().__init__()
        self.in_channels = in_channels
        out_channels = in_channels if out_channels is None else out_channels
        self.out_channels = out_channels
        self.use_conv_shortcut = conv_shortcut
        self.norm1 = Normalize(in_channels)
        self.conv1 = nn.Conv2d(in_channels, out_channels, kernel_size=3, stride=1, padding=1)
        if temb_channels > 0:
            self.temb_proj = nn.Linear(temb_channels, out_channels)
        self.norm2 = Normalize(out_channels)
        self.dropout = nn.Dropout(dropout)
        self.conv2 = nn.Conv2d(out_channels, out_channels, kernel_size=3, stride=1, padding=1)
        if self.in_channels != self.out_channels:
            if self.use_conv_shortcut:
                self.conv_shortcut = nn.Conv2d(in_channels, out_channels, kernel_size=3, stride=1, padding=1)
            else:
                self.nin_shortcut = nn.Conv2d(in_channels, out_channels, kernel_size=1, stride=1, padding=0)


class AttnBlock(nn.Module):
    def __init__(self, in_channels):
        super().__init__()
        self.in_channels = in_channels
        self.norm = Normalize(in_channels)
        self.q = nn.Conv2d(in_channels, in_channels, kernel_size=1, stride=1, padding=0)
        self.k = nn.Conv2d(in_channels, in_channels, kernel_size=1, stride=1, padding=0)
        self.v = nn.Conv2d(in_channels, in_channels, kernel_size=1, stride=1, padding=0)
        self.proj_out = nn.Conv2d(in_channels, in_channels, kernel_size=1, stride=1, padding=0)


def make_attn(in_channels, attn_type="vanilla"):
    assert attn_type in ["vanilla", "linear", "none"], f'attn_type {attn_type} unknown'
    if attn_type == "vanilla":
        return AttnBlock(in_channels)
    if attn_type == "none":
        return nn.Identity(in_channels)
    raise NotImplementedError("sdb200 VAE: linear attention is outside the hot path")


def _fingerprint(module):
    """(first parameter's address, device, sum of parameter versions): changes when parameters are replaced, moved or
    written in place (load through a parent module, EMA copy_to, ...)."""
    ps = module.__dict__.get("_param_list")
    if ps is None:
        ps = module.__dict__["_param_list"] = list(module.parameters())
    return (ps[0].data_ptr(), ps[0].device, sum(p._version for p in ps))


FUSED_ATTN_CHANNELS = (256, 512)     # head widths of tc_attention_wide_kernel


class _VaeNet(nn.Module):
    """Packing and block execution shared by Encoder and Decoder."""
    fused_attention = True           # False: AttnBlock as three GEMMs + row softmax per image (the round-1 path, kept for A/B)

    def __init__(self):
        super().__init__()
        # a parent's load_state_dict recurses through _load_from_state_dict and never reaches the override below
        self.register_load_state_dict_post_hook(lambda module, incompatible_keys: module._invalidate())

    def _invalidate(self):
        self._packed = {}
        self.__dict__.pop("_param_list", None)
        self.__dict__.pop("_fp_seen", None)

    def _check_weights(self):
        fp = _fingerprint(self)
        if fp != self.__dict__.get("_fp_seen"):
            if self.__dict__.get("_fp_seen") is not None:
                self._invalidate()
            self.__dict__["_fp_seen"] = fp

    def load_state_dict(self, *a, **k):
        r = super().load_state_dict(*a, **k)
        self._invalidate()
        return r

    def _apply(self, fn, *a, **k):
        r = super()._apply(fn, *a, **k)
        self._invalidate()
        return r

    def _pack(self, mode):
        self._check_weights()
        if mode in self._packed:
            return self._packed[mode]
        P = {}
        for m in self.modules():
            if isinstance(m, ResnetBlock):
                P[("c1", id(m))] = PackedConv(m.conv1.weight, m.conv1.bias, mode)
                P[("c2", id(m))] = PackedConv(m.conv2.weight, m.conv2.bias, mode)
                if hasattr(m, "nin_shortcut"):
                    P[("sc", id(m))] = PackedConv(m.nin_shortcut.weight, m.nin_shortcut.bias, mode)
                elif hasattr(m, "conv_shortcut"):
                    P[("sc", id(m))] = PackedConv(m.conv_shortcut.weight, m.conv_shortcut.bias, mode)
            elif isinstance(m, AttnBlock):
                Cc = m.in_channels
                for name in ("q", "k", "proj_out"):
                    conv = getattr(m, name)
                    P[(name, id(m))] = PackedLinear(conv.weight.reshape(Cc, Cc), conv.bias, mode)
                # V is produced transposed ([C, tokens]) by swapping GEMM operands, so its bias (per output ROW)
                # is added after P.V instead: softmax rows sum to 1, so P (V + 1 b^T) = P V + b^T.
                P[("v", id(m))] = PackedLinear(m.v.weight.reshape(Cc, Cc), None, mode)
                P[("vb", id(m))] = m.v.bias.detach().float().contiguous()
                if mode == "bf16" and Cc in FUSED_ATTN_CHANNELS:
                    # fused path: one [3C, C] projection (q | k | v side by side), then the wide-head flash kernel
                    P[("qkv", id(m))] = PackedLinear(torch.cat([m.q.weight, m.k.weight, m.v.weight], 0).reshape(3 * Cc, Cc),
                                                     torch.cat([m.q.bias, m.k.bias, m.v.bias], 0), mode)
            elif isinstance(m, Upsample):
                P[("up", id(m))] = PackedConv(m.conv.weight, m.conv.bias, mode, up2=True)
            elif isinstance(m, Downsample):
                P[("down", id(m))] = PackedConv(m.conv.weight, m.conv.bias, mode, stride=2, pad=0, pad_hi=1)
        P["conv_in"] = PackedConv(self.conv_in.weight, self.conv_in.bias, mode)
        P["conv_out"] = PackedConv(self.conv_out.weight, self.conv_out.bias, mode)
        self._packed[mode] = P
        return P

    @staticmethod
    def _gn(norm, x, mode, act, out_dtype, want_raw=False):
        return ops.groupnorm(x, norm.weight, norm.bias, norm.eps, act=act, out_dtype=out_dtype,
                             groups=norm.num_groups, exact=(mode == "fp32"), want_raw=want_raw)

    def _resnet(self, rb, P, mode, x):
        """ResnetBlock.forward with temb=None (model.py:123-143).  Every conv whose output feeds a GroupNorm also emits
        that GroupNorm's column statistics (want_stats), and the 1x1 nin_shortcut's bf16 operand comes out of norm1's pass."""
        c1, c2 = P[("c1", id(rb))], P[("c2", id(rb))]
        sc = P.get(("sc", id(rb)))
        raw = None
        if sc is not None and sc.in_dtype == torch.bfloat16:
            hn, raw = self._gn(rb.norm1, x, mode, 1, c1.in_dtype, want_raw=True)
        else:
            hn = self._gn(rb.norm1, x, mode, 1, c1.in_dtype)
        h = engine.conv(hn, c1, want_stats=True)
        h = self._gn(rb.norm2, h, mode, 1, c2.in_dtype)
        if sc is not None:
            xs = engine.conv(raw if raw is not None else x, sc)
        else:
            xs = x
        return engine.conv(h, c2, residual=xs, want_stats=True)

    def _attn(self, ab, P, mode, x):
        """AttnBlock.forward (model.py:180-204): single head, d = C, scores materialised per image
        (as the reference's torch.bmm does), all three contractions on the GEMM kernels."""
        B, Hh, Ww, Cc = x.shape
        S = Hh * Ww
        odt = engine.op_dtype(mode)
        hn = self._gn(ab.norm, x, mode, 0, odt).reshape(B * S, Cc)
        if ("qkv", id(ab)) in P and self.fused_attention:
            # bf16 mode, C = 256 / 512: flash-style kernel, no [S, S] score matrix, no per-image loop
            qkv = engine.linear(hn, P[("qkv", id(ab))], out_dtype=odt)                          # [B*S, 3C]
            W3 = 3 * Cc
            o = ops.attention_wide(qkv, qkv[:, Cc:], qkv[:, 2 * Cc:], B, S, S, Cc, float(int(Cc) ** (-0.5)),
                                   (S * W3, W3), (S * W3, W3), (S * W3, W3))
            # rows_per_item: the measured launch plan of this shape (tc_plans, keyed per image) applies
            out = engine.linear(o.reshape(B * S, Cc), P[("proj_out", id(ab))], residual=x.reshape(B * S, Cc), rows_per_item=S)
            return out.reshape(B, Hh, Ww, Cc)
        q = engine.linear(hn, P[("q", id(ab))], out_dtype=odt)
        k = engine.linear(hn, P[("k", id(ab))], out_dtype=odt)
        scale = float(int(Cc) ** (-0.5))
        o = torch.empty((B * S, Cc), dtype=odt, device=x.device)
        wv = P[("v", id(ab))]
        for b in range(B):
            qb, kb, hb = q[b * S:(b + 1) * S], k[b * S:(b + 1) * S], hn[b * S:(b + 1) * S]
            if mode == "bf16":
                vT = ops.gemm_tc(wv.w, hb, out_dtype=odt)                                   # [C, S] = Wv @ hn^T
                sc = ops.gemm_tc(qb, kb)                                                    # [S, S] fp32
                pm = ops.softmax_rows(sc, scale, out_dtype=odt)
                ops.gemm_tc(pm, vT, bias=P[("vb", id(ab))], out=o[b * S:(b + 1) * S], out_dtype=odt)
            else:
                v = ops.gemm_simt(hb, wv.w, P[("vb", id(ab))])                              # [S, C]
                sc = ops.gemm_simt(qb, kb)
                pm = ops.softmax_rows(sc, scale)
                ops.gemm_simt(pm, v, b_kn=True, out=o[b * S:(b + 1) * S])
        out = engine.linear(o, P[("proj_out", id(ab))], residual=x.reshape(B * S, Cc), rows_per_item=S)
        return out.reshape(B, Hh, Ww, Cc)


class Encoder(_VaeNet):
    """ldm/modules/diffusionmodules/model.py:370-465 — same constructor kwargs and state-dict keys
    (`conv_in`, `down.L.block.K.*`, `down.L.attn.K.*`, `down.L.downsample.conv`, `mid.*`, `norm_out`, `conv_out`)."""

    def __init__(self, *, ch, out_ch, ch_mult=(1, 2, 4, 8), num_res_blocks, attn_resolutions, dropout=0.0,
                 resamp_with_conv=True, in_channels, resolution, z_channels, double_z=True, use_linear_attn=False,
                 attn_type="vanilla", compute_mode=None, **ignore_kwargs):
        super().__init__()
        if use_linear_attn:
            attn_type = "linear"
        self.ch = ch
        self.temb_ch = 0
        self.num_resolutions = len(ch_mult)
        self.num_res_blocks = num_res_blocks
        self.resolution = resolution
        self.in_channels = in_channels
        self.compute_mode = compute_mode or engine.default_mode()
        self.conv_in = nn.Conv2d(in_channels, self.ch, kernel_size=3, stride=1, padding=1)
        curr_res = resolution
        in_ch_mult = (1,) + tuple(ch_mult)
        self.in_ch_mult = in_ch_mult
        self.down = nn.ModuleList()
        for i_level in range(self.num_resolutions):
            block = nn.ModuleList()
            attn = nn.ModuleList()
            block_in = ch * in_ch_mult[i_level]
            block_out = ch * ch_mult[i_level]
            for i_block in range(self.num_res_blocks):
                block.append(ResnetBlock(in_channels=block_in, out_channels=block_out, temb_channels=self.temb_ch, dropout=dropout))
                block_in = block_out
                if curr_res in attn_resolutions:
                    attn.append(make_attn(block_in, attn_type=attn_type))
            down = nn.Module()
            down.block = block
            down.attn = attn
            if i_level != self.num_resolutions - 1:
                down.downsample = Downsample(block_in, resamp_with_conv)
                curr_res = curr_res // 2
            self.down.append(down)
        self.mid = nn.Module()
        self.mid.block_1 = ResnetBlock(in_channels=block_in, out_channels=block_in, temb_channels=self.temb_ch, dropout=dropout)
        self.mid.attn_1 = make_attn(block_in, attn_type=attn_type)
        self.mid.block_2 = ResnetBlock(in_channels=block_in, out_channels=block_in, temb_channels=self.temb_ch, dropout=dropout)
        self.norm_out = Normalize(block_in)
        self.conv_out = nn.Conv2d(block_in, 2 * z_channels if double_z else z_channels, kernel_size=3, stride=1, padding=1)
        self._packed = {}

    def _forward_nhwc(self, x, mode):
        """x [N,H,W,in_channels] fp32 -> [N,H/2^(L-1),W/2^(L-1),2*z_channels] fp32 (Encoder.forward, model.py:434-465)."""
        P = self._pack(mode)
        ci = P["conv_in"]
        h = engine.conv(x if ci.in_dtype == torch.float32 else ops.cast_concat(x, None, out_dtype=torch.bfloat16), ci, want_stats=True)
        for i_level in range(self.num_resolutions):
            for i_block in range(self.num_res_blocks):
                h = self._resnet(self.down[i_level].block[i_block], P, mode, h)
                if len(self.down[i_level].attn) > 0 and isinstance(self.down[i_level].attn[i_block], AttnBlock):
                    h = self._attn(self.down[i_level].attn[i_block], P, mode, h)
            if i_level != self.num_resolutions - 1:
                pc = P[("down", id(self.down[i_level].downsample))]
                hin = h if pc.in_dtype == torch.float32 else ops.cast_concat(h, None, out_dtype=torch.bfloat16)
                h = engine.conv(hin, pc, want_stats=True)
        h = self._resnet(self.mid.block_1, P, mode, h)
        if isinstance(self.mid.attn_1, AttnBlock):
            h = self._attn(self.mid.attn_1, P, mode, h)
        h = self._resnet(self.mid.block_2, P, mode, h)
        co = P["conv_out"]
        h = self._gn(self.norm_out, h, mode, 1, co.in_dtype)
        return engine.conv(h, co)

    @torch.no_grad()
    def forward(self, x):
        """x [N, in_channels, H, W] -> [N, 2*z_channels, h, w] (fp32 in, fp32 out)."""
        from ._lib import require_cuda
        with torch.cuda.device(x.device):
            require_cuda(x)
            h = ops.nchw_to_nhwc(x.float().contiguous())
            out = ops.nhwc_to_nchw(self._forward_nhwc(h, self.compute_mode))
        return out if x.dtype == torch.float32 else out.to(x.dtype)


class DiagonalGaussianDistribution(object):
    """ldm/modules/distributions/distributions.py:24-65; mean / logvar / std / var / sample come out of one kernel."""

    def __init__(self, parameters, deterministic=False):
        self.parameters = parameters
        self.deterministic = deterministic
        self._moments = parameters.float().contiguous()
        self.mean, self.logvar, self.std, self.var, _ = ops.diag_gaussian(self._moments)
        if self.deterministic:
            self.var = self.std = torch.zeros_like(self.mean)

    def sample(self, noise=None):
        """mean + std * randn (distributions.py:35-37); `noise` lets a caller supply the draw (tests, per-sample seeds)."""
        if noise is None:
            noise = torch.randn(self.mean.shape, device=self.mean.device)
        if self.deterministic:
            return self.mean.clone()
        return ops.diag_gaussian(self._moments, noise.float().contiguous())[4]

    def kl(self, other=None):
        if self.deterministic:
            return torch.Tensor([0.])
        if other is None:
            return 0.5 * torch.sum(torch.pow(self.mean, 2) + self.var - 1.0 - self.logvar, dim=[1, 2, 3])
        return 0.5 * torch.sum(torch.pow(self.mean - other.mean, 2) / other.var + self.var / other.var - 1.0
                               - self.logvar + other.logvar, dim=[1, 2, 3])

    def nll(self, sample, dims=[1, 2, 3]):
        if self.deterministic:
            return torch.Tensor([0.])
        logtwopi = 1.8378770664093453
        return 0.5 * torch.sum(logtwopi + self.logvar + torch.pow(sample - self.mean, 2) / self.var, dim=dims)

    def mode(self):
        return self.mean


class Decoder(_VaeNet):
    """ldm/modules/diffusionmodules/model.py:468-574."""

    def __init__(self, *, ch, out_ch, ch_mult=(1, 2, 4, 8), num_res_blocks, attn_resolutions, dropout=0.0,
                 resamp_with_conv=True, in_channels, resolution, z_channels, give_pre_end=False, tanh_out=False,
                 use_linear_attn=False, attn_type="vanilla", compute_mode=None, **ignorekwargs):
        super().__init__()
        if use_linear_attn:
            attn_type = "linear"
        if tanh_out or give_pre_end:
            raise NotImplementedError("sdb200 Decoder: tanh_out / give_pre_end are outside the hot path")
        self.ch = ch
        self.temb_ch = 0
        self.num_resolutions = len(ch_mult)
        self.num_res_blocks = num_res_blocks
        self.resolution = resolution
        self.in_channels = in_channels
        self.give_pre_end = give_pre_end
        self.tanh_out = tanh_out
        self.compute_mode = compute_mode or engine.default_mode()
        block_in = ch * ch_mult[self.num_resolutions - 1]
        curr_res = resolution // 2 ** (self.num_resolutions - 1)
        self.z_shape = (1, z_channels, curr_res, curr_res)
        self.conv_in = nn.Conv2d(z_channels, block_in, kernel_size=3, stride=1, padding=1)
        self.mid = nn.Module()
        self.mid.block_1 = ResnetBlock(in_channels=block_in, out_channels=block_in, temb_channels=self.temb_ch, dropout=dropout)
        self.mid.attn_1 = make_attn(block_in, attn_type=attn_type)
        self.mid.block_2 = ResnetBlock(in_channels=block_in, out_channels=block_in, temb_channels=self.temb_ch, dropout=dropout)
        self.up = nn.ModuleList()
        for i_level in reversed(range(self.num_resolutions)):
            block = nn.ModuleList()
            attn = nn.ModuleList()
            block_out = ch * ch_mult[i_level]
            for i_block in range(self.num_res_blocks + 1):
                block.append(ResnetBlock(in_channels=block_in, out_channels=block_out, temb_channels=self.temb_ch, dropout=dropout))
                block_in = block_out
                if curr_res in attn_resolutions:
                    attn.append(make_attn(block_in, attn_type=attn_type))
            up = nn.Module()
            up.block = block
            up.attn = attn
            if i_level != 0:
                up.upsample = Upsample(block_in, resamp_with_conv)
                curr_res = curr_res * 2
            self.up.insert(0, up)
        self.norm_out = Normalize(block_in)
        self.conv_out = nn.Conv2d(block_in, out_ch, kernel_size=3, stride=1, padding=1)
        self._packed = {}

    def _forward_nhwc(self, z, mode):
        P = self._pack(mode)
        h = engine.conv(z, P["conv_in"], want_stats=True)
        h = self._resnet(self.mid.block_1, P, mode, h)
        if isinstance(self.mid.attn_1, AttnBlock):
            h = self._attn(self.mid.attn_1, P, mode, h)
        h = self._resnet(self.mid.block_2, P, mode, h)
        for i_level in reversed(range(self.num_resolutions)):
            for i_block in range(self.num_res_blocks + 1):
                h = self._resnet(self.up[i_level].block[i_block], P, mode, h)
                if len(self.up[i_level].attn) > 0 and isinstance(self.up[i_level].attn[i_block], AttnBlock):
                    h = self._attn(self.up[i_level].attn[i_block], P, mode, h)
            if i_level != 0:
                pc = P[("up", id(self.up[i_level].upsample))]
                if pc.use_tc:
                    h = engine.conv_up2(ops.cast_concat(h, None, out_dtype=torch.bfloat16), pc, want_stats=True)
                else:
                    h = engine.conv(h, pc, up=2)
        co = P["conv_out"]
        h = self._gn(self.norm_out, h, mode, 1, co.in_dtype)
        return engine.conv(h, co)

    @torch.no_grad()
    def forward(self, z):
        """z [N, z_channels, h, w] -> [N, out_ch, 8h, 8w] (fp32 in, fp32 out)."""
        from ._lib import require_cuda
        with torch.cuda.device(z.device):
            require_cuda(z)
            self.last_z_shape = z.shape
            h = ops.nchw_to_nhwc(z.float().contiguous())
            out = ops.nhwc_to_nchw(self._forward_nhwc(h, self.compute_mode))
        return out if z.dtype == torch.float32 else out.to(z.dtype)


class _FirstStage(nn.Module):
    """What AutoencoderKL and VQModel share: Encoder / Decoder compute mode, checkpoint loading, the fp32 SIMT packing
    of the 1x1 quant_conv / post_quant_conv, and the micro-batched encode / decode loops."""

    @property
    def compute_mode(self):
        return self.decoder.compute_mode

    @compute_mode.setter
    def compute_mode(self, m):
        self.decoder.compute_mode = m
        self.encoder.compute_mode = m

    def init_from_ckpt(self, path, ignore_keys=list()):
        sd = torch.load(path, map_location="cpu")["state_dict"]
        for k in list(sd.keys()):
            for ik in ignore_keys:
                if k.startswith(ik):
                    del sd[k]
        self.load_state_dict(sd, strict=False)

    def _invalidate(self):
        self.decoder._invalidate()
        self.encoder._invalidate()
        self._pq = None
        self._q = None

    def load_state_dict(self, *a, **k):
        r = super().load_state_dict(*a, **k)
        self._invalidate()
        return r

    def _apply(self, fn, *a, **k):
        r = super()._apply(fn, *a, **k)
        self._invalidate()
        return r

    _pq = None
    _q = None

    def _packed_1x1(self, slot, conv):
        """quant_conv / post_quant_conv packed for the fp32 SIMT kernel (C_in = 3 ... 8), re-packed whenever the layer's
        parameters were replaced or written in place."""
        fp = (conv.weight.data_ptr(), conv.weight._version, conv.bias.data_ptr(), conv.bias._version)
        cur = getattr(self, slot)
        if cur is None or cur[0] != fp:
            cur = (fp, PackedConv(conv.weight, conv.bias, "fp32"))
            setattr(self, slot, cur)
        return cur[1]

    def _encode_quant_conv(self, x):
        """Encoder then quant_conv, in micro-batches of `micro_batch` images: x [N,C,H,W] -> [N,C',h,w] fp32 NCHW."""
        from ._lib import require_cuda
        with torch.cuda.device(x.device):
            require_cuda(x)
            mode = self.encoder.compute_mode
            qc = self._packed_1x1("_q", self.quant_conv)                                   # tiny C_in: SIMT fp32 kernel in both modes
            xf = x.float().contiguous()
            outs = []
            for i in range(0, xf.shape[0], self.micro_batch):
                h = self.encoder._forward_nhwc(ops.nchw_to_nhwc(xf[i:i + self.micro_batch].contiguous()), mode)
                outs.append(ops.nhwc_to_nchw(engine.conv(h, qc)))
            return outs[0] if len(outs) == 1 else torch.cat(outs, 0)

    def _decode_post_quant(self, z, to_nhwc):
        """post_quant_conv then Decoder on z [N,C,h,w], in micro-batches of `micro_batch` images (activations at 512^2
        are ~0.5 GB/image); results are identical because nothing on the path reduces over the batch.  `to_nhwc` turns
        one NCHW fp32 micro-batch into the NHWC fp32 operand of post_quant_conv."""
        from ._lib import require_cuda
        with torch.cuda.device(z.device):
            require_cuda(z)
            mode = self.decoder.compute_mode
            pq = self._packed_1x1("_pq", self.post_quant_conv)                             # tiny C_in: SIMT fp32 kernel in both modes
            zf = z.float().contiguous()
            N = zf.shape[0]
            outs = []
            for i in range(0, N, self.micro_batch):
                h = engine.conv(to_nhwc(zf[i:i + self.micro_batch].contiguous()), pq)
                outs.append(ops.nhwc_to_nchw(self.decoder._forward_nhwc(h, mode)))
            out = outs[0] if len(outs) == 1 else torch.cat(outs, 0)
        return out if z.dtype == torch.float32 else out.to(z.dtype)


class AutoencoderKL(_FirstStage):
    """ldm/models/autoencoder.py:292-350: decode (hot path), encode and forward ('next' row f3).  The loss / Lightning
    training hooks are out of scope (SURVEY.md §2.1); their state-dict keys are tolerated with strict=False."""

    def __init__(self, ddconfig, lossconfig=None, embed_dim=4, ckpt_path=None, ignore_keys=[], image_key="image",
                 colorize_nlabels=None, monitor=None, compute_mode=None, micro_batch=8):
        super().__init__()
        self.image_key = image_key
        self.encoder = Encoder(**ddconfig, compute_mode=compute_mode)
        self.decoder = Decoder(**ddconfig, compute_mode=compute_mode)
        assert ddconfig["double_z"]
        self.quant_conv = nn.Conv2d(2 * ddconfig["z_channels"], 2 * embed_dim, 1)
        self.post_quant_conv = nn.Conv2d(embed_dim, ddconfig["z_channels"], 1)
        self.embed_dim = embed_dim
        self.micro_batch = micro_batch
        if monitor is not None:
            self.monitor = monitor
        if ckpt_path is not None:
            self.init_from_ckpt(ckpt_path, ignore_keys=ignore_keys)

    @torch.no_grad()
    def encode(self, x):
        """AutoencoderKL.encode (autoencoder.py:331-335): Encoder, quant_conv (1x1, 8->8), posterior.
        x [N,3,H,W] in [-1,1] -> DiagonalGaussianDistribution over [N,embed_dim,H/8,W/8]."""
        moments = self._encode_quant_conv(x)
        with torch.cuda.device(moments.device):
            return DiagonalGaussianDistribution(moments)

    @torch.no_grad()
    def decode(self, z):
        """AutoencoderKL.decode (autoencoder.py:337-340): post_quant_conv (1x1, 4->4) then Decoder."""
        return self._decode_post_quant(z, ops.nchw_to_nhwc)

    def forward(self, input, sample_posterior=True):
        """autoencoder.py:342-349: (reconstruction, posterior)."""
        posterior = self.encode(input)
        z = posterior.sample() if sample_posterior else posterior.mode()
        return self.decode(z), posterior


class VQModel(_FirstStage):
    """ldm/models/autoencoder.py VQModel (inference): Encoder, quant_conv (z_channels -> embed_dim), VectorQuantizer2
    (`quantize`, n_embed codes of embed_dim), post_quant_conv (embed_dim -> z_channels), Decoder; the reference's
    constructor kwargs and state-dict keys (`quantize.embedding.weight`, ...).  The loss, Lightning training hooks,
    batch resizing and the LR schedule are out of scope: their kwargs are accepted and ignored and `loss.*` keys are
    tolerated with strict=False."""

    def __init__(self, ddconfig, lossconfig, n_embed, embed_dim, ckpt_path=None, ignore_keys=[], image_key="image",
                 colorize_nlabels=None, monitor=None, batch_resize_range=None, scheduler_config=None, lr_g_factor=1.0,
                 remap=None, sane_index_shape=False, use_ema=False, compute_mode=None, micro_batch=8):
        super().__init__()
        if use_ema:
            raise NotImplementedError("sdb200 VQModel: use_ema (LitEma training copy) is not built")
        from .quantize import VectorQuantizer2
        self.embed_dim = embed_dim
        self.n_embed = n_embed
        self.image_key = image_key
        self.encoder = Encoder(**ddconfig, compute_mode=compute_mode)
        self.decoder = Decoder(**ddconfig, compute_mode=compute_mode)
        self.quantize = VectorQuantizer2(n_embed, embed_dim, beta=0.25, remap=remap, sane_index_shape=sane_index_shape)
        self.quant_conv = nn.Conv2d(ddconfig["z_channels"], embed_dim, 1)
        self.post_quant_conv = nn.Conv2d(embed_dim, ddconfig["z_channels"], 1)
        self.micro_batch = micro_batch
        self.batch_resize_range = batch_resize_range
        self.scheduler_config = scheduler_config
        self.lr_g_factor = lr_g_factor
        self.use_ema = use_ema
        if monitor is not None:
            self.monitor = monitor
        if ckpt_path is not None:
            self.init_from_ckpt(ckpt_path, ignore_keys=ignore_keys)

    @torch.no_grad()
    def encode(self, x):
        """(quant, emb_loss, (None, None, indices)): Encoder, quant_conv, quantize."""
        return self.quantize(self.encode_to_prequant(x))

    @torch.no_grad()
    def encode_to_prequant(self, x):
        """Encoder then quant_conv: x [N,3,H,W] -> [N,embed_dim,h,w] fp32."""
        return self._encode_quant_conv(x)

    @torch.no_grad()
    def decode(self, quant):
        """post_quant_conv then Decoder."""
        return self._decode_post_quant(quant, ops.nchw_to_nhwc)

    def decode_code(self, code_b):
        # the reference calls quantize.embed_code, which VectorQuantizer2 does not define
        raise NotImplementedError("VQModel.decode_code: VectorQuantizer2 has no embed_code; use "
                                  "decode(quantize.get_codebook_entry(indices, shape))")

    def forward(self, input, return_pred_indices=False):
        quant, diff, (_, _, ind) = self.encode(input)
        dec = self.decode(quant)
        if return_pred_indices:
            return dec, diff, ind
        return dec, diff


class VQModelInterface(VQModel):
    """ldm/models/autoencoder.py VQModelInterface, the first stage of the VQ latent-diffusion models: encode stops
    before the quantizer; decode quantizes (unless force_not_quantize) and decodes.  On the decode path the quantizer
    writes z_q channels-last straight into post_quant_conv's operand."""

    def __init__(self, embed_dim, *args, **kwargs):
        super().__init__(*args, embed_dim=embed_dim, **kwargs)
        self.embed_dim = embed_dim

    @torch.no_grad()
    def encode(self, x):
        return self.encode_to_prequant(x)

    @torch.no_grad()
    def decode(self, h, force_not_quantize=False):
        from ._lib import require_cuda
        require_cuda(h)
        if force_not_quantize:
            return self._decode_post_quant(h, ops.nchw_to_nhwc)
        to_nhwc = lambda z: self.quantize._quantize(z, zq_layout="nhwc", want_idx=False, want_loss=False)[0]
        return self._decode_post_quant(h, to_nhwc)


class IdentityFirstStage(nn.Module):
    """ldm/models/autoencoder.py IdentityFirstStage: the first stage of pixel-space models."""

    def __init__(self, *args, vq_interface=False, **kwargs):
        self.vq_interface = vq_interface
        super().__init__()

    def encode(self, x, *args, **kwargs):
        return x

    def decode(self, x, *args, **kwargs):
        return x

    def quantize(self, x, *args, **kwargs):
        if self.vq_interface:
            return x, None, [None, None, None]
        return x

    def forward(self, x, *args, **kwargs):
        return x


AutoEncoderKL = AutoencoderKL   # VAE/autoencoder.py spells it with a capital E
