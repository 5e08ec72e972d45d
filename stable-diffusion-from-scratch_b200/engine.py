"""Execution helpers shared by the drop-in modules: weight packing and mode dispatch.

Two compute modes (the constructor/env switch SURVEY.md §8b asks for, not a signature change):
  "bf16": tcgen05 tensor-core kernels; bf16 operands are produced by the norm/cast kernels, every
          contraction accumulates in fp32 (TMEM) and writes the fp32 residual stream.
  "fp32": SIMT FFMA kernels, fp32 everywhere (the <= 1e-5 parity mode).
There is no other path: both modes run hand-written kernels from libsdb200.so.
"""
import os

import torch

from . import ops

MODES = ("bf16", "fp32")


def default_mode():
    return os.environ.get("SDB200_MODE", "bf16")


def op_dtype(mode):
    return torch.bfloat16 if mode == "bf16" else torch.float32


def head_pad(d):
    """Heads are stored padded to a multiple of 64 channels for the tcgen05 attention kernel."""
    return (d + 63) // 64 * 64


class PackedConv:
    """A conv layer's weights repacked tap-major [kh*kw, Cout, Cin] for one compute mode."""

    def __init__(self, weight, bias, mode, stride=1, pad=None, up2=False, pad_hi=None):
        Cout, Cin, kh, kw = weight.shape
        self.cout, self.cin, self.kh, self.kw = Cout, Cin, kh, kw
        self.stride = stride
        self.pad = (kh // 2) if pad is None else pad
        self.pad_hi = self.pad if pad_hi is None else pad_hi      # bottom/right padding (asymmetric for the VAE Downsample)
        # the tensor-core path needs whole 16-byte channel rows; tiny-C layers stay on the SIMT kernel
        self.use_tc = (mode == "bf16") and (Cin % 8 == 0) and (Cin >= 32)
        dt = torch.bfloat16 if self.use_tc else torch.float32
        self.w = ops.pack_conv_weight(weight, dt)
        self.bias = None if bias is None else bias.detach().float().contiguous()
        # conv that follows a nearest-2x upsampling: folded sub-pixel weights (tensor-core path only)
        self.w_up2 = ops.fold_upsample_weights(weight, dt) if (up2 and self.use_tc and kh == 3 and kw == 3 and stride == 1) else None

    @property
    def in_dtype(self):
        return torch.bfloat16 if self.use_tc else torch.float32


class PackedWeights:
    """Mixin for an nn.Module that keeps per-mode packed copies of its parameters in `self._packed`: the copies are dropped
    when a state dict is loaded, when the module is moved or cast (`_apply`), and when a parameter is changed in place
    (`_check_weights`, a fingerprint of the first parameter's storage and every parameter's `_version`).  Call
    `_init_packing()` in `__init__` and `_check_weights()` before every use of the packed copies."""

    def _init_packing(self):
        self._packed = {}
        self.register_load_state_dict_post_hook(lambda module, incompatible_keys: module._invalidate())

    def _invalidate(self):
        self._packed = {}
        self.__dict__.pop("_param_list", None)
        self.__dict__.pop("_fp_seen", None)

    def _apply(self, fn, *a, **k):
        r = super()._apply(fn, *a, **k)
        self._invalidate()
        return r

    def _check_weights(self):
        ps = self.__dict__.get("_param_list")
        if ps is None:
            ps = self.__dict__["_param_list"] = list(self.parameters())
        fp = (ps[0].data_ptr(), ps[0].device, sum(p._version for p in ps))
        if fp != self.__dict__.get("_fp_seen"):
            if self.__dict__.get("_fp_seen") is not None:
                self._invalidate()
            self.__dict__["_fp_seen"] = fp


class PackedLinear:
    def __init__(self, weight, bias, mode, geglu=False):
        self.n, self.k = weight.shape
        self.use_tc = (mode == "bf16") and (self.k % 8 == 0)
        self.geglu = geglu
        self.block_n = 0
        w = weight.detach().float()
        b = None if bias is None else bias.detach().float()
        if geglu and self.use_tc:
            self.block_n = 256 if (self.n // 2) % 128 == 0 else 128
            w, b = ops.pack_geglu_weight(w, b, self.block_n)
        self.w = w.to(torch.bfloat16 if self.use_tc else torch.float32).contiguous()
        self.bias = None if b is None else b.contiguous()


# Packed weights (PackedConv / PackedLinear) are written once, long before any launch that reads them: the tcgen05 kernels may
# fetch their first weight tiles before the programmatic-dependent-launch wait (sdb_tc_args.b_const).  SDB200_B_CONST=0 = off.
B_CONST = os.environ.get("SDB200_B_CONST", "0") == "1"


def conv(x, pc, rowvec=None, residual=None, out_dtype=torch.float32, up=1, want_stats=False):
    """x [N,H,W,Cin] in pc.in_dtype (fp32 for the SIMT path, bf16 for tcgen05) -> [N,OH,OW,Cout].
    want_stats: the output feeds a GroupNorm — let the tcgen05 epilogue also emit its column statistics."""
    if pc.use_tc:
        assert up == 1
        return ops.conv_tc(x, pc.w, pc.bias, pc.kh, pc.kw, stride=pc.stride, pad=pc.pad, rowvec=rowvec,
                           residual=residual, out_dtype=out_dtype, want_stats=want_stats, pad_hi=pc.pad_hi, b_const=B_CONST)
    return ops.conv_simt(x, pc.w, pc.bias, pc.kh, pc.kw, stride=pc.stride, pad=pc.pad, up=up, rowvec=rowvec,
                         residual=residual, out_dtype=out_dtype, pad_hi=pc.pad_hi)


def conv_up2(x, pc, want_stats=False):
    """conv `pc` applied to the nearest-2x upsampling of x [N,H,W,Cin] (bf16 on the tensor-core path)."""
    if pc.w_up2 is not None:
        return ops.conv_up2_tc(x, pc.w_up2, pc.bias, want_stats=want_stats, b_const=B_CONST)
    return conv(x, pc, up=2)


def linear(x, pl, residual=None, out_dtype=torch.float32, col_group=0, col_group_stride=0, rows_per_item=0, out=None):
    """x [rows, K] -> [rows, N] (or [rows, N/2] for a GEGLU layer)."""
    rows = x.numel() // x.shape[-1]
    x2 = x.reshape(rows, x.shape[-1])
    if pl.use_tc:
        return ops.gemm_tc(x2, pl.w, pl.bias, residual=residual, out_dtype=out_dtype, geglu=pl.geglu,
                           col_group=col_group, col_group_stride=col_group_stride, block_n=pl.block_n,
                           rows_per_item=rows_per_item, out=out, b_const=B_CONST)
    assert col_group == 0
    if pl.geglu:
        h = ops.gemm_simt(x2, pl.w, pl.bias)
        g = ops.geglu(h, out_dtype=out_dtype)
        return g
    return ops.gemm_simt(x2, pl.w, pl.bias, residual=residual, out_dtype=out_dtype)


def attention_fp32(q, k, v, B, H, Sq, Sk, d, scale, ld=None):
    """fp32 unfused attention: scores = q k^T (batched over (b, h)), row softmax, out = P v.
    q [B*Sq, H*d], k/v [B*Sk, H*d] fp32 -> [B*Sq, H*d] fp32.  ld: the row stride of q, k and v in elements when they are
    column blocks of one wider tensor (e.g. the q | k | v projection), else H*d."""
    Cc = H * d
    ld = Cc if ld is None else ld
    scores = torch.empty((B, H, Sq, Sk), dtype=torch.float32, device=q.device)
    ops.gemm_simt(q, k, out=scores, M=Sq, N=Sk, K=d, lda=ld, ldb=ld, ldc=Sk, batch=(B, H),
                  sa=(Sq * ld, d), sb=(Sk * ld, d), sc=(H * Sq * Sk, Sq * Sk))
    P = ops.softmax_rows(scores, scale)
    out = torch.empty((B * Sq, Cc), dtype=torch.float32, device=q.device)
    ops.gemm_simt(P, v, out=out, b_kn=True, M=Sq, N=d, K=Sk, lda=Sk, ldb=ld, ldc=Cc, batch=(B, H),
                  sa=(H * Sq * Sk, Sq * Sk), sb=(Sk * ld, d), sc=(Sq * Cc, d))
    return out
