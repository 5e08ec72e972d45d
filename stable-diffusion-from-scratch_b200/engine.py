"""Execution helpers shared by the drop-in modules: weight packing and mode dispatch.

Two compute modes (the constructor/env switch SURVEY.md §8b asks for, not a signature change):
  "bf16": tcgen05 tensor-core kernels; bf16 operands are produced by the norm/cast kernels, every
          contraction accumulates in fp32 (TMEM) and writes the fp32 residual stream.
  "fp32": SIMT FFMA kernels, fp32 everywhere (the <= 1e-5 parity mode).
There is no other path: both modes run hand-written kernels from libsdb200.so.
"""
import os
import weakref

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
    when a state dict is loaded (also through a parent module), when the module is moved or cast (`_apply`), and when a
    parameter is changed in place (`_check_weights`, a fingerprint of the first parameter's storage and every parameter's
    `_version`).  Call `_init_packing()` in `__init__`, `_check_weights()` once per public call and `packed(mode)` for the
    copies; a subclass implements `_build_pack(mode)`."""

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

    def packed(self, mode):
        P = self._packed.get(mode)
        if P is None:
            if mode not in MODES:
                raise ValueError("compute_mode must be one of %s" % (MODES,))
            P = self._packed[mode] = self._build_pack(mode)
        return P


class TensorMemo:
    """Values derived from tensors the owner does not own (a projection of the caller's conditioning, a table built from
    schedule buffers).  An entry stays valid only while each source tensor is the same live object (weakref), unwritten
    since (`_version`) and in the same place (`data_ptr`: `Module.to()` moves a Parameter without changing either of the
    others).  At `capacity` entries, a new one first drops entries whose sources died, then clears the memo."""

    def __init__(self, capacity):
        self.capacity = capacity
        self._entries = {}           # key -> (((weakref, _version, data_ptr) per source tensor), value)

    def get(self, tensors, key, build):
        """The value stored under `key` for these live `tensors`, else `build()`, stored."""
        hit = self._entries.get(key)
        if hit is not None and len(hit[0]) == len(tensors) and all(
                r() is t and v == t._version and p == t.data_ptr() for (r, v, p), t in zip(hit[0], tensors)):
            return hit[1]
        stamp = tuple((weakref.ref(t), t._version, t.data_ptr()) for t in tensors)
        value = build()
        if key not in self._entries and len(self._entries) >= self.capacity:
            self._entries = {k: e for k, e in self._entries.items() if all(r() is not None for r, _, _ in e[0])}
            if len(self._entries) >= self.capacity:
                self._entries.clear()
        self._entries[key] = (stamp, value)
        return value

    def clear(self):
        self._entries.clear()


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


def attention_fp32(q, k, v, B, H, Sq, Sk, d, scale, o_strides=None, causal=False):
    """fp32 unfused attention: scores = q k^T (batched over (b, h)), row softmax (causal: query i sees keys 0 .. i),
    out = P v.  q [B*Sq, >= H*d], k / v [B*Sk, >= H*d] fp32 row views (e.g. column blocks of the q | k | v projection,
    each read at its own row stride) -> [B*Sq, H*d] fp32.  o_strides = (batch, seq, head) element strides of another
    output layout."""
    Cc = H * d
    ldq, ldk, ldv = q.stride(0), k.stride(0), v.stride(0)
    scores = torch.empty((B, H, Sq, Sk), dtype=torch.float32, device=q.device)
    ops.gemm_simt(q, k, out=scores, M=Sq, N=Sk, K=d, lda=ldq, ldb=ldk, ldc=Sk, batch=(B, H),
                  sa=(Sq * ldq, d), sb=(Sk * ldk, d), sc=(H * Sq * Sk, Sq * Sk))
    P = ops.softmax_rows_causal(scores, scale, Sq) if causal else ops.softmax_rows(scores, scale)
    out = torch.empty((B * Sq, Cc), dtype=torch.float32, device=q.device)
    o_bs, o_ss, o_hs = o_strides if o_strides is not None else (Sq * Cc, Cc, d)
    ops.gemm_simt(P, v, out=out, b_kn=True, M=Sq, N=d, K=Sk, lda=Sk, ldb=ldv, ldc=o_ss, batch=(B, H),
                  sa=(H * Sq * Sk, Sq * Sk), sb=(Sk * ldv, d), sc=(o_bs, o_hs))
    return out
