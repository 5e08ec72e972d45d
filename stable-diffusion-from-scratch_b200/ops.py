"""Tensor-level wrappers over the C-ABI (include/sdb200.h).

Every function enqueues hand-written sm_100a kernels from libsdb200.so on the current CUDA stream.
torch is used for allocation (`torch.empty`) and pointers only.  Activations are channels-last:
images [N, H, W, C], tokens [rows, C].
"""
import ctypes as C
import os

import torch

from . import _lib
from ._lib import BF16, F32, AttnArgs, SimtArgs, TcArgs, check, dtype_code, ptr, require_cuda, stream_ptr


def _L():
    return _lib.load()


# ---- layout ---------------------------------------------------------------------------------------
def nchw_to_nhwc(x, out_dtype=torch.float32, pad_to=0, split=False, x1=None):
    """[N,C,H,W] fp32 -> [N,H,W,C] (or [N,H,W,pad_to] with zero channels appended).
    split=True (bf16 output, pad_to >= 2C): channels C..2C-1 hold the bf16 rounding residual x - bf16(x) of channels 0..C-1.
    x1 [N,C1,H,W] fp32: a second source whose channels follow x's (C = C + C1), i.e. the layout change of torch.cat([x, x1], 1)
    in the same pass."""
    require_cuda(x, x1)
    assert x.dtype == torch.float32 and x.is_contiguous()
    N, Cc, H, W = x.shape
    C1 = 0
    if x1 is not None:
        assert x1.dtype == torch.float32 and x1.is_contiguous() and x1.dim() == 4
        assert x1.shape[0] == N and tuple(x1.shape[2:]) == (H, W), "nchw_to_nhwc: x1 %s does not match x %s" % (
            tuple(x1.shape), tuple(x.shape))
        C1 = x1.shape[1]
    Ct = Cc + C1
    Cd = max(Ct, pad_to)
    out = torch.empty((N, H, W, Cd), dtype=out_dtype, device=x.device)
    if split:
        assert out_dtype == torch.bfloat16 and Cd >= 2 * Ct
    if x1 is not None:
        check(_L().sdb_nchw_concat_to_nhwc(ptr(x), Cc, ptr(x1), C1, ptr(out), dtype_code(out_dtype), Cd, int(split), N, H * W,
                                           stream_ptr()), "nchw_concat_to_nhwc")
    elif split:
        check(_L().sdb_nchw_to_nhwc_split(ptr(x), ptr(out), N, Cc, Cd, H * W, stream_ptr()), "nchw_to_nhwc_split")
    else:
        check(_L().sdb_nchw_to_nhwc(ptr(x), ptr(out), dtype_code(out_dtype), N, Cc, Cd, H * W, stream_ptr()), "nchw_to_nhwc")
    return out


def nhwc_to_nchw(x):
    require_cuda(x)
    assert x.dtype == torch.float32 and x.is_contiguous()
    N, H, W, Cc = x.shape
    out = torch.empty((N, Cc, H, W), dtype=torch.float32, device=x.device)
    check(_L().sdb_nhwc_to_nchw(ptr(x), ptr(out), N, Cc, H * W, stream_ptr()), "nhwc_to_nchw")
    return out


# ---- normalisation ----------------------------------------------------------------------------------
_gn_counters = {}
_USE_COLSTATS = os.environ.get("SDB200_COLSTATS", "1") != "0"     # measurement switch


def _gn_ticket_buffer(dev, n):
    """Persistent zeroed ticket counters (one int per sample) for the GroupNorm statistics kernel; the kernel
    leaves them zero again, so one buffer per (device, stream) serves every call."""
    key = (dev.index, torch.cuda.current_stream(dev).cuda_stream)
    buf = _gn_counters.get(key)
    if buf is None or buf.numel() < n:
        buf = torch.zeros(max(n, 1024), dtype=torch.int32, device=dev)
        _gn_counters[key] = buf
    return buf


def groupnorm(x0, gamma, beta, eps, act=0, out_dtype=torch.float32, x1=None, groups=32, exact=False, want_raw=False):
    """GroupNorm(groups) over the channel-concat of x0 (and x1) [N,H,W,C*], optional SiLU.
    want_raw=True also returns the un-normalised bf16 concat (written by the same pass).
    gamma / beta: [C] shared by the batch, or [N, C] per-sample rows (scale_shift_affine)."""
    require_cuda(x0, x1, gamma, beta)
    assert x0.dtype == torch.float32 and x0.is_contiguous()
    N, H, W, C0 = x0.shape
    gbs = 0
    if gamma.dim() == 2:
        assert gamma.shape == beta.shape and gamma.shape[0] == N and gamma.stride(1) == 1 and beta.stride() == gamma.stride()
        gbs = gamma.stride(0)
    C1 = 0
    if x1 is not None:
        assert x1.dtype == torch.float32 and x1.is_contiguous() and x1.shape[:3] == x0.shape[:3]
        C1 = x1.shape[3]
    Ct = C0 + C1
    lib = _L()
    cs0 = getattr(x0, "_sdb_cs", None)
    cs1 = getattr(x1, "_sdb_cs", None) if x1 is not None else None
    if cs0 is not None and (x1 is None or cs1 is not None) and _USE_COLSTATS:
        # statistics were produced by the conv(s) that wrote x0 / x1: finalize them and make ONE pass over the tensor
        ws = torch.empty(N * groups * 8 + 256, dtype=torch.uint8, device=x0.device)
        out = torch.empty((N, H, W, Ct), dtype=out_dtype, device=x0.device)
        raw = torch.empty((N, H, W, Ct), dtype=torch.bfloat16, device=x0.device) if want_raw else None
        lay0 = (C.c_longlong * 4)(*cs0[1:5])
        lay1 = (C.c_longlong * 4)(*cs1[1:5]) if cs1 else None
        check(lib.sdb_groupnorm_from_colstats(ptr(x0), C0, ptr(cs0[0]), lay0, ptr(x1), C1, ptr(cs1[0]) if cs1 else 0, lay1,
                                              N, H * W, groups, float(eps), ptr(gamma), ptr(beta), gbs,
                                              int(act), int(bool(exact)), ptr(out), dtype_code(out_dtype), ptr(raw), ptr(ws),
                                              stream_ptr()), "groupnorm_from_colstats")
        return (out, raw) if want_raw else out
    ws_bytes = lib.sdb_groupnorm_ws_bytes(N, H * W, Ct, groups)
    if ws_bytes < 0:
        raise _lib.SdbError("groupnorm: unsupported shape N=%d HW=%d C=%d" % (N, H * W, Ct))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x0.device)
    out = torch.empty((N, H, W, Ct), dtype=out_dtype, device=x0.device)
    raw = torch.empty((N, H, W, Ct), dtype=torch.bfloat16, device=x0.device) if want_raw else None
    check(lib.sdb_groupnorm_nhwc(ptr(x0), C0, ptr(x1), C1, N, H * W, groups, float(eps), ptr(gamma), ptr(beta), gbs,
                                 int(act), int(bool(exact)), ptr(out), dtype_code(out_dtype), ptr(raw), ptr(ws),
                                 ptr(_gn_ticket_buffer(x0.device, N)), stream_ptr()),
          "groupnorm")
    return (out, raw) if want_raw else out


def scale_shift_affine(gamma, beta, ss):
    """Per-sample GroupNorm affine rows for `norm(h) * (1 + scale) + shift` (openai_model/model.py:244-248):
    ss [N, 2C] fp32 (any row stride) = (scale | shift) -> (gamma * (1 + scale), beta * (1 + scale) + shift), each [N, C]."""
    require_cuda(gamma, beta, ss)
    N, C2 = ss.shape
    Cc = C2 // 2
    assert ss.dtype == torch.float32 and ss.stride(1) == 1 and gamma.numel() == Cc
    go = torch.empty((N, Cc), dtype=torch.float32, device=ss.device)
    bo = torch.empty((N, Cc), dtype=torch.float32, device=ss.device)
    check(_L().sdb_scale_shift_affine(ptr(gamma), ptr(beta), ptr(ss), ss.stride(0), N, Cc, ptr(go), ptr(bo), stream_ptr()),
          "scale_shift_affine")
    return go, bo


def avgpool2x2(x, out_dtype=torch.float32):
    """x [N,H,W,C] fp32 -> [N,H/2,W/2,C]: avg_pool2d(kernel 2, stride 2) (openai_model/model.py:88-93)."""
    require_cuda(x)
    assert x.dtype == torch.float32 and x.is_contiguous()
    N, H, W, Cc = x.shape
    out = torch.empty((N, H // 2, W // 2, Cc), dtype=out_dtype, device=x.device)
    check(_L().sdb_avgpool2x2(ptr(x), N, H, W, Cc, ptr(out), dtype_code(out_dtype), stream_ptr()), "avgpool2x2")
    return out


def layernorm(x, gamma, beta, eps=1e-5, out_dtype=torch.float32):
    """LayerNorm over the last dim of x [..., C] fp32."""
    require_cuda(x, gamma, beta)
    assert x.dtype == torch.float32 and x.is_contiguous()
    Cc = x.shape[-1]
    rows = x.numel() // Cc
    out = torch.empty(x.shape, dtype=out_dtype, device=x.device)
    check(_L().sdb_layernorm(ptr(x), rows, Cc, float(eps), ptr(gamma), ptr(beta), ptr(out), dtype_code(out_dtype), stream_ptr()),
          "layernorm")
    return out


# ---- elementwise ------------------------------------------------------------------------------------
def cast_concat(x0, x1=None, up=1, out_dtype=torch.bfloat16):
    require_cuda(x0, x1)
    assert x0.dtype == torch.float32 and x0.is_contiguous()
    N, H, W, C0 = x0.shape
    C1 = 0 if x1 is None else x1.shape[3]
    out = torch.empty((N, H * up, W * up, C0 + C1), dtype=out_dtype, device=x0.device)
    check(_L().sdb_cast_concat(ptr(x0), C0, ptr(x1), C1, N, H, W, up, ptr(out), dtype_code(out_dtype), stream_ptr()),
          "cast_concat")
    return out


def upsample_bilinear2x(x, out_dtype=torch.float32):
    require_cuda(x)
    assert x.dtype == torch.float32 and x.is_contiguous()
    N, H, W, Cc = x.shape
    out = torch.empty((N, 2 * H, 2 * W, Cc), dtype=out_dtype, device=x.device)
    check(_L().sdb_upsample_bilinear2x(ptr(x), N, H, W, Cc, ptr(out), dtype_code(out_dtype), stream_ptr()), "upsample_bilinear2x")
    return out


def activation(x, act, out_dtype=torch.float32):
    require_cuda(x)
    assert x.dtype == torch.float32 and x.is_contiguous()
    out = torch.empty(x.shape, dtype=out_dtype, device=x.device)
    check(_L().sdb_activation(ptr(x), ptr(out), dtype_code(out_dtype), x.numel(), act, stream_ptr()), "activation")
    return out


def geglu(h, out_dtype=torch.float32):
    require_cuda(h)
    assert h.dtype == torch.float32 and h.is_contiguous()
    inner = h.shape[-1] // 2
    rows = h.numel() // h.shape[-1]
    out = torch.empty(h.shape[:-1] + (inner,), dtype=out_dtype, device=h.device)
    check(_L().sdb_geglu(ptr(h), rows, inner, ptr(out), dtype_code(out_dtype), stream_ptr()), "geglu")
    return out


def softmax_rows(s, scale, out_dtype=torch.float32):
    """softmax(scale * s) over the last dim; s fp32 contiguous."""
    require_cuda(s)
    assert s.dtype == torch.float32 and s.is_contiguous()
    Lk = s.shape[-1]
    rows = s.numel() // Lk
    out = torch.empty(s.shape, dtype=out_dtype, device=s.device)
    check(_L().sdb_softmax_rows(ptr(s), rows, Lk, Lk, float(scale), ptr(out), dtype_code(out_dtype), Lk, stream_ptr()), "softmax_rows")
    return out


def softmax_rows_causal(s, scale, Sq, out_dtype=torch.float32):
    """softmax(scale * s) over the last dim with a causal mask: row r is query r % Sq and sees keys 0 .. r % Sq."""
    require_cuda(s)
    assert s.dtype == torch.float32 and s.is_contiguous()
    Lk = s.shape[-1]
    rows = s.numel() // Lk
    out = torch.empty(s.shape, dtype=out_dtype, device=s.device)
    check(_L().sdb_softmax_rows_causal(ptr(s), rows, Lk, int(Sq), Lk, float(scale), ptr(out), dtype_code(out_dtype), Lk, stream_ptr()),
          "softmax_rows_causal")
    return out


def add(a, b):
    require_cuda(a, b)
    assert a.dtype == b.dtype == torch.float32 and a.shape == b.shape and a.is_contiguous() and b.is_contiguous()
    out = torch.empty_like(a)
    check(_L().sdb_add(ptr(a), ptr(b), ptr(out), a.numel(), stream_ptr()), "add")
    return out


def add_rowvec(x, rowvec, out_dtype=torch.float32):
    """x [N,H,W,C] fp32 + rowvec [N,C] (row stride = rowvec.stride(0)) broadcast over pixels."""
    require_cuda(x, rowvec)
    assert x.dtype == torch.float32 and x.is_contiguous() and rowvec.dtype == torch.float32 and rowvec.stride(1) == 1
    N, H, W, Cc = x.shape
    out = torch.empty(x.shape, dtype=out_dtype, device=x.device)
    check(_L().sdb_add_rowvec(ptr(x), ptr(rowvec), rowvec.stride(0), N, H * W, Cc, ptr(out), dtype_code(out_dtype), stream_ptr()),
          "add_rowvec")
    return out


def timestep_embedding(t, freqs, round_fp16=True):
    """t fp32 [B], freqs fp32 [half] -> [B, 2*half] = [cos | sin] (optionally rounded through fp16)."""
    require_cuda(t, freqs)
    assert t.dtype == torch.float32 and freqs.dtype == torch.float32
    B, half = t.shape[0], freqs.shape[0]
    emb = torch.empty((B, 2 * half), dtype=torch.float32, device=t.device)
    check(_L().sdb_timestep_embedding(ptr(t), ptr(freqs), B, half, int(bool(round_fp16)), ptr(emb), stream_ptr()), "timestep_embedding")
    return emb


def gather_rows(table, idx):
    require_cuda(table, idx)
    assert table.dtype == torch.float32 and idx.dtype == torch.int64 and table.is_contiguous()
    B, dim = idx.shape[0], table.shape[1]
    out = torch.empty((B, dim), dtype=torch.float32, device=table.device)
    check(_L().sdb_gather_rows(ptr(table), ptr(idx), B, dim, ptr(out), stream_ptr()), "gather_rows")
    return out


def skinny_linear(x, W, bias=None, act_in=0, act_out=0):
    """y = act_out(act_in(x) @ W^T + bias); x fp32 [M<=32, K], W fp32 or bf16 [N, K] (fp32 accumulation either way)."""
    require_cuda(x, W, bias)
    assert x.dtype == torch.float32 and W.dtype in (torch.float32, torch.bfloat16) and x.is_contiguous() and W.is_contiguous()
    M, K = x.shape
    N = W.shape[0]
    y = torch.empty((M, N), dtype=torch.float32, device=x.device)
    fn = _L().sdb_skinny_linear if W.dtype == torch.float32 else _L().sdb_skinny_linear_bf16w
    for i in range(0, M, 32):   # the kernel holds at most 32 rows in shared memory
        m = min(32, M - i)
        check(fn(ptr(x) + 4 * i * K, m, K, ptr(W), ptr(bias), N, act_in, act_out, ptr(y) + 4 * i * N, stream_ptr()), "skinny_linear")
    return y


def _f32c(name, t, like=None):
    if t is None:
        return
    if t.dtype != torch.float32 or not t.is_contiguous():
        raise _lib.SdbError("%s must be a contiguous fp32 tensor (got %s, contiguous=%s)" % (name, t.dtype, t.is_contiguous()))
    if like is not None and t.numel() != like.numel():
        raise _lib.SdbError("%s has %d elements, expected %d" % (name, t.numel(), like.numel()))


def ddim_step(x, e_cond, sqrt_at, sqrt_aprev, dir_coef, sigma_t, sqrt_one_minus_at, e_uncond=None, cfg_scale=1.0,
              noise=None, temperature=1.0):
    """One fused DDIM update; the five scalars are the fp32 per-step coefficients (see DDIMSampler.derived_coefficients).
    Every tensor operand must be contiguous fp32 with x's element count (the kernel reads n fp32 values from each)."""
    require_cuda(x, e_cond, e_uncond, noise)
    _f32c("x", x)
    _f32c("e_cond", e_cond, x)
    _f32c("e_uncond", e_uncond, x)
    _f32c("noise", noise, x)
    x_prev = torch.empty_like(x)
    pred_x0 = torch.empty_like(x)
    check(_L().sdb_ddim_step(ptr(x), ptr(e_cond), ptr(e_uncond), float(cfg_scale), ptr(noise), float(sqrt_at), float(sqrt_aprev),
                             float(dir_coef), float(sigma_t), float(sqrt_one_minus_at), float(temperature), ptr(x_prev),
                             ptr(pred_x0), x.numel(), stream_ptr()), "ddim_step")
    return x_prev, pred_x0


def ddim_xprev(pred_x0, e_cond, sqrt_aprev, dir_coef, sigma_t, e_uncond=None, cfg_scale=1.0, noise=None, temperature=1.0):
    """x_prev from a GIVEN pred_x0 (quantize_denoised branch of p_sample_ddim, ldm/diffusion/ddim.py:198-205)."""
    require_cuda(pred_x0, e_cond, e_uncond, noise)
    _f32c("pred_x0", pred_x0)
    _f32c("e_cond", e_cond, pred_x0)
    _f32c("e_uncond", e_uncond, pred_x0)
    _f32c("noise", noise, pred_x0)
    x_prev = torch.empty_like(pred_x0)
    check(_L().sdb_ddim_xprev(ptr(pred_x0), ptr(e_cond), ptr(e_uncond), float(cfg_scale), ptr(noise), float(sqrt_aprev),
                              float(dir_coef), float(sigma_t), float(temperature), ptr(x_prev), pred_x0.numel(), stream_ptr()),
          "ddim_xprev")
    return x_prev


def ddpm_step(x, t, table, eps=None, x0=None, noise=None, clip=False, temperature=1.0, want_x_prev=True, want_x0=False):
    """One fused ancestral update (LatentDiffusion.p_sample arithmetic, see include/sdb200.h sdb_ddpm_step).
    x / eps / x0 / noise: contiguous fp32 [B, ...] with x's element count; t: int64 [B] on the device; table: fp32 [5, T]
    (LatentDiffusion.ddpm_table).  x0 given replaces predict_start_from_noise (eps is then unused).  noise None: x_prev is
    the posterior mean.  Returns (x_prev or None, x0 or None)."""
    require_cuda(x, t, table, eps, x0, noise)
    _f32c("x", x)
    _f32c("eps", eps, x)
    _f32c("x0", x0, x)
    _f32c("noise", noise, x)
    _f32c("table", table)
    B = x.shape[0]
    if t.dtype != torch.int64 or t.numel() != B or not t.is_contiguous():
        raise _lib.SdbError("t must be a contiguous int64 tensor of %d timesteps (got %s %s)" % (B, t.dtype, tuple(t.shape)))
    if table.dim() != 2 or table.shape[0] != 5:
        raise _lib.SdbError("table must be [5, T] (got %s)" % (tuple(table.shape),))
    x_prev = torch.empty_like(x) if want_x_prev else None
    x0_out = torch.empty_like(x) if want_x0 else None
    check(_L().sdb_ddpm_step(ptr(x), ptr(eps), ptr(x0), ptr(noise), ptr(t), ptr(table), table.shape[1], int(bool(clip)),
                             float(temperature), ptr(x_prev), ptr(x0_out), B, x.numel() // B if B else 0, stream_ptr()), "ddpm_step")
    return x_prev, x0_out


def inpaint_blend(x0, noise, a, c, mask, img):
    """(a[b]*x0 + c[b]*noise) * mask + (1 - mask) * img: q_sample + the mask blend of ddim_sampling in one kernel
    (ldm/diffusion/ddim.py:144-149, ldm/diffusion/ddpm.py:407-412).  x0 / noise / img [B,C,H,W]; mask [B,1,H,W] or [B,C,H,W]."""
    require_cuda(x0, noise, a, c, mask, img)
    _f32c("x0", x0)
    _f32c("noise", noise, x0)
    _f32c("img", img, x0)
    _f32c("a", a)
    _f32c("c", c)
    _f32c("mask", mask)
    B, Cc = x0.shape[0], x0.shape[1]
    HW = x0.numel() // (B * Cc)
    Cm = mask.numel() // (B * HW)
    if a.numel() != B or c.numel() != B or Cm * B * HW != mask.numel() or Cm not in (1, Cc):
        raise _lib.SdbError("inpaint_blend: mask %s does not broadcast over x0 %s" % (tuple(mask.shape), tuple(x0.shape)))
    out = torch.empty_like(x0)
    check(_L().sdb_inpaint_blend(ptr(x0), ptr(noise), ptr(a), ptr(c), ptr(mask), ptr(img), B, Cc, Cm, HW, ptr(out), stream_ptr()),
          "inpaint_blend")
    return out


# ---- vector quantisation ------------------------------------------------------------------------------
_LAYOUTS = {"nchw": 0, "nhwc": 1}


def vq_quantize(z, codebook, beta=0.25, z_layout="nchw", zq_layout="nchw", want_zq=True, want_idx=True, want_loss=True):
    """VectorQuantizer2.forward arithmetic (see include/sdb200.h sdb_vq_quantize) on contiguous fp32 tensors.
    z [N,D,H,W] ("nchw") or [N,H,W,D] ("nhwc"); codebook [n_e, D].  Returns (z_q in zq_layout, idx int64 [N*H*W] in
    (n, h, w) order, loss fp32 0-d tensor), each None when not wanted."""
    require_cuda(z, codebook)
    _f32c("z", z)
    _f32c("codebook", codebook)
    if z_layout not in _LAYOUTS or zq_layout not in _LAYOUTS:
        raise _lib.SdbError("vq_quantize: layouts are 'nchw' or 'nhwc' (got %r, %r)" % (z_layout, zq_layout))
    if z.dim() != 4 or codebook.dim() != 2:
        raise _lib.SdbError("vq_quantize: z must be 4-d and the codebook [n_e, D] (got %s, %s)"
                            % (tuple(z.shape), tuple(codebook.shape)))
    if z_layout == "nchw":
        N, D, H, W_ = z.shape
    else:
        N, H, W_, D = z.shape
    n_e = codebook.shape[0]
    if codebook.shape[1] != D:
        raise _lib.SdbError("vq_quantize: codebook %s does not match D=%d of z" % (tuple(codebook.shape), D))
    M = N * H * W_
    lib = _L()
    ws_bytes = lib.sdb_vq_ws_bytes(M, n_e)
    if ws_bytes < 0:
        raise _lib.SdbError("vq_quantize: unsupported shape M=%d n_e=%d" % (M, n_e))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=z.device)
    zq = None
    if want_zq:
        zq = torch.empty((N, D, H, W_) if zq_layout == "nchw" else (N, H, W_, D), dtype=torch.float32, device=z.device)
    idx = torch.empty(M, dtype=torch.int64, device=z.device) if want_idx else None
    loss = torch.empty((), dtype=torch.float32, device=z.device) if want_loss else None
    # the GroupNorm kernels' ticket counters: zero between launches, so one buffer per stream serves both
    counters = _gn_ticket_buffer(z.device, 1) if want_loss else None
    check(lib.sdb_vq_quantize(ptr(z), _LAYOUTS[z_layout], N, H * W_, D, ptr(codebook), n_e, float(beta), ptr(zq),
                              _LAYOUTS[zq_layout], ptr(idx), ptr(loss), ptr(ws), ptr(counters), stream_ptr()), "vq_quantize")
    return zq, idx, loss


def vq_codebook_gather(idx, codebook, shape, out_layout="nchw"):
    """codebook[idx] as an fp32 image: idx int64 with N*H*W entries in (n, h, w) order, shape = (N, H, W) ->
    [N,D,H,W] ("nchw") or [N,H,W,D] ("nhwc").  Out-of-range indices give NaN rows."""
    require_cuda(idx, codebook)
    _f32c("codebook", codebook)
    N, H, W_ = (int(s) for s in shape)
    if idx.dtype != torch.int64 or not idx.is_contiguous() or idx.numel() != N * H * W_:
        raise _lib.SdbError("vq_codebook_gather: idx must be a contiguous int64 tensor of %d indices (got %s %s)"
                            % (N * H * W_, idx.dtype, tuple(idx.shape)))
    if out_layout not in _LAYOUTS:
        raise _lib.SdbError("vq_codebook_gather: layouts are 'nchw' or 'nhwc' (got %r)" % (out_layout,))
    n_e, D = codebook.shape
    out = torch.empty((N, D, H, W_) if out_layout == "nchw" else (N, H, W_, D), dtype=torch.float32, device=codebook.device)
    check(_L().sdb_vq_codebook_gather(ptr(idx), idx.numel(), ptr(codebook), n_e, D, ptr(out), _LAYOUTS[out_layout], H * W_,
                                      stream_ptr()), "vq_codebook_gather")
    return out


# ---- patch-distributed fold / unfold (LatentDiffusion.split_input_params) -----------------------------------------------
def patch_grid(h, w, ks, stride):
    """(Ly, Lx): the crops of ks at `stride` that fit in h x w, as torch.nn.Unfold counts them."""
    return (h - ks[0]) // stride[0] + 1, (w - ks[1]) // stride[1] + 1


def patch_unfold(x, ks, stride):
    """x [B,C,H,W] -> its Ly*Lx crops of ks at `stride` as one batch [L*B, C, ks[0], ks[1]] fp32, crop-major (row l*B + b):
    unfold(x).view(B, C, *ks, L)[..., l] for every l, a pure copy (see include/sdb200.h sdb_patch_unfold)."""
    require_cuda(x)
    xf = x.float().contiguous()
    if xf.dim() != 4:
        raise _lib.SdbError("patch_unfold: x must be 4-d (got %s)" % (tuple(x.shape),))
    B, C, H, W_ = xf.shape
    Ly, Lx = patch_grid(H, W_, ks, stride)
    out = torch.empty((max(Ly * Lx, 0) * B, C, ks[0], ks[1]), dtype=torch.float32, device=x.device)
    check(_L().sdb_patch_unfold(ptr(xf), B, C, H, W_, int(ks[0]), int(ks[1]), int(stride[0]), int(stride[1]), ptr(out),
                                stream_ptr()), "patch_unfold")
    return out


def patch_fold(o, B, grid, stride, out_hw, wpix, wcrop=None):
    """Crops o [L*B, C, KH, KW] (crop-major) of a Ly x Lx `grid` at `stride` -> fold(o * w) / fold(w) as [B, C, *out_hw] fp32,
    w = wpix [KH*KW] per pixel, times wcrop [L] per crop when given (see include/sdb200.h sdb_patch_fold)."""
    require_cuda(o, wpix, wcrop)
    _f32c("o", o)
    _f32c("wpix", wpix)
    _f32c("wcrop", wcrop)
    if o.dim() != 4 or o.shape[0] % B or wpix.numel() != o.shape[2] * o.shape[3]:
        raise _lib.SdbError("patch_fold: crops %s do not match B=%d and a weight table of %d" % (tuple(o.shape), B, wpix.numel()))
    _, C, KH, KW = o.shape
    Ly, Lx = grid
    L = o.shape[0] // B
    if wcrop is not None and wcrop.numel() != L:
        raise _lib.SdbError("patch_fold: %d crop weights for %d crops" % (wcrop.numel(), L))
    out = torch.empty((B, C, out_hw[0], out_hw[1]), dtype=torch.float32, device=o.device)
    check(_L().sdb_patch_fold(ptr(o), B, C, KH, KW, int(Ly), int(Lx), int(stride[0]), int(stride[1]), int(out_hw[0]),
                              int(out_hw[1]), ptr(wpix), ptr(wcrop), L, ptr(out), stream_ptr()), "patch_fold")
    return out


def diag_gaussian(moments, noise=None):
    """moments [N,2C,H,W] fp32 -> (mean, logvar, std, var, sample or None), each [N,C,H,W]
    (DiagonalGaussianDistribution, ldm/modules/distributions/distributions.py:24-37)."""
    require_cuda(moments, noise)
    assert moments.dtype == torch.float32 and moments.is_contiguous() and moments.shape[1] % 2 == 0
    N, C2, H, W = moments.shape
    shape = (N, C2 // 2, H, W)
    outs = [torch.empty(shape, dtype=torch.float32, device=moments.device) for _ in range(4)]
    sample = None
    if noise is not None:
        assert noise.dtype == torch.float32 and noise.is_contiguous() and tuple(noise.shape) == shape
        sample = torch.empty(shape, dtype=torch.float32, device=moments.device)
    check(_L().sdb_diag_gaussian(ptr(moments), ptr(noise), N, C2 // 2, H * W, ptr(outs[0]), ptr(outs[1]), ptr(outs[2]),
                                 ptr(outs[3]), ptr(sample), stream_ptr()), "diag_gaussian")
    return outs[0], outs[1], outs[2], outs[3], sample


def q_sample(x0, noise, a, c):
    """out[b] = a[b] * x0[b] + c[b] * noise[b] (fp32; DDIMSampler.stochastic_encode, ldm/diffusion/ddim.py:218-222)."""
    require_cuda(x0, noise, a, c)
    for t in (x0, noise, a, c):
        assert t.dtype == torch.float32 and t.is_contiguous()
    B = x0.shape[0]
    assert noise.shape == x0.shape and a.numel() == B and c.numel() == B
    out = torch.empty_like(x0)
    check(_L().sdb_q_sample(ptr(x0), ptr(noise), ptr(a), ptr(c), B, x0.numel() // B, ptr(out), stream_ptr()), "q_sample")
    return out


# ---- weight packing (host side, once per load) ----------------------------------------------------------
def pack_conv_weight(w, dtype):
    """OIHW [Cout,Cin,kh,kw] -> tap-major [kh*kw, Cout, Cin] contiguous ("RSKC")."""
    Cout, Cin, kh, kw = w.shape
    return w.detach().permute(2, 3, 0, 1).reshape(kh * kw, Cout, Cin).to(dtype).contiguous()


def pack_geglu_weight(w, b, block_n):
    """Interleave value/gate rows per block_n tile: tile t = [value rows t*h..(t+1)*h | gate rows ...], h = block_n/2."""
    two_inner, K = w.shape
    inner = two_inner // 2
    h = block_n // 2
    assert inner % h == 0
    wv, wg = w[:inner].reshape(inner // h, h, K), w[inner:].reshape(inner // h, h, K)
    wp = torch.cat([wv, wg], dim=1).reshape(two_inner, K).contiguous()
    bv, bg = b[:inner].reshape(inner // h, h), b[inner:].reshape(inner // h, h)
    bp = torch.cat([bv, bg], dim=1).reshape(two_inner).contiguous()
    return wp, bp


# ---- fp32 SIMT contraction ----------------------------------------------------------------------------
def conv_simt(x, w_rskc, bias, kh, kw, stride=1, pad=0, up=1, rowvec=None, residual=None, out_dtype=torch.float32, pad_hi=None):
    """x [N,IH,IW,Cin] fp32 (logical input is the nearest-`up`x upsampling of x), w [kh*kw,Cout,Cin] fp32."""
    require_cuda(x, w_rskc, bias, rowvec, residual)
    assert x.dtype == torch.float32 and w_rskc.dtype == torch.float32 and x.is_contiguous() and w_rskc.is_contiguous()
    N, IH, IW, Cin = x.shape
    taps, Cout, Cin2 = w_rskc.shape
    assert Cin2 == Cin and taps == kh * kw
    pad_hi = pad if pad_hi is None else pad_hi          # bottom/right zero padding (VAE Downsample pads (0,1,0,1))
    OH = (IH * up + pad + pad_hi - kh) // stride + 1
    OW = (IW * up + pad + pad_hi - kw) // stride + 1
    out = torch.empty((N, OH, OW, Cout), dtype=out_dtype, device=x.device)
    a = SimtArgs()
    a.A, a.B, a.out = ptr(x), ptr(w_rskc), ptr(out)
    a.bias, a.rowvec, a.residual = ptr(bias), ptr(rowvec), ptr(residual)
    a.lda, a.ldb, a.ldc = Cin, Cin, Cout
    a.ldr = Cout
    a.ldv = rowvec.stride(0) if rowvec is not None else 0
    a.M, a.N, a.K = N * OH * OW, Cout, taps * Cin
    a.alpha = 1.0
    a.b_kn = 0
    a.nb1 = a.nb2 = 1
    a.kh, a.kw, a.stride, a.pad, a.up = kh, kw, stride, pad, up
    a.NB, a.IH, a.IW, a.Cin, a.OH, a.OW = N, IH, IW, Cin, OH, OW
    a.out_dtype = dtype_code(out_dtype)
    if residual is not None:
        assert residual.dtype == torch.float32 and residual.shape == out.shape and residual.is_contiguous()
    check(_L().sdb_simt_contract(C.byref(a), stream_ptr()), "simt conv")
    return out


def gemm_simt(A, B, bias=None, residual=None, alpha=1.0, b_kn=False, out=None, out_dtype=torch.float32,
              M=None, N=None, K=None, lda=None, ldb=None, ldc=None, batch=(1, 1),
              sa=(0, 0), sb=(0, 0), sc=(0, 0)):
    """out[M,N] = alpha * A[M,K] @ (B[N,K]^T or B[K,N]) + bias + residual, two-level batched, explicit strides."""
    require_cuda(A, B, bias, residual, out)
    assert A.dtype == torch.float32 and B.dtype == torch.float32
    if M is None:
        M, K = A.shape[-2], A.shape[-1]
        N = B.shape[-1] if b_kn else B.shape[-2]
    lda = lda if lda is not None else A.stride(-2)
    ldb = ldb if ldb is not None else B.stride(-2)
    if out is None:
        out = torch.empty((M, N), dtype=out_dtype, device=A.device)
    ldc = ldc if ldc is not None else out.stride(-2)
    a = SimtArgs()
    a.A, a.B, a.out = ptr(A), ptr(B), ptr(out)
    a.bias, a.rowvec, a.residual = ptr(bias), 0, ptr(residual)
    a.lda, a.ldb, a.ldc = lda, ldb, ldc
    a.ldr = residual.stride(-2) if residual is not None else 0
    a.ldv = 0
    a.M, a.N, a.K = M, N, K
    a.alpha = float(alpha)
    a.b_kn = int(bool(b_kn))
    a.nb1, a.nb2 = batch
    a.sa1, a.sa2 = sa
    a.sb1, a.sb2 = sb
    a.sc1, a.sc2 = sc
    a.kh = 0
    a.out_dtype = dtype_code(out.dtype)
    check(_L().sdb_simt_contract(C.byref(a), stream_ptr()), "simt gemm")
    return out


# ---- tcgen05 contraction -----------------------------------------------------------------------------
def _plan_table():
    if os.environ.get("SDB200_TC_PLANS", "1") == "0":
        return {}
    from .tc_plans import PLANS
    return PLANS


_PLANS = None


def _apply_plan(a, kind, rows_per_sample):
    """Fill (variant, block_n, split_k) from the measured plan table when the caller left all three on auto.
    Keyed by the per-sample geometry only, so the plan (and a sample's bits) is independent of the batch size."""
    global _PLANS
    if a.split_k or a.variant or (a.block_n and not a.geglu):
        return
    if _PLANS is None:
        _PLANS = _plan_table()
    key = (kind, int(rows_per_sample), a.N, a.K, a.taps, a.stride if a.taps else 0, a.geglu, int(bool(a.residual)),
           a.out_dtype, a.col_group)
    hit = _PLANS.get(key)
    if hit is not None:
        if a.geglu:                      # the tile width is baked into the packed GEGLU weights
            if hit[1] == a.block_n:
                a.variant = hit[0]
        else:
            a.variant, a.block_n, a.split_k = hit[0], hit[1], hit[2]


def _tc_launch(a, what):
    """Give the call its split-K workspace (if the plan splits) and enqueue it."""
    lib = _L()
    need = lib.sdb_tc_workspace_bytes(C.byref(a))
    if need < 0:
        check(-1, what)
    ws = None
    if need > 0:
        ws = torch.empty(need, dtype=torch.uint8, device=torch.device("cuda", torch.cuda.current_device()))
        a.ws, a.ws_bytes = ws.data_ptr(), need
    check(lib.sdb_tc_contract(C.byref(a), stream_ptr()), what)


def conv_tc(x, w_rskc, bias, kh, kw, stride=1, pad=0, rowvec=None, residual=None, out_dtype=torch.float32,
            split_k=0, block_n=0, out=None, phase=None, variant=0, want_stats=False, stats_into=None, pad_hi=None, b_const=False):
    """x [N,IH,IW,Cin] bf16, w [kh*kw,Cout,Cin] bf16 -> [N,OH,OW,Cout].

    phase=(sh, sw, oh, ow, OHF, OWF, pad_h, pad_w) writes this conv's OHxOW result into the strided
    sub-lattice of a larger [N,OHF,OWF,Cout] `out` (sub-pixel decomposition of upsample+conv).
    """
    require_cuda(x, w_rskc, bias, rowvec, residual, out)
    assert x.dtype == torch.bfloat16 and w_rskc.dtype == torch.bfloat16 and x.is_contiguous() and w_rskc.is_contiguous()
    N, IH, IW, Cin = x.shape
    taps, Cout, Cin2 = w_rskc.shape
    assert Cin2 == Cin and taps == kh * kw
    a = TcArgs()
    if phase is None:
        pad_hi = pad if pad_hi is None else pad_hi      # bottom/right padding: TMA zero-fills whatever lies past the image
        OH = (IH + pad + pad_hi - kh) // stride + 1
        OW = (IW + pad + pad_hi - kw) // stride + 1
        pad_h = pad_w = pad
        if out is None:
            out = torch.empty((N, OH, OW, Cout), dtype=out_dtype, device=x.device)
        a.out_sh = a.out_sw = 1
        a.out_oh = a.out_ow = 0
        a.OHF, a.OWF = OH, OW
    else:
        sh, sw, o_h, o_w, OHF, OWF, pad_h, pad_w = phase
        OH, OW = IH, IW
        assert out is not None and tuple(out.shape) == (N, OHF, OWF, Cout)
        a.out_sh, a.out_sw, a.out_oh, a.out_ow, a.OHF, a.OWF = sh, sw, o_h, o_w, OHF, OWF
    a.A, a.B, a.out = ptr(x), ptr(w_rskc), ptr(out)
    a.bias, a.rowvec, a.residual = ptr(bias), ptr(rowvec), ptr(residual)
    a.lda, a.ldb, a.ldc = Cin, Cin, Cout
    a.ldr = Cout
    a.ldv = rowvec.stride(0) if rowvec is not None else 0
    a.M, a.N, a.K = N * OH * OW, Cout, taps * Cin
    a.out_dtype = dtype_code(out.dtype)
    a.geglu = 0
    a.col_group = a.col_group_stride = 0
    a.split_k = split_k
    a.block_n = block_n
    a.variant = variant
    a.taps, a.kw, a.stride, a.pad_h, a.pad_w = taps, kw, stride, pad_h, pad_w
    a.NB, a.IH, a.IW, a.Cin, a.OH, a.OW = N, IH, IW, Cin, OH, OW
    a.cout_pad = Cout
    a.b_const = int(bool(b_const))        # weights written by no earlier launch of the stream: fetched before the PDL wait
    if residual is not None:
        assert residual.dtype == torch.float32 and residual.is_contiguous()
    _apply_plan(a, "conv", OH * OW)
    cs = None
    if stats_into is not None:
        # one phase of an upsampling conv: its slot region inside the caller's statistics buffer (see conv_up2_tc)
        cs_t, total_slots, first_slot = stats_into
        a.colstats, a.colstats_slots = cs_t.data_ptr() + 4 * first_slot * Cout, total_slots
    elif want_stats and phase is None and out.dtype == torch.float32:
        # per-(32-row slot, channel) sums of the stored values, written by the epilogue: the statistics pass of the
        # GroupNorm that reads `out` next (ops.groupnorm picks them up from the tensor)
        slots, spi = tc_colstats_layout(a)
        if slots > 0:
            cs = torch.empty((2, slots, Cout), dtype=torch.float32, device=x.device)
            a.colstats, a.colstats_slots = cs.data_ptr(), slots
    _tc_launch(a, "tc conv")
    if cs is not None:
        out._sdb_cs = (cs, slots, spi, 1, 0)          # (buffer, slots, slots per sample, regions, region stride)
    return out


def tc_colstats_layout(a):
    slots, spi = C.c_longlong(0), C.c_longlong(0)
    check(_L().sdb_tc_colstats_layout(C.byref(a), C.byref(slots), C.byref(spi)), "tc colstats layout")
    return slots.value, spi.value


UP2_PHASES = ((0, 0), (0, 1), (1, 0), (1, 1))


def fold_upsample_weights(w, dtype):
    """Nearest-2x upsampling followed by a 3x3 / pad 1 conv (openai_model/model.py:119-131; ldm/.../model.py:44-59) equals,
    for each output phase (py, px), a 2x2 conv over the LOW-resolution input whose taps are sums of the 3x3 taps that land
    on the same source pixel: 4/9 of the multiply-adds and no 4x intermediate.  w [Cout,Cin,3,3] -> 4 x [4, Cout, Cin]."""
    rows = {0: ((0,), (1, 2)), 1: ((0, 1), (2,))}      # phase -> 3x3 taps hitting source offset (-1 + phase) and (0 + phase)
    wf = w.detach().float()
    out = []
    for py, px in UP2_PHASES:
        taps = []
        for a_ in (0, 1):
            for b_ in (0, 1):
                acc = None
                for ky in rows[py][a_]:
                    for kx in rows[px][b_]:
                        acc = wf[:, :, ky, kx] if acc is None else acc + wf[:, :, ky, kx]
                taps.append(acc)
        out.append(torch.stack(taps, 0).to(dtype).contiguous())
    return out


def conv_up2_tc(x, w_phases, bias, want_stats=False, b_const=False):
    """conv3x3(pad 1) of the nearest-2x upsampling of x [N,H,W,Cin] bf16 as four sub-pixel 2x2 convs -> [N,2H,2W,Cout] fp32."""
    require_cuda(x, bias)
    N, H, W, Cin = x.shape
    Cout = w_phases[0].shape[1]
    out = torch.empty((N, 2 * H, 2 * W, Cout), dtype=torch.float32, device=x.device)
    cs = None
    for p, (py, px) in enumerate(UP2_PHASES):
        ph = (2, 2, py, px, 2 * H, 2 * W, 1 - py, 1 - px)
        if want_stats and p == 0:
            # probe the layout of one phase (all four share it), then give each phase its own slot region
            probe = TcArgs()
            _fill_conv_args(probe, x, w_phases[0], bias, out, 2, 2, 1, ph)
            _apply_plan(probe, "conv", H * W)
            slots, spi = tc_colstats_layout(probe)
            if slots > 0:
                cs = torch.empty((2, 4 * slots, Cout), dtype=torch.float32, device=x.device)
        conv_tc(x, w_phases[p], bias, 2, 2, stride=1, pad=0, out=out, phase=ph, b_const=b_const,
                stats_into=(cs, 4 * slots, p * slots) if cs is not None else None)
    if cs is not None:
        out._sdb_cs = (cs, 4 * slots, spi, 4, slots)
    return out


def _fill_conv_args(a, x, w_rskc, bias, out, kh, kw, stride, phase):
    """Geometry part of conv_tc's argument block (enough for plan / layout queries)."""
    N, IH, IW, Cin = x.shape
    taps, Cout, _ = w_rskc.shape
    sh, sw, o_h, o_w, OHF, OWF, pad_h, pad_w = phase
    a.out_sh, a.out_sw, a.out_oh, a.out_ow, a.OHF, a.OWF = sh, sw, o_h, o_w, OHF, OWF
    a.A, a.B, a.out = ptr(x), ptr(w_rskc), ptr(out)
    a.bias = ptr(bias)
    a.lda, a.ldb, a.ldc, a.ldr = Cin, Cin, Cout, Cout
    a.M, a.N, a.K = N * IH * IW, Cout, taps * Cin
    a.out_dtype = dtype_code(out.dtype)
    a.taps, a.kw, a.stride, a.pad_h, a.pad_w = taps, kw, stride, pad_h, pad_w
    a.NB, a.IH, a.IW, a.Cin, a.OH, a.OW = N, IH, IW, Cin, IH, IW
    a.cout_pad = Cout


def gemm_tc(A, W, bias=None, residual=None, out_dtype=torch.float32, geglu=False, col_group=0, col_group_stride=0,
            split_k=0, block_n=0, out=None, ldc=None, M=None, lda=None, rows_per_item=0, variant=0, b_const=False):
    """out[M,N] = A[M,K] @ W[N,K]^T + bias + residual; A, W bf16 (K contiguous)."""
    require_cuda(A, W, bias, residual, out)
    assert A.dtype == torch.bfloat16 and W.dtype == torch.bfloat16 and W.is_contiguous()
    K = A.shape[-1]
    if M is None:
        M = A.numel() // K
    N = W.shape[0]
    assert W.shape[1] == K
    n_out = N // 2 if geglu else N
    if out is None:
        width = (N // col_group) * col_group_stride if col_group else n_out
        if col_group:
            out = torch.zeros((M, width), dtype=out_dtype, device=A.device)   # pad columns must read as 0
        else:
            out = torch.empty((M, width), dtype=out_dtype, device=A.device)
    a = TcArgs()
    a.A, a.B, a.out = ptr(A), ptr(W), ptr(out)
    a.bias, a.rowvec, a.residual = ptr(bias), 0, ptr(residual)
    a.lda = lda if lda is not None else K
    a.ldb = K
    a.ldc = ldc if ldc is not None else out.stride(-2)
    a.ldr = residual.stride(-2) if residual is not None else 0
    a.ldv = 0
    a.M, a.N, a.K = M, N, K
    a.out_dtype = dtype_code(out.dtype)
    a.geglu = int(bool(geglu))
    a.col_group, a.col_group_stride = col_group, col_group_stride
    a.split_k = split_k
    a.block_n = block_n
    a.variant = variant
    a.taps = 0
    a.rows_per_item = int(rows_per_item)
    a.b_const = int(bool(b_const))        # W written by no earlier launch of the stream: fetched before the PDL wait
    if rows_per_item:
        _apply_plan(a, "gemm", rows_per_item)
    _tc_launch(a, "tc gemm")
    return out


def attention_tc(q, k, v, B, H, Sq, Sk, d, dpad, scale, q_strides, k_strides, v_strides, out=None, o_strides=None, dense=False,
                 causal=False):
    """q/k/v: bf16 tensors (any views) whose (batch, seq, head) element strides are given; heads stored padded to dpad
    channels, or (dense=True) with their d channels only.
    Returns out [B, Sq, H*d] bf16; o_strides = (batch, seq, head) element strides of another output layout."""
    require_cuda(q, k, v)
    assert q.dtype == k.dtype == v.dtype == torch.bfloat16
    if out is None:
        out = torch.empty((B, Sq, H * d), dtype=torch.bfloat16, device=q.device)
    a = AttnArgs()
    a.q, a.k, a.v, a.out = ptr(q), ptr(k), ptr(v), ptr(out)
    a.q_bs, a.q_ss, a.q_hs = q_strides
    a.k_bs, a.k_ss, a.k_hs = k_strides
    a.v_bs, a.v_ss, a.v_hs = v_strides
    a.o_bs, a.o_ss, a.o_hs = o_strides if o_strides is not None else (Sq * H * d, H * d, d)
    a.B, a.H, a.Sq, a.Sk, a.d, a.dpad = B, H, Sq, Sk, d, dpad
    a.scale = float(scale)
    a.dense = int(bool(dense))
    a.causal = int(bool(causal))
    check(_L().sdb_attention_fwd(C.byref(a), stream_ptr()), "attention_fwd")
    return out


def attention_wide(q, k, v, B, Sq, Sk, d, scale, q_strides, k_strides, v_strides, out=None):
    """One wide head (d = 256 / 512, the VAE AttnBlock): q / k / v bf16 views with (batch, seq) element strides, channels
    contiguous.  Returns out [B, Sq, d] bf16."""
    require_cuda(q, k, v, out)
    assert q.dtype == k.dtype == v.dtype == torch.bfloat16
    if out is None:
        out = torch.empty((B, Sq, d), dtype=torch.bfloat16, device=q.device)
    check(_L().sdb_attention_wide_fwd(ptr(q), ptr(k), ptr(v), ptr(out), q_strides[0], q_strides[1], k_strides[0], k_strides[1],
                                      v_strides[0], v_strides[1], Sq * d, d, B, Sq, Sk, d, float(scale), stream_ptr()), "attention_wide_fwd")
    return out
