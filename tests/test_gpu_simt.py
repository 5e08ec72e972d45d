"""GPU: fp32 SIMT contraction kernel (conv / gemm / batched attention path) vs float64 torch math."""
import pytest
import torch
import torch.nn.functional as F

from gpu_util import nchw, nhwc, randn, rel

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("N,H,W,Cin,Cout,k,stride,pad,up", [
    (2, 16, 16, 64, 96, 3, 1, 1, 1), (1, 9, 7, 4, 320, 3, 1, 1, 1), (2, 8, 8, 3, 128, 3, 1, 1, 1),
    (2, 16, 16, 64, 64, 3, 2, 1, 1), (1, 8, 8, 32, 48, 3, 1, 1, 2), (3, 6, 6, 128, 40, 1, 1, 0, 1),
    (1, 1, 1, 512, 512, 3, 1, 1, 1), (2, 5, 5, 320, 4, 3, 1, 1, 1)])
def test_conv_simt(cuda, N, H, W, Cin, Cout, k, stride, pad, up):
    from sdb200 import ops
    x = randn(N, H, W, Cin, seed=1)
    w = randn(Cout, Cin, k, k, seed=2) * (Cin * k * k) ** -0.5
    b = randn(Cout, seed=3)
    xin = nchw(x).double()
    if up == 2:
        xin = F.interpolate(xin, scale_factor=2, mode="nearest")
    ref = nhwc(F.conv2d(xin, w.double(), b.double(), stride=stride, padding=pad))
    rv = randn(N, Cout + 8, seed=4)
    res = randn(*ref.shape, seed=5)
    out = ops.conv_simt(x, ops.pack_conv_weight(w, torch.float32), b, k, k, stride=stride, pad=pad, up=up)
    assert out.shape == ref.shape and rel(out, ref) < 2e-6
    out2 = ops.conv_simt(x, ops.pack_conv_weight(w, torch.float32), b, k, k, stride=stride, pad=pad, up=up,
                         rowvec=rv[:, 3:3 + Cout], residual=res)
    ref2 = ref + rv[:, None, None, 3:3 + Cout].double() + res.double()
    assert rel(out2, ref2) < 2e-6


@pytest.mark.parametrize("M,N,K", [(128, 64, 64), (77, 320, 768), (1000, 130, 72), (5, 7, 9), (256, 2560, 320)])
def test_gemm_simt(cuda, M, N, K):
    from sdb200 import ops
    A, B, bias, res = randn(M, K, seed=1), randn(N, K, seed=2) * K ** -0.5, randn(N, seed=3), randn(M, N, seed=4)
    ref = A.double() @ B.double().T + bias.double() + res.double()
    assert rel(ops.gemm_simt(A, B, bias, residual=res), ref) < 2e-6
    Bkn = B.T.contiguous()
    assert rel(ops.gemm_simt(A, Bkn, bias, residual=res, b_kn=True), ref) < 2e-6
    assert rel(ops.gemm_simt(A, B, None, alpha=0.5), 0.5 * (A.double() @ B.double().T)) < 2e-6


@pytest.mark.parametrize("B,H,Sq,Sk,d", [(2, 8, 64, 64, 40), (1, 2, 100, 77, 32), (2, 4, 16, 16, 64)])
def test_attention_fp32_row_views(cuda, B, H, Sq, Sk, d):
    from sdb200.engine import attention_fp32
    C = H * d
    q, k, v = randn(B * Sq, C, seed=1), randn(B * Sk, C, seed=2), randn(B * Sk, C, seed=3)
    scale = d ** -0.5
    o = attention_fp32(q, k, v, B, H, Sq, Sk, d, scale)
    qh = q.double().view(B, Sq, H, d).transpose(1, 2)
    kh = k.double().view(B, Sk, H, d).transpose(1, 2)
    vh = v.double().view(B, Sk, H, d).transpose(1, 2)
    ref = (torch.softmax(qh @ kh.transpose(-1, -2) * scale, -1) @ vh).transpose(1, 2).reshape(B * Sq, C)
    assert rel(o, ref) < 2e-6
    # fused-qkv layout (column views of one [rows, 3C] tensor), as the UNet uses it
    qkv = torch.cat([q, q * 0.5 + 1, q * 2 - 1], 1).contiguous() if Sq == Sk else None
    if qkv is not None:
        o2 = attention_fp32(qkv, qkv[:, C:], qkv[:, 2 * C:], B, H, Sq, Sq, d, scale)
        k2, v2 = (q * 0.5 + 1).double().view(B, Sq, H, d).transpose(1, 2), (q * 2 - 1).double().view(B, Sq, H, d).transpose(1, 2)
        s2 = qh @ k2.transpose(-1, -2) * scale
        ref2 = (torch.softmax(s2, -1) @ v2).transpose(1, 2).reshape(B * Sq, C)
        assert rel(o2, ref2) < 2e-6
        # causal (CLIP's text tower): query i sees keys 0 .. i
        o3 = attention_fp32(qkv, qkv[:, C:], qkv[:, 2 * C:], B, H, Sq, Sq, d, scale, causal=True)
        mask = torch.ones(Sq, Sq, dtype=torch.bool, device=q.device).triu(1)
        ref3 = (torch.softmax(s2.masked_fill(mask, float("-inf")), -1) @ v2).transpose(1, 2).reshape(B * Sq, C)
        assert rel(o3, ref3) < 2e-6
