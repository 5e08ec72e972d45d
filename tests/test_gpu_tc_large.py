"""GPU: the tcgen05 contraction at UNet scale (multi-wave persistent scheduling, every epilogue mode), in BOTH kernel
variants (CTA-pair persistent / one-CTA), against fp32 torch math on the same bf16-rounded operands."""
import pytest
import torch
import torch.nn.functional as F

from gpu_util import nchw, nhwc, randn, rel

pytestmark = pytest.mark.gpu


@pytest.fixture(params=[2, 1], ids=["pair", "single"])
def variant(request, cuda):
    """the sdb_tc_args.variant every call passes: an explicit variant also keeps the measured launch plans (which would
    pick their own kernel) out of the way"""
    return request.param


@pytest.mark.parametrize("N,H,W,Cin,Cout", [(8, 64, 64, 320, 320), (8, 32, 32, 640, 640), (8, 16, 16, 1280, 1280), (8, 8, 8, 1280, 1280),
                                            (3, 40, 24, 128, 256)])
def test_conv_large(variant, N, H, W, Cin, Cout):
    from sdb200 import ops
    x = randn(N, H, W, Cin, seed=1).to(torch.bfloat16)
    w = (randn(Cout, Cin, 3, 3, seed=2) * (Cin * 9) ** -0.5).to(torch.bfloat16)
    b = randn(Cout, seed=3)
    rv = randn(N, 2 * Cout, seed=4)
    res = randn(N, H, W, Cout, seed=5)
    ref = nhwc(F.conv2d(nchw(x.float()), w.float(), b, padding=1)) + rv[:, None, None, Cout:] + res
    out = ops.conv_tc(x, ops.pack_conv_weight(w, torch.bfloat16), b, 3, 3, pad=1, rowvec=rv[:, Cout:], residual=res, variant=variant)
    assert rel(out, ref) < 3e-5
    out_b = ops.conv_tc(x, ops.pack_conv_weight(w, torch.bfloat16), b, 3, 3, pad=1, rowvec=rv[:, Cout:], residual=res,
                        out_dtype=torch.bfloat16, variant=variant)
    assert rel(out_b, ref) < 4e-3


@pytest.mark.parametrize("M,N,K", [(32768, 320, 320), (32768, 320, 1280), (8192, 640, 2560), (2048, 1280, 5120), (616, 640, 768)])
def test_gemm_large(variant, M, N, K):
    from sdb200 import ops
    A = randn(M, K, seed=1).to(torch.bfloat16)
    W = (randn(N, K, seed=2) * K ** -0.5).to(torch.bfloat16)
    bias, res = randn(N, seed=3), randn(M, N, seed=4)
    ref = A.float() @ W.float().T + bias + res
    assert rel(ops.gemm_tc(A, W, bias, residual=res, variant=variant), ref) < 2e-5
    # padded-head bf16 output (q/k/v projections)
    d = N // 8
    dp = (d + 63) // 64 * 64
    pad = ops.gemm_tc(A, W, out_dtype=torch.bfloat16, col_group=d, col_group_stride=dp, variant=variant)
    pv = pad.view(M, 8, dp)
    assert rel(pv[:, :, :d].reshape(M, N), A.float() @ W.float().T) < 4e-3
    assert float(pv[:, :, d:].abs().max()) == 0.0 if dp > d else True


@pytest.mark.parametrize("M,C", [(32768, 320), (8192, 640), (2048, 1280)])
def test_geglu_large(variant, M, C):
    from sdb200 import ops
    from sdb200.engine import PackedLinear
    A = randn(M, C, seed=1).to(torch.bfloat16)
    W = (randn(8 * C, C, seed=2) * C ** -0.5)
    b = randn(8 * C, seed=3)
    pl = PackedLinear(W, b, "bf16", geglu=True)
    h = A.float() @ W.to(torch.bfloat16).float().T + b
    ref = h[:, :4 * C] * F.gelu(h[:, 4 * C:])
    out = ops.gemm_tc(A, pl.w, pl.bias, out_dtype=torch.bfloat16, geglu=True, block_n=pl.block_n, variant=variant)
    assert out.shape == (M, 4 * C)
    assert rel(out, ref) < 4e-3
