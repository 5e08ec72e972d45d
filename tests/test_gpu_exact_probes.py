"""GPU: exact-arithmetic probes of the tcgen05 contraction, the SIMT contraction and the attention kernels.

The rel-L2 checks of the other kernel tests cannot see an error confined to one tile: one 128-row block of a 32768-row
bf16 output can be 6 % off and still pass 4e-3.  Here the operands are small integers (activations in [-2, 2], weights
in {-1, 0, 1}, bias / time-embedding row / residual in [-4, 4]), so every partial sum is an integer below 2^16 and the
correct result is exact in fp32 in any summation order.  Whatever the tiling, split-K or epilogue, the kernel must then
match an fp64 reference bit for bit (fp32 outputs), or that reference rounded to bf16 (bf16 outputs, which exercises the
round-to-nearest-even ties of every store path).  Attention gets probes whose answers are known in closed form: a
permutation (each query picks out one key), a uniform softmax (exact ones channel and means), and staircases of logits
around the lazy-rescale threshold.

Every measured launch plan (tc_plans.PLANS) is run through the wrapper production uses, and a spy on ops._tc_launch checks
that the plan was the one launched; an eager SD UNet forward and VAE decode check that every plan key is still reached.
If a probe ever differs by +-1 or less, suspect the assumption that the tcgen05 fp32 accumulator keeps every integer bit
of these sums before suspecting an index bug: index bugs give large differences.
"""
import contextlib
import math

import pytest
import torch
import torch.nn.functional as F

from gpu_util import nchw, nhwc

pytestmark = pytest.mark.gpu


# ---- operands and exact references ----------------------------------------------------------------------------------------
def _ints(shape, lo, hi, seed, dtype=torch.float32, density=None):
    g = torch.Generator().manual_seed(seed)
    t = torch.randint(lo, hi + 1, shape, generator=g).float()
    if density is not None:
        t = t * (torch.rand(shape, generator=g) < density).float()
    return t.to(dtype).cuda()


def act(shape, seed):
    return _ints(shape, -2, 2, seed, torch.bfloat16)


def wts(shape, seed, density=None, dtype=torch.bfloat16):
    return _ints(shape, -1, 1, seed, dtype, density)


def vec(shape, seed):
    return _ints(shape, -4, 4, seed)


def exact(ref):
    """fp64 reference -> its integer values (cuDNN may pick Winograd / FFT, which leave tiny non-integer residues)."""
    r = ref.round()
    assert float((ref - r).abs().max()) <= 1e-6, "reference is not integer-valued"
    assert float(r.abs().max()) < 2 ** 24
    return r


def assert_exact(out, ref):
    """fp32: bit-identical to the integer reference; bf16: identical to its round-to-nearest-even rounding."""
    want = ref.float().to(out.dtype)
    if not torch.equal(out, want):
        bad = (out.float() != want.float()).nonzero()
        raise AssertionError("%d of %d elements differ, first at %s: got %s, want %s" % (
            bad.shape[0], out.numel(), tuple(bad[0].tolist()), out[tuple(bad[0])].item(), want[tuple(bad[0])].item()))


def bf16_ulp(x):
    """one bf16 ulp at |x| (fp64).  Floored at the ulp of 2^-100: the attention kernels clamp their exponentials at 2^-125
    instead of flushing them to zero, so a probability that should underflow can leave a contribution of that order."""
    a = x.double().abs().clamp_min(2.0 ** -100)
    return torch.exp2(torch.floor(torch.log2(a)) - 7)


def assert_within_ulp(out, ref, what=""):
    err = (out.double() - ref.double()).abs()
    bad = err > bf16_ulp(ref)
    assert not bool(bad.any()), "%s: %d elements beyond one bf16 ulp, worst %.3g" % (what, int(bad.sum()), float(err.max()))


def canvas(rows, cols, ld, dtype, spare=37, device="cuda"):
    """A NaN-filled [rows + spare, ld] buffer and its [rows, cols] view: nothing outside the view may be written."""
    buf = torch.full((rows + spare, ld), float("nan"), dtype=dtype, device=device)
    return buf, buf[:rows, :cols]


def assert_outside_untouched(buf, rows, cols):
    mask = torch.ones(buf.shape, dtype=torch.bool, device=buf.device)
    mask[:rows, :cols] = False
    assert bool(buf[mask].float().isnan().all()), "the kernel wrote outside its output"


@contextlib.contextmanager
def switch(name, value):
    """run with a library switch (sdb_tc_set_tma_epilogue, ...) set, restoring it afterwards"""
    from sdb200 import _lib
    fn = getattr(_lib.load(), name)
    prev = fn(value)
    try:
        yield
    finally:
        fn(prev)


def plan_key(a):
    """the tc_plans key of a launch's argument block, as ops._apply_plan forms it"""
    rows = a.OH * a.OW if a.taps else a.rows_per_item
    return ("conv" if a.taps else "gemm", rows, a.N, a.K, a.taps, a.stride if a.taps else 0, a.geglu, int(bool(a.residual)),
            a.out_dtype, a.col_group)


@pytest.fixture
def launches(monkeypatch, cuda):
    """records (key, variant, block_n, split_k) of every tcgen05 launch as ops hands it to the library"""
    from sdb200 import ops
    rec = []
    orig = ops._tc_launch

    def spy(a, what):
        rec.append((plan_key(a), a.variant, a.block_n, a.split_k))
        return orig(a, what)
    monkeypatch.setattr(ops, "_tc_launch", spy)
    return rec


# ---- A.1: every measured launch plan, through the production wrappers -------------------------------------------------------
def _plan_cases():
    from sdb200.tc_plans import PLANS
    cases = []
    for key in sorted(PLANS):
        batches = (2,) if key[1] == 262144 else (8, 3)
        for nb in batches:
            cases.append(pytest.param(key, nb, id="%s-%d-%d-%d-t%d-r%d-o%d-b%d" % (key[0], key[1], key[2], key[3], key[4], key[7], key[8], nb)))
    return cases


def _run_plan_entry(key, nb, seed):
    """(callable that runs the entry through its production wrapper, exact reference, canvas check or None)"""
    from sdb200 import ops
    kind, rows, N, K, taps, stride, geglu, res_flag, odt, cg = key
    assert stride in (0, 1) and not geglu and not cg
    out_dtype = torch.bfloat16 if odt else torch.float32
    side = int(round(math.sqrt(rows)))
    bias = vec((N,), seed + 2)
    if kind == "gemm":
        M = nb * rows
        A = act((M, K), seed)
        W = wts((N, K), seed + 1)
        res = vec((M, N), seed + 3) if res_flag else None
        ref = A.double() @ W.double().T + bias.double()
        if res is not None:
            ref = ref + res.double()
        ld = N + 8
        buf, view = canvas(M, N, ld, out_dtype)

        def run():
            buf.fill_(float("nan"))
            ops.gemm_tc(A, W, bias, residual=res, out_dtype=out_dtype, out=view, ldc=ld, rows_per_item=rows)
            return view
        return run, exact(ref), lambda: assert_outside_untouched(buf, M, N)
    assert side * side == rows
    if taps == 4:
        Cin = K // 4
        x = act((nb, side, side, Cin), seed)
        w = wts((N, Cin, 3, 3), seed + 1)
        wph = ops.fold_upsample_weights(w, torch.bfloat16)
        ref = F.conv2d(F.interpolate(nchw(x.double()), scale_factor=2, mode="nearest"), w.double(), bias.double(), padding=1)
        assert not res_flag and not odt
        return (lambda: ops.conv_up2_tc(x, wph, bias)), exact(nhwc(ref)), None
    k = 3 if taps == 9 else 1
    Cin = K // taps
    x = act((nb, side, side, Cin), seed)
    w = wts((N, Cin, k, k), seed + 1)
    wp = ops.pack_conv_weight(w, torch.bfloat16)
    rv = vec((nb, N), seed + 4) if taps == 9 and not odt else None      # the ResBlock conv carries the time-embedding row
    res = vec((nb, side, side, N), seed + 3) if res_flag else None
    ref = nhwc(F.conv2d(nchw(x.double()), w.double(), bias.double(), padding=k // 2))
    if rv is not None:
        ref = ref + rv.double()[:, None, None, :]
    if res is not None:
        ref = ref + res.double()
    M = nb * rows
    buf, _ = canvas(M, N, N, out_dtype)
    out = buf[:M].view(nb, side, side, N)

    def run():
        buf.fill_(float("nan"))
        ops.conv_tc(x, wp, bias, k, k, pad=k // 2, rowvec=rv, residual=res, out_dtype=out_dtype, out=out)
        return out
    return run, exact(ref), lambda: assert_outside_untouched(buf, M, N)


@pytest.mark.parametrize("key,nb", _plan_cases())
def test_plan_entry_exact(launches, key, nb):
    """Each PLANS entry at batch 8 and a ragged 3 (the 512^2 VAE entries at 2), TMA epilogue on and off, and for the
    (one-CTA, 160, no split) plans tail split on and off: bit-exact, nothing written outside, and launched with its plan."""
    from sdb200.tc_plans import PLANS
    plan = PLANS[key][:3]
    run, ref, untouched = _run_plan_entry(key, nb, seed=sum(key[1:4]) % 1000 + nb)
    tails = (1, 0) if plan == (1, 160, 1) else (1,)
    for tma in (1, 0):
        for tail in tails:
            del launches[:]
            with switch("sdb_tc_set_tma_epilogue", tma), switch("sdb_tc_set_tail_split", tail):
                out = run()
                torch.cuda.synchronize()
            assert launches, "no tcgen05 launch"
            for k_, v_, bn_, sk_ in launches:
                assert k_ == key, (k_, key)
                assert (v_, bn_, sk_) == plan, ("launched", (v_, bn_, sk_), "plan", plan)
            assert_exact(out, ref)
            if untouched is not None:
                untouched()


# ---- A.2: a heuristic matrix beside the plans (explicit variant, so no plan applies) ------------------------------------
GEMM_SHAPES = [(1000, 320, 320), (333, 200, 1280), (77, 640, 768), (2100, 1280, 640)]
OUTPUTS = [("f32", torch.float32, False), ("f32+res", torch.float32, True), ("bf16", torch.bfloat16, False),
           ("bf16+res", torch.bfloat16, True)]


@pytest.mark.parametrize("variant", [2, 1], ids=["pair", "single"])
@pytest.mark.parametrize("block_n", [32, 64, 128, 160, 256])
def test_gemm_matrix_exact(cuda, variant, block_n):
    """ragged M, N not a multiple of the tile, split_k 1 / 2 / 5, fp32 / bf16 outputs with and without residual, both
    epilogues; the output is a view with ldc > N inside a NaN canvas"""
    from sdb200 import ops
    for si, (M, N, K) in enumerate(GEMM_SHAPES):
        A = act((M, K), 10 + si)
        W = wts((N, K), 20 + si)
        bias = vec((N,), 30 + si)
        res = vec((M, N), 40 + si)
        base = A.double() @ W.double().T + bias.double()
        for name, odt, with_res in OUTPUTS:
            ref = exact(base + res.double() if with_res else base)
            ld = N + 8
            buf, view = canvas(M, N, ld, odt)
            for sk in (1, 2, 5):
                for tma in (1, 0):
                    buf.fill_(float("nan"))
                    with switch("sdb_tc_set_tma_epilogue", tma):
                        ops.gemm_tc(A, W, bias, residual=res if with_res else None, out_dtype=odt, out=view, ldc=ld,
                                    split_k=sk, block_n=block_n, variant=variant)
                    try:
                        assert_exact(view, ref)
                        assert_outside_untouched(buf, M, N)
                    except AssertionError as e:
                        raise AssertionError("M=%d N=%d K=%d %s split_k=%d tma=%d: %s" % (M, N, K, name, sk, tma, e))


@pytest.mark.parametrize("variant", [2, 1], ids=["pair", "single"])
@pytest.mark.parametrize("block_n", [64, 128, 256])
def test_geglu_exact(cuda, variant, block_n):
    """GEGLU: the pre-activation is exact, so value * gelu(gate) may differ from its fp64 value by one bf16 ulp.  The
    epilogue's erf approximation (common.cuh gelu_erf_fast) is 4e-5 relative at gate = -3 but 0.6 % at -4 and 5 % at -5,
    where gelu is below 1.3e-4: there the bound is 1e-6 * |value| absolute instead."""
    from sdb200 import ops
    M, inner, K = 1000, 1280, 320
    A = act((M, K), 41)
    W = torch.cat([wts((inner, K), 42), wts((inner, K), 43, density=0.1)])
    b = vec((2 * inner,), 44)
    wp, bp = ops.pack_geglu_weight(W, b, block_n)
    h = exact(A.double() @ W.double().T + b.double())
    val, gate = h[:, :inner], h[:, inner:]
    ref = val * F.gelu(gate)
    for tma in (1, 0):
        with switch("sdb_tc_set_tma_epilogue", tma):
            out = ops.gemm_tc(A, wp, bp, out_dtype=torch.bfloat16, geglu=True, block_n=block_n, variant=variant)
        err = (out.double() - ref).abs()
        tol = torch.where(gate > -3.5, bf16_ulp(ref), bf16_ulp(ref) + 1e-6 * val.abs())
        assert bool((err <= tol).all()), "GEGLU: %d elements out of bound (tma=%d)" % (int((err > tol).sum()), tma)


# (N, H, W, Cin, Cout, k, stride, pad, pad_hi): 1x1, 3x3, the VAE Downsample (stride 2, padding (0, 1, 0, 1)), maps
# smaller than a tile (several images per tile) and ragged ones, the LDM-BSR / VQ-f4 widths
CONV_GEOMS = [(3, 20, 12, 320, 160, 1, 1, 0, 0), (3, 24, 20, 160, 320, 3, 1, 1, 1), (8, 8, 8, 640, 640, 3, 1, 1, 1),
              (3, 8, 8, 320, 160, 3, 1, 1, 1), (2, 33, 31, 128, 128, 3, 2, 0, 1), (5, 16, 16, 640, 320, 3, 1, 1, 1)]
CONV_OUTPUTS = [("f32", torch.float32, False, False), ("f32+res", torch.float32, True, False), ("f32+rv+res", torch.float32, True, True),
                ("bf16", torch.bfloat16, False, False), ("bf16+res", torch.bfloat16, True, False)]


@pytest.mark.parametrize("variant", [2, 1], ids=["pair", "single"])
@pytest.mark.parametrize("geom", CONV_GEOMS, ids=lambda g: "x".join(map(str, g)))
def test_conv_matrix_exact(cuda, variant, geom):
    from sdb200 import ops
    nb, H, W_, Cin, Cout, k, stride, pad, pad_hi = geom
    x = act((nb, H, W_, Cin), 1)
    w = wts((Cout, Cin, k, k), 2)
    wp = ops.pack_conv_weight(w, torch.bfloat16)
    bias, rv = vec((Cout,), 3), vec((nb, Cout), 4)
    xd = F.pad(nchw(x.double()), (pad, pad_hi, pad, pad_hi))
    base = nhwc(F.conv2d(xd, w.double(), bias.double(), stride=stride))
    OH, OW = base.shape[1:3]
    res = vec((nb, OH, OW, Cout), 5)
    M = nb * OH * OW
    for name, odt, with_res, with_rv in CONV_OUTPUTS:
        ref = base + res.double() if with_res else base
        if with_rv:
            ref = ref + rv.double()[:, None, None, :]
        ref = exact(ref)
        buf, _ = canvas(M, Cout, Cout, odt)
        out = buf[:M].view(nb, OH, OW, Cout)
        for block_n in (0, 64, 160) if Cout % 160 == 0 else (0, 64, 128):
            for sk in (1, 2, 5):
                for tma in (1, 0):
                    buf.fill_(float("nan"))
                    with switch("sdb_tc_set_tma_epilogue", tma):
                        ops.conv_tc(x, wp, bias, k, k, stride=stride, pad=pad, pad_hi=pad_hi, rowvec=rv if with_rv else None,
                                    residual=res if with_res else None, out_dtype=odt, out=out, split_k=sk, block_n=block_n,
                                    variant=variant)
                    try:
                        assert_exact(out, ref)
                        assert_outside_untouched(buf, M, Cout)
                    except AssertionError as e:
                        raise AssertionError("%s block_n=%d split_k=%d tma=%d: %s" % (name, block_n, sk, tma, e))


@pytest.mark.parametrize("variant", [2, 1], ids=["pair", "single"])
@pytest.mark.parametrize("d,H", [(40, 8), (80, 8), (160, 8), (32, 10)])
def test_col_group_exact(cuda, variant, d, H):
    """q | k | v projection into padded heads: head h of each third lands in columns [h * dp, h * dp + d), pad columns 0"""
    from sdb200 import ops
    from sdb200.engine import head_pad
    dp = head_pad(d)
    M, K = 1000, 320
    A = act((M, K), 6)
    W = wts((3 * H * d, K), 7)
    ref = exact(A.double() @ W.double().T)
    for tma in (1, 0):
        with switch("sdb_tc_set_tma_epilogue", tma):
            out = ops.gemm_tc(A, W, out_dtype=torch.bfloat16, col_group=d, col_group_stride=dp, variant=variant)
        pv = out.view(M, 3 * H, dp)
        assert_exact(pv[:, :, :d].reshape(M, 3 * H * d), ref)
        assert bool((pv[:, :, d:] == 0).all()), "pad columns written"


def _pick_tile(OW, OH, NB=8, stride=1):
    """csrc/tc_contract.cu pick_tile: the tw x th x tn = 128 pixel block with the fewest tiles at a nominal batch of 8"""
    best = None
    w = 128
    while w >= 1:
        if w * stride <= 256:
            h = 128 // w
            while h >= 1:
                if h * stride <= 256 and 128 // (w * h) <= 256:
                    n = 128 // (w * h)
                    tiles = -(-OW // w) * -(-OH // h) * -(-NB // n)
                    if best is None or tiles < best[0]:
                        best = (tiles, w, h, n)
                h //= 2
        w //= 2
    return best[1:]


def _slot_sums(out, split, stride=1):
    """fp64 per-(32-row slot, column) sum and sum of squares of the stored output, in the slot layout of the launch"""
    nb, OH, OW, C = out.shape
    o = out.double().reshape(-1, C)
    if split > 1:                                  # the reduction kernel: one slot per 32 consecutive output rows
        o = o.view(-1, 32, C)
        return o.sum(1), (o * o).sum(1)
    tw, th, tn = _pick_tile(OW, OH, 8, stride)
    tiles_w, tiles_h = -(-OW // tw), -(-OH // th)
    m_tiles = tiles_w * tiles_h * -(-nb // tn)
    mt = torch.arange(m_tiles, device=out.device)[:, None]
    r = torch.arange(128, device=out.device)[None, :]
    in_, rem = r // (th * tw), r % (th * tw)
    img = (mt // (tiles_w * tiles_h)) * tn + in_
    oh = ((mt // tiles_w) % tiles_h) * th + rem // tw
    ow = (mt % tiles_w) * tw + rem % tw
    valid = (img < nb) & (oh < OH) & (ow < OW)
    idx = torch.where(valid, (img * OH + oh) * OW + ow, torch.full_like(img, o.shape[0]))
    g = torch.cat([o, o.new_zeros(1, C)])[idx.flatten()].view(m_tiles * 4, 32, C)
    return g.sum(1), (g * g).sum(1)


@pytest.mark.parametrize("variant", [2, 1], ids=["pair", "single"])
@pytest.mark.parametrize("geom,split", [((3, 16, 16, 320, 320, 1), 1), ((8, 8, 8, 640, 640, 3), 1), ((3, 8, 8, 640, 1280, 3), 3),
                                        ((2, 32, 32, 320, 320, 3), 1), ((2, 48, 40, 128, 256, 3), 1), ((4, 16, 16, 640, 640, 3), 2)],
                         ids=lambda v: "x".join(map(str, v)) if isinstance(v, tuple) else "sk%d" % v)
def test_colstats_exact(cuda, variant, geom, split):
    """GroupNorm column statistics emitted by the epilogue / split-K reduction: every slot's sum and sum of squares equal
    the fp64 sums of the stored output bit for bit (sparse weights keep every sum of squares below 2^24)."""
    from sdb200 import ops
    nb, H, W_, Cin, Cout, k = geom
    x = act((nb, H, W_, Cin), 11)
    w = wts((Cout, Cin, k, k), 12, density=4.0 / (Cin * k * k))
    wp = ops.pack_conv_weight(w, torch.bfloat16)
    bias, rv, res = vec((Cout,), 13), vec((nb, Cout), 14), vec((nb, H, W_, Cout), 15)
    ref = exact(nhwc(F.conv2d(nchw(x.double()), w.double(), bias.double(), padding=k // 2)) + rv.double()[:, None, None, :] + res.double())
    for tma in (1, 0):
        with switch("sdb_tc_set_tma_epilogue", tma):
            out = ops.conv_tc(x, wp, bias, k, k, pad=k // 2, rowvec=rv, residual=res, variant=variant, split_k=split, want_stats=True)
        assert_exact(out, ref)
        cs = getattr(out, "_sdb_cs", None)
        assert cs is not None, "no column statistics for this launch"
        s1, s2 = _slot_sums(out, split)
        assert float(s2.max()) < 2 ** 24, "probe precondition: slot sums of squares must be exact in fp32"
        n = s1.shape[0]
        assert cs[1] >= n
        assert torch.equal(cs[0][0, :n], s1.float()), "column sums differ (tma=%d)" % tma
        assert torch.equal(cs[0][1, :n], s2.float()), "column sums of squares differ (tma=%d)" % tma


# ---- A.3: the fp32 SIMT contraction ------------------------------------------------------------------------------------
@pytest.mark.parametrize("geom", [(3, 20, 12, 64, 96, 3, 1, 1, 1, 1), (2, 33, 31, 32, 64, 3, 2, 0, 1, 1), (2, 9, 7, 48, 40, 3, 1, 1, 1, 2),
                                  (3, 16, 16, 128, 64, 1, 1, 0, 0, 1)], ids=lambda g: "x".join(map(str, g)))
def test_conv_simt_exact(cuda, geom):
    from sdb200 import ops
    nb, H, W_, Cin, Cout, k, stride, pad, pad_hi, up = geom
    x = act((nb, H, W_, Cin), 21).float()
    w = wts((Cout, Cin, k, k), 22, dtype=torch.float32)
    bias = vec((Cout,), 23)
    xin = nchw(x.double())
    if up > 1:
        xin = F.interpolate(xin, scale_factor=up, mode="nearest")
    base = nhwc(F.conv2d(F.pad(xin, (pad, pad_hi, pad, pad_hi)), w.double(), bias.double(), stride=stride))
    rv, res = vec((nb, Cout), 24), vec(tuple(base.shape), 25)
    wp = ops.pack_conv_weight(w, torch.float32)
    out = ops.conv_simt(x, wp, bias, k, k, stride=stride, pad=pad, pad_hi=pad_hi, up=up)
    assert_exact(out, exact(base))
    out = ops.conv_simt(x, wp, bias, k, k, stride=stride, pad=pad, pad_hi=pad_hi, up=up, rowvec=rv, residual=res)
    assert_exact(out, exact(base + rv.double()[:, None, None, :] + res.double()))


@pytest.mark.parametrize("b_kn", [False, True])
@pytest.mark.parametrize("M,N,K", [(1000, 320, 320), (77, 200, 768), (129, 33, 1000)])
def test_gemm_simt_exact(cuda, b_kn, M, N, K):
    from sdb200 import ops
    A = act((M, K), 31).float()
    W = wts((N, K), 32, dtype=torch.float32)
    bias, res = vec((N,), 33), vec((M, N), 34)
    B = W.T.contiguous() if b_kn else W
    ref = exact(A.double() @ W.double().T + bias.double() + res.double())
    ld = N + 5
    buf, view = canvas(M, N, ld, torch.float32)
    ops.gemm_simt(A, B, bias, residual=res, b_kn=b_kn, out=view, ldc=ld)
    assert_exact(view, ref)
    assert_outside_untouched(buf, M, N)


# ---- B: attention probes -----------------------------------------------------------------------------------------------
def _code_bits(n):
    return max(1, math.ceil(math.log2(n))) if n > 1 else 0


def _codes(n, bits):
    """[n, bits] the +-1 binary code of each index"""
    j = torch.arange(n)[:, None]
    return ((j >> torch.arange(bits)[None, :]) & 1).float() * 2 - 1


def _attn(q, k, v, scale, layout, causal=False):
    """q [B,Sq,H,d], k / v [B,Sk,H,d] bf16 -> attention_tc output [B,Sq,H,d] through the dense or the padded head layout"""
    from sdb200 import ops
    from sdb200.engine import head_pad
    B, Sq, H, d = q.shape
    Sk = k.shape[1]
    dp = head_pad(d)
    if layout == "dense":
        st = lambda S: (S * H * d, H * d, d)   # noqa: E731
        out = ops.attention_tc(q.contiguous(), k.contiguous(), v.contiguous(), B, H, Sq, Sk, d, dp, scale, st(Sq), st(Sk), st(Sk),
                               dense=True, causal=causal)
    else:
        def padded(t):
            p = torch.zeros(t.shape[0], t.shape[1], H, dp, dtype=torch.bfloat16, device=t.device)
            p[..., :d] = t
            return p
        st = lambda S: (S * H * dp, H * dp, dp)   # noqa: E731
        out = ops.attention_tc(padded(q), padded(k), padded(v), B, H, Sq, Sk, d, dp, scale, st(Sq), st(Sk), st(Sk), causal=causal)
    return out.view(B, Sq, H, d)


def _perm_probe(B, H, Sq, Sk, d, seed):
    """keys carry the +-1 code of their index, query i carries 64 * code(sigma(i)): with scale 1 the best key beats the second
    best by 128 logits (185 log2 units), so every other probability underflows to 0 and row i is v[sigma(i)]"""
    bits = _code_bits(Sk)
    assert bits <= d
    g = torch.Generator().manual_seed(seed)
    sigma = torch.stack([torch.stack([torch.randperm(Sk, generator=g)[:Sq] if Sq <= Sk else torch.randint(0, Sk, (Sq,), generator=g)
                                      for _ in range(H)], 1) for _ in range(B)])          # [B, Sq, H]
    k = torch.zeros(B, Sk, H, d)
    k[..., :bits] = _codes(Sk, bits)[None, :, None, :]
    q = torch.zeros(B, Sq, H, d)
    q[..., :bits] = 64 * _codes(Sk, bits)[sigma]
    v = torch.randint(-4, 5, (B, Sk, H, d), generator=g).float()
    want = torch.gather(v, 1, sigma[..., None].expand(B, Sq, H, d))
    return q.bfloat16().cuda(), k.bfloat16().cuda(), v.bfloat16().cuda(), want.cuda()


def _uniform_probe(B, H, Sq, Sk, d, seed, leak_guard):
    """q = 0 (or, leak_guard, every real key at logit -112 so a zero key past Sk would take the mass): channel 0 of V is 1,
    the other channels integers in [-4, 4], so the output is (1, mean of V)"""
    g = torch.Generator().manual_seed(seed)
    q = torch.zeros(B, Sq, H, d)
    k = torch.zeros(B, Sk, H, d)
    v = torch.randint(-4, 5, (B, Sk, H, d), generator=g).float()
    v[..., 0] = 1
    if leak_guard:
        q[..., d - 1] = 1
        k[..., d - 1] = -112         # * scale 1 * log2(e) = -161.6 log2 units
    return q.bfloat16().cuda(), k.bfloat16().cuda(), v.bfloat16().cuda(), v.cuda()


ATTN_COVER = [  # (d, B, H, Sq, Sk): every d sees a ragged Sq, a ragged Sk and a multi-tile Sk
    (32, 2, 3, 77, 300), (32, 2, 3, 300, 4096), (32, 2, 3, 129, 129),
    (40, 2, 3, 300, 77), (40, 2, 3, 1, 4096), (40, 2, 3, 129, 300),
    (64, 2, 3, 77, 4096), (64, 2, 3, 300, 129), (64, 2, 3, 128, 1),
    (80, 2, 3, 129, 300), (80, 2, 3, 77, 4096), (80, 2, 3, 300, 128),
    (160, 2, 3, 300, 77), (160, 2, 3, 129, 4096), (160, 2, 3, 1, 300)]


@pytest.mark.parametrize("layout", ["dense", "padded"])
@pytest.mark.parametrize("d,B,H,Sq,Sk", ATTN_COVER)
def test_attention_permutation_probe(cuda, layout, d, B, H, Sq, Sk):
    q, k, v, want = _perm_probe(B, H, Sq, Sk, d, seed=d + Sq + Sk)
    out = _attn(q, k, v, 1.0, layout)
    assert_within_ulp(out, want, "permutation")


@pytest.mark.parametrize("leak_guard", [False, True], ids=["q0", "leak_guard"])
@pytest.mark.parametrize("d,B,H,Sq,Sk", ATTN_COVER)
def test_attention_uniform_probe(cuda, leak_guard, d, B, H, Sq, Sk):
    q, k, v, vf = _uniform_probe(B, H, Sq, Sk, d, seed=d + Sk, leak_guard=leak_guard)
    out = _attn(q, k, v, 1.0, "dense")
    assert bool((out[..., 0] == 1).all()), "row sums: channel 0 is not exactly 1 (min %s)" % float(out[..., 0].float().min())
    mean = vf.double().mean(1, keepdim=True).expand(B, Sq, H, d)
    assert_within_ulp(out, mean, "uniform")


@pytest.mark.parametrize("d", [32, 40, 64, 80, 160])
@pytest.mark.parametrize("S", [77, 300, 1000])
def test_attention_causal_uniform_probe(cuda, d, S):
    """causal uniform: row i is the prefix mean of V over keys 0 .. i, channel 0 exactly 1"""
    B, H = 2, 3
    q, k, v, vf = _uniform_probe(B, H, S, S, d, seed=S + d, leak_guard=False)
    out = _attn(q, k, v, 1.0, "dense", causal=True)
    assert bool((out[..., 0] == 1).all())
    prefix = vf.double().cumsum(1) / torch.arange(1, S + 1, device=vf.device, dtype=torch.float64)[None, :, None, None]
    assert_within_ulp(out, prefix, "causal prefix mean")


@pytest.mark.parametrize("short_kernel", [1, 0], ids=["kv1", "tile_walk"])
@pytest.mark.parametrize("Sk", [1, 50, 64, 65, 77, 80, 81, 128])
@pytest.mark.parametrize("d", [32, 40, 64, 80])
def test_attention_short_keys_probes(cuda, short_kernel, Sk, d):
    """Sk <= 128 with the one-key-tile kernel enabled and disabled: permutation and leak-guarded uniform probes"""
    B, H, Sq = 2, 3, 300
    with switch("sdb_attention_set_short_key_kernel", short_kernel):
        q, k, v, want = _perm_probe(B, H, Sq, Sk, d, seed=Sk + d)
        assert_within_ulp(_attn(q, k, v, 1.0, "dense"), want, "permutation")
        q, k, v, vf = _uniform_probe(B, H, Sq, Sk, d, seed=Sk, leak_guard=True)
        out = _attn(q, k, v, 1.0, "dense")
    assert bool((out[..., 0] == 1).all()), "row sums: channel 0 min %s" % float(out[..., 0].float().min())
    assert_within_ulp(out, vf.double().mean(1, keepdim=True).expand(B, Sq, H, d), "uniform")


def _staircase(kind, delta, T):
    """per-key-tile logit (log2 units) of the staircase probes"""
    t = torch.arange(T).float()
    if kind == "rise":
        return delta * t
    if kind == "fall":
        return delta * (T - 1 - t)
    s = torch.zeros(T)
    s[-1] = 3 * delta                 # one late spike
    return s


@pytest.mark.parametrize("kind", ["rise", "fall", "spike"])
@pytest.mark.parametrize("delta", [7.75, 8.0, 8.25])
@pytest.mark.parametrize("d", [40, 64, 160])
def test_attention_staircase_probe(cuda, kind, delta, d):
    """logits constant within each 128-key tile, stepping by delta log2 units per tile (below, at and above the lazy
    rescale threshold of 8): V channel t is the indicator of key tile t, so output channel t is that tile's softmax mass"""
    B, H, Sq, T = 2, 3, 200, 10
    Sk = 128 * T
    assert T + 1 <= d
    lg = _staircase(kind, delta, T)
    q = torch.zeros(B, Sq, H, d)
    q[..., 0] = delta if kind == "rise" or kind == "fall" else 3 * delta
    kk = torch.zeros(B, Sk, H, d)
    tile = torch.arange(Sk) // 128
    kk[..., 0] = (lg / q[0, 0, 0, 0])[tile][None, :, None]      # small integers: exact in bf16
    v = torch.zeros(B, Sk, H, d)
    v[:, torch.arange(Sk), :, tile] = 1
    v[..., T] = 1
    qb, kb, vb = q.bfloat16().cuda(), kk.bfloat16().cuda(), v.bfloat16().cuda()
    scale = math.log(2.0)           # logits in log2 units
    out = _attn(qb, kb, vb, scale, "dense").double()
    s = (qb.double().transpose(1, 2) @ kb.double().transpose(1, 2).transpose(-1, -2)) * scale
    ref = (torch.softmax(s, -1) @ vb.double().transpose(1, 2)).transpose(1, 2)
    mass, rmass = out[..., :T], ref[..., :T]
    big = rmass > 1e-6
    assert bool(((mass - rmass).abs() <= 0.01 * rmass)[big].all()), "tile masses off by more than 1 %%: worst %.3g" % float(
        ((mass - rmass).abs() / rmass.clamp_min(1e-30))[big].max())
    assert bool(((mass - rmass).abs() <= 1e-6)[~big].all())
    assert_within_ulp(out[..., T], torch.ones_like(out[..., T]), "ones channel")


@pytest.mark.parametrize("d", [256, 512])
@pytest.mark.parametrize("Sq,Sk", [(77, 300), (300, 129), (129, 4096), (1, 77)])
def test_attention_wide_probes(cuda, d, Sq, Sk):
    """tc_attention_wide_kernel (one head of d = 256 / 512): permutation and leak-guarded uniform probes, q | k | v as column
    blocks of one projection output"""
    from sdb200 import ops
    B = 2

    def run(q, k, v):
        S = max(Sq, Sk)
        qkv = torch.zeros(B * S, 3 * d, dtype=torch.bfloat16, device="cuda")
        qkv[:B * Sq, :d] = q.reshape(B * Sq, d)
        qkv[:B * Sk, d:2 * d] = k.reshape(B * Sk, d)
        qkv[:B * Sk, 2 * d:] = v.reshape(B * Sk, d)
        W3 = 3 * d
        return ops.attention_wide(qkv[:B * Sq, :d], qkv[:B * Sk, d:2 * d], qkv[:B * Sk, 2 * d:], B, Sq, Sk, d, 1.0,
                                  (Sq * W3, W3), (Sk * W3, W3), (Sk * W3, W3))
    q, k, v, want = _perm_probe(B, 1, Sq, Sk, d, seed=d + Sk)
    assert_within_ulp(run(q, k, v), want.view(B, Sq, d), "permutation")
    q, k, v, vf = _uniform_probe(B, 1, Sq, Sk, d, seed=Sk, leak_guard=True)
    out = run(q, k, v)
    assert bool((out[..., 0] == 1).all())
    assert_within_ulp(out, vf.double().mean(1, keepdim=True).expand(B, Sq, 1, d).reshape(B, Sq, d), "uniform")


# ---- C: every plan key is reached by production ------------------------------------------------------------------------
def test_every_plan_is_reached(launches):
    """An eager SD-1.x UNet forward (64x64 latent, 77-token context) and a VAE decode to 512x512, batch 1, bf16 mode:
    every PLANS key is hit, and every hit launched with its plan.  A refactor that orphans a measured plan fails here."""
    from oracle import weights as W
    from oracle.golden import load_golden
    from sdb200.autoencoder import AutoencoderKL
    from sdb200.openai_model import UNetModel
    from sdb200.tc_plans import PLANS
    gu = load_golden("unet_sd.pt")
    net = UNetModel(**gu["cfg"], compute_mode="bf16")
    net.load_state_dict(W.make_state_dict(gu["key_shapes"], gu["seed"]))
    net = net.cuda()
    net(W.seeded_randn((1, 4, 64, 64), 1).cuda(), torch.tensor([500], device="cuda"), W.seeded_randn((1, 77, 768), 2).cuda())
    del net
    gv = load_golden("vae_sd_z64.pt")
    vae = AutoencoderKL(ddconfig=gv["ddconfig"], embed_dim=4, compute_mode="bf16")
    vae.load_state_dict(W.make_state_dict(gv["key_shapes"], gv["seed"]), strict=False)
    vae = vae.cuda()
    vae.decode(W.seeded_randn((1, 4, 64, 64), 3).cuda())
    torch.cuda.synchronize()
    hit = {}
    for key, v_, bn_, sk_ in launches:
        if key in PLANS:
            hit.setdefault(key, set()).add((v_, bn_, sk_))
    missing = sorted(set(PLANS) - set(hit))
    assert not missing, "plan keys no launch reached: %s" % missing
    for key, got in hit.items():
        assert got == {PLANS[key][:3]}, (key, got, PLANS[key][:3])
    print("plan keys hit: %d of %d" % (len(hit), len(PLANS)))
