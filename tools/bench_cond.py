#!/usr/bin/env python
"""Cost of the conditioning stages of sdb200.encoders on one GPU.

    python tools/bench_cond.py [--reps 5] [--iters 20]

(a) Text tower: BERTEmbedder(n_embed 1280, n_layer 32) (the LDM text-to-image conditioner) on [B, 77] token ids, bf16,
    B = 8 and 16 (16 = the CFG batch of 8 images), per call; beside it the same tower as an eager fp32 torch expression
    (F.linear / softmax / layer_norm, TF32 off) on the same inputs.  Its share of a batch-8 DDIM-50 sample: one B = 16
    encoder call over (that call + 50 UNet steps), the UNet step being one call of the LDM text-to-image UNet
    (SD UNet layout with context_dim 1280) on a [16, 4, 32, 32] latent with a [16, 77, 1280] context, bf16, timed here.
(b) SpatialRescaler(n_stages=2, bilinear, 0.5, 182 -> 3), the semantic-synthesis conditioner, on [8, 182, 256, 256] and
    [8, 182, 512, 512] inputs: the two fused launches against torch's F.interpolate x 2 + nn.Conv2d(182, 3, 1) on the same
    inputs.  Achieved bytes/s over the algorithmic bytes (stage 1 reads the input and writes the half-size map, stage 2
    reads that and writes the 3-channel quarter-size map).  Both inputs are larger than the 126 MB L2.
Every timing: CUDA events around `iters` back-to-back calls after a warm-up, repeated `reps` times alternating the compared
variants; medians with the range.  Prints one JSON line with the GPU name and power limit; writes nothing.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=20).stdout.strip()
        return [s.strip() for s in out.split(",")[:3]]
    except Exception as e:          # the timing does not depend on it; say why it is missing
        return [None, "unavailable (%s)" % e, None]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--iters", type=int, default=20)
    a = ap.parse_args()

    import torch
    import torch.nn.functional as F
    if not torch.cuda.is_available():
        sys.exit("bench_cond.py needs a CUDA device")
    import __graft_entry__ as ge
    ge.build()
    from sdb200 import encoders as E
    from sdb200.openai_model import UNetModel
    from sdb200.pipeline import SD_UNET_CONFIG

    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    torch.cuda.set_device(0)
    name, power, max_sm = gpu_info()

    def timed(fn, iters):
        fn()
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(iters):
            fn()
        e.record()
        e.synchronize()
        return s.elapsed_time(e) / iters

    def alternate(fns, iters):
        """{name: (median ms, min, max)} over `reps` rounds, the variants alternating inside each round."""
        res = {k: [] for k in fns}
        for _ in range(a.reps):
            for k, fn in fns.items():
                res[k].append(timed(fn, iters))
        return {k: (sorted(v)[len(v) // 2], min(v), max(v)) for k, v in res.items()}

    out = {"gpu": name, "power_limit": power, "clocks_max_sm": max_sm, "reps": a.reps, "iters": a.iters}

    # (a) the text tower
    torch.manual_seed(0)
    bert = E.BERTEmbedder(1280, 32, use_tokenizer=False, compute_mode="bf16").cuda()
    sd = {k: v.detach() for k, v in bert.state_dict().items()}

    def torch_tower(ids):
        p = "transformer."
        B, S = ids.shape
        x = sd[p + "token_emb.weight"][ids] + sd[p + "pos_emb.emb.weight"][:S][None]
        for i in range(64):
            q_ = "%sattn_layers.layers.%d." % (p, i)
            h = F.layer_norm(x, (1280,), sd[q_ + "0.weight"], sd[q_ + "0.bias"])
            if i % 2 == 0:
                q, k, v = (F.linear(h, sd[q_ + "1.to_%s.weight" % n]).view(B, S, 8, 64).transpose(1, 2) for n in "qkv")
                att = torch.softmax((q @ k.transpose(-1, -2)) * 0.125, dim=-1) @ v
                x = F.linear(att.transpose(1, 2).reshape(B, S, 512), sd[q_ + "1.to_out.weight"], sd[q_ + "1.to_out.bias"]) + x
            else:
                h = F.gelu(F.linear(h, sd[q_ + "1.net.0.0.weight"], sd[q_ + "1.net.0.0.bias"]))
                x = F.linear(h, sd[q_ + "1.net.2.weight"], sd[q_ + "1.net.2.bias"]) + x
        return F.layer_norm(x, (1280,), sd[p + "norm.weight"], sd[p + "norm.bias"])

    text = {}
    with torch.no_grad():
        for B in (8, 16):
            ids = torch.randint(0, 30522, (B, 77), device="cuda")
            rel = float((bert(ids).double() - torch_tower(ids).double()).norm() / torch_tower(ids).double().norm())
            t = alternate({"sdb200_bf16": lambda: bert(ids), "torch_fp32_eager": lambda: torch_tower(ids)}, a.iters)
            text["B%d" % B] = {"ms": t, "rel_l2_vs_torch_fp32": rel}
        unet = UNetModel(**dict(SD_UNET_CONFIG, context_dim=1280), compute_mode="bf16").cuda()
        x = torch.randn(16, 4, 32, 32, device="cuda")
        tt = torch.full((16,), 500, device="cuda", dtype=torch.long)
        ctx = torch.randn(16, 77, 1280, device="cuda")
        step = alternate({"unet_step_b16": lambda: unet(x, tt, context=ctx)}, a.iters)["unet_step_b16"]
    enc16 = text["B16"]["ms"]["sdb200_bf16"][0]
    text["unet_step_b16_ms"] = step
    text["share_of_ddim50_b8_sample"] = enc16 / (enc16 + 50 * step[0])
    out["text_tower_1280x32_S77"] = text
    del bert, unet, sd

    # (b) SpatialRescaler 182 -> 3, two bilinear stages
    sr = E.SpatialRescaler(2, "bilinear", 0.5, in_channels=182, out_channels=3).cuda()
    conv = sr.channel_mapper
    resc = {}
    with torch.no_grad():
        for H in (256, 512):
            xin = torch.randn(8, 182, H, H, device="cuda")
            fused = lambda: sr(xin)
            ref = lambda: conv(F.interpolate(F.interpolate(xin, scale_factor=0.5, mode="bilinear"), scale_factor=0.5,
                                             mode="bilinear"))
            rel = float((fused().double() - ref().double()).norm() / ref().double().norm())
            t = alternate({"sdb200_fused": fused, "torch_interp2_conv": ref}, max(2, a.iters // 4))
            nbytes = 4 * 8 * (182 * H * H + 2 * 182 * (H // 2) ** 2 + 3 * (H // 4) ** 2)
            resc["8x182x%dx%d" % (H, H)] = {
                "ms": t, "algorithmic_bytes": nbytes, "input_bytes": 4 * 8 * 182 * H * H, "exceeds_126MB_L2": True,
                "GBps": {k: nbytes / (v[0] * 1e-3) / 1e9 for k, v in t.items()}, "rel_l2_vs_torch": rel}
            del xin
    out["spatial_rescaler_182to3_2stages"] = resc
    print(json.dumps(out))


if __name__ == "__main__":
    main()
