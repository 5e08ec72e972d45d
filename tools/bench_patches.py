#!/usr/bin/env python
"""LatentDiffusion's split_input_params branch on the LDM-BSR super-resolution shapes: the crops of a call run as one batch
against the reference's per-crop loop over the same modules.

    python tools/bench_patches.py [--reps 5] [--steps 100] [--launches 1000] [--batches 1 4]

Models (procedural weights, bf16): the UNet of the LDM-BSR config (in 6, out 3, model_channels 160, attention_resolutions
[16, 8], num_res_blocks 2, channel_mult [1, 2, 2, 4], num_head_channels 32, concat conditioning on the LR image,
cond_stage_key "LR_image") and the VQ-f4 first stage (ch 128, ch_mult [1, 2, 4], num_res_blocks 2, attn_resolutions [],
n_embed 8192, embed_dim 3).  Geometry: a 3 x 256^2 latent, ks 128, stride 64, vqf 4 -> 9 crops, a 1024^2 image.
For batch B in `batches`, each timed `reps` times, alternating the two variants, medians with ranges:
  (a) one apply_model            batched (one UNet call on 9B crops)  vs  the loop (9 calls on B crops)
  (b) one split decode_first_stage  batched (one decode of 9B crops) vs  the loop (9 decodes of B crops)
  (c) DDIM-`steps` (eta 0) + decode, images/s, both variants
The outputs of the two variants are compared in the same run and must be identical.
  (d) sdb_patch_fold alone on the batch-4 decode geometry ([36, 3, 512, 512] crops -> [4, 3, 1024, 1024]), `launches`
      launches replayed from one CUDA graph, against the reference's torch expression fold(o * weighting) / normalization
      (normalization precomputed) on the same GPU; bytes moved = crops read + image written, against the 6499 GB/s copy
      peak measured for this repository (DESIGN.md).  The 163 MB working set exceeds the 126 MB L2, so it is not
      L2-resident between launches.
Prints one JSON line with the GPU name and power limit; writes nothing.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

COPY_PEAK_GBS = 6499.0
SPLIT = {"ks": (128, 128), "stride": (64, 64), "vqf": 4, "patch_distributed_vq": True, "tie_braker": False,
         "clip_max_weight": 0.5, "clip_min_weight": 0.01, "clip_max_tie_weight": 0.5, "clip_min_tie_weight": 0.01}
UNET = dict(image_size=128, in_channels=6, out_channels=3, model_channels=160, attention_resolutions=[16, 8], num_res_blocks=2,
            channel_mult=[1, 2, 2, 4], num_head_channels=32)
VQ_DD = dict(double_z=False, z_channels=3, resolution=256, in_channels=3, out_ch=3, ch=128, ch_mult=(1, 2, 4),
             num_res_blocks=2, attn_resolutions=[], dropout=0.0)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip()
        return [s.strip() for s in out.split(",")[:2]]
    except Exception as e:          # the timing does not depend on it; say why it is missing
        return [None, "unavailable (%s)" % e]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--launches", type=int, default=1000)
    ap.add_argument("--batches", type=int, nargs="+", default=[1, 4])
    a = ap.parse_args()

    import torch
    import torch.nn.functional as F
    if not torch.cuda.is_available():
        sys.exit("bench_patches.py needs a CUDA device")
    import __graft_entry__ as ge
    ge.build()
    from oracle import weights as W
    from sdb200 import ops
    from sdb200.autoencoder import VQModelInterface
    from sdb200.pipeline import LatentDiffusion

    torch.cuda.set_device(0)
    med = lambda v: sorted(v)[len(v) // 2]

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        r = fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), r

    fs = VQModelInterface(3, ddconfig=VQ_DD, lossconfig=None, n_embed=8192, compute_mode="bf16")
    fs.load_state_dict(W.make_state_dict(W.key_shapes_of(fs), 3))
    ld = LatentDiffusion(unet_config=UNET, first_stage_config=False, first_stage_model=fs, conditioning_key="concat",
                         compute_mode="bf16", scale_factor=1.0, channels=3, image_size=256, cond_stage_key="LR_image")
    ld.model.diffusion_model.load_state_dict(W.make_state_dict(W.key_shapes_of(ld.model.diffusion_model), 5))
    ld = ld.cuda()
    ld.split_input_params = dict(SPLIT)

    # ---- the reference's per-crop loop (ldm/diffusion/ddpm.py get_fold_unfold, apply_model, decode_first_stage) ---------
    def fold_unfold(x, ks, st, uf=1):
        h, w = x.shape[-2:]
        Ly, Lx = (h - ks[0]) // st[0] + 1, (w - ks[1]) // st[1] + 1
        fks, fst, out = (ks[0] * uf, ks[0] * uf), (st[0] * uf, st[1] * uf), (h * uf, w * uf)
        fold = lambda t: F.fold(t, out, fks, stride=fst)
        weighting = ld.get_weighting(ks[0] * uf, ks[1] * uf, Ly, Lx, x.device).to(x.dtype)
        normalization = fold(weighting).view(1, 1, *out)
        return fold, (lambda t: F.unfold(t, ks, stride=st)), normalization, weighting.view(1, 1, fks[0], fks[1], Ly * Lx)

    def loop_apply(x, t, c):
        ks, st = SPLIT["ks"], SPLIT["stride"]
        fold, unfold, norm, wt = fold_unfold(x, ks, st)
        z = unfold(x).view(x.shape[0], -1, ks[0], ks[1], wt.shape[-1])
        cc = unfold(c).view(c.shape[0], -1, ks[0], ks[1], wt.shape[-1])
        o = torch.stack([ld.model(z[..., i], t, c_concat=[cc[..., i]]) for i in range(z.shape[-1])], axis=-1)
        return fold((o * wt).view(o.shape[0], -1, o.shape[-1])) / norm

    def loop_decode(z):
        ks, st = SPLIT["ks"], SPLIT["stride"]
        ks, st = (min(ks[0], z.shape[2]), min(ks[1], z.shape[3])), (min(st[0], z.shape[2]), min(st[1], z.shape[3]))
        fold, unfold, norm, wt = fold_unfold(z, ks, st, uf=SPLIT["vqf"])
        zc = unfold(z).view(z.shape[0], -1, ks[0], ks[1], wt.shape[-1])
        o = torch.stack([fs.decode(zc[..., i]) for i in range(zc.shape[-1])], axis=-1)
        return fold((o * wt).view(o.shape[0], -1, o.shape[-1])) / norm

    def sr_sample(B, lr, x_T, loop):
        if loop:
            ld.apply_model = lambda x, t, c, return_ids=False: loop_apply(x, t, c)
        try:
            z, _ = ld.sample_log(lr, B, ddim=True, ddim_steps=a.steps, shape=(3, 256, 256), x_T=x_T, eta=0.0)
            return loop_decode(z) if loop else ld.decode_first_stage(z)
        finally:
            ld.__dict__.pop("apply_model", None)

    name, power = gpu_info()
    res = {"metric": "split_input_params", "reps": a.reps, "ddim_steps": a.steps, "crops": 9, "latent": [3, 256, 256],
           "image": [3, 1024, 1024], "ks": 128, "stride": 64, "vqf": 4, "compute_mode": "bf16"}
    for B in a.batches:
        x = W.seeded_randn((B, 3, 256, 256), 11).cuda()
        lr = W.seeded_randn((B, 3, 256, 256), 12).cuda()
        t = torch.full((B,), 500, device="cuda", dtype=torch.long)
        cases = {
            "apply_model_ms": (lambda: ld.apply_model(x, t, lr), lambda: loop_apply(x, t, lr)),
            "decode_ms": (lambda: ld.decode_first_stage(x), lambda: loop_decode(x)),
            "ddim_sr_ms": (lambda: sr_sample(B, lr, x, False), lambda: sr_sample(B, lr, x, True)),
        }
        row = {}
        for key, (fb, fl) in cases.items():
            fb(), fl()                                            # warm-up
            tb, tl = [], []
            same = True
            for _ in range(a.reps):
                ms, ob = timed(fb)
                tb.append(ms)
                ms, ol = timed(fl)
                tl.append(ms)
                same = same and bool(torch.equal(ob, ol))
            assert same, "%s: the batched path and the per-crop loop differ at batch %d" % (key, B)
            row[key] = {"batched": round(med(tb), 3), "batched_range": [round(min(tb), 3), round(max(tb), 3)],
                        "loop": round(med(tl), 3), "loop_range": [round(min(tl), 3), round(max(tl), 3)],
                        "loop_over_batched": round(med(tl) / med(tb), 3), "identical": same}
        d = row["ddim_sr_ms"]
        row["ddim_sr_images_per_s"] = {"batched": round(1e3 * B / d["batched"], 4), "loop": round(1e3 * B / d["loop"], 4)}
        res["b%d" % B] = row
        del x, lr
        torch.cuda.empty_cache()

    # (d) the fold kernel alone, batch-4 decode geometry
    B, L, C, K = 4, 9, 3, 512
    o5 = torch.randn(B, C, K, K, L, device="cuda")
    o = o5.permute(4, 0, 1, 2, 3).contiguous().view(L * B, C, K, K)
    wpix, wcrop = ld._patch_weights(K, K, 3, 3, o.device)
    args = (B, (3, 3), (256, 256), (1024, 1024), wpix, wcrop)
    wt = ld.get_weighting(K, K, 3, 3, o.device)
    tfold = lambda v: F.fold(v, (1024, 1024), (K, K), stride=(256, 256))
    norm = tfold(wt).view(1, 1, 1024, 1024)
    wt = wt.view(1, 1, K, K, L)
    torch_expr = lambda: tfold((o5 * wt).view(B, -1, L)) / norm
    assert torch.equal(ops.patch_fold(o, *args), torch_expr()), "sdb_patch_fold differs from the torch expression"
    n = a.launches
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(n):
            ops.patch_fold(o, *args)
    graph.replay()
    torch_expr()
    tk, tt = [], []
    for _ in range(a.reps):
        tk.append(1e3 * timed(graph.replay)[0] / n)
        tt.append(1e3 * timed(lambda: [torch_expr() for _ in range(20)])[0] / 20)
    us = med(tk)
    nbytes = 4 * (o.numel() + B * C * 1024 * 1024)
    res["fold_b4_decode"] = {
        "kernel_us": round(us, 2), "kernel_us_range": [round(min(tk), 2), round(max(tk), 2)],
        "torch_us": round(med(tt), 2), "torch_us_range": [round(min(tt), 2), round(max(tt), 2)],
        "bytes": nbytes, "gb_per_s": round(nbytes / (us * 1e-6) / 1e9, 1),
        "copy_peak_share": round(nbytes / (us * 1e-6) / 1e9 / COPY_PEAK_GBS, 3), "launches": n,
        "l2_resident": "no: 163 MB of crops + image per launch against a 126 MB L2"}
    res.update({"gpu": name, "power_limit": power})
    print(json.dumps(res))


if __name__ == "__main__":
    main()
