#!/usr/bin/env python
"""Cost of image conditioning ("concat" / "hybrid" keys) on the SD-1.x UNet.

    python tools/bench_conditioning.py [--batch 8] [--steps 20] [--reps 5] [--launches 1000] [--warmup 3]

SD-1.x UNet with the procedural weights of oracle/weights.py (tests/golden/unet_sd.pt seed), bf16 compute mode, CUDA graph on,
a 64x64x4 latent and a 77x768 context per sample.  The 9-channel model has the same weights except conv_in (4 + 5 channels:
latent | mask | masked-image latent).  Timed with CUDA events:
  (a) one UNet call: the 4-channel model's forward against the 9-channel model's forward_concat, `steps` calls each;
  (b) one DDIM step with classifier-free guidance 7.5 on the 9-channel hybrid LatentDiffusion: the 2B dict path (one call
      at batch 2B) against the two-call path (uncond and cond at batch B);
  (c) the layout kernel alone: the fused two-source sdb_nchw_concat_to_nhwc against torch.cat + sdb_nchw_to_nhwc_split, each
      `launches` times replayed from one CUDA graph.
(a) and (b) alternate their two variants `--reps` times; medians are reported with every value.  The JSON line also has the
number of aten::cat ops in one eager forward_concat call (torch.profiler, outside the timed windows) and the GPU's name and
power limit.  Writes nothing.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip()
        name, power = [s.strip() for s in out.split(",")[:2]]
        return name, power
    except Exception as e:          # the timing does not depend on it; say why it is missing
        return None, "unavailable (%s)" % e


def timed(fn, n):
    import torch
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    s.record()
    for _ in range(n):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / n


def summary(v):
    return {"median": round(statistics.median(v), 4), "min": round(min(v), 4), "max": round(max(v), 4),
            "all": [round(x, 4) for x in v]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--launches", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_conditioning.py needs a CUDA device")
    from oracle import weights as W
    from oracle.golden import load_golden
    from sdb200 import ops
    from sdb200.ddim import DDIMSampler
    from sdb200.openai_model import UNetModel
    from sdb200.pipeline import LatentDiffusion

    g = load_golden("unet_sd.pt")
    B = a.batch

    def unet(cin):
        net = UNetModel(**dict(g["cfg"], in_channels=cin), compute_mode="bf16")
        net.load_state_dict(W.make_state_dict(W.key_shapes_of(net), g["seed"]))
        net = net.cuda()
        net.use_cuda_graph = True
        return net

    net4, net9 = unet(4), unet(9)
    x = W.seeded_randn((B, 4, 64, 64), 1).cuda()
    cc = torch.cat([(W.seeded_randn((B, 1, 64, 64), 2) > 0).float(), W.seeded_randn((B, 4, 64, 64), 3)], 1).cuda()
    ctx = W.seeded_randn((B, 77, 768), 4).cuda()
    uctx = W.seeded_randn((B, 77, 768), 5).cuda()
    t = torch.full((B,), 500, device="cuda", dtype=torch.long)

    # (a) UNet call, 4-channel crossattn vs 9-channel hybrid
    run4 = lambda: net4(x, t, ctx)
    run9 = lambda: net9.forward_concat(x, [cc], t, context=ctx)
    for _ in range(a.warmup):
        run4(), run9()
    a4, a9 = [], []
    for _ in range(a.reps):
        a4.append(timed(run4, a.steps))
        a9.append(timed(run9, a.steps))

    # aten::cat in one eager 9-channel call (the concat is inside the layout kernel)
    net9.use_cuda_graph = False
    run9()
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU]) as prof:
        run9()
        torch.cuda.synchronize()
    n_cat = sum(ev.count for ev in prof.key_averages() if ev.key == "aten::cat")
    net9.use_cuda_graph = True

    # (b) DDIM step with CFG on the hybrid model: 2B dict path vs two calls
    ld = LatentDiffusion(first_stage_config=False, unet=net9, conditioning_key="hybrid").cuda()
    c = {"c_concat": [cc], "c_crossattn": [ctx]}
    uc = {"c_concat": [cc], "c_crossattn": [uctx]}
    s2b, s2 = DDIMSampler(ld), DDIMSampler(ld)
    s2._cfg_dict_pairable = lambda c_, uc_: False
    for s in (s2b, s2):
        s.make_schedule(50, ddim_eta=0.0, verbose=False)
    step = lambda s: s.p_sample_ddim(x, c, t, index=25, unconditional_guidance_scale=7.5, unconditional_conditioning=uc)
    for _ in range(a.warmup):
        step(s2b), step(s2)
    b2b, b2 = [], []
    for _ in range(a.reps):
        b2b.append(timed(lambda: step(s2b), a.steps))
        b2.append(timed(lambda: step(s2), a.steps))
    same = torch.equal(step(s2b)[0], step(s2)[0])

    # (c) the layout kernel alone, from a CUDA graph
    m, z = cc[:, :1].contiguous(), cc[:, 1:].contiguous()
    fused = lambda: ops.nchw_to_nhwc(x, out_dtype=torch.bfloat16, pad_to=32, split=True, x1=cc)
    unfused = lambda: ops.nchw_to_nhwc(torch.cat([x, m, z], 1), out_dtype=torch.bfloat16, pad_to=32, split=True)
    assert torch.equal(fused(), unfused())

    def graph_of(fn):
        st = torch.cuda.Stream()
        st.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(st):
            for _ in range(3):
                fn()
        torch.cuda.current_stream().wait_stream(st)
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            for _ in range(a.launches):
                fn()
        return gr

    gf, gu = graph_of(fused), graph_of(unfused)
    gf.replay(), gu.replay()
    cf, cu = [], []
    for _ in range(a.reps):
        cf.append(timed(gf.replay, 1) * 1000.0 / a.launches)
        cu.append(timed(gu.replay, 1) * 1000.0 / a.launches)

    name, power = gpu_info()
    print(json.dumps({
        "bench": "conditioning", "gpu": name, "power_limit": power, "batch": B, "latent": [4, 64, 64], "compute_mode": "bf16",
        "cuda_graph": True, "steps": a.steps, "reps": a.reps,
        "a_unet_ms": {"crossattn_4ch_forward": summary(a4), "hybrid_9ch_forward_concat": summary(a9)},
        "a_ratio_9ch_over_4ch": round(statistics.median(a9) / statistics.median(a4), 4),
        "aten_cat_in_9ch_call": n_cat,
        "b_ddim_cfg_step_ms": {"dict_2b_one_call": summary(b2b), "two_calls": summary(b2)},
        "b_ratio_2b_over_two_calls": round(statistics.median(b2b) / statistics.median(b2), 4),
        "b_2b_equals_two_calls": same,
        "c_layout_us_per_launch": {"fused_two_source": summary(cf), "cat_then_layout": summary(cu)},
        "c_launches": a.launches,
    }))


if __name__ == "__main__":
    main()
