#!/usr/bin/env python
"""PLMS against DDIM on the SD-1.x UNet: wall time, per-step sampler overhead, and the fused PLMS update kernel alone.

    python tools/bench_plms.py [--batch 8] [--steps 50] [--reps 5] [--launches 1000] [--warmup 2]

SD-1.x UNet with the procedural weights of oracle/weights.py (tests/golden/unet_sd.pt key shapes and seed), bf16 compute
mode, CUDA graph on, a 64x64x4 latent and a 77x768 context per sample.  Timed with CUDA events, without guidance and with
classifier-free guidance at scale 7.5 (one 2B UNet call per model evaluation):
  (a) PLMSSampler.sample and DDIMSampler.sample, `steps` steps each (PLMS makes steps + 1 model evaluations);
  (b) overhead_ms per step: PLMS time minus steps + 1 bare UNet calls, over steps; DDIM time minus steps bare calls, over
      steps.  (a) and (b) alternate PLMS, DDIM and the two bare runs `--reps` times; medians are reported with every value,
      and overhead_spread_ms (max - min over the reps) is the run-to-run spread of each overhead;
  (c) sdb_plms_step alone at order 4 with guidance (x, e, e_uncond and three history tensors read; e, pred_x0 and x_prev
      written, as the sampler requests them), `launches` launches issued from Python and replayed from one CUDA graph.
      At batch 8 these tensors (about 5 MB) stay in L2 between launches, so (c) measures launch cost, not HBM bandwidth.
Prints one JSON line with the GPU's name and power limit.  Writes nothing.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from bench_ancestral import HBM_GBS, gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--launches", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=2)
    a = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_plms.py needs a CUDA device")
    import __graft_entry__ as ge
    ge.build()
    from oracle import weights as W
    from oracle.golden import load_golden
    from sdb200 import ops
    from sdb200.ddim import DDIMSampler
    from sdb200.pipeline import LatentDiffusion
    from sdb200.plms import PLMSSampler

    torch.cuda.set_device(0)
    g = load_golden("unet_sd.pt")
    ld = LatentDiffusion(unet_config=g["cfg"], first_stage_config=False, compute_mode="bf16")
    ld.model.diffusion_model.load_state_dict(W.make_state_dict(g["key_shapes"], g["seed"]))
    ld = ld.cuda()
    ld.model.diffusion_model.use_cuda_graph = True
    B, S = a.batch, a.steps
    x = W.seeded_randn((B, 4, 64, 64), 1).cuda()
    ctx = W.seeded_randn((B, 77, 768), 2).cuda()
    uctx = W.seeded_randn((B, 77, 768), 3).cuda()
    ts = torch.full((B,), 500, device="cuda", dtype=torch.long)

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    med = lambda v: sorted(v)[len(v) // 2]
    r4 = lambda v: round(v, 4)
    # one sampler of each kind for all runs: the 2B conditioning is built once, so the UNet projects its context once
    plms, ddim = PLMSSampler(ld), DDIMSampler(ld)
    result = {"metric": "plms_vs_ddim", "batch": B, "latent": [4, 64, 64], "context": [77, 768], "mode": "bf16",
              "cuda_graph": True, "steps": S, "reps": a.reps}
    for label, scale in (("no_cfg", 1.0), ("cfg7.5", 7.5)):
        kw = dict(conditioning=ctx, x_T=x, verbose=False)
        if scale != 1.0:
            kw.update(unconditional_guidance_scale=scale, unconditional_conditioning=uctx)
            x_in, t_in, c_in = torch.cat([x] * 2), torch.cat([ts] * 2), torch.cat([uctx, ctx])
        else:
            x_in, t_in, c_in = x, ts, ctx
        run_plms = lambda: plms.sample(S, B, (4, 64, 64), **kw)
        run_ddim = lambda: ddim.sample(S, B, (4, 64, 64), **kw)

        def bare(n):
            for _ in range(n):
                ld.apply_model(x_in, t_in, c_in)

        for _ in range(a.warmup):                        # graphs, schedule tables, allocator
            run_plms()
            run_ddim()
            bare(2)
        t_plms, t_ddim, t_b1, t_b0, o_plms, o_ddim = [], [], [], [], [], []
        for _ in range(a.reps):
            t_plms.append(timed(run_plms))
            t_ddim.append(timed(run_ddim))
            t_b1.append(timed(lambda: bare(S + 1)))
            t_b0.append(timed(lambda: bare(S)))
            o_plms.append((t_plms[-1] - t_b1[-1]) / S)
            o_ddim.append((t_ddim[-1] - t_b0[-1]) / S)
        result[label] = {
            "plms_ms": r4(med(t_plms)), "ddim_ms": r4(med(t_ddim)), "plms_over_ddim": round(med(t_plms) / med(t_ddim), 4),
            "expected_ratio_from_model_calls": round((S + 1) / S, 4),
            "bare_unet_ms_per_call": r4(med(t_b0) / S),
            "overhead_ms_plms": r4(med(o_plms)), "overhead_ms_ddim": r4(med(o_ddim)),
            "overhead_spread_ms_plms": r4(max(o_plms) - min(o_plms)), "overhead_spread_ms_ddim": r4(max(o_ddim) - min(o_ddim)),
            "plms_ms_all": [r4(v) for v in t_plms], "ddim_ms_all": [r4(v) for v in t_ddim],
            "bare_s_plus_1_ms_all": [r4(v) for v in t_b1], "bare_s_ms_all": [r4(v) for v in t_b0],
            "overhead_ms_plms_all": [r4(v) for v in o_plms], "overhead_ms_ddim_all": [r4(v) for v in o_ddim],
        }

    # (c) the kernel alone: order 4 with guidance, the outputs the sampler requests
    shape = (B, 4, 64, 64)
    e, eu = torch.randn(shape, device="cuda"), torch.randn(shape, device="cuda")
    olds = [torch.randn(shape, device="cuda") for _ in range(3)]
    coef = plms.derived_coefficients(10)

    def kernel():
        for _ in range(a.launches):
            ops.plms_step(x, e, 4, coef[0], coef[1], coef[2], coef[3], coef[4], e_uncond=eu, cfg_scale=7.5, e_old=olds,
                          want_e=True)

    kernel()
    ms_issued = timed(kernel)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        kernel()
    graph.replay()
    ms_graph = timed(graph.replay)
    graph_us = 1e3 * ms_graph / a.launches
    nbytes = 9 * 4 * x.numel()
    gbs = nbytes / (graph_us * 1e-6) / 1e9
    name, power = gpu_info()
    result.update({
        "kernel": "sdb_plms_step order 4, cfg, 6 tensors read, 3 written",
        "kernel_launches": a.launches,
        "kernel_us_per_launch_issued": round(1e3 * ms_issued / a.launches, 3),
        "kernel_us_per_launch_graph": round(graph_us, 3),
        "kernel_bytes": nbytes,
        "kernel_gbs": round(gbs, 1),
        "kernel_fraction_of_hbm": round(gbs / HBM_GBS, 4),
        "hbm_gbs_reference": HBM_GBS,
        "kernel_note": "tensors of %.1f MB stay in L2 between launches: launch-bound, not an HBM bandwidth figure" % (nbytes / 1e6),
        "gpu": name, "power_limit": power,
    })
    print(json.dumps(result))


if __name__ == "__main__":
    main()
