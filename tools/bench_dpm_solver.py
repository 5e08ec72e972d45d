#!/usr/bin/env python
"""DPM-Solver++(2M) against DDIM-50 and PLMS-50 on the SD-1.x UNet: wall time, per-step sampler overhead, and the fused
DPM-Solver update kernel alone.

    python tools/bench_dpm_solver.py [--batch 8] [--dpm-steps 10,15,20,25] [--reps 5] [--launches 1000] [--warmup 2]

SD-1.x UNet with the procedural weights of oracle/weights.py (tests/golden/unet_sd.pt key shapes and seed), bf16 compute
mode, CUDA graph on, a 64x64x4 latent and a 77x768 context per sample.  Timed with CUDA events, without guidance and with
classifier-free guidance at scale 7.5 (one 2B UNet call per model evaluation):
  (a) DPMSolverSampler.sample at each S of --dpm-steps (S model evaluations), DDIMSampler.sample and PLMSSampler.sample at
      50 steps (50 and 51 evaluations);
  (b) overhead_ms per step: each sampler's time minus as many bare UNet calls as it makes evaluations, over its steps.
      (a) and (b) alternate every sampler and every bare run `--reps` times; medians are reported with every value, and
      overhead_spread_ms (max - min over the reps) is the run-to-run spread of each overhead;
  (c) sdb_dpm_solver_step alone at order 3 with guidance (x, e, e_uncond and two history tensors read; x_next and m0
      written, as the sampler requests them), `launches` launches issued from Python and replayed from one CUDA graph.
      At batch 8 these tensors (about 3.7 MB) stay in L2 between launches, so (c) measures launch cost, not HBM bandwidth.
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
    ap.add_argument("--dpm-steps", default="10,15,20,25")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--launches", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=2)
    a = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_dpm_solver.py needs a CUDA device")
    import __graft_entry__ as ge
    ge.build()
    from oracle import weights as W
    from oracle.golden import load_golden
    from sdb200 import ops
    from sdb200.ddim import DDIMSampler
    from sdb200.dpm_solver import DPM_Solver, DPMSolverSampler
    from sdb200.pipeline import LatentDiffusion
    from sdb200.plms import PLMSSampler

    torch.cuda.set_device(0)
    g = load_golden("unet_sd.pt")
    ld = LatentDiffusion(unet_config=g["cfg"], first_stage_config=False, compute_mode="bf16")
    ld.model.diffusion_model.load_state_dict(W.make_state_dict(g["key_shapes"], g["seed"]))
    ld = ld.cuda()
    ld.model.diffusion_model.use_cuda_graph = True
    B, S_ref = a.batch, 50
    dpm_steps = [int(s) for s in a.dpm_steps.split(",")]
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
    dpm, ddim, plms = DPMSolverSampler(ld), DDIMSampler(ld), PLMSSampler(ld)
    result = {"metric": "dpm_solver_vs_ddim_plms", "batch": B, "latent": [4, 64, 64], "context": [77, 768], "mode": "bf16",
              "cuda_graph": True, "dpm_solver": "order 2, multistep, time_uniform, lower_order_final", "reps": a.reps}
    for label, scale in (("no_cfg", 1.0), ("cfg7.5", 7.5)):
        kw = dict(conditioning=ctx, x_T=x, verbose=False)
        if scale != 1.0:
            kw.update(unconditional_guidance_scale=scale, unconditional_conditioning=uctx)
            x_in, t_in, c_in = torch.cat([x] * 2), torch.cat([ts] * 2), torch.cat([uctx, ctx])
        else:
            x_in, t_in, c_in = x, ts, ctx

        def bare(n):
            for _ in range(n):
                ld.apply_model(x_in, t_in, c_in)

        # name -> (run, model evaluations, steps)
        runs = {"ddim50": (lambda: ddim.sample(S_ref, B, (4, 64, 64), **kw), S_ref, S_ref),
                "plms50": (lambda: plms.sample(S_ref, B, (4, 64, 64), **kw), S_ref + 1, S_ref)}
        for S in dpm_steps:
            runs["dpm%d" % S] = ((lambda S=S: dpm.sample(S, B, (4, 64, 64), **kw)), S, S)
        n_bare = sorted({n for _, n, _ in runs.values()})
        for _ in range(a.warmup):                        # graphs, schedule tables, allocator
            for fn, _, _ in runs.values():
                fn()
            bare(2)
        t_run = {k: [] for k in runs}
        t_bare = {n: [] for n in n_bare}
        for _ in range(a.reps):
            for k, (fn, _, _) in runs.items():
                t_run[k].append(timed(fn))
            for n in n_bare:
                t_bare[n].append(timed(lambda: bare(n)))
        res = {"bare_unet_ms_per_call": r4(med(t_bare[S_ref]) / S_ref)}
        for k, (_, n, steps) in runs.items():
            over = [(t - b) / steps for t, b in zip(t_run[k], t_bare[n])]
            res[k] = {"ms": r4(med(t_run[k])), "model_calls": n, "overhead_ms_per_step": r4(med(over)),
                      "overhead_spread_ms": r4(max(over) - min(over)), "ms_all": [r4(v) for v in t_run[k]],
                      "bare_ms_all": [r4(v) for v in t_bare[n]], "overhead_ms_all": [r4(v) for v in over]}
        for S in dpm_steps:
            res["dpm%d" % S].update({
                "over_ddim50": round(med(t_run["dpm%d" % S]) / med(t_run["ddim50"]), 4),
                "over_plms50": round(med(t_run["dpm%d" % S]) / med(t_run["plms50"]), 4),
                "model_call_ratio_vs_ddim50": round(S / S_ref, 4)})
        result[label] = res

    # (c) the kernel alone: order 3 with guidance, the outputs the sampler requests
    shape = (B, 4, 64, 64)
    e, eu = torch.randn(shape, device="cuda"), torch.randn(shape, device="cuda")
    m1, m2 = torch.randn(shape, device="cuda"), torch.randn(shape, device="cuda")
    solver = DPM_Solver(None, dpm.noise_schedule)
    tg = solver.get_time_steps("time_uniform", 1., 1e-3, 20)
    coef = solver.update_coefficients([tg[i].reshape(1) for i in range(7, 10)], tg[10].reshape(1), 3)

    def kernel():
        for _ in range(a.launches):
            ops.dpm_solver_step(x, e, 3, coef, e_uncond=eu, cfg_scale=7.5, m1=m1, m2=m2)

    kernel()
    ms_issued = timed(kernel)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        kernel()
    graph.replay()
    ms_graph = timed(graph.replay)
    graph_us = 1e3 * ms_graph / a.launches
    nbytes = 7 * 4 * x.numel()
    gbs = nbytes / (graph_us * 1e-6) / 1e9
    name, power = gpu_info()
    result.update({
        "kernel": "sdb_dpm_solver_step order 3, cfg, 5 tensors read, 2 written",
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
