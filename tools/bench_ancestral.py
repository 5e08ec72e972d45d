#!/usr/bin/env python
"""Cost of the ancestral sampler's per-step work on top of the UNet (LatentDiffusion.p_sample_loop).

    python tools/bench_ancestral.py [--batch 8] [--steps 200] [--launches 1000] [--warmup 10] [--profile FILE]

SD-1.x UNet with the procedural weights of oracle/weights.py (tests/golden/unet_sd.pt key shapes and seed), bf16 compute
mode, CUDA graph on, a 64x64x4 latent and a 77x768 context per sample.  Timed with CUDA events:
  (a) p_sample_loop(timesteps=steps): UNet + noise draw + fused sdb_ddpm_step per step;
  (b) `steps` bare UNet calls on the same inputs;
  (c) sdb_ddpm_step alone (eps, noise, clamp on), `launches` back-to-back launches, issued from Python and replayed
      from one CUDA graph (the graph time is the kernels' own; kernel_gbs is taken from it).
Prints one JSON line: per-step ms of (a) and (b), overhead_ms = (a - b) / steps and its share of the UNet step, the
kernel's time per launch and its bytes (x, eps, noise read, x_prev written, 4 B each) over that time against 6499 GB/s,
and the GPU's name and power limit.  (a) and (b) alternate `--reps` times; the medians are reported with every value.  The step's tensors (2 MB at batch 8) stay in L2 between launches, so (c) measures
launch-bound, L2-resident behaviour, not HBM bandwidth.  Writes nothing, except with --profile FILE: then nothing is
timed; 20 steps of p_sample_loop run under torch.profiler and the per-op CUDA/CPU table is written to FILE (run it as a
separate process from the timing run: tracing slows the host).
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

HBM_GBS = 6499.0


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip()
        name, power = [s.strip() for s in out.split(",")[:2]]
        return name, power
    except Exception as e:          # the timing does not depend on it; say why it is missing
        return None, "unavailable (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--launches", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--reps", type=int, default=3, help="(a) and (b) are timed this many times, alternated; medians reported")
    ap.add_argument("--profile", metavar="FILE", default=None)
    a = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_ancestral.py needs a CUDA device")
    import __graft_entry__ as ge
    ge.build()
    from oracle import weights as W
    from oracle.golden import load_golden
    from sdb200 import ops
    from sdb200.pipeline import LatentDiffusion

    torch.cuda.set_device(0)
    g = load_golden("unet_sd.pt")
    ld = LatentDiffusion(unet_config=g["cfg"], first_stage_config=False, compute_mode="bf16")
    ld.model.diffusion_model.load_state_dict(W.make_state_dict(g["key_shapes"], g["seed"]))
    ld = ld.cuda()
    ld.model.diffusion_model.use_cuda_graph = True
    B = a.batch
    shape = (B, 4, 64, 64)
    x = W.seeded_randn(shape, 1).cuda()
    ctx = W.seeded_randn((B, 77, 768), 2).cuda()
    ts = torch.full((B,), 500, device="cuda", dtype=torch.long)

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    def loop():
        ld.p_sample_loop(ctx, shape, x_T=x, timesteps=a.steps, verbose=False)

    def bare():
        for _ in range(a.steps):
            ld.apply_model(x, ts, ctx)

    table = ld.ddpm_table()
    eps, noise = torch.randn(shape, device="cuda"), torch.randn(shape, device="cuda")

    def kernel():
        for _ in range(a.launches):
            ops.ddpm_step(x, ts, table, eps=eps, noise=noise, clip=True)

    ld.p_sample_loop(ctx, shape, x_T=x, timesteps=a.warmup, verbose=False)      # graphs, schedule table, allocator
    for _ in range(a.warmup):
        ld.apply_model(x, ts, ctx)
        ops.ddpm_step(x, ts, table, eps=eps, noise=noise, clip=True)
    if a.profile:
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            ld.p_sample_loop(ctx, shape, x_T=x, timesteps=20, verbose=False)
            torch.cuda.synchronize()
        with open(a.profile, "w") as f:
            f.write(prof.key_averages().table(sort_by="self_cuda_time_total", row_limit=40))
            f.write("\n")
            f.write(prof.key_averages().table(sort_by="self_cpu_time_total", row_limit=40))
        return
    loops, bares = [], []
    for _ in range(a.reps):
        loops.append(timed(loop) / a.steps)
        bares.append(timed(bare) / a.steps)
    ms_kernel = timed(kernel)
    # the same launches captured in one CUDA graph: replay time is the kernels' own, without the Python / ctypes issue cost
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        kernel()
    graph.replay()
    ms_graph = timed(graph.replay)

    med = lambda v: sorted(v)[len(v) // 2]
    loop_step, bare_step = med(loops), med(bares)
    overhead = loop_step - bare_step
    kernel_us = 1e3 * ms_kernel / a.launches
    graph_us = 1e3 * ms_graph / a.launches
    nbytes = 4 * 4 * x.numel()
    gbs = nbytes / (graph_us * 1e-6) / 1e9
    name, power = gpu_info()
    print(json.dumps({
        "metric": "ancestral_sampler_overhead",
        "batch": B, "latent": [4, 64, 64], "context": [77, 768], "mode": "bf16", "cuda_graph": True, "steps": a.steps,
        "loop_ms_per_step": round(loop_step, 4),
        "unet_ms_per_step": round(bare_step, 4),
        "reps": a.reps, "loop_ms_per_step_all": [round(v, 4) for v in loops], "unet_ms_per_step_all": [round(v, 4) for v in bares],
        "overhead_ms": round(overhead, 4),
        "overhead_pct_of_unet_step": round(100.0 * overhead / bare_step, 3),
        "kernel_launches": a.launches,
        "kernel_us_per_launch_issued": round(kernel_us, 3),
        "kernel_us_per_launch_graph": round(graph_us, 3),
        "kernel_bytes": nbytes,
        "kernel_gbs": round(gbs, 1),
        "kernel_fraction_of_hbm": round(gbs / HBM_GBS, 4),
        "hbm_gbs_reference": HBM_GBS,
        "gpu": name, "power_limit": power,
    }))


if __name__ == "__main__":
    main()
