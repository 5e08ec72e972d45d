#!/usr/bin/env python
"""bench.py — 512 px DDIM-50 images/s of the sdb200 hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl sdb200|reference] [--batch B]

A "step" = one pass of the whole hot path over one batch: DDIM-50 (50 UNet calls + 50 fused DDIM
updates) + VAE decode to 512x512, SD-1.x shapes, random-init weights, synthetic latents/context.
Under torchrun (N > 1) every rank samples its own batch (weak scaling) and the decoded images are
all-gathered with NCCL; time is bracketed by barrier + synchronize and taken as the max over ranks.
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

UNET_GFLOP_PER_SAMPLE = 803.27      # SURVEY.md §8d (algorithmic, once-through), latent 64x64
VAE_GFLOP_PER_IMAGE = 2514.52
DDIM_STEPS = 50


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="sdb200", choices=["sdb200", "reference"])
    ap.add_argument("--batch", type=int, default=8, help="images per GPU per step")
    ap.add_argument("--mode", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--ddim-steps", type=int, default=DDIM_STEPS)
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--micro-batch", type=int, default=0, help="c4-strong: images per UNet call (0 = min(32, per-GPU share))")
    ap.add_argument("--config", default="c2", choices=["c2", "c3", "c5", "c4-strong"],
                    help="BASELINE.json config: c2 = DDIM-50 + decode, batch 8 per GPU (the headline, default); c3 = VAE decode "
                         "64x64x4 -> 512x512x3, batch 16; c5 = one UNet step on a 96x96 latent, batch sweep 1..32; c4-strong = the "
                         "full pipeline at a FIXED global batch of 64 sharded over the GPUs (strong scaling)")
    return ap.parse_args()


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1341.2), d.get("hbm_gbs", 6499.0), "measured"
    return 1400.0, 6650.0, "fallback"


class ClockSampler(threading.Thread):
    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.stop_flag = False
        self.max_mhz = None

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for n, v in zip(names, out[2:]):
                    if "Active" in v and "Not" not in v:
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


# ------------------------------------------------------------------------------------------------------
# CPU reference arm: the oracle restatement of the reference's own PyTorch path, on the host cores
# ------------------------------------------------------------------------------------------------------
_CPU_REF_STATE = {}


def cpu_reference_images_per_s(ddim_steps, repeats=1):
    """Bounded sample: one fp32 UNet call (B=1, 64x64 latent, 77x768 context) and one VAE decode
    (1x4x64x64 -> 512x512) of the oracle restatement; images/s = 1 / (ddim_steps * t_unet + t_decode)."""
    import torch
    from oracle import restate as R
    from oracle import weights as W
    from oracle.golden import load_golden
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    if not _CPU_REF_STATE:          # random-init weights of the reference's shapes, generated once per process
        gu, gv = load_golden("unet_sd.pt"), load_golden("vae_sd_z16.pt")
        _CPU_REF_STATE["sdu"] = W.make_state_dict(gu["key_shapes"], 1)
        _CPU_REF_STATE["sdv"] = W.make_state_dict(gv["key_shapes"], 2)
    sdu, sdv = _CPU_REF_STATE["sdu"], _CPU_REF_STATE["sdv"]
    x, ctx = W.seeded_randn((1, 4, 64, 64), 3), W.seeded_randn((1, 77, 768), 4)
    t = torch.tensor([500])
    tu, td = [], []
    with torch.no_grad():
        for _ in range(repeats):
            t0 = time.perf_counter()
            R.unet_forward(sdu, R.SD_UNET_CFG, x, t, ctx)
            tu.append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            R.autoencoder_decode(sdv, R.SD_VAE_DDCONFIG, x)
            td.append(time.perf_counter() - t0)
    t_unet, t_dec = min(tu), min(td)
    return 1.0 / (ddim_steps * t_unet + t_dec), cores, t_unet, t_dec


def workload_config(ddim_steps, per_gpu_batch, global_batch):
    """`config` of the C2 workload: the SAME dict in both arms (the driver compares them key by key)."""
    return {"workload": "SD-1.x UNet DDIM-%d + VAE decode, 64x64x4 latent -> 512x512x3, ctx 77x768, batch %d per GPU" % (ddim_steps, per_gpu_batch),
            "global_batch": global_batch, "per_gpu_batch": per_gpu_batch,
            "l2": "no flush between steps: one step touches 1.7 GB of bf16 weights per UNet call x 50 calls + activations, far more than the 126 MB L2"}


def run_reference(a):
    """Reference arm: the reference's own CPU PyTorch path (its oracle restatement — the Python reference cannot travel to
    the GPU box) on all host threads, same metric / unit / workload as the sdb200 arm.  One "step" of the workload is a
    batch of `--batch` images (DDIM-50 + decode); each of the W + K steps times a BOUNDED SAMPLE of it — one UNet call and
    one VAE decode at B=1 — and extrapolates t_image = ddim_steps * t_unet + t_decode (nothing on the path reduces over
    the batch).  The K timed samples are averaged."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    B = a.batch
    world = max(1, a.gpus)
    per_image = []
    for i in range(max(0, a.warmup) + max(1, a.steps)):
        ips1, cores, t_unet, t_dec = cpu_reference_images_per_s(a.ddim_steps, repeats=1)
        if i >= a.warmup:
            per_image.append((1.0 / ips1, t_unet, t_dec))
    t_img = sum(p[0] for p in per_image) / len(per_image)
    t_unet = sum(p[1] for p in per_image) / len(per_image)
    t_dec = sum(p[2] for p in per_image) / len(per_image)
    ips = 1.0 / t_img
    sample = "oracle restatement of the reference PyTorch path, fp32, %d host threads; per step 1 UNet call B=1 (%.2f s) + 1 VAE " \
             "decode B=1 (%.2f s), extrapolated: t_image = %d*t_unet + t_decode, step = %d images" % (cores, t_unet, t_dec, a.ddim_steps, B)
    line = {
        "impl": "reference", "metric": "512px DDIM-50 images/sec", "value": ips, "unit": "images/s", "n_gpus": a.gpus,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1000.0 * t_img * B, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(a.ddim_steps, B, B * world),
        "note": "host CPU only (one process, rank 0): the value does not grow with n_gpus",
        "cpu_baseline": {"value": ips, "unit": "images/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": ips, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------
# sdb200 arm
# ------------------------------------------------------------------------------------------------------
def run_sdb200(a):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import __graft_entry__ as ge
    if rank == 0:
        ge.build()
    if world > 1:
        dist.barrier()
    from sdb200 import _lib
    from sdb200.distributed import gather_images, per_sample_randn, shard_range
    from sdb200.pipeline import LatentDiffusion
    lib = _lib.load()

    B = a.batch
    GB = B * world
    torch.manual_seed(0)
    ld = LatentDiffusion(compute_mode=a.mode)
    # random-init weights; zero_module'd layers re-initialised so eps is not identically 0
    for m in ld.modules():
        if isinstance(m, (torch.nn.Conv2d, torch.nn.Linear)) and float(m.weight.detach().abs().max()) == 0.0:
            m.reset_parameters()
    ld = ld.to(dev)
    unet = ld.model.diffusion_model
    unet.use_cuda_graph = not a.no_graph

    lo, hi = shard_range(GB, rank, world)
    x_host = per_sample_randn(range(lo, hi), (4, 64, 64), 1000).pin_memory()
    c_host = per_sample_randn(range(lo, hi), (77, 768), 2000).pin_memory()
    img_host = torch.empty((hi - lo, 3, 512, 512), dtype=torch.float32).pin_memory()

    def one_step_device(x_T, ctx):
        # a fresh conditioning tensor per batch: the UNet projects the context's K / V once per DDIM-50 run (the
        # context is the same for its 50 calls) and must not carry them over from the previous batch
        ctx = ctx.clone()
        z, img = ld.txt2img(ctx, hi - lo, ddim_steps=a.ddim_steps, shape=(4, 64, 64), x_T=x_T)
        if world > 1:
            img = gather_images(img, GB)
        return img

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    x_dev, c_dev = x_host.to(dev), c_host.to(dev)
    for _ in range(a.warmup):
        one_step_device(x_dev, c_dev)
    sync_all()

    # ---- timed region 1: inputs resident in HBM ("value") ----
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = lib.sdb_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    ev0.record()
    for _ in range(a.steps):
        one_step_device(x_dev, c_dev)
    ev1.record()
    sync_all()
    ms = ev0.elapsed_time(ev1)
    launches_eager = lib.sdb_launch_count() - l0

    # ---- timed region 2: end to end through the public API with HOST buffers ("e2e") ----
    sync_all()
    ev2, ev3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev2.record()
    for _ in range(a.steps):
        xd = x_host.to(dev, non_blocking=True)
        cd = c_host.to(dev, non_blocking=True)
        img = one_step_device(xd, cd)
        img_host.copy_(img[lo:hi] if world > 1 else img, non_blocking=True)
    ev3.record()
    sync_all()
    ms_e2e = ev2.elapsed_time(ev3)
    sampler.stop_flag = True

    t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = float(t[0]), float(t[1])

    # ---- UNet step latency + roofline of the dominant kernel (tcgen05 contraction), device events ----
    roof, roof_hbm, unet_ms, launches_per_unet = None, None, None, None
    if rank == 0:
        unet.use_cuda_graph = not a.no_graph
        tt = torch.full((B,), 500, device=dev, dtype=torch.long)
        for _ in range(3):
            unet(x_dev, tt, c_dev)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            unet(x_dev, tt, c_dev)
        e1.record()
        torch.cuda.synchronize()
        unet_ms = e0.elapsed_time(e1) / 10
        unet.use_cuda_graph = False
        # per-launch durations: every kernel alone on the device (the side streams of the graph — time embedding, ResBlock skip
        # convs — overlap launches, which speeds the step up but makes the overlapped kernels' own brackets longer)
        side = (unet.emb_side_stream, unet.skip_side_stream)
        unet.emb_side_stream = unet.skip_side_stream = False
        try:
            roof, roof_hbm, launches_per_unet = roofline_pass(lambda: unet(x_dev, tt, c_dev), "unet")
        finally:
            unet.emb_side_stream, unet.skip_side_stream = side
        unet.use_cuda_graph = not a.no_graph

    if rank == 0:
        tf_peak, hbm_peak, which = peaks()
        ips = GB * a.steps / (ms / 1000.0)
        ips_e2e = GB * a.steps / (ms_e2e / 1000.0)
        flop_per_image = (a.ddim_steps * UNET_GFLOP_PER_SAMPLE + VAE_GFLOP_PER_IMAGE) * 1e9
        # launches: eager count is exact; under graph replay the UNet's launches are replayed, not re-issued
        if launches_per_unet is not None and not a.no_graph:
            gl = int(launches_eager + a.steps * a.ddim_steps * launches_per_unet)
        else:
            gl = int(launches_eager)
        line = {
            "metric": "512px DDIM-50 images/sec", "value": ips, "unit": "images/s", "n_gpus": world, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": a.mode if a.mode != "fp32" else "f32", "data": "synthetic",
            "config": workload_config(a.ddim_steps, B, GB),
            "run": {"cuda_graph": not a.no_graph,
                    "context_kv": "to_k/to_v of the context projected once per DDIM-50 run (every batch), not per UNet call"},
            "unet_step_ms": unet_ms,
            "model_tflops_per_gpu": ips / world * flop_per_image / 1e12,
            "model_frac_of_tensor_peak": ips / world * flop_per_image / 1e12 / tf_peak,
            "e2e": {"value": ips_e2e, "unit": "images/s", "h2d_bytes_per_step": int(x_host.numel() * 4 + c_host.numel() * 4),
                    "d2h_bytes_per_step": int(img_host.numel() * 4)},
            "gpu_launches": gl,
            "clocks": sampler.summary(),
            "roofline": roof,
            "roofline_hbm": roof_hbm,
            "peaks": {"bf16_tflops": tf_peak, "hbm_gbs": hbm_peak, "source": which},
        }
        if not a.skip_cpu_baseline:
            cips, cores, t_unet, t_dec = cpu_reference_images_per_s(a.ddim_steps)
            line["cpu_baseline"] = {"value": cips, "unit": "images/s", "cores": cores, "kind": "port",
                                    "sample": "oracle restatement (fp32 PyTorch CPU): 1 UNet call B=1 %.2f s + 1 VAE decode B=1 %.2f s; "
                                              "images/s = 1/(%d*t_unet+t_dec)" % (t_unet, t_dec, a.ddim_steps)}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def roofline_pass(run, label):
    """One eager call of `run` with CUDA events around every launch of (a) the tcgen05 contraction — the dominant kernel — and
    (b) the GroupNorm / LayerNorm kernels, the bandwidth class.  Tensor roofline: achieved = algorithmic FLOP (2*M*N*K*taps,
    from the launch arguments) / summed launch durations, against the measured sustained bf16 peak.  HBM roofline: achieved =
    algorithmic bytes (each element read once as fp32 and written once in the output dtype, plus the raw bf16 copy when the
    same pass emits one) / summed launch durations, against the measured copy bandwidth."""
    import torch
    from sdb200 import _lib
    lib = _lib.load()
    tc, bw, at = [], [], []
    names = ("sdb_tc_contract", "sdb_groupnorm_nhwc", "sdb_groupnorm_from_colstats", "sdb_layernorm", "sdb_attention_fwd")
    orig = {n: getattr(lib, n) for n in names}

    def ev_pair():
        return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    replay_tc, replay_bw = [], []          # the launches of each class with their original arguments, in issue order

    def w_tc(argp, stream):
        a = argp._obj
        e0, e1 = ev_pair()
        e0.record()
        rc = orig["sdb_tc_contract"](argp, stream)
        e1.record()
        tc.append((2.0 * a.M * a.N * a.K, e0, e1))
        replay_tc.append(type(a).from_buffer_copy(a))
        return rc

    def w_gn(*args):          # x0, C0, x1, C1, N, HW, groups, eps, gamma, beta, gbs, act, exact, out, out_dtype, raw, ...
        e0, e1 = ev_pair()
        e0.record()
        rc = orig["sdb_groupnorm_nhwc"](*args)
        e1.record()
        replay_bw.append(("sdb_groupnorm_nhwc", args))
        elems = float(args[4]) * args[5] * (args[1] + args[3])
        bw.append((elems * (4 + (2 if args[14] == 1 else 4) + (2 if args[15] else 0)), e0, e1, "gn"))
        return rc

    def w_gc(*args):          # x0, C0, cs0, lay0, x1, C1, cs1, lay1, N, HW, groups, eps, gamma, beta, gbs, act, exact, out, out_dtype, raw, ...
        e0, e1 = ev_pair()
        e0.record()
        rc = orig["sdb_groupnorm_from_colstats"](*args)
        e1.record()
        replay_bw.append(("sdb_groupnorm_from_colstats", args))
        elems = float(args[8]) * args[9] * (args[1] + args[5])
        bw.append((elems * (4 + (2 if args[18] == 1 else 4) + (2 if args[19] else 0)), e0, e1, "gn_colstats"))
        return rc

    def w_ln(*args):          # x, rows, C, eps, gamma, beta, out, out_dtype, stream
        e0, e1 = ev_pair()
        e0.record()
        rc = orig["sdb_layernorm"](*args)
        e1.record()
        replay_bw.append(("sdb_layernorm", args))
        bw.append((float(args[1]) * args[2] * (4 + (2 if args[7] == 1 else 4)), e0, e1, "ln"))
        return rc

    def w_at(argp, stream):
        a = argp._obj
        e0, e1 = ev_pair()
        e0.record()
        rc = orig["sdb_attention_fwd"](argp, stream)
        e1.record()
        at.append((4.0 * a.B * a.H * a.Sq * a.Sk * a.d, float(a.B) * a.H * a.Sq * (80 if a.Sk <= 80 else ((a.Sk + 127) // 128) * 128), e0, e1,
                   "self" if a.Sq == a.Sk else "cross"))
        return rc

    for _ in range(2):
        run()
    torch.cuda.synchronize()
    l0 = lib.sdb_launch_count()
    lib.sdb_tc_contract, lib.sdb_groupnorm_nhwc, lib.sdb_groupnorm_from_colstats, lib.sdb_layernorm = w_tc, w_gn, w_gc, w_ln
    lib.sdb_attention_fwd = w_at
    try:
        # park the device behind a ~0.1 s spin so the host enqueues the whole call ahead of it: the events then
        # bracket kernel execution only, not host launch gaps
        torch.cuda._sleep(int(2e8))
        run()
        torch.cuda.synchronize()
    finally:
        for n in names:
            setattr(lib, n, orig[n])
    launches = lib.sdb_launch_count() - l0

    # Second measurement of each class, without the per-launch event brackets: the class's launches are re-issued BACK TO BACK with
    # their original arguments and in their original order (nothing else in between, so consecutive launches overlap through
    # programmatic dependent launch as they do inside the captured graph), 5 passes between ONE pair of events, the device parked
    # while the host runs ahead.  A pass streams the same 1.7 GB of weights through L2 as the real step; activations are not
    # L2-warm (their producers do not run), which is pessimistic.  No allocation happens between the call above and the re-issue, so
    # every pointer in the saved arguments still refers to memory of the same size in the caching allocator.
    import ctypes as C

    def reissue(items, call, passes=5):
        if not items:
            return None
        st = _lib.stream_ptr()
        for it in items:
            call(it, st)
        torch.cuda.synchronize()
        e0, e1 = ev_pair()
        torch.cuda._sleep(int(2e8))
        e0.record()
        for _ in range(passes):
            for it in items:
                call(it, st)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / passes

    ms_tc_b2b = reissue(replay_tc, lambda a, st: orig["sdb_tc_contract"](C.byref(a), st))
    ms_bw_b2b = reissue(replay_bw, lambda it, st: orig[it[0]](*it[1]))
    tf_peak, hbm_peak, which = peaks()
    roof = roof_hbm = None
    if tc:
        flop = sum(r[0] for r in tc)
        ms = sum(r[1].elapsed_time(r[2]) for r in tc)
        ach = flop / (ms / 1000.0) / 1e12
        traffic = None
        tp = os.path.join(ROOT, "profiles", "r02_tc_traffic.json")      # ncu dram bytes per launch of the same kernels
        if not os.path.exists(tp):
            tp = os.path.join(ROOT, "profiles", "r01_tc_traffic.json")
        if os.path.exists(tp) and label == "unet":
            try:
                traffic = json.load(open(tp))["dram_bytes_per_launch"]
            except Exception:
                traffic = None
        roof = {"bound": "tensor", "kernel": "tc_contract_pair_kernel / tc_contract_kernel (tcgen05 implicit-GEMM conv + GEMM), %s" % label,
                "achieved": ach, "peak": tf_peak, "unit": "TFLOP/s", "frac": ach / tf_peak, "traffic": traffic, "launches": len(tc),
                "sum_ms": ms, "algorithmic_gflop": flop / 1e9, "peak_source": which + " (sustained cuBLAS bf16)",
                "method": "sum of per-launch CUDA-event brackets (each bracket carries the event pair's own ~1-2 us: conservative)"}
        if ms_tc_b2b:
            # headline figures = the back-to-back measurement; the per-launch brackets are kept beside it
            roof["bracketed"] = {"sum_ms": roof["sum_ms"], "achieved": roof["achieved"], "frac": roof["frac"], "method": roof["method"]}
            roof["sum_ms"] = ms_tc_b2b
            roof["achieved"] = flop / (ms_tc_b2b / 1000.0) / 1e12
            roof["frac"] = roof["achieved"] / tf_peak
            roof["method"] = ("the %d contraction launches of one call re-issued back to back with their original arguments, in issue order, "
                              "5 passes between ONE pair of CUDA events (device parked while the host runs ahead); average launch "
                              "duration = sum_ms / launches" % len(tc))
    if bw:
        by, ms = sum(r[0] for r in bw), sum(r[1].elapsed_time(r[2]) for r in bw)
        ach = by / (ms / 1000.0) / 1e9
        per = {}
        for b_, e0, e1, kind in bw:
            d = per.setdefault(kind, [0.0, 0.0, 0])
            d[0] += b_
            d[1] += e0.elapsed_time(e1)
            d[2] += 1
        roof_hbm = {"bound": "hbm", "kernel": "GroupNorm(+SiLU) / LayerNorm kernels (gn_apply, gn_cluster, layernorm), %s" % label,
                    "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak, "traffic": None, "launches": len(bw),
                    "sum_ms": ms, "algorithmic_mbytes": by / 1e6, "peak_source": which + " (device copy)",
                    "by_kernel": {k: {"GB/s": v[0] / (v[1] / 1000.0) / 1e9, "ms": v[1], "launches": v[2]} for k, v in per.items()},
                    "convention": "fp32 read once + output written once (bf16 operand, + the raw bf16 copy when emitted)",
                    "method": "sum of per-launch CUDA-event brackets (15-20 us kernels: the ~1-2 us of the event pair deflates this figure)"}
        if ms_bw_b2b:
            roof_hbm["bracketed"] = {"sum_ms": roof_hbm["sum_ms"], "achieved": roof_hbm["achieved"], "frac": roof_hbm["frac"], "method": roof_hbm["method"]}
            roof_hbm["sum_ms"] = ms_bw_b2b
            roof_hbm["achieved"] = by / (ms_bw_b2b / 1000.0) / 1e9
            roof_hbm["frac"] = roof_hbm["achieved"] / hbm_peak
            roof_hbm["method"] = ("the %d GroupNorm / LayerNorm launches of one call re-issued back to back with their original arguments, in issue "
                                  "order, 5 passes between ONE pair of CUDA events" % len(bw))
    if at and roof is not None:
        # attention kernels: tensor roofline on the algorithmic 4*B*H*Sq*Sk*d FLOP, and the exponential rate against the
        # MUFU.EX2 pipe (16 per clock and SM, measured: profiles/r01_xu_rate.txt) at the clock sampled during the timed region
        ms_a = sum(r[2].elapsed_time(r[3]) for r in at)
        fl_a = sum(r[0] for r in at)
        ex_a = sum(r[1] for r in at)
        per = {}
        for fl, ex, e0, e1, kind in at:
            d = per.setdefault(kind, [0.0, 0.0, 0.0, 0])
            d[0] += fl; d[1] += ex; d[2] += e0.elapsed_time(e1); d[3] += 1
        mufu_peak = 16.0 * 148 * 1.92e9
        roof["attention"] = {"kernel": "tc_attention_kernel / tc_attention_kv1_kernel", "launches": len(at), "sum_ms": ms_a,
                             "achieved": fl_a / (ms_a / 1000.0) / 1e12, "unit": "TFLOP/s", "frac": fl_a / (ms_a / 1000.0) / 1e12 / tf_peak,
                             "exp_per_s": ex_a / (ms_a / 1000.0), "mufu_frac": ex_a / (ms_a / 1000.0) / mufu_peak,
                             "mufu_peak": "16 ex2 / clk / SM x 148 SMs x 1.92 GHz",
                             "by_kind": {k: {"TFLOP/s": v[0] / (v[2] / 1000.0) / 1e12, "mufu_frac": v[1] / (v[2] / 1000.0) / mufu_peak,
                                             "ms": v[2], "launches": v[3]} for k, v in per.items()}}
    return roof, roof_hbm, launches


# ------------------------------------------------------------------------------------------------------
# the other BASELINE.json configs, driver-runnable: --config c3 | c5 | c4-strong
# ------------------------------------------------------------------------------------------------------
def _dist_setup():
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import __graft_entry__ as ge
    if rank == 0:
        ge.build()
    if world > 1:
        dist.barrier()
    return rank, world, local, dev


def _reinit_zero_modules(mod):
    import torch
    for m in mod.modules():
        if isinstance(m, (torch.nn.Conv2d, torch.nn.Linear)) and float(m.weight.detach().abs().max()) == 0.0:
            m.reset_parameters()


def _timed_steps(fn, steps, warmup, world):
    """W untimed + K timed calls of fn bracketed by barrier + synchronize, CUDA events, MAX over ranks (ms for the K steps)."""
    import torch
    import torch.distributed as dist

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    for _ in range(max(3, warmup)):
        fn()
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    sync_all()
    t = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t[0])


def run_c3(a):
    """BASELINE configs[2]: VAE decode 64x64x4 -> 512x512x3, batch 16 per GPU (micro-batches of 8): images/s, tensor roofline of
    the contractions and HBM roofline of the GroupNorm passes of one decode."""
    import torch
    rank, world, local, dev = _dist_setup()
    from sdb200 import _lib
    from sdb200.autoencoder import AutoencoderKL
    from sdb200.distributed import per_sample_randn, shard_range
    from sdb200.pipeline import SD_VAE_DDCONFIG
    lib = _lib.load()
    B = 16 if a.batch == 8 else a.batch
    torch.manual_seed(0)
    vae = AutoencoderKL(ddconfig=SD_VAE_DDCONFIG, embed_dim=4, compute_mode=a.mode).to(dev)
    lo, hi = shard_range(B * world, rank, world)
    z_host = per_sample_randn(range(lo, hi), (4, 64, 64), 4000).pin_memory()
    img_host = torch.empty((B, 3, 512, 512), dtype=torch.float32).pin_memory()
    z_dev = z_host.to(dev)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = lib.sdb_launch_count()
    ms = _timed_steps(lambda: vae.decode(z_dev), a.steps, a.warmup, world)
    launches = int((lib.sdb_launch_count() - l0) * a.steps / (a.steps + max(3, a.warmup)))

    def e2e():
        img = vae.decode(z_host.to(dev, non_blocking=True))
        img_host.copy_(img, non_blocking=True)
    ms_e2e = _timed_steps(e2e, a.steps, 1, world)
    sampler.stop_flag = True
    if rank != 0:
        return
    roof, roof_hbm, _ = roofline_pass(lambda: vae.decode(z_dev[:8]), "vae decode, batch 8")
    tf_peak, hbm_peak, which = peaks()
    ips = B * world * a.steps / (ms / 1000.0)
    line = {
        "metric": "VAE decode 512px images/sec", "value": ips, "unit": "images/s", "n_gpus": world, "steps": a.steps, "warmup": max(3, a.warmup),
        "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": a.mode if a.mode != "fp32" else "f32", "data": "synthetic",
        "config": {"workload": "ldm VAE Decoder, latent 64x64x4 -> 512x512x3, batch %d per GPU (BASELINE.json configs[2])" % B,
                   "global_batch": B * world, "per_gpu_batch": B, "micro_batch": vae.micro_batch,
                   "l2": "one decode touches ~5 GB of activations per micro-batch, far beyond the 126 MB L2; no flush"},
        "model_tflops_per_gpu": ips / world * VAE_GFLOP_PER_IMAGE / 1e3,
        "model_frac_of_tensor_peak": ips / world * VAE_GFLOP_PER_IMAGE / 1e3 / tf_peak,
        "e2e": {"value": B * world * a.steps / (ms_e2e / 1000.0), "unit": "images/s", "h2d_bytes_per_step": int(z_host.numel() * 4),
                "d2h_bytes_per_step": int(img_host.numel() * 4)},
        "gpu_launches": launches, "clocks": sampler.summary(), "roofline": roof, "roofline_hbm": roof_hbm,
        "peaks": {"bf16_tflops": tf_peak, "hbm_gbs": hbm_peak, "source": which},
    }
    print(json.dumps(line))


def run_c5(a):
    """BASELINE configs[4]: one UNet step on a 96x96x4 latent (9216 tokens at the top level), batch sweep 1..32: step latency,
    achieved TFLOP/s against the algorithmic 2148.12 GFLOP/sample, and the per-kernel rooflines at batch 8."""
    import torch
    rank, world, local, dev = _dist_setup()
    if rank != 0:
        return
    from sdb200 import _lib
    from sdb200.openai_model import UNetModel
    from sdb200.pipeline import SD_UNET_CONFIG
    lib = _lib.load()
    GF96 = 2148.12
    torch.manual_seed(0)
    net = UNetModel(**SD_UNET_CONFIG, compute_mode=a.mode)
    _reinit_zero_modules(net)
    net = net.to(dev)
    net.use_cuda_graph = not a.no_graph
    tf_peak, hbm_peak, which = peaks()
    sampler = ClockSampler(local)
    sampler.start()
    sweep = []
    launches = 0
    for B in (1, 2, 4, 8, 16, 32):
        x = torch.randn(B, 4, 96, 96, device=dev)
        t = torch.full((B,), 500, device=dev, dtype=torch.long)
        c = torch.randn(B, 77, 768, device=dev)
        ms = _timed_steps(lambda: net(x, t, c), max(a.steps, 5), a.warmup, 1) / max(a.steps, 5)
        tf = B * GF96 / ms
        sweep.append({"batch": B, "ms": ms, "tflops": tf, "frac_of_tensor_peak": tf / tf_peak})
        if B == 8:
            x_host, c_host = x.cpu().pin_memory(), c.cpu().pin_memory()
            out_host = torch.empty((B, 4, 96, 96)).pin_memory()

            def e2e():
                out_host.copy_(net(x_host.to(dev, non_blocking=True), t, c_host.to(dev, non_blocking=True)), non_blocking=True)
            ms_e2e = _timed_steps(e2e, max(a.steps, 5), 1, 1) / max(a.steps, 5)
            net.use_cuda_graph = False
            side = (net.emb_side_stream, net.skip_side_stream)      # per-launch durations: every kernel alone on the device
            net.emb_side_stream = net.skip_side_stream = False
            try:
                roof, roof_hbm, launches = roofline_pass(lambda: net(x, t, c), "unet 96x96, batch 8")
            finally:
                net.emb_side_stream, net.skip_side_stream = side
            net.use_cuda_graph = not a.no_graph
    sampler.stop_flag = True
    b8 = [r for r in sweep if r["batch"] == 8][0]
    line = {
        "metric": "UNet step latency ms (96x96 latent, batch 8)", "value": b8["ms"], "unit": "ms", "n_gpus": 1, "steps": max(a.steps, 5),
        "warmup": max(3, a.warmup), "ms_per_step": b8["ms"], "higher_is_better": False, "scaling": "weak", "vs_baseline": None,
        "dtype": a.mode if a.mode != "fp32" else "f32", "data": "synthetic",
        "config": {"workload": "SD-1.x UNetModel forward, latent 96x96x4 (768 px), ctx 77x768, batch sweep 1-32 (BASELINE.json configs[4])",
                   "global_batch": 8, "cuda_graph": not a.no_graph, "algorithmic_gflop_per_sample": GF96,
                   "l2": "1.7 GB of bf16 weights streamed per call; no flush"},
        "sweep": sweep,
        "e2e": {"value": ms_e2e, "unit": "ms", "h2d_bytes_per_step": int(8 * 4 * 96 * 96 * 4 + 8 * 77 * 768 * 4), "d2h_bytes_per_step": int(8 * 4 * 96 * 96 * 4)},
        "gpu_launches": int(launches * max(a.steps, 5)), "clocks": sampler.summary(), "roofline": roof, "roofline_hbm": roof_hbm,
        "peaks": {"bf16_tflops": tf_peak, "hbm_gbs": hbm_peak, "source": which},
    }
    print(json.dumps(line))


def run_c4_strong(a):
    """BASELINE configs[3] as STRONG scaling: a fixed global batch of 64 images (DDIM-50 + decode), sample i seeded by its global
    index, sharded contiguously over the N GPUs, each rank running its 64/N samples in batches of 8; one NCCL all-gather of
    the decoded images at the end."""
    import torch
    rank, world, local, dev = _dist_setup()
    from sdb200 import _lib
    from sdb200.distributed import gather_images, per_sample_randn, shard_range
    from sdb200.pipeline import LatentDiffusion
    lib = _lib.load()
    GB = 64
    torch.manual_seed(0)
    ld = LatentDiffusion(compute_mode=a.mode)
    _reinit_zero_modules(ld)
    ld = ld.to(dev)
    ld.model.diffusion_model.use_cuda_graph = not a.no_graph
    lo, hi = shard_range(GB, rank, world)
    x_host = per_sample_randn(range(lo, hi), (4, 64, 64), 1000).pin_memory()
    c_host = per_sample_randn(range(lo, hi), (77, 768), 2000).pin_memory()
    # micro-batch: the whole per-GPU share up to 32 images per UNet call.  A sample's bits do not depend on the batch it is in
    # (tests/test_gpu_models.py); 32 images per call are ~7 % cheaper per image than 8 per call (measured: 15.6 vs 14.6 images/s
    # at N = 1).  --micro-batch 8 reproduces the per-call batch of the weak-scaling line.
    mb = min(a.micro_batch if a.micro_batch > 0 else 32, hi - lo)

    def step():
        imgs = []
        for i in range(0, hi - lo, mb):
            xd = x_host[i:i + mb].to(dev, non_blocking=True)
            cd = c_host[i:i + mb].to(dev, non_blocking=True)
            imgs.append(ld.txt2img(cd, xd.shape[0], ddim_steps=a.ddim_steps, shape=(4, 64, 64), x_T=xd)[1])
        img = torch.cat(imgs, 0) if len(imgs) > 1 else imgs[0]
        return gather_images(img, GB) if world > 1 else img
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = lib.sdb_launch_count()
    # warm-up: W >= 3 passes over ONE micro-batch (graph capture, weight packing), then the timed full-batch steps
    xw, cw = x_host[:mb].to(dev), c_host[:mb].to(dev)
    for _ in range(max(3, a.warmup)):
        ld.txt2img(cw, xw.shape[0], ddim_steps=a.ddim_steps, shape=(4, 64, 64), x_T=xw)
    import torch.distributed as dist
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.steps):
        step()
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0])
    sampler.stop_flag = True
    if rank == 0:
        tf_peak, hbm_peak, which = peaks()
        ips = GB * a.steps / (ms / 1000.0)
        flop_per_image = (a.ddim_steps * UNET_GFLOP_PER_SAMPLE + VAE_GFLOP_PER_IMAGE) * 1e9
        line = {
            "metric": "512px DDIM-50 images/sec", "value": ips, "unit": "images/s", "n_gpus": world, "steps": a.steps, "warmup": max(3, a.warmup),
            "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": a.mode if a.mode != "fp32" else "f32", "data": "synthetic",
            "config": {"workload": "SD-1.x UNet DDIM-%d + VAE decode, 64x64x4 latent -> 512x512x3, ctx 77x768, FIXED global batch 64 sharded "
                                   "over the GPUs, %d images per UNet call (BASELINE.json configs[3])" % (a.ddim_steps, mb),
                       "global_batch": GB, "per_gpu_batch": hi - lo, "micro_batch": mb, "cuda_graph": not a.no_graph,
                       "warmup_note": "warm-up passes run one micro-batch (graph capture, packing); every timed step runs the full 64",
                       "l2": "1.7 GB bf16 weights streamed per UNet call; no flush"},
            "model_tflops_per_gpu": ips / world * flop_per_image / 1e12,
            "model_frac_of_tensor_peak": ips / world * flop_per_image / 1e12 / tf_peak,
            "e2e": {"value": ips, "unit": "images/s", "h2d_bytes_per_step": int(x_host.numel() * 4 + c_host.numel() * 4), "d2h_bytes_per_step": 0,
                    "note": "inputs start in pinned host memory and are copied per micro-batch inside the timed region; the gathered "
                            "images stay on the device"},
            "gpu_launches": int(lib.sdb_launch_count() - l0), "clocks": sampler.summary(),
            "limiting_term": "per-GPU work is 64/N images in calls of min(32, 64/N); the per-image UNet cost is 1.22 ms at 32 per call and "
                             "1.24-1.31 ms at 8 per call (N = 8, the weak-scaling point), so strong scaling is within ~7 % of linear; the "
                             "all-gather of 201 MB of fp32 images is the only collective",
            "peaks": {"bf16_tflops": tf_peak, "hbm_gbs": hbm_peak, "source": which},
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    elif a.config == "c3":
        run_c3(a)
    elif a.config == "c5":
        run_c5(a)
    elif a.config == "c4-strong":
        run_c4_strong(a)
    else:
        run_sdb200(a)


if __name__ == "__main__":
    main()
