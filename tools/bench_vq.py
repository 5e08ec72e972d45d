#!/usr/bin/env python
"""Cost of the VQ first stage's quantizer (sdb_vq_quantize) against the reference's torch expression, and its share of
a VQModelInterface decode.

    python tools/bench_vq.py [--launches 200] [--reps 5] [--decode-iters 10]

(a) For D = 3, n_e in {8192, 16384} and M in {4096, 32768} latent pixels (1 and 8 images of 64x64): per-launch time of
    ops.vq_quantize (NCHW in, NCHW z_q, int64 indices, the loss), `launches` launches replayed from one CUDA graph, timed
    with CUDA events; beside it the reference's expression (VectorQuantizer2.forward: fp32 distance matrix, argmin, gather,
    loss, straight-through) in eager torch on the same inputs, TF32 off, and the share of rows where the two pick the
    same code.  Derived: code-distance pairs per second, and the FP32-pipe share = M * n_e * (2D + 2) flop over
    148 SMs * 128 lanes * 2 flop * the maximum SM clock read in the same run (clocks.max.sm).
(b) VQModelInterface.decode of batch 8 (3x64x64 latents -> 3x256x256 images; ch=128, ch_mult=(1,2,4), 2 res blocks,
    attn_type none, n_embed 8192), bf16, with and without force_not_quantize: the quantizer's share of a decode.
Every timing is repeated `reps` times, alternating the compared variants; medians are reported with the range.  The
inputs (<= 0.4 MB) stay in L2.  Prints one JSON line with the GPU name and power limit; writes nothing.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SMS, LANES = 148, 128


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=20).stdout.strip()
        return [s.strip() for s in out.split(",")[:4]]
    except Exception as e:          # the timing does not depend on it; say why it is missing
        return [None, "unavailable (%s)" % e, None, None]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--decode-iters", type=int, default=10)
    a = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_vq.py needs a CUDA device")
    import __graft_entry__ as ge
    ge.build()
    from oracle import weights as W
    from sdb200 import ops
    from sdb200.autoencoder import VQModelInterface

    torch.backends.cuda.matmul.allow_tf32 = False
    torch.cuda.set_device(0)
    med = lambda v: sorted(v)[len(v) // 2]

    def timed(fn, n=1):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    def torch_quantize(z, Wc, beta=0.25):
        D = Wc.shape[1]
        zh = z.permute(0, 2, 3, 1).contiguous()
        zf = zh.view(-1, D)
        d = torch.sum(zf ** 2, dim=1, keepdim=True) + torch.sum(Wc ** 2, dim=1) - 2 * torch.einsum("bd,dn->bn", zf, Wc.t())
        idx = torch.argmin(d, dim=1)
        e = Wc[idx].view(zh.shape)
        loss = torch.mean((e - zh) ** 2) + beta * torch.mean((e - zh) ** 2)
        return (zh + (e - zh)).permute(0, 3, 1, 2).contiguous(), idx, loss

    name, power, clk_max, clk_now = gpu_info()
    clk_hz = float(clk_max.split()[0]) * 1e6 if clk_max else None
    D = 3
    rows = []
    for n_img in (1, 8):
        for n_e in (8192, 16384):
            M = n_img * 64 * 64
            g = torch.Generator().manual_seed(n_e + n_img)
            z = torch.randn(n_img, D, 64, 64, generator=g).cuda()
            Wc = (torch.rand(n_e, D, generator=g) * 2 - 1).cuda()
            ops.vq_quantize(z, Wc)
            torch_quantize(z, Wc)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                for _ in range(a.launches):
                    ops.vq_quantize(z, Wc)
            graph.replay()
            t_k, t_t = [], []
            for _ in range(a.reps):
                t_k.append(1e3 * timed(graph.replay) / a.launches)
                t_t.append(1e3 * timed(lambda: torch_quantize(z, Wc), max(10, a.launches // 10)))
            _, idx_k, _ = ops.vq_quantize(z, Wc)
            _, idx_t, _ = torch_quantize(z, Wc)
            us = med(t_k)
            flop = M * n_e * (2 * D + 2)
            rows.append({
                "M": M, "n_e": n_e, "D": D,
                "kernel_us": round(us, 2), "kernel_us_range": [round(min(t_k), 2), round(max(t_k), 2)],
                "torch_us": round(med(t_t), 2), "torch_us_range": [round(min(t_t), 2), round(max(t_t), 2)],
                "speedup": round(med(t_t) / us, 2),
                "index_agreement": round(float((idx_k == idx_t).double().mean()), 6),
                "gpairs_per_s": round(M * n_e / (us * 1e-6) / 1e9, 1),
                "fp32_pipe_share": round(flop / (SMS * LANES * 2 * clk_hz * us * 1e-6), 4) if clk_hz else None,
            })

    # (b) decode of batch 8 with the f4 first stage
    dd = dict(double_z=False, z_channels=3, resolution=256, in_channels=3, out_ch=3, ch=128, ch_mult=(1, 2, 4),
              num_res_blocks=2, attn_resolutions=[], dropout=0.0, attn_type="none")
    fs = VQModelInterface(3, ddconfig=dd, lossconfig=None, n_embed=8192, compute_mode="bf16")
    fs.load_state_dict(W.make_state_dict(W.key_shapes_of(fs), 3))
    fs = fs.cuda()
    h = W.seeded_randn((8, 3, 64, 64), 4).cuda()
    fs.decode(h)
    fs.decode(h, force_not_quantize=True)
    t_q, t_nq = [], []
    for _ in range(a.reps):
        t_q.append(timed(lambda: fs.decode(h), a.decode_iters))
        t_nq.append(timed(lambda: fs.decode(h, force_not_quantize=True), a.decode_iters))
    q, nq = med(t_q), med(t_nq)
    print(json.dumps({
        "metric": "vq_quantize",
        "quantize": rows, "launches": a.launches, "reps": a.reps,
        "decode_b8_bf16_ms": round(q, 3), "decode_b8_bf16_ms_range": [round(min(t_q), 3), round(max(t_q), 3)],
        "decode_b8_bf16_force_not_quantize_ms": round(nq, 3),
        "decode_b8_bf16_force_not_quantize_ms_range": [round(min(t_nq), 3), round(max(t_nq), 3)],
        "quantizer_share_of_decode_pct": round(100.0 * (q - nq) / q, 2),
        "sm_clock_for_fp32_share": "clocks.max.sm %s (clocks.sm at read time %s)" % (clk_max, clk_now),
        "gpu": name, "power_limit": power,
    }))


if __name__ == "__main__":
    main()
