#!/usr/bin/env python
"""Shape sweep of the fused view-attention pair (fwd + bwd) through the C ABI.

    python tools/bench_shapes.py [--only NAME,...] [--iters K] [--out gpurun_out/shapes.json]

One JSON line per shape: ms per launch (CUDA events on the launching stream, L2 flushed by a
256 MB memset between iterations), algorithmic bytes (SURVEY.md 8d) and fraction of the measured
HBM peak.  Shapes: the BASELINE.json stress sweep (1 M points x {8,16,32,64} views x 128 ch), ragged
counts, bf16 storage, and the per-step shapes of the shipped configs (SURVEY.md Appendix E:
S3DIS 4 x 40 k spheres x ~8 views x 64 ch, KITTI-360 80 k x ~20 views x 128 ch, C = 32 / 512 branches).
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

SHAPES = [
    # name, points, mean views, channels, dtype, counts, idx
    ("stress_v8", 1_000_000, 8, 128, "f32", "uniform", "randperm"),
    ("stress_v16", 1_000_000, 16, 128, "f32", "uniform", "randperm"),
    ("stress_v32", 1_000_000, 32, 128, "f32", "uniform", "randperm"),
    ("stress_v64", 1_000_000, 64, 128, "f32", "uniform", "randperm"),
    ("stress_v32_ragged", 1_000_000, 32, 128, "f32", "ragged", "randperm"),
    ("stress_v32_bf16", 1_000_000, 32, 128, "bf16", "uniform", "randperm"),
    ("stress_v32_bf16_ragged", 1_000_000, 32, 128, "bf16", "ragged", "randperm"),
    ("stress_v8_ragged", 1_000_000, 8, 128, "f32", "ragged", "randperm"),
    ("s3dis_160k_v8_c64", 160_000, 8, 64, "f32", "ragged", "randperm"),
    ("s3dis_160k_v8_c64_bf16", 160_000, 8, 64, "bf16", "ragged", "randperm"),
    ("kitti_80k_v20_c128", 80_000, 20, 128, "f32", "ragged", "randperm"),
    ("pyramid_160k_v8_c32", 160_000, 8, 32, "f32", "ragged", "randperm"),
    ("early_160k_v8_c512", 160_000, 8, 512, "f32", "ragged", "randperm"),
    ("sphere_40k_v8_c64", 40_000, 8, 64, "f32", "ragged", "randperm"),
    ("big_1m_v8_c64", 1_000_000, 8, 64, "f32", "ragged", "randperm"),
    ("big_1m_v8_c64_bf16", 1_000_000, 8, 64, "bf16", "ragged", "randperm"),
]


def algorithmic_bytes(N, V, C, G, s):
    fwd = V * (C * s + 4 + 4 * G) + N * (8 + C * s)
    both = V * (3 * C * s + 8 + 12 * G) + N * (2 * C * s + 16)
    return fwd, both - fwd


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default="")
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--groups", type=int, default=4)
    ap.add_argument("--out", default="")
    ap.add_argument("--path", default="auto", choices=["auto", "stream", "ring", "lane"],
                    help="kernels of the pair: auto = the library's per-shape choice, stream = streaming kernels for "
                         "both passes, ring = ring forward + lane backward, lane = streaming forward + lane backward "
                         "(ring / lane only where they apply)")
    args = ap.parse_args()
    from deepviewagg_b200.host_api import ViewAttentionHostPlan
    from deepviewagg_b200 import _lib
    assert _lib.load().dva_view_attention_set_path({"auto": 0, "stream": 1, "ring": 2, "lane": 3}[args.path]) == 0
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        peak = 6650.0
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    only = set(filter(None, args.only.split(",")))
    G = args.groups
    lines = []
    for name, N, v, C, dt, counts_mode, idx_mode in SHAPES:
        if only and name not in only:
            continue
        tdtype = torch.float32 if dt == "f32" else torch.bfloat16
        s = 4 if dt == "f32" else 2
        gen = torch.Generator(device=dev).manual_seed(1234)
        if counts_mode == "uniform":
            counts = torch.full((N,), v, dtype=torch.long, device=dev)
        else:
            counts = torch.poisson(torch.full((N,), float(v), device=dev), generator=gen).clamp(0, 4 * v).long()
            counts[torch.rand(N, device=dev, generator=gen) < 0.1] = 0
        ptr = torch.cat([torch.zeros(1, dtype=torch.long, device=dev), counts.cumsum(0)])
        V = int(ptr[-1].item())
        plan = ViewAttentionHostPlan(N, V, V, C, G, dtype=tdtype, idx_dtype=torch.int32, gating=True,
                                     group_scaling=True, device=dev)
        plan.ptr.copy_(ptr)
        plan.x.copy_(torch.randn(V, C, device=dev, generator=gen).to(tdtype))
        plan.idx.copy_((torch.randperm(V, device=dev, generator=gen) if idx_mode == "randperm"
                        else torch.arange(V, device=dev)).int())
        plan.compat.copy_(torch.randn(V, G, device=dev, generator=gen))
        plan.gate[0].fill_(1.0)
        plan.gate[1].fill_(0.0)
        plan.gout.copy_(torch.randn(N, C, device=dev, generator=gen).to(tdtype))
        for _ in range(args.warmup):
            plan.forward_device()
            plan.backward_device()
        torch.cuda.synchronize()
        K = args.iters
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(K)]
        for k in range(K):
            flush.zero_()
            ev[k][0].record()
            plan.forward_device()
            ev[k][1].record()
            plan.backward_device()
            ev[k][2].record()
        torch.cuda.synchronize()
        fwd = statistics.median(ev[k][0].elapsed_time(ev[k][1]) for k in range(K))
        bwd = statistics.median(ev[k][1].elapsed_time(ev[k][2]) for k in range(K))
        bf, bb = algorithmic_bytes(N, V, C, G, s)
        line = {"shape": name, "points": N, "views_total": V, "channels": C, "groups": G, "dtype": dt,
                "counts": counts_mode, "idx": idx_mode, "path": args.path,
                "fwd_ms": round(fwd, 4), "bwd_ms": round(bwd, 4),
                "fwd_frac": round(bf / (fwd * 1e-3) / 1e9 / peak, 4),
                "bwd_frac": round(bb / (bwd * 1e-3) / 1e9 / peak, 4),
                "step_frac": round((bf + bb) / ((fwd + bwd) * 1e-3) / 1e9 / peak, 4),
                "mpoints_per_s": round(N / ((fwd + bwd) * 1e-3) / 1e6, 2), "peak_gbs": peak}
        print(json.dumps(line), flush=True)
        lines.append(line)
        del plan
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for ln in lines:
                f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
