#!/usr/bin/env python
"""bench.py -- Mpoints/s through the fused view-aggregation forward+backward (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (named in config.workload): the synthetic stress case the metric is quoted on --
1 M points x 32 views x 128 channels fp32 per GPU, Group-pool variant (scores given), gating on,
group scaling on, rows gathered through a random permutation (worst-case locality; SURVEY 8d).
One step = one fused forward + one fused backward over one batch.  Weak scaling: every rank owns an
independent batch; the only collective is the NCCL all-reduce of the pool-parameter gradient bucket
(SURVEY 8e: ~160 KB -- the gate gradients the kernels produce live at its head), issued on a side
stream so that it overlaps the next step's forward.

Timing: a measurement is EXACTLY --steps steps between two CUDA events, bracketed by a barrier and a
device synchronisation on both sides, max over ranks.  By default it is taken once, so the timed steps
are exactly --steps; --rounds R repeats it R times (0: as many rounds as add up to >= 2.5 s) and the
MEDIAN round is reported; every round, the mean and per-rank step statistics are in `consistency`.

--dump-outputs DIR writes what the timed path returned in its last timed step (out [N,C], gx [V,C],
gcompat [V,G], ggate [2,G]) as DIR/<name>.npy in float32, each array capped at 16 MB by a fixed seeded
sample of its rows, so that two builds run with the same arguments can be compared output for output.

value : device-resident throughput (inputs in HBM), CUDA events, max over ranks.
e2e   : the same step through the host-buffer API (deepviewagg_b200.host_api): pinned host inputs
        -> H2D -> fwd -> bwd -> D2H of every result, copies inside the timed region.
roofline : dominant kernel (backward) -- algorithmic bytes / mean launch time vs measured HBM peak.
cpu_baseline / --impl reference : the oracle port of the reference's PyTorch path timed on the host
        cores of this box (the reference is pure Python; its own modules cannot travel to the box).
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "Mpoints/s through view-agg fwd+bwd"
UNIT = "Mpoints/s"

# stdout carries exactly ONE line, the JSON result.  Libraries write to file descriptor 1 behind
# Python's back (NCCL prints "NCCL version ..." there at communicator creation), so fd 1 is pointed
# at stderr for the whole run and the result goes to a private duplicate of the original stdout.
_RESULT_FD = None


def capture_stdout():
    global _RESULT_FD
    if _RESULT_FD is None:
        sys.stdout.flush()
        _RESULT_FD = os.dup(1)
        os.dup2(2, 1)


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        os.write(_RESULT_FD, line)


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=30)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--points", type=int, default=1_000_000)
    p.add_argument("--views", type=int, default=32)
    p.add_argument("--channels", type=int, default=128)
    p.add_argument("--groups", type=int, default=4)
    p.add_argument("--dtype", default="f32", choices=["f32", "bf16"])
    p.add_argument("--idx", default="randperm", choices=["randperm", "arange", "none"])
    p.add_argument("--counts", default="uniform", choices=["uniform", "ragged"])
    p.add_argument("--rounds", type=int, default=1, help="timed repetitions of the K-step region, median reported "
                                                         "(0 = from a 2.5 s budget)")
    p.add_argument("--dump-outputs", default="", metavar="DIR", help="write the outputs of the last timed step as "
                                                                      "DIR/<name>.npy (float32, sampled rows)")
    p.add_argument("--sweep", default="", help="comma list of views per point (BASELINE config #5: 8,16,32,64): extra "
                                               "device-resident measurements under roofline_detail.sweep")
    p.add_argument("--no-variant-b", action="store_true", help="skip the variant-B side measurement (QKVBimodalCSRPool: scores "
                                                              "from K [V,G*D] and Q [N,G*D]; roofline_detail.variant_b)")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-modules", action="store_true", help="skip the whole-module side measurements (roofline_detail.modules)")
    p.add_argument("--no-cpu-baseline", action="store_true")
    return p.parse_args()


def algorithmic_bytes(N, V, C, G, s):
    """SURVEY.md 8(d): 4-byte row index per view, 8-byte pointer per point, fp32 scores."""
    fwd = V * (C * s + 4 + 4 * G) + N * (8 + C * s)
    both = V * (3 * C * s + 8 + 12 * G) + N * (2 * C * s + 16)
    return fwd, both - fwd


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ---------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------
_Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
      "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
      "clocks_event_reasons.sw_power_cap")
_REASONS = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]


class ClockSampler:
    """SM clocks / throttle reasons of the given GPUs, sampled in-process through NVML from a
    background thread of rank 0 (no nvidia-smi children: at N = 8 eight of them initialising NVML
    inside a sub-second timed window was one of the round-1 scaling suspects).  start() is called
    >= 2 s before the timed region; mark()/unmark() delimit the samples that count as "under load"."""

    def __init__(self, gpu_indices, period_s=0.05):
        self.gpus, self.period = list(gpu_indices), period_s
        self.rows, self._stop, self._thread, self._on = [], None, None, False
        self.backend = None

    def _loop_nvml(self):
        import pynvml as nv
        hs = [nv.nvmlDeviceGetHandleByIndex(i) for i in self.gpus]
        bits = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        mx = [nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM) for h in hs]
        while not self._stop.is_set():
            for g, h, m in zip(self.gpus, hs, mx):
                try:
                    sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    self.rows.append((self._on, g, float(sm), float(m), [k for k, b in bits.items() if r & b]))
                except Exception:
                    pass
            self._stop.wait(self.period)

    def start(self):
        import threading
        self._stop = threading.Event()
        try:
            import pynvml as nv
            nv.nvmlInit()
            self.backend = "nvml (in-process thread, rank 0)"
            self._thread = threading.Thread(target=self._loop_nvml, daemon=True)
            self._thread.start()
        except Exception:
            self.backend = None

    def mark(self):
        self._on = True

    def unmark(self):
        self._on = False

    def stop(self):
        if self._thread is not None:
            self._stop.set()
            self._thread.join(timeout=5)
        rows = [r for r in self.rows if r[0]] or self.rows
        if not rows:  # NVML unavailable: one immediate nvidia-smi query so the key is never empty
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={_Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=30)
                for r in out.stdout.splitlines():
                    f = [c.strip() for c in r.split(",")]
                    if f and f[0].isdigit() and int(f[0]) in self.gpus:
                        rows.append((True, int(f[0]), float(f[1]), float(f[2]),
                                     [n for n, v in zip(_REASONS, f[4:8]) if v == "Active"]))
                self.backend = "nvidia-smi (one query after the timed region)"
            except Exception:
                pass
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        per_gpu = {}
        for _, g, sm, _, _ in rows:
            per_gpu.setdefault(g, []).append(sm)
        return {"sm_mhz": statistics.median(r[2] for r in rows), "sm_max_mhz": max(r[3] for r in rows),
                "reasons": sorted({x for r in rows for x in r[4]}), "samples": len(rows),
                "per_gpu_sm_mhz_median": {str(g): statistics.median(v) for g, v in sorted(per_gpu.items())},
                "source": self.backend}


# ---------------------------------------------------------------------------------------------------
# CPU arm: oracle port of the reference path (pooling.py:285-300 chain + modules.py:518 gather)
# ---------------------------------------------------------------------------------------------------
def cpu_problem(n_points, views, C, G, seed=1234):
    gen = torch.Generator().manual_seed(seed)
    V = n_points * views
    return dict(
        x=torch.randn(V, C, generator=gen), idx=torch.randperm(V, generator=gen),
        compat=torch.randn(V, G, generator=gen), ptr=torch.arange(0, V + 1, views),
        gw=torch.ones(1, G), gb=torch.zeros(1, G), gout=torch.randn(n_points, C, generator=gen))


def cpu_step(pr, G):
    from oracle import pooling_oracle as O
    x = pr["x"].requires_grad_(True)
    c = pr["compat"].requires_grad_(True)
    gw = pr["gw"].requires_grad_(True)
    gb = pr["gb"].requires_grad_(True)
    out, _ = O.view_attention(x, c, pr["ptr"], G, idx=pr["idx"], gate_weight=gw, gate_bias=gb,
                              group_scaling=True)
    torch.autograd.grad(out, [x, c, gw, gb], grad_outputs=pr["gout"])


REFERENCE_SAMPLE_POINTS = 100_000     # fixed: identical `config` on every box and at every N


def cpu_threads():
    """Threads the CPU arm may really use: logical CPUs this process is allowed on, capped by the
    cgroup CPU quota (os.cpu_count() reports the host's CPUs even inside a limited container)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except Exception:
        pass
    return n


def cpu_best_threads(views, C, G):
    """The reference arm gets its best thread count: a quick probe (one warm step + one timed step of
    20 000 points each) at {all, 64, 32, 16} allowed threads.  Round 1 ran 128 threads over dozens of
    small torch ops and measured seconds of size-independent cost per step; the sample itself is fixed."""
    avail = cpu_threads()
    cands = sorted({t for t in (avail, 64, 32, 16) if t <= avail}, reverse=True)
    if len(cands) == 1:
        return cands[0], {}
    pr = cpu_problem(20_000, views, C, G)
    probe = {}
    for t in cands:
        torch.set_num_threads(t)
        cpu_step(pr, G)
        t0 = time.perf_counter()
        cpu_step(pr, G)
        probe[t] = time.perf_counter() - t0
    best = min(probe, key=probe.get)
    return best, {str(k): round(v, 3) for k, v in probe.items()}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    C, G, v = args.channels, args.groups, args.views
    threads, probe = cpu_best_threads(v, C, G)
    torch.set_num_threads(threads)
    n = REFERENCE_SAMPLE_POINTS
    pr = cpu_problem(n, v, C, G)
    for _ in range(args.warmup):
        cpu_step(pr, G)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_step(pr, G)
    dt = time.perf_counter() - t0
    val = n * args.steps / dt / 1e6
    sample = (f"{n} points x {v} views x {C} ch fp32 per step (fixed sample), fwd+bwd, oracle port of "
              f"pooling.py:285-300 + modules.py:518 on torch CPU, {threads} threads (best of probe {probe})")
    cfg = workload_config(args, int(os.environ.get("WORLD_SIZE", str(args.gpus))))   # the GPU arm's config, verbatim
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def workload_config(args, world):
    return {"workload": f"synthetic stress: {args.points} points x {args.views} views x {args.channels} ch "
                        f"per GPU, Group-pool variant A (scores given), G={args.groups}, gating, "
                        f"group_scaling, idx={args.idx}, counts={args.counts}",
            "points_per_gpu": args.points, "views": args.views, "channels": args.channels,
            "groups": args.groups, "idx": args.idx, "counts": args.counts, "parallelism": f"dp{world}",
            "sample_points": REFERENCE_SAMPLE_POINTS,   # points per step of the CPU reference arm / cpu_baseline leg
            "parity_tolerance": ("fp32: outputs and gradients within 1e-4 relative of the oracle (tests/test_gpu_config_size.py)"
                                 if args.dtype == "f32" else
                                 "bf16 storage, fp32 accumulate: within 1.6e-2 of the tensor's max (2 bf16 ulps) of the fp32 "
                                 "oracle -- reported separately from the 1e-4 fp32 bar"),
            "l2": "inputs (>16 GB per step) exceed the 126 MB L2; no explicit flush needed"}


DUMP_BYTES_PER_ARRAY = 16 << 20      # four arrays: at most 64 MB per dump


def dump_outputs(out_dir, arrays):
    """Write each [rows, cols] device array as out_dir/<name>.npy in float32.  An array larger than
    DUMP_BYTES_PER_ARRAY is replaced by a sample of its rows: the first rows of a seeded permutation,
    in ascending order, so the same shape always samples the same rows."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.reshape(t.shape[0], -1)
        keep = max(1, DUMP_BYTES_PER_ARRAY // (4 * t.shape[1]))
        if t.shape[0] > keep:
            rows = torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values
            t = t[rows.to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def ncu_traffic(args):
    """DRAM bytes per launch measured by ncu for this exact workload (profiles/ncu_traffic.json), or {}."""
    key = (f"points={args.points} views={args.views} channels={args.channels} groups={args.groups} "
           f"dtype={args.dtype} idx={args.idx} counts={args.counts}")
    try:
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "ncu_traffic.json")) as f:
            return json.load(f).get(key, {})
    except (OSError, ValueError):
        return {}


# ---------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------
def main():
    args = parse()
    capture_stdout()
    if args.impl == "reference":
        run_reference_arm(args)
        return

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    from deepviewagg_b200.distributed import bind_to_gpu_numa_node
    numa_info = bind_to_gpu_numa_node(local)         # CPU affinity + memory policy before any pinned allocation
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    from deepviewagg_b200 import _lib
    from deepviewagg_b200.host_api import ViewAttentionHostPlan

    N, v, C, G = args.points, args.views, args.channels, args.groups
    tdtype = torch.float32 if args.dtype == "f32" else torch.bfloat16
    s = 4 if args.dtype == "f32" else 2
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    if args.counts == "uniform":
        counts = torch.full((N,), v, dtype=torch.long, device=dev)
    else:  # clamp(Poisson(v), 0, 4v) with 10 % unseen points (SURVEY 8d)
        counts = torch.poisson(torch.full((N,), float(v), device=dev), generator=gen).clamp(0, 4 * v).long()
        counts[torch.rand(N, device=dev, generator=gen) < 0.1] = 0
    ptr = torch.cat([torch.zeros(1, dtype=torch.long, device=dev), counts.cumsum(0)])
    V = int(ptr[-1].item())
    idx_dtype = None if args.idx == "none" else torch.int32
    plan = ViewAttentionHostPlan(N, V, V, C, G, dtype=tdtype, idx_dtype=idx_dtype, gating=True,
                                 group_scaling=True, device=dev)
    plan.ptr.copy_(ptr)
    plan.x.copy_(torch.randn(V, C, device=dev, generator=gen).to(tdtype))
    if args.idx == "randperm":
        plan.idx.copy_(torch.randperm(V, device=dev, generator=gen).int())
    elif args.idx == "arange":
        plan.idx.copy_(torch.arange(V, device=dev).int())
    plan.compat.copy_(torch.randn(V, G, device=dev, generator=gen))
    plan.gate[0].fill_(1.0)
    plan.gate[1].fill_(0.0)
    plan.gout.copy_(torch.randn(N, C, device=dev, generator=gen).to(tdtype))
    torch.cuda.synchronize()

    # ---- the path's only exchange: the pool-parameter gradient bucket (SURVEY 8e) ------------------
    # GroupBimodalCSRPool(in_map=8, in_mod=C, G) has 40 236 parameters at C = 128 (161 KB fp32); the
    # kernels of this step produce the last 2*G of them (G.weight, G.bias), written straight into the
    # bucket; the rest stands in for the encoder gradients a full model step would add.  Two buckets
    # alternate so that the all-reduce of step k (side stream) overlaps forward + backward of step k+1.
    n_bucket = 2 * C * C + 4 * C + 7212 + 2 * G      # E_mod (2 layers + BN) + E_map/E_score + gate
    buckets = [torch.zeros(n_bucket, dtype=torch.float32, device=dev) for _ in range(2)]
    gate_views = [bk[n_bucket - 2 * G:].view(2, G) for bk in buckets]
    side = torch.cuda.Stream(device=dev) if dist is not None else None
    ar_done = [None, None]
    main_stream = torch.cuda.current_stream(dev)
    step_no = [0]

    def step(ev=None):
        k = step_no[0] % 2
        step_no[0] += 1
        if ev is not None:
            ev[0].record()
        plan.forward_device()
        if ev is not None:
            ev[1].record()
        if ar_done[k] is not None:                      # bucket k is being reduced since step-2
            main_stream.wait_event(ar_done[k])
        plan.ggate = gate_views[k]
        plan.backward_device()
        if ev is not None:
            ev[2].record()
        if dist is not None:
            side.wait_stream(main_stream)
            with torch.cuda.stream(side):
                dist.all_reduce(buckets[k])
                ar_done[k] = torch.cuda.Event()
                ar_done[k].record(side)

    def drain():
        if side is not None:
            main_stream.wait_stream(side)

    W_ = max(args.warmup, 3)
    for _ in range(W_):
        step()
    drain()
    torch.cuda.synchronize()

    K = args.steps
    # one measurement = exactly K steps; --rounds 0 sizes the rounds so that the timed regions total >= 2.5 s
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    rounds = args.rounds
    if rounds <= 0:
        e0.record()
        for _ in range(K):
            step()
        drain()
        e1.record()
        torch.cuda.synchronize()
        probe_ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(probe_ms, op=dist.ReduceOp.MAX)
        rounds = int(min(40, max(3, -(-2500.0 // float(probe_ms.item())))))

    sampler = ClockSampler(list(range(int(os.environ.get("LOCAL_WORLD_SIZE", str(world))))) if world > 1
                           else [local]) if rank == 0 else None
    if sampler is not None:
        sampler.start()
    # >= 2 s of the same work before the first timed round: the sampler is up, clocks are settled
    t_pre = time.perf_counter()
    while time.perf_counter() - t_pre < 2.0:
        for _ in range(K):
            step()
        drain()
        torch.cuda.synchronize()

    ev = [[[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(K)] for _ in range(rounds)]
    round_ms = []
    launches = 0
    for r in range(rounds):
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        launches0 = _lib.launch_count()
        if sampler is not None:
            sampler.mark()
        e0.record()
        for k in range(K):
            step(ev[r][k])
        drain()                                          # the last all-reduces finish inside the region
        e1.record()
        torch.cuda.synchronize()
        if sampler is not None:
            sampler.unmark()
        launches = _lib.launch_count() - launches0
        if dist is not None:
            dist.barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        round_ms.append(float(t.item()))
    clocks = sampler.stop() if sampler is not None else None
    if rank == 0 and args.dump_outputs:       # before the side measurements reuse the plan's buffers
        dump_outputs(args.dump_outputs, {"out": plan.out, "gx": plan.gx, "gcompat": plan.gcompat, "ggate": plan.ggate})
    pts = torch.tensor([float(N)], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(pts, op=dist.ReduceOp.SUM)
    total_points = float(pts.item())
    elapsed_ms = statistics.median(round_ms)
    value = total_points * K / (elapsed_ms * 1e-3) / 1e6

    # per-rank step statistics (ms, event-timed start of step k -> start of step k+1) so a straggler is named
    own = []
    for r in range(rounds):
        for k in range(K - 1):
            own.append(ev[r][k][0].elapsed_time(ev[r][k + 1][0]))
    own_t = torch.tensor([min(own), statistics.median(own), max(own)] if own else [0.0, 0.0, 0.0],
                         device=dev, dtype=torch.float64)
    if dist is not None:
        allr = [torch.zeros_like(own_t) for _ in range(world)]
        dist.all_gather(allr, own_t)
    else:
        allr = [own_t]
    per_rank = [{"rank": i, "min": float(t[0]), "median": float(t[1]), "max": float(t[2])} for i, t in enumerate(allr)]
    consistency = {"rounds": rounds, "steps_per_round": K, "round_ms": round_ms,
                   "timed_region_s": sum(round_ms) * 1e-3,
                   "mean_ms_per_step": sum(round_ms) / (rounds * K), "median_ms_per_step": elapsed_ms / K,
                   "min_ms_per_step": min(round_ms) / K, "max_ms_per_step": max(round_ms) / K,
                   "per_rank_step_ms": per_rank,
                   "allreduce": {"elements": n_bucket, "bytes": 4 * n_bucket,
                                 "where": "side stream, overlaps the next step; drained inside the timed region"}
                   if dist is not None else None,
                   "numa": numa_info}

    flat = [e for r in ev for e in r]
    fwd_ms = statistics.mean(e[0].elapsed_time(e[1]) for e in flat)
    bwd_ms = statistics.mean(e[1].elapsed_time(e[2]) for e in flat)
    b_fwd, b_bwd = algorithmic_bytes(N, V, C, G, s)
    peak, peak_src = hbm_peak()
    ach_bwd = b_bwd / (bwd_ms * 1e-3) / 1e9
    ach_fwd = b_fwd / (fwd_ms * 1e-3) / 1e9
    ach_step = (b_fwd + b_bwd) / ((fwd_ms + bwd_ms) * 1e-3) / 1e9
    traffic = ncu_traffic(args)
    roofline = {"bound": "hbm", "kernel": "view_attention_bwd_kernel", "achieved": ach_bwd, "peak": peak,
                "unit": "GB/s", "frac": ach_bwd / peak, "traffic": traffic.get("view_attention_bwd_kernel"),
                "traffic_source": traffic.get("source"), "peak_source": peak_src,
                "algorithmic_bytes_per_launch": b_bwd, "ms_per_launch": bwd_ms}
    extra_roof = {
        "fwd": {"kernel": "view_attention_fwd_kernel", "achieved": ach_fwd, "frac": ach_fwd / peak,
                "traffic": traffic.get("view_attention_fwd_kernel"),
                "algorithmic_bytes_per_launch": b_fwd, "ms_per_launch": fwd_ms},
        "fwd_plus_bwd": {"achieved": ach_step, "frac": ach_step / peak,
                         "algorithmic_bytes": b_fwd + b_bwd, "ms": fwd_ms + bwd_ms}}

    # ---- e2e: host buffers, copies inside the timed region ---------------------------------------
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(args, plan, dist, dev, world, N, V, n_bucket)

    if rank == 0 and world == 1 and args.sweep:
        extra_roof["sweep"] = run_sweep(args, dev, peak, [int(t) for t in args.sweep.split(",") if t])
    if rank == 0 and world == 1 and not args.no_variant_b:
        try:
            extra_roof["variant_b"] = run_variant_b(args, plan, dev, peak, N, V)
        except Exception as e:
            extra_roof["variant_b"] = {"error": f"{type(e).__name__}: {e}"}
    if rank == 0 and world == 1 and not args.no_modules:
        try:
            extra_roof["modules"] = run_module_workloads(dev, peak)
        except Exception as e:  # the graded line must survive a failure of this side measurement
            extra_roof["modules"] = {"error": f"{type(e).__name__}: {e}"}

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # bounded sample: one warm-up + two timed steps of the reference arm's fixed 100 000-point sample
        threads, probe = cpu_best_threads(v, C, G)
        torch.set_num_threads(threads)
        n_cpu = REFERENCE_SAMPLE_POINTS
        pr = cpu_problem(n_cpu, v, C, G)
        cpu_step(pr, G)
        reps = 2
        t0 = time.perf_counter()
        for _ in range(reps):
            cpu_step(pr, G)
        dt = (time.perf_counter() - t0) / reps
        cpu_baseline = {"value": n_cpu / dt / 1e6, "unit": UNIT, "cores": threads, "kind": "port",
                        "sample": f"{n_cpu} points x {v} views x {C} ch fp32 (fixed sample), fwd+bwd, oracle port "
                                  f"of pooling.py:285-300 + modules.py:518 on torch CPU, {threads} threads (best "
                                  f"of probe {probe}), {reps} timed steps after 1 warm-up"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K,
            "warmup": W_, "ms_per_step": elapsed_ms / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
            "config": workload_config(args, world), "clocks": clocks, "e2e": e2e,
            "gpu_launches": int(launches), "roofline": roofline, "roofline_detail": extra_roof,
            "cpu_baseline": cpu_baseline, "consistency": consistency,
        }
        emit(line)
    if dist is not None:
        dist.destroy_process_group()


MODULE_WORKLOADS = {
    # BASELINE.json configs #1 / #3: a whole GroupBimodalCSRPool training step (DeepSetFeat map encoder,
    # E_mod, E_score, fused attention; forward + backward of inputs and parameters)
    "module_s3dis": dict(points=160_000, mean_views=8, channels=64),
    "module_kitti360": dict(points=80_000, mean_views=20, channels=128),
}


def run_module_workloads(dev, peak, steps=20, warmup=5):
    """ms / step of the full pool module at the shipped-config shapes, against the module's own
    algorithmic-byte floor: every input read once, every output / input gradient written once, the view
    features re-read once in backward:  V (3 C s + 96) + N (2 C s + 8)  bytes per step, s = 4."""
    from deepviewagg_b200.modules.multimodal.pooling import GroupBimodalCSRPool
    out = {}
    for name, c in MODULE_WORKLOADS.items():
        N, v, C = c["points"], c["mean_views"], c["channels"]
        gen = torch.Generator(device=dev).manual_seed(4321)
        counts = torch.poisson(torch.full((N,), float(v), device=dev), generator=gen).clamp(0, 4 * v).long()
        counts[torch.rand(N, device=dev, generator=gen) < 0.1] = 0
        ptr = torch.cat([torch.zeros(1, dtype=torch.long, device=dev), counts.cumsum(0)])
        V = int(ptr[-1].item())
        torch.manual_seed(0)
        m = GroupBimodalCSRPool(in_map=8, in_mod=C, num_groups=4, use_mod=False, gating=True, group_scaling=True,
                                map_encoder="DeepSetFeat", use_num=True).to(dev).train()
        x_mod = torch.randn(V, C, device=dev, generator=gen).requires_grad_(True)
        x_map = torch.rand(V, 8, device=dev, generator=gen).requires_grad_(True)
        w = torch.randn(N, C, device=dev, generator=gen)

        def step():
            o = m(None, x_mod, x_map, ptr)
            torch.autograd.backward(o, w)
            x_mod.grad = None
            x_map.grad = None
            for p_ in m.parameters():
                p_.grad = None

        for _ in range(warmup):
            step()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            step()
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / steps
        bytes_ = V * (3 * C * 4 + 96) + N * (2 * C * 4 + 8)
        out[name] = {"points": N, "views": V, "channels": C, "ms_per_step": ms, "mpoints_per_s": N / ms / 1e3,
                     "algorithmic_bytes": bytes_, "achieved_gbs": bytes_ / (ms * 1e-3) / 1e9,
                     "frac": bytes_ / (ms * 1e-3) / 1e9 / peak, "steps": steps,
                     "what": "GroupBimodalCSRPool(use_mod=False, DeepSetFeat, use_num) train step, fwd + bwd, fp32"}
        del m, x_mod, x_map, w
    return out


def run_sweep(args, dev, peak, views_list, steps=10, warmup=3):
    """BASELINE.json config #5: the same fused pair at N points x v views for every v of the sweep (uniform counts,
    random permutation), device-resident, median over `steps` launches."""
    from deepviewagg_b200.host_api import ViewAttentionHostPlan
    tdtype = torch.float32 if args.dtype == "f32" else torch.bfloat16
    s = 4 if args.dtype == "f32" else 2
    N, C, G = args.points, args.channels, args.groups
    out = {}
    for v in views_list:
        V = N * v
        gen = torch.Generator(device=dev).manual_seed(99 + v)
        plan = ViewAttentionHostPlan(N, V, V, C, G, dtype=tdtype, idx_dtype=torch.int32, gating=True, group_scaling=True,
                                     device=dev)
        plan.ptr.copy_(torch.arange(0, V + 1, v, device=dev))
        plan.x.copy_(torch.randn(V, C, device=dev, generator=gen).to(tdtype))
        plan.idx.copy_(torch.randperm(V, device=dev, generator=gen).int())
        plan.compat.copy_(torch.randn(V, G, device=dev, generator=gen))
        plan.gate[0].fill_(1.0)
        plan.gate[1].fill_(0.0)
        plan.gout.copy_(torch.randn(N, C, device=dev, generator=gen).to(tdtype))
        fw, bw = [], []
        for i in range(warmup + steps):
            e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            e[0].record(); plan.forward_device(); e[1].record(); plan.backward_device(); e[2].record()
            torch.cuda.synchronize()
            if i >= warmup:
                fw.append(e[0].elapsed_time(e[1])); bw.append(e[1].elapsed_time(e[2]))
        f_ms, b_ms = statistics.median(fw), statistics.median(bw)
        bf, bb = algorithmic_bytes(N, V, C, G, s)
        out[str(v)] = {"fwd_ms": f_ms, "bwd_ms": b_ms, "mpoints_per_s": N / (f_ms + b_ms) / 1e3,
                       "fwd_frac": bf / (f_ms * 1e-3) / 1e9 / peak, "bwd_frac": bb / (b_ms * 1e-3) / 1e9 / peak,
                       "step_frac": (bf + bb) / ((f_ms + b_ms) * 1e-3) / 1e9 / peak}
        del plan
        torch.cuda.empty_cache()
    return out


def run_variant_b(args, plan, dev, peak, N, V, D=8, steps=10, warmup=3):
    """Variant B of SURVEY 8(d) (QKVBimodalCSRPool, pooling.py:499-530) on the headline shape: the scores are not
    given but computed from keys K [V, G*D] (one row per view) and queries Q [N, G*D] (one row per point, never
    expanded to the views); the backward also emits dK and dQ.  Two launches each way (dva_qk_scores_* then the fused
    attention pair, compat [V,G] = 16 B per view in between).  Bytes: variant A + (V + N) G D 4 (read K, Q) forward,
    + the same again backward (write dK, dQ), as SURVEY 8(d) counts them -- the 16 B per view of compat traffic the
    two-launch pipeline adds is NOT credited."""
    from deepviewagg_b200 import _lib
    lib = _lib.load()
    G, C = args.groups, args.channels
    s = 4 if args.dtype == "f32" else 2
    gen = torch.Generator(device=dev).manual_seed(4242)
    K = torch.randn(V, G * D, device=dev, generator=gen)
    Q = torch.randn(N, G * D, device=dev, generator=gen)
    dK, dQ = torch.empty_like(K), torch.empty_like(Q)
    scale = 1.0 / math.sqrt(D)
    st = torch.cuda.current_stream(dev).cuda_stream

    def fwd():
        _lib.check(lib.dva_qk_scores_fwd(K.data_ptr(), Q.data_ptr(), plan.ptr.data_ptr(), plan.compat.data_ptr(),
                                         N, V, G, D, scale, st), "dva_qk_scores_fwd")
        plan.forward_device()

    def bwd():
        plan.backward_device()
        _lib.check(lib.dva_qk_scores_bwd(K.data_ptr(), Q.data_ptr(), plan.ptr.data_ptr(), plan.gcompat.data_ptr(),
                                         dK.data_ptr(), dQ.data_ptr(), N, V, G, D, scale, st), "dva_qk_scores_bwd")
    fw, bw = [], []
    for i in range(warmup + steps):
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        e[0].record(); fwd(); e[1].record(); bwd(); e[2].record()
        torch.cuda.synchronize()
        if i >= warmup:
            fw.append(e[0].elapsed_time(e[1])); bw.append(e[1].elapsed_time(e[2]))
    f_ms, b_ms = statistics.median(fw), statistics.median(bw)
    bf, bb = algorithmic_bytes(N, V, C, G, s)
    qk = (V + N) * G * D * 4
    bf, bb = bf + qk, bb + qk
    return {"what": "qk_scores + fused attention, fwd + bwd incl. dK, dQ (QKVBimodalCSRPool, nc_qk = %d, dim_scaling)" % D,
            "fwd_ms": f_ms, "bwd_ms": b_ms, "mpoints_per_s": N / (f_ms + b_ms) / 1e3,
            "algorithmic_bytes": bf + bb, "fwd_frac": bf / (f_ms * 1e-3) / 1e9 / peak,
            "bwd_frac": bb / (b_ms * 1e-3) / 1e9 / peak, "step_frac": (bf + bb) / ((f_ms + b_ms) * 1e-3) / 1e9 / peak,
            "launches_per_step": 4}


def run_e2e(args, plan, dist, dev, world, N, V, n_bucket):
    """Same step through the host-buffer API. Pinned buffers for the whole batch (x alone is
    V*C*s bytes); if the host cannot hold them the e2e leg is skipped with a reason."""
    try:
        import psutil
        avail = psutil.virtual_memory().available
    except Exception:
        avail = None
    need = sum(t.numel() * t.element_size() for t in (plan.x, plan.gx, plan.compat, plan.gcompat,
                                                      plan.gout, plan.out, plan.ptr))
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    if avail is not None and need * local_world * 1.3 > avail:
        return {"value": None, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "skipped": f"host RAM: need {need * local_world / 2**30:.0f} GiB pinned, "
                           f"{avail / 2**30:.0f} GiB available"}
    from deepviewagg_b200.host_api import ViewAttentionHostPipeline
    # two slots when host RAM and HBM allow it: step k+1 copies in while step k copies out
    depth = 2
    free_hbm = torch.cuda.mem_get_info(dev)[0]
    out_bytes = sum(t.numel() * t.element_size() for t in (plan.gx, plan.gcompat, plan.out))
    if free_hbm < need * 1.2 or (avail is not None and (need + out_bytes) * local_world * 1.3 > avail):
        depth = 1
    pipe = ViewAttentionHostPipeline(depth, N, V, V, args.channels, args.groups, dtype=plan.dtype,
                                     idx_dtype=plan.idx.dtype if plan.idx is not None else None,
                                     gating=True, first_plan=plan, device=dev)
    ins, outs0 = plan.host_buffers(pin=True)
    outs = [outs0] + [pipe.plans[k].host_buffers(pin=True)[1] for k in range(1, depth)]
    for k, h in ins.items():           # fill the caller-side buffers with this rank's data
        h.copy_(getattr(plan, k))
    torch.cuda.synchronize()
    # every slot reduces its own full-size parameter-gradient bucket (gate gradients at the tail)
    for pl in pipe.plans:
        pl.bucket = torch.zeros(n_bucket, dtype=torch.float32, device=dev)
        pl.ggate = pl.bucket[n_bucket - 2 * args.groups:].view(2, args.groups)
    reduce_grads = (lambda p: dist.all_reduce(p.bucket)) if dist is not None else None

    def timed(n_steps, use_depth):
        """n_steps full host-buffer steps; returns (ms, h2d, d2h)."""
        if dist is not None:
            dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for i in range(n_steps):
            if use_depth == 1:
                h2d, d2h = plan.run_host(ins, outs[0])
                if reduce_grads is not None:
                    reduce_grads(plan)
            else:
                _, h2d, d2h = pipe.submit(ins, outs[i % depth], after_step=reduce_grads)
        if use_depth > 1:
            pipe.drain()
        b.record()
        torch.cuda.synchronize()
        ms = torch.tensor([a.elapsed_time(b)], device=dev, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), h2d, d2h

    timed(depth, depth)                 # warm-up every slot (page-locks are already in place)
    seq_steps = 2
    seq_ms, h2d, d2h = timed(seq_steps, 1)
    steps = max(2, min(args.steps, 8))
    ms, h2d, d2h = timed(steps, depth)
    val = world * N * steps / (ms * 1e-3) / 1e6
    # the pipelined results must be the single-stream results
    torch.cuda.synchronize()
    same = all(torch.equal(outs[0][k], outs[j][k]) for j in range(1, depth) for k in ("out", "gcompat"))
    return {"value": val, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
            "steps": steps, "ms_per_step": ms / steps, "pipeline_depth": depth,
            "single_stream": {"value": world * N * seq_steps / (seq_ms * 1e-3) / 1e6,
                              "ms_per_step": seq_ms / seq_steps, "steps": seq_steps},
            "slots_agree": bool(same),
            "api": "deepviewagg_b200.host_api.ViewAttentionHostPipeline.submit (pinned host buffers, "
                   "every step: H2D of all inputs, fwd, bwd, D2H of all results)"}


if __name__ == "__main__":
    main()
