#!/usr/bin/env python
"""Headline benchmark of the B200 duplicate-detection hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload of the headline line (BASELINE.json configs[1]): batched fingerprint forward of 10 000 synthetic clips x 64
frames @ 64x64 per GPU, bf16 frames resident in HBM, random-init weights of the reference architecture. One "step" = one
pass of `model.fingerprint_packed` over all clips of the rank. Launched under torchrun for N > 1 (one rank per GPU, clips
sharded, no data-path collective in the forward => weak scaling).

One JSON line on stdout (rank 0):
  value        whole-job videos/s, device-resident inputs, product defaults (one pipeline, 65 536-frame conv passes); CUDA events
               around exactly K steps after W warm-up steps, max over ranks
  e2e          the same metric through the public API `model.fingerprint_host` with HOST (pinned) uint8 frames,
               host<->device copies inside the timed region
  roofline     dominant kernel, from per-stage CUDA-event times taken INSIDE a hot multi-step loop (library stage
               profiler, single pipeline so that stages do not overlap); sum of stages is printed beside that loop's step time
  cpu_baseline the oracle's reference-semantics B=1 loop on the box's host cores (N = 1 only)
  join         all-pairs cosine threshold join, 262 144 rows per GPU (weak scaling; second half of the BASELINE metric). The
               sharded joins (this and cfg4) synchronise with the host several times per call: warm-up until two calls agree
               within 10 %, then the MEDIAN of five calls (max over ranks each); mean, per-call and warm-up lists are printed
  cfg3_varlen  BASELINE configs[2]: 10 000 clips of 16-300 frames (+ a few > 500-frame inputs through subsample()),
               LPT-sharded over the ranks, uint8 frames in HBM, parity spot-check against the oracle inside the run
  cfg4_join    BASELINE configs[3]: 1 048 576 rows in total, row-block sharded, NCCL all-gather overlapped with the
               local block (strong scaling), parity spot-check against an fp32 matmul
  cfg5_topk    BASELINE configs[4]: top-10 of 100 000 queries (sharded) against 10 000 000 database rows
`--dump-outputs DIR` (git ignores bench_outputs/) writes the embeddings the last timed step returned (rank 0) as
DIR/embeddings.npy, float32; the inputs are seeded, so two builds run with the same arguments can be compared output for
output.
`--impl reference` times the reference algorithm's CPU path (oracle port; the reference itself is not installable on the
GPU box) on the same config.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_CLIPS = 10_000
T_FRAMES = 64
FLOPS_PER_FRAME = 39_806_976
METRIC = "fingerprint videos/s (64 frames@64^2)"


def clip_flops(t: int) -> int:  # SURVEY.md section 8d
    return FLOPS_PER_FRAME * t + 4096 * t * t + 524_288


FLOPS_PER_CLIP = clip_flops(T_FRAMES)

# algorithmic FLOPs per clip of each profiled stage (2 FLOP per MAC), T = 64
_T = T_FRAMES
STAGE_FLOPS = {
    "conv1_stem": 2 * 1024 * 32 * 75 * _T,
    "conv2_igemm": 2 * 256 * 64 * 288 * _T,
    "stem_fused": 2 * (1024 * 32 * 75 + 256 * 64 * 288) * _T,   # conv1 + conv2 in one kernel
    "conv3_igemm": 2 * 64 * 128 * 576 * _T,
    "conv4_igemm_pool": 2 * 16 * 256 * 1152 * _T,
    "conv34_fused": 2 * (64 * 128 * 576 + 16 * 256 * 1152) * _T,
    "token_embed_gemm": 2 * (256 * 128 + 128 * 256) * _T,
    "qkv_gemm": 4 * 2 * 256 * 768 * _T,
    "attention": 4 * 4 * _T * _T * 256,
    "out_proj_gemm": 4 * 2 * 256 * 256 * _T,
    "mlp1_gemm_gelu": 4 * 2 * 256 * 1024 * _T,
    "mlp2_gemm": 4 * 2 * 1024 * 256 * _T,
    "ffn_fused": 4 * 2 * 2 * 256 * 1024 * _T,                   # both MLP GEMMs in one kernel
    "pool_logits_gemm": 2 * 256 * 256 * _T,
}
# algorithmic HBM bytes per clip of the stages whose binding roofline is memory, not the tensor pipe
STAGE_BYTES = {
    "conv1_stem": (24576 + 65536) * _T,
    "conv2_igemm": (65536 + 32768) * _T,
    "stem_fused": (24576 + 32768) * _T,           # bf16 frame in, 16x16x64 out (conv1's output never leaves the SM)
    "conv3_igemm": (32768 + 16384) * _T,
    "conv34_fused": (32768 + 512) * _T,
    "temporal_conv": 2 * (1024 + 1024) * _T,      # two blocks, fp32 stream in + out
    "layernorm": 8 * (1024 + 512 + 1024 + 512) * _T,
}


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(hbm=float(p["hbm_gbs"]), tc_burst=float(p["bf16_tflops"]), tc_sustained=float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), source="measured")
    except Exception:
        return dict(hbm=6650.0, tc_burst=1590.0, tc_sustained=1400.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 50 ms; only the samples that fall INSIDE a timed region
    (host timestamps taken around it) are reported. Started before the warm-up so nvidia-smi's start-up is not lost."""

    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50", "-i", str(self.index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True,
            )
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def window(self, t_begin: float, t_end: float):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        inside = [r for t, r in list(self.rows) if t_begin <= t <= t_end + 0.05 and len(r) >= 6]
        rows = inside if inside else [r for _, r in self.rows[-3:] if len(r) >= 6]
        sm = [float(r[0]) for r in rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in rows for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "samples_inside_timed_region": len(inside)}

    def stop(self):
        if self.proc is None:
            return
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()


def dist_setup():
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("NCCL_DEBUG", "WARN")  # keep stdout to the one JSON line
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return world, rank, local


def barrier(world):
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(x: float, world: int, dev) -> float:
    if world == 1:
        return x
    import torch.distributed as dist

    t = torch.tensor([x], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def sum_over_ranks(x: float, world: int, dev) -> float:
    if world == 1:
        return x
    import torch.distributed as dist

    t = torch.tensor([x], dtype=torch.float64, device=dev)
    dist.all_reduce(t)
    return float(t.item())


def timed_ms_each(fn, reps: int, world: int, dev):
    """For the sharded joins, whose every call synchronises with the host about ten times (candidate counts, NCCL size
    exchange): (median, mean, per-repetition list) of the repetition time, each repetition taken as the max over ranks.
    A one-off host stall of 100+ ms inside one repetition was observed on shared boxes (2 GPUs: 97.9 ms mean against 24 ms in
    every other run), so the MEDIAN is reported as the time and the mean and the list are printed next to it."""
    barrier(world)
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
    evs[0].record()
    for r in range(reps):
        fn()
        evs[r + 1].record()
    barrier(world)
    each = torch.tensor([evs[r].elapsed_time(evs[r + 1]) for r in range(reps)], dtype=torch.float64, device=dev)
    if world > 1:
        import torch.distributed as dist

        dist.all_reduce(each, op=dist.ReduceOp.MAX)
    each = each.tolist()
    return float(np.median(each)), float(np.mean(each)), [round(t, 2) for t in each]


def warm_until_steady(fn, world: int, dev, min_calls: int = 3, max_calls: int = 12):
    """Warm-up for the sharded joins: at least `min_calls` calls, then until two consecutive calls (max over ranks) agree
    within 10 %. The first calls of a process pay NCCL's connection set-up and the allocator's first big blocks; on some
    2-GPU boxes the per-call time kept falling for seven calls (182, 103, 109, 87, 33 ms after three warm-up calls)."""
    prev, times = None, []
    for k in range(max_calls):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier(world)
        a.record()
        fn()
        b.record()
        barrier(world)
        t = max_over_ranks(a.elapsed_time(b), world, dev)
        times.append(round(t, 2))
        if k + 1 >= min_calls and prev is not None and abs(t - prev) <= 0.1 * t:
            break
        prev = t
    return times


def timed_ms(fn, reps: int, world: int, dev) -> float:
    """CUDA-event time per repetition on the current stream, barrier + synchronize on both sides, max over ranks."""
    barrier(world)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    barrier(world)
    return max_over_ranks(a.elapsed_time(b) / reps, world, dev)


# --------------------------------------------------------------------------------------------------
# CPU reference arm (oracle port of the reference's --device cpu path: B=1 forward loop, fingerprint.py:244-249)
# --------------------------------------------------------------------------------------------------
def cpu_reference_rate(budget_s: float, max_clips: int):
    from oracle.forward_oracle import forward_oracle
    from oracle.weights import make_state_dict

    sd = make_state_dict(0, "default")
    g = torch.Generator().manual_seed(4321)
    clip = torch.rand((1, T_FRAMES, 3, 64, 64), generator=g)
    forward_oracle(sd, clip)  # warm-up
    n, t0 = 0, time.perf_counter()
    while n < max_clips and (time.perf_counter() - t0 < budget_s or n < 4):
        forward_oracle(sd, clip)
        n += 1
    dt = time.perf_counter() - t0
    return n / dt, n, dt


def run_reference(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    torch.set_num_threads(os.cpu_count() or 1)  # torchrun pins OMP_NUM_THREADS=1; the reference arm gets every host core
    threads = torch.get_num_threads()
    per_step = max(4.0, min(20.0, 120.0 / max(1, args.steps + args.warmup)))
    if args.ref_budget:   # tests: a shorter bounded sample per step
        per_step = args.ref_budget
    for _ in range(args.warmup):
        cpu_reference_rate(per_step / 4, 64)
    clips, secs = 0, 0.0
    for _ in range(args.steps):
        _, n, dt = cpu_reference_rate(per_step, 512)
        clips += n
        secs += dt
    value = clips / secs
    sample = f"{clips} clips x {T_FRAMES} frames in {secs:.1f}s, B=1 forwards (oracle port of the reference CPU path; the reference itself cannot be shipped to the GPU box)"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "videos/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 * secs / max(1, args.steps), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": {"workload": f"fingerprint forward, {T_FRAMES} frames @ 64x64 per clip, bounded sample of the 10k-clip workload"},
        "cpu_baseline": {"value": value, "unit": "videos/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "videos/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "world_size_env": world,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# synthetic data
# --------------------------------------------------------------------------------------------------
def make_join_data(n: int, dev, seed: int = 11):
    """Unit vectors with planted near-duplicates on both sides of 0.95 (SURVEY.md section 8d, cfg 4)."""
    g = torch.Generator(device=dev).manual_seed(seed)
    E = torch.randn((n, 256), generator=g, device=dev)
    E = E / E.norm(dim=1, keepdim=True)
    n_dup = n // 50
    src = torch.randint(0, n, (n_dup,), generator=g, device=dev)
    dst = torch.randint(0, n, (n_dup,), generator=g, device=dev)
    sigma = torch.tensor([0.0, 0.005, 0.0145, 0.0205, 0.03], device=dev)[torch.randint(0, 5, (n_dup,), generator=g, device=dev)]
    v = E[src] + sigma[:, None] * torch.randn((n_dup, 256), generator=g, device=dev)
    E[dst] = v / v.norm(dim=1, keepdim=True)
    return E.contiguous()


def make_unit_rows(n: int, dev, seed: int, chunk: int = 1 << 20):
    g = torch.Generator(device=dev).manual_seed(seed)
    E = torch.empty((n, 256), dtype=torch.float32, device=dev)
    for s in range(0, n, chunk):
        e = min(n, s + chunk)
        x = torch.randn((e - s, 256), generator=g, device=dev)
        E[s:e] = x / x.norm(dim=1, keepdim=True)
    return E


def join_roofline(n_total: int, ms: float, world: int, peaks):
    """The score matrix of a self join is symmetric and the product screens its upper triangle only (every block of it
    on ONE rank, mirrored pairs emitted by the re-score kernel), so the EXECUTED tensor work is (n^2 + n) / 2 dot products;
    the algorithmic figure SURVEY.md section 8(d) defines is 512 FLOP for each of the n^2 ordered pairs the reference
    computes. The roofline fraction is taken on the executed work; both are printed."""
    executed = (n_total * (n_total + 1) / 2) * 512 / (ms / 1000.0) / 1e12 / world
    algorithmic = n_total * n_total * 512 / (ms / 1000.0) / 1e12 / world
    return {"bound": "tensor", "achieved": executed, "peak": peaks["tc_burst"], "unit": "TFLOP/s per GPU (executed: upper triangle)",
            "frac": executed / peaks["tc_burst"], "frac_of_sustained": executed / peaks["tc_sustained"],
            "algorithmic_tflops_per_gpu": algorithmic, "algorithmic_over_peak": algorithmic / peaks["tc_burst"], "traffic": None}


# --------------------------------------------------------------------------------------------------
# BASELINE configs[2..4]
# --------------------------------------------------------------------------------------------------
def bench_cfg3_varlen(vfp, model, world, rank, dev, peaks, n_videos: int, reps: int):
    """10 000 clips, lengths randint(16, 301) seed 7, plus a few decoded inputs longer than max_frames that go through the
    scanner's subsampling rule; clips LPT-sharded over the ranks (strong scaling, no collective); uint8 frames in HBM."""
    from video_fingerprint_b200 import sharding

    rng = np.random.default_rng(7)
    lengths = rng.integers(16, 301, size=n_videos).tolist()
    decoded_long = [750, 1203, 2000, 5000][: max(0, min(4, n_videos // 100))]   # decoded frame counts > max_frames = 500
    scanner = vfp.VideoFingerprintScanner(model=model, config={"model_type": "attention"})
    kept_long = [scanner.subsample(t) for t in decoded_long]
    for j, keep in enumerate(kept_long):            # the first few videos are the long ones
        lengths[j] = len(keep)
    parts = sharding.partition_clips(lengths, world)
    mine = parts[rank]
    my_len = [lengths[i] for i in mine]
    total = sum(my_len)
    g = torch.Generator(device=dev).manual_seed(7000 + rank)
    frames = torch.empty((total, 3, 64, 64), dtype=torch.uint8, device=dev)
    off = 0
    for i, t in zip(mine, my_len):
        if i < len(decoded_long):   # a long input: synthesise the decoded video, keep the frames subsample() selects
            full = torch.randint(0, 256, (decoded_long[i], 3, 64, 64), generator=g, device=dev, dtype=torch.uint8)
            frames[off : off + t] = full[torch.tensor(kept_long[i], device=dev)]
        off += t
    chunk = 1 << 15
    first_short = sum(t for i, t in zip(mine, my_len) if i < len(decoded_long))
    for s in range(first_short, total, chunk):
        e = min(total, s + chunk)
        frames[s:e] = torch.randint(0, 256, (e - s, 3, 64, 64), generator=g, device=dev, dtype=torch.uint8)
    torch.cuda.synchronize()
    emb = model.fingerprint_packed(frames, my_len)   # warm-up
    ms = timed_ms(lambda: model.fingerprint_packed(frames, my_len), reps, world, dev)
    flops = sum_over_ranks(float(sum(clip_flops(t) for t in my_len)), world, dev)
    frames_all = sum_over_ranks(float(total), world, dev)
    max_frames_rank = max_over_ranks(float(total), world, dev)
    parity = None
    if rank == 0:   # spot check against the oracle's B=1 forward on the host: shortest, longest, a subsampled one, two more
        from oracle.forward_oracle import forward_oracle

        sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
        cu = np.concatenate([[0], np.cumsum(my_len)])
        picks = sorted({int(np.argmin(my_len)), int(np.argmax(my_len)), 0, len(mine) // 2, len(mine) - 1})
        worst = 1.0
        for c in picks:
            clip = frames[cu[c] : cu[c + 1]].cpu().float().div_(255.0).unsqueeze(0)
            want = forward_oracle(sd, clip)[0].double()
            got = emb[c].cpu().double()
            worst = min(worst, float(torch.dot(want, got) / (want.norm() * got.norm())))
        parity = {"clips_checked": len(picks), "lengths": [my_len[c] for c in picks], "min_cosine_vs_oracle": worst, "ok": worst >= 0.9999}
    del frames
    return {
        "value": n_videos / (ms / 1000.0), "unit": "videos/s", "videos": n_videos, "frames": int(frames_all), "ms": ms, "scaling": "strong",
        "frames_per_s": frames_all / (ms / 1000.0), "max_frames_on_a_rank": int(max_frames_rank),
        "lengths": "randint(16, 301) seed 7; first %d videos are decoded inputs of %s frames reduced by subsample() to %s" % (len(decoded_long), decoded_long, [len(k) for k in kept_long]),
        "roofline": {"bound": "tensor", "achieved": flops / (ms / 1000.0) / 1e12 / world, "peak": peaks["tc_sustained"], "unit": "TFLOP/s per GPU",
                     "frac": flops / (ms / 1000.0) / 1e12 / world / peaks["tc_sustained"]},
        "parity": parity, "input": "uint8 frames resident in HBM, LPT partition by frame count, no collective",
    }


def bench_cfg4_join(vfp, world, rank, dev, peaks, n_total: int, reps: int):
    """All-pairs threshold join over n_total rows in total: rank r owns rows [r n/G, (r+1) n/G); the timed region holds the
    all-gather (overlapped with the rank's own diagonal block) and the row-block join against all columns."""
    from video_fingerprint_b200 import sharding

    E = make_join_data(n_total, dev, seed=11)     # same matrix on every rank (same seed); a rank only USES its rows
    lo, hi = sharding.row_block(n_total, world, rank)
    local = E[lo:hi].contiguous()
    res = {}

    def step():
        res["out"] = sharding.sharded_threshold_join_device(local, 0.95)

    warm = warm_until_steady(step, world, dev)   # 4 GPUs: first call 90 ms against 54 ms in steady state (scripts/dev_sharded_join_phases.py)
    ms, ms_mean, ms_each = timed_ms_each(step, max(reps, 5), world, dev)
    i, j, s, _ = res["out"]
    pairs = int(sum_over_ranks(float(i.numel()), world, dev))
    # parity: 512 sampled rows against ALL columns in fp32 (blocked matmul on rank 0), threshold band excluded. A rank's
    # list also holds mirrored pairs of other ranks' rows, so the sampled rows' pairs are collected from every rank.
    gsel = torch.Generator(device=dev).manual_seed(5)
    rows = torch.randint(0, n_total, (512,), generator=gsel, device=dev).unique()
    sel = torch.isin(i, rows)
    mine = torch.stack([i[sel], j[sel]], dim=1)
    allp, _ = sharding.all_gather_rows(mine) if world > 1 else (mine, None)
    parity = None
    if rank == 0:
        S = E[rows] @ E.T
        want, near = set(), set()
        for a, b in (S >= 0.95 - 1e-5).nonzero().tolist():
            key = (int(rows[a]), b)
            (near if abs(float(S[a, b]) - 0.95) < 1e-5 else want).add(key)
        got = [tuple(p) for p in allp.tolist()]
        gset = set(got)
        parity = {"rows_checked": int(rows.numel()), "pairs_expected": len(want), "missing": len(want - gset), "unexpected": len(gset - want - near),
                  "duplicates": len(got) - len(gset), "ok": len(want - gset) == 0 and len(gset - want - near) == 0 and len(got) == len(gset)}
        del S
    gpairs = (n_total * n_total) / (ms / 1000.0) / 1e9
    del E
    return {
        "value": gpairs, "unit": "Gpairs/s", "n": n_total, "rows_per_gpu": hi - lo, "threshold": 0.95, "pairs_found": pairs, "ms": ms, "ms_mean": ms_mean, "ms_each": ms_each, "warmup_ms": warm, "timing": "median of 5 calls, each the max over ranks, after a warm-up that runs until two calls agree within 10 %", "scaling": "strong",
        "roofline": join_roofline(n_total, ms, world, peaks),
        "parity": parity,
        "note": "one GPU joins n x n" if world == 1 else f"row-block sharded over {world} GPUs: NCCL all-gather of the fp32 shards overlapped with the own-column block, then the remaining columns; all inside the timed region",
    }


def bench_cfg5_topk(vfp, world, rank, dev, peaks, n_db: int, n_q: int, k: int, reps: int):
    """Flat inner-product top-k, queries sharded over the ranks, database replicated (SURVEY.md section 8e). The database is
    resident before the timed region (the reference's index.add, fingerprint.py:525); the search (index.search, :528) is timed."""
    db = make_unit_rows(n_db, dev, seed=21)
    gq = torch.Generator(device=dev).manual_seed(22)
    Q = torch.randn((n_q, 256), generator=gq, device=dev)
    Q = Q / Q.norm(dim=1, keepdim=True)
    n_copy = n_q // 100                                       # 1 % of the queries are noisy copies of database rows
    src = torch.randint(0, n_db, (n_copy,), generator=gq, device=dev)
    v = db[src] + 0.01 * torch.randn((n_copy, 256), generator=gq, device=dev)
    Q[:n_copy] = v / v.norm(dim=1, keepdim=True)
    n_tie = min(1000, n_copy, n_db // 4)                             # exact duplicates inside the database => exact score ties
    db[n_db - n_tie :] = db[src[:n_tie]]
    per = -(-n_q // world)
    q_local = Q[rank * per : min(n_q, (rank + 1) * per)].contiguous()
    res = {}

    def step():
        res["out"] = vfp.topk_inner_product_device(q_local, db, k)

    step()
    ms = timed_ms(step, reps, world, dev)
    S, I = res["out"]
    parity = None
    if rank == 0:
        nchk = min(64, q_local.shape[0])
        ref = q_local[:nchk] @ db.T
        ts, ti = torch.topk(ref, k + 8, dim=1)
        ts, ti = ts.cpu().numpy(), ti.cpu().numpy()
        gotS, gotI = S[:nchk].cpu().numpy(), I[:nchk].cpu().numpy()
        exact = flips = bad = 0
        for r in range(nchk):
            order = np.lexsort((ti[r], -ts[r]))[:k]
            wi, ws = ti[r][order], ts[r][order]
            if np.array_equal(wi, gotI[r]):
                exact += 1
            elif np.allclose(ws, gotS[r], atol=2e-6) and all(abs(ref[r, int(a)].item() - float(b)) <= 2e-6 for a, b in zip(gotI[r], gotS[r])):
                flips += 1   # same scores to fp32 summation order; indices differ only among (near-)ties
            else:
                bad += 1
        parity = {"queries_checked": nchk, "identical": exact, "tie_order_only": flips, "wrong": bad, "ok": bad == 0}
        del ref
    tfl = 2.0 * n_q * n_db * 256 / (ms / 1000.0) / 1e12 / world
    del db, Q
    return {
        "value": n_q / (ms / 1000.0), "unit": "queries/s", "n_db": n_db, "n_q": n_q, "k": k, "ms": ms, "scaling": "strong", "queries_per_gpu": int(q_local.shape[0]),
        "gpairs_per_s": n_q * n_db / (ms / 1000.0) / 1e9,
        "roofline": {"bound": "tensor", "achieved": tfl, "peak": peaks["tc_burst"], "unit": "TFLOP/s per GPU", "frac": tfl / peaks["tc_burst"],
                     "frac_of_sustained": tfl / peaks["tc_sustained"]},
        "parity": parity, "note": "queries sharded, database replicated and resident; fp32-exact results (bf16 tensor-core screen + fp32 re-score + exactness proof)",
    }


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Each array as float32 out_dir/<name>.npy. An array larger than its share of 64 MB is reduced to a fixed sample of
    its rows (seeded: the same rows in every run for the same shape)."""
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_LIMIT_BYTES // len(arrays)
    for name, t in arrays.items():
        a = t.detach().float().cpu().numpy()
        if a.nbytes > share:
            rows = np.random.default_rng(0).choice(a.shape[0], share // (a.nbytes // a.shape[0]), replace=False)
            a = a[np.sort(rows)]
        np.save(os.path.join(out_dir, name + ".npy"), a)


# --------------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------------
def run_ours(args):
    import video_fingerprint_b200 as vfp
    from video_fingerprint_b200 import _native, sharding

    world, rank, local = dist_setup()
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    lib = _native.load()
    for kv in args.tuning:
        k, v = kv.split("=")
        if lib.vfp_set_tuning(int(k), int(v)) != 0:
            raise SystemExit(f"bench.py: vfp_set_tuning({k}, {v}) rejected")
    peaks = load_peaks()

    n_clips = args.clips
    torch.manual_seed(0)
    model = vfp.create_model("attention").eval()
    if args.frames_per_pass:
        model.frames_per_pass = args.frames_per_pass
    if args.pipelines:
        model.pipelines = args.pipelines
    lib.vfp_set_tuning(9, int(model.pipelines))
    lengths = [T_FRAMES] * n_clips
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    frames = torch.empty((n_clips * T_FRAMES, 3, 64, 64), dtype=torch.bfloat16, device=dev)
    chunk = 64 * T_FRAMES
    for s in range(0, frames.shape[0], chunk):  # generate in slices: torch.rand has no bf16 generator path for 15 GB at once
        e = min(frames.shape[0], s + chunk)
        frames[s:e] = torch.rand((e - s, 3, 64, 64), generator=g, device=dev, dtype=torch.float32).to(torch.bfloat16)
    torch.cuda.synchronize()

    def step():
        return model.fingerprint_packed(frames, lengths)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(3, args.warmup)):
        emb = step()
    barrier(world)
    stage_ms = (C.c_double * 32)()
    launches = C.c_uint64(0)
    lib.vfp_profile_read(stage_ms, 32, C.byref(launches), 1)  # reset the launch counter
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(world)
    t_begin = time.perf_counter()
    ev0.record()
    for _ in range(args.steps):
        emb = step()
    ev1.record()
    barrier(world)
    t_end = time.perf_counter()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.window(t_begin, t_end) if rank == 0 else None
    lib.vfp_profile_read(stage_ms, 32, C.byref(launches), 1)
    gpu_launches = int(launches.value)
    ms = max_over_ranks(ms, world, dev)
    value = world * n_clips * args.steps / (ms / 1000.0)

    # ---- per-kernel times INSIDE a hot loop: the library's stage profiler (CUDA events between the stages on the launching
    # stream) stays on for `prof_steps` back-to-back steps that directly follow the timed region, so the clocks are the
    # power-capped ones of a long run. Profiling forces ONE pipeline (stages of two passes in flight would overlap and the
    # event pairs would measure queueing), hence the loop is timed on its own and sum(stages) is compared with ITS step time.
    prof_steps = max(2, min(args.steps, 5))
    lib.vfp_profile_enable(1)
    step()   # first profiled step re-sizes nothing but settles the single-pipeline schedule
    torch.cuda.synchronize()
    lib.vfp_profile_read(stage_ms, 32, C.byref(launches), 1)
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tp_begin = time.perf_counter()
    p0.record()
    for _ in range(prof_steps):
        step()
    p1.record()
    torch.cuda.synchronize()
    tp_end = time.perf_counter()
    prof_ms_per_step = p0.elapsed_time(p1) / prof_steps
    lib.vfp_profile_read(stage_ms, 32, C.byref(launches), 1)
    lib.vfp_profile_enable(0)
    prof_clocks = sampler.window(tp_begin, tp_end) if rank == 0 else None
    n_stage = lib.vfp_profile_num_stages()
    stages = {lib.vfp_profile_stage_name(i).decode(): stage_ms[i] / prof_steps for i in range(n_stage)}

    # ---- end-to-end through the public API with host uint8 frames (pinned), copies inside the timed region ----
    e2e = None
    if not args.no_e2e:
        host = torch.empty((n_clips * T_FRAMES, 3, 64, 64), dtype=torch.uint8, pin_memory=True)
        blk = min(host.shape[0], 64 * T_FRAMES * 16)
        host[:blk].random_(0, 256)
        for s in range(blk, host.shape[0], blk):   # replicate the random block (filling 7.9 GB with the CPU generator takes too long)
            e = min(host.shape[0], s + blk)
            host[s:e] = host[: e - s]
        out_host = torch.empty((n_clips, 256), dtype=torch.float32, pin_memory=True)

        def e2e_step():
            model.fingerprint_host(host, lengths, chunk_frames=500 * T_FRAMES, out=out_host)   # returns after the D2H copy

        e2e_step()
        barrier(world)
        t0 = time.perf_counter()
        e2e_steps = max(1, min(args.steps, 3))
        for _ in range(e2e_steps):
            e2e_step()
        barrier(world)
        dt = max_over_ranks(time.perf_counter() - t0, world, dev)
        e2e = {
            "value": world * n_clips * e2e_steps / dt, "unit": "videos/s",
            "h2d_bytes_per_step": n_clips * T_FRAMES * 12288, "d2h_bytes_per_step": n_clips * 256 * 4,
            "input": "uint8 frames in pinned host memory through model.fingerprint_host (500-clip chunks, double-buffered on a copy stream)", "steps": e2e_steps,
            "pcie_gbs": n_clips * T_FRAMES * 12288 * e2e_steps / dt / 1e9,
        }
        del host
    del frames
    torch.cuda.empty_cache()

    # ---- similarity join, weak scaling (second half of the BASELINE metric): join_n rows per GPU ----
    join = None
    if not args.no_join:
        n_local = args.join_n
        E_local = make_join_data(n_local, dev, seed=11 + rank)
        res = {}

        def join_step():
            res["out"] = sharding.sharded_threshold_join_device(E_local, 0.95)

        j_warm = warm_until_steady(join_step, world, dev)
        jms, j_mean, j_each = timed_ms_each(join_step, 5, world, dev)
        n_total = res["out"][3]
        pairs_found = int(sum_over_ranks(float(res["out"][0].numel()), world, dev))
        gpairs = (n_total * n_total) / (jms / 1000.0) / 1e9
        join = {
            "value": gpairs, "unit": "Gpairs/s (ordered pairs of the n x n matrix the reference computes)", "n": n_total, "rows_per_gpu": n_local, "threshold": 0.95,
            "pairs_found": pairs_found, "ms": jms, "ms_mean": j_mean, "ms_each": j_each, "warmup_ms": j_warm, "timing": "median of 5 calls, each the max over ranks, after a warm-up that runs until two calls agree within 10 %", "scaling": "weak",
            "roofline": join_roofline(n_total, jms, world, peaks),
            "note": ("one GPU joins n x n" if world == 1 else
                     f"row-block sharded: NCCL all-gather of {world} x ({n_local}, 256) fp32 shards overlapped with the own-column block + the remaining columns, all inside the timed region"),
        }
        del E_local, res
        torch.cuda.empty_cache()

    def guarded(fn, *a):
        try:
            out = fn(*a)
        except Exception as exc:  # the side configurations never take the headline line down
            out = {"error": repr(exc)}
        torch.cuda.empty_cache()
        return out

    cfg3 = guarded(bench_cfg3_varlen, vfp, model, world, rank, dev, peaks, args.cfg3_videos, 3) if not args.no_cfg3 else None
    cfg4 = guarded(bench_cfg4_join, vfp, world, rank, dev, peaks, args.cfg4_rows, 3) if not args.no_cfg4 else None
    cfg5 = guarded(bench_cfg5_topk, vfp, world, rank, dev, peaks, args.cfg5_db, args.cfg5_q, 10, 2) if not args.no_cfg5 else None

    if rank == 0:
        sampler.stop()
    if rank != 0:
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"embeddings": emb})
    # ---- roofline of the dominant kernel ----
    known = [k for k in stages if (k in STAGE_FLOPS or k in STAGE_BYTES) and stages[k] > 0]
    dom = max(known, key=lambda k: stages[k])
    sum_stages = sum(stages.values())
    conv_pass = min(65536, n_clips * T_FRAMES)   # the library's default conv pass (vfp_set_tuning key 3)
    conv_launches = -(-n_clips * T_FRAMES // conv_pass)
    dom_ms = stages[dom]
    tflops = STAGE_FLOPS.get(dom, 0) * n_clips / (dom_ms / 1000.0) / 1e12
    gbs = STAGE_BYTES.get(dom, 0) * n_clips / (dom_ms / 1000.0) / 1e9
    frac_t, frac_h = tflops / peaks["tc_sustained"], gbs / peaks["hbm"]
    hbm_bound = frac_h > frac_t  # the binding roofline is the one the kernel sits closer to
    # DRAM bytes of the stem from the committed `ncu --set full` capture (profiles/r02_ncu_full_conv_join.txt: dram__bytes_read.sum
    # + dram__bytes_write.sum = 402.76 + 485.82 MB for a launch over 16 384 frames), scaled to the frames of one launch here
    ncu_traffic = {"stem_fused": (402.76e6 + 485.82e6) * conv_pass / 16384}
    whole_tfl = value / world * FLOPS_PER_CLIP / 1e12
    roofline = {
        "bound": "hbm" if hbm_bound else "tensor", "kernel": dom,
        "achieved": gbs if hbm_bound else tflops, "peak": peaks["hbm"] if hbm_bound else peaks["tc_sustained"],
        "unit": "GB/s" if hbm_bound else "TFLOP/s", "frac": frac_h if hbm_bound else frac_t,
        "frac_of_burst": None if hbm_bound else tflops / peaks["tc_burst"],
        "traffic": ncu_traffic.get(dom) if (n_clips * T_FRAMES) >= 16384 else None,
        "traffic_note": "bytes per launch (one conv pass of %d frames; ncu capture of a 16 384-frame launch, scaled) ; algorithmic bytes per launch = %.1f MB" % (conv_pass, STAGE_BYTES.get(dom, 0) / T_FRAMES * conv_pass / 1e6),
        "peak_source": f"{peaks['source']} ({'HBM copy bandwidth' if hbm_bound else 'sustained bf16: the kernel is timed inside a long hot loop'})",
        "timing": f"stage events inside a {prof_steps}-step hot loop that follows the timed region (single pipeline): {prof_ms_per_step:.2f} ms/step, sum of stages {sum_stages:.2f} ms",
        "profiled_ms_per_step": prof_ms_per_step, "sum_of_stages_ms": sum_stages, "profile_clocks": prof_clocks,
        "other_roofline": {"tensor_tflops": tflops, "tensor_frac": frac_t, "hbm_gbs": gbs, "hbm_frac": frac_h},
        "launches_per_step": conv_launches, "ms_per_step_in_kernel": dom_ms,
        "algorithmic_per_clip": {"flops": STAGE_FLOPS.get(dom), "bytes": STAGE_BYTES.get(dom)},
        "whole_step": {"achieved": whole_tfl, "unit": "TFLOP/s", "frac": whole_tfl / peaks["tc_sustained"], "frac_of_burst": whole_tfl / peaks["tc_burst"]},
        "per_stage": {
            k: {"ms": round(stages[k], 3),
                "tflops": round(STAGE_FLOPS[k] * n_clips / (stages[k] / 1000.0) / 1e12, 1) if k in STAGE_FLOPS and stages[k] > 0 else None,
                "gbs": round(STAGE_BYTES[k] * n_clips / (stages[k] / 1000.0) / 1e9, 1) if k in STAGE_BYTES and stages[k] > 0 else None}
            for k in stages if stages[k] > 0
        },
    }
    line = {
        "metric": METRIC, "value": value, "unit": "videos/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {
            "workload": f"batched fingerprint forward: {n_clips} synthetic clips x {T_FRAMES} frames @ 64x64 per GPU, bf16 frames resident in HBM, random-init weights (BASELINE configs[1])",
            "frames_per_pass": model.frames_per_pass, "pipelines": model.pipelines,
            "l2": f"inputs ({n_clips * T_FRAMES * 24576 / 1e9:.1f} GB) and per-pass activations exceed the 126 MB L2; no flush needed",
            "parallelism": f"clips sharded over {world} GPU(s), no data-path collective",
        },
        "e2e": e2e, "gpu_launches": gpu_launches, "roofline": roofline, "stage_ms_per_step": {k: v for k, v in stages.items() if v > 0},
        "join": join, "cfg3_varlen": cfg3, "cfg4_join": cfg4, "cfg5_topk": cfg5, "clocks": clocks,
    }
    if not args.no_cpu and world == 1:
        r, n, dt = cpu_reference_rate(args.cpu_seconds, 2048)
        line["cpu_baseline"] = {
            "value": r, "unit": "videos/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{n} clips x {T_FRAMES} frames in {dt:.1f}s, B=1 forward loop of oracle/forward_oracle.py (restatement of the reference --device cpu path) on host cores",
        }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--clips", type=int, default=N_CLIPS)
    ap.add_argument("--frames-per-pass", type=int, default=0, help="frames per token pass (default: the model's)")
    ap.add_argument("--pipelines", type=int, default=0, help="token passes in flight (default: the model's)")
    ap.add_argument("--join-n", type=int, default=262_144)
    ap.add_argument("--cfg3-videos", type=int, default=10_000)
    ap.add_argument("--cfg4-rows", type=int, default=1_048_576)
    ap.add_argument("--cfg5-db", type=int, default=10_000_000)
    ap.add_argument("--cfg5-q", type=int, default=100_000)
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--tuning", action="append", default=[], help="experiment: key=value passed to vfp_set_tuning")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-join", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--ref-budget", type=float, default=0.0, help="reference arm: seconds of CPU work per step (default: 4-20 s from --steps)")
    ap.add_argument("--no-cfg3", action="store_true")
    ap.add_argument("--no-cfg4", action="store_true")
    ap.add_argument("--no-cfg5", action="store_true")
    ap.add_argument("--forward-only", action="store_true", help="skip e2e, joins, cfg 3-5 and the CPU baseline (kernel experiments)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the embeddings of the last timed step to DIR/embeddings.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.forward_only:
        args.no_e2e = args.no_join = args.no_cpu = args.no_cfg3 = args.no_cfg4 = args.no_cfg5 = True
    if args.impl == "reference":
        run_reference(args)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    run_ours(args)
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        import torch.distributed as dist

        dist.destroy_process_group()


if __name__ == "__main__":
    main()
