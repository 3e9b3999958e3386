"""Dev helper: the attention model on clips read in place (fingerprint_views) against the copying paths.

    python scripts/dev_forward_views_time.py                # card, separate, varlen, strided, decoded
    python scripts/dev_forward_views_time.py --only strided

separate - 10 000 x 64-frame bf16 clips, each its own allocation (the bench.py corpus shape): m.fingerprint_clips(clips)
           (concatenates them first), m.fingerprint_views(clips) (reads them where they are), and m.fingerprint_packed on
           the same frames already packed into one tensor. All three must be bit-identical.
varlen   - 2 048 bf16 clips of 16 - 300 frames, each its own allocation, the same three ways.
strided  - 256 preprocessed decoder-layout uint8 videos of 1 200 - 3 000 frames; the scanner keeps every skip-th frame up to
           500 (VideoFingerprintScanner.subsample). fingerprint_views of the `frames[::skip][:500]` views against gathering
           those frames into one tensor first (torch.cat of the views) + fingerprint_packed.
decoded  - 32 decoded 320 x 240 videos of 300 - 1 000 frames (host arrays, slices of one seeded pool) through
           scanner.extract_fingerprints_from_decoded (one fingerprint_views call) against a loop of
           extract_fingerprint_from_decoded (one forward per video).
Each pair of runs is alternated `--rounds` times in this one process; a round is CUDA events around `--reps` calls after a
warm-up call (the scanner paths end in a device-to-host copy, which synchronises). Every printed line is a JSON object."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    import torch

    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001 - the card name alone is still worth printing
        out = f"unavailable ({e})"
    return {"card": name, "power_limit_and_max_sm_clock": out}


def timed(fn, reps):
    import torch

    out = fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, out


def alternate(case, runs, rounds, reps, extra):
    """Time every (name, fn) of `runs` once per round, alternating; print one line per run -> {name: last output}."""
    ms = {name: [] for name, _ in runs}
    outs = {}
    for _ in range(rounds):
        for name, fn in runs:
            t, outs[name] = timed(fn, reps)
            ms[name].append(t)
    for name, _ in runs:
        med = statistics.median(ms[name])
        line = {"case": case, "run": name, **extra, "ms_median": round(med, 3), "ms_rounds": [round(t, 3) for t in ms[name]],
                "videos_per_s": round(extra["videos"] / med * 1e3)}
        print(json.dumps(line), flush=True)
    return outs


def same_rows(a, b):
    import numpy as np

    return all((x is None and y is None) or (x is not None and y is not None and np.array_equal(x, y)) for x, y in zip(a, b))


def separate_case(m, lengths, case, args):
    import torch

    gen = torch.Generator("cuda").manual_seed(len(lengths))
    clips = [torch.rand((t, 3, 64, 64), device="cuda", generator=gen).to(torch.bfloat16) for t in lengths]
    packed = torch.cat(clips)
    extra = {"videos": len(lengths), "frames": sum(lengths)}
    outs = alternate(case, [("clips", lambda: m.fingerprint_clips(clips)), ("views", lambda: m.fingerprint_views(clips)),
                            ("packed", lambda: m.fingerprint_packed(packed, lengths))], args.rounds, args.reps, extra)
    same = torch.equal(outs["clips"], outs["packed"]) and torch.equal(outs["views"], outs["packed"])
    print(json.dumps({"case": case, "bit_identical": same}), flush=True)
    return same


def strided_case(vfp, m, args):
    import torch

    sc = vfp.VideoFingerprintScanner(model=m, config={"model_type": "attention"})
    g = torch.Generator().manual_seed(4321)
    lengths = [int(t) for t in torch.randint(1200, 3001, (args.strided_videos,), generator=g)]
    pool = torch.randint(0, 256, (sum(lengths), 64, 64, 3), dtype=torch.uint8, device="cuda", generator=torch.Generator("cuda").manual_seed(5))
    views, f = [], 0
    for t in lengths:
        keep = sc.subsample(t)
        views.append(pool[f : f + keep[-1] + 1 : keep[1] - keep[0]])
        f += t
    kept = [int(v.shape[0]) for v in views]

    def gather():
        return m.fingerprint_packed(torch.cat(views), kept)

    extra = {"videos": len(views), "frames": sum(kept)}
    outs = alternate("strided", [("gather+packed", gather), ("views", lambda: m.fingerprint_views(views))], args.rounds, args.reps, extra)
    same = torch.equal(outs["gather+packed"], outs["views"])
    print(json.dumps({"case": "strided", "bit_identical": same}), flush=True)
    return same


def decoded_case(vfp, m, args):
    import numpy as np

    sc = vfp.VideoFingerprintScanner(model=m, config={"model_type": "attention"})
    rng = np.random.default_rng(99)
    lengths = rng.integers(300, 1001, args.decoded_videos).tolist()
    pool = rng.integers(0, 256, (1000 + args.decoded_videos, 240, 320, 3), dtype=np.uint8)
    videos = [pool[i : i + t] for i, t in enumerate(lengths)]   # host views: decoded frames as a decoder hands them over
    extra = {"videos": len(videos), "frames": sum(lengths), "size": "320x240"}
    outs = alternate("decoded", [("per_video_loop", lambda: [sc.extract_fingerprint_from_decoded(v) for v in videos]),
                                 ("batched", lambda: sc.extract_fingerprints_from_decoded(videos))],
                     args.rounds, max(1, args.reps // 5), extra)
    same = same_rows(outs["per_video_loop"], outs["batched"])
    print(json.dumps({"case": "decoded", "bit_identical": same}), flush=True)
    return same


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", choices=["separate", "varlen", "strided", "decoded"])
    ap.add_argument("--n", type=int, default=10_000, help="64-frame clips of the separate case")
    ap.add_argument("--varlen-clips", type=int, default=2048)
    ap.add_argument("--strided-videos", type=int, default=256)
    ap.add_argument("--decoded-videos", type=int, default=32)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    import torch

    import video_fingerprint_b200 as vfp

    assert torch.cuda.is_available(), "this script times the B200 path; there is nothing to time without a GPU"
    print(json.dumps(card()), flush=True)
    torch.manual_seed(0)
    m = vfp.create_model("attention").eval()
    ok = True
    if args.only in (None, "separate"):
        ok &= separate_case(m, [64] * args.n, "separate", args)
        torch.cuda.empty_cache()
    if args.only in (None, "varlen"):
        g = torch.Generator().manual_seed(1234)
        ok &= separate_case(m, [int(t) for t in torch.randint(16, 301, (args.varlen_clips,), generator=g)], "varlen", args)
        torch.cuda.empty_cache()
    if args.only in (None, "strided"):
        ok &= strided_case(vfp, m, args)
        torch.cuda.empty_cache()
    if args.only in (None, "decoded"):
        ok &= decoded_case(vfp, m, args)
    if not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
