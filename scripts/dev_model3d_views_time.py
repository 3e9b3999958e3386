"""Dev helper: the 3-D CNN model on clips read in place (fingerprint_views) against the copying paths.

    python scripts/dev_model3d_views_time.py              # card, varlen, hwc, scanner, decoded
    python scripts/dev_model3d_views_time.py --only varlen

varlen   - the seeded corpus of scripts/dev_model3d_varlen_time.py (8 192 bf16 clips, T ~ U[10, 128], frame_stride 16) through
           m.fingerprint_clips(clips) (concatenates the clips), m.fingerprint_packed(frames, lengths) on the already
           concatenated frames, and m.fingerprint_views(clips) (reads the clips where they are). All three must be bit-identical.
scanner  - 1 024 preprocessed uint8 videos of 300 - 1 000 frames at the default clip_length 128 (3 windows each) through
           scanner.extract_fingerprints_3d_from_frames (copies every window, then concatenates them) and through the same
           rule on fingerprint_views of the windows in place.
hwc      - the varlen lengths as uint8 frames: fingerprint_views on planar (T, 3, 64, 64) views against the same frames in
           decoder layout (T, 64, 64, 3); both must be bit-identical.
decoded  - 64 decoded 320 x 240 videos of 300 - 1 000 frames (host arrays, slices of one seeded pool) through
           scanner.extract_fingerprints_3d_from_decoded, against preprocess_frames_device of every frame + permute +
           extract_fingerprints_3d_from_frames.
Times are CUDA events around `--reps` calls after warm-up (the scanner paths end in a device-to-host copy, which
synchronises); every printed line is also a JSON object on stdout."""
import argparse
import json
import os
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


def timed(fn, reps, warmup=2):
    import torch

    for _ in range(warmup):
        out = fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, out


def same_rows(a, b):
    import numpy as np

    return all((x is None and y is None) or (x is not None and y is not None and np.array_equal(x, y)) for x, y in zip(a, b))


def varlen(m, n, reps):
    import torch

    g = torch.Generator().manual_seed(1234)
    lengths = [int(t) for t in torch.randint(10, 129, (n,), generator=g)]
    total = sum(lengths)
    frames = torch.rand(total, 3, 64, 64, device="cuda").to(torch.bfloat16)
    starts = [0]
    for t in lengths:
        starts.append(starts[-1] + t)
    clips = [frames[starts[i] : starts[i + 1]] for i in range(n)]
    rows = [("clips", lambda: m.fingerprint_clips(clips)), ("packed", lambda: m.fingerprint_packed(frames, lengths)),
            ("views", lambda: m.fingerprint_views(clips))]
    outs = {}
    for name, fn in rows:
        ms, outs[name] = timed(fn, reps)
        print(json.dumps({"case": "varlen", "run": name, "clips": n, "frames": total, "ms": round(ms, 3),
                          "videos_per_s": round(n / ms * 1e3), "frames_per_s": round(total / ms * 1e3)}), flush=True)
    same = torch.equal(outs["clips"], outs["packed"]) and torch.equal(outs["views"], outs["packed"])
    print(json.dumps({"case": "varlen", "bit_identical": same}), flush=True)
    return same


def hwc_case(m, n, reps):
    import torch

    g = torch.Generator().manual_seed(1234)
    lengths = [int(t) for t in torch.randint(10, 129, (n,), generator=g)]
    total = sum(lengths)
    planar = torch.randint(0, 256, (total, 3, 64, 64), dtype=torch.uint8, device="cuda", generator=torch.Generator("cuda").manual_seed(3))
    hwc = planar.permute(0, 2, 3, 1).contiguous()
    starts = [0]
    for t in lengths:
        starts.append(starts[-1] + t)
    outs = {}
    for name, buf in (("planar_u8", planar), ("hwc_u8", hwc)):
        clips = [buf[starts[i] : starts[i + 1]] for i in range(n)]
        ms, outs[name] = timed(lambda: m.fingerprint_views(clips), reps)
        print(json.dumps({"case": "hwc", "run": name, "clips": n, "frames": total, "ms": round(ms, 3),
                          "videos_per_s": round(n / ms * 1e3), "frames_per_s": round(total / ms * 1e3)}), flush=True)
    same = torch.equal(outs["planar_u8"], outs["hwc_u8"])
    print(json.dumps({"case": "hwc", "bit_identical": same}), flush=True)
    return same


def scanner_case(vfp, m, n_videos, reps):
    import torch

    sc = vfp.VideoFingerprintScanner(model=m, config={"model_type": "3d", "frame_stride": m.frame_stride})
    g = torch.Generator().manual_seed(4321)
    lengths = [int(t) for t in torch.randint(300, 1001, (n_videos,), generator=g)]
    pool = torch.randint(0, 256, (sum(lengths), 3, 64, 64), dtype=torch.uint8, device="cuda", generator=torch.Generator("cuda").manual_seed(5))
    videos, f = [], 0
    for t in lengths:
        videos.append(pool[f : f + t])
        f += t
    clip_length = sc.config.get("clip_length", 128)

    def views_rule():   # the rule of extract_fingerprints_3d_from_frames, its windows read in place
        views, spans = [], []
        for v, fr in enumerate(videos):
            starts = sc.window_starts_3d(int(fr.shape[0]))
            spans.append((v, len(views), len(starts)))
            views += [fr[s : s + clip_length] for s in starts]
        emb = m.fingerprint_views(views).cpu().numpy()
        result = [None] * len(videos)
        sc._combine_windows_3d(emb, spans, lengths, result)
        return result

    windows = sum(len(sc.window_starts_3d(t)) for t in lengths)
    outs = {}
    for name, fn in (("frames", lambda: sc.extract_fingerprints_3d_from_frames(videos)), ("views", views_rule)):
        ms, outs[name] = timed(fn, reps, warmup=1)
        print(json.dumps({"case": "scanner", "run": name, "videos": n_videos, "frames": sum(lengths), "windows": windows,
                          "ms": round(ms, 3), "videos_per_s": round(n_videos / ms * 1e3)}), flush=True)
    same = same_rows(outs["frames"], outs["views"])
    print(json.dumps({"case": "scanner", "bit_identical": same}), flush=True)
    return same


def decoded_case(vfp, m, n_videos, reps):
    import numpy as np
    import torch

    sc = vfp.VideoFingerprintScanner(model=m, config={"model_type": "3d", "frame_stride": m.frame_stride})
    rng = np.random.default_rng(99)
    lengths = rng.integers(300, 1001, n_videos).tolist()
    pool = rng.integers(0, 256, (1000 + n_videos, 240, 320, 3), dtype=np.uint8)
    videos = [pool[i : i + t] for i, t in enumerate(lengths)]   # host views: decoded frames as a decoder hands them over

    def full_path():
        planar = [vfp.preprocess_frames_device(v).permute(0, 3, 1, 2).contiguous() for v in videos]
        return sc.extract_fingerprints_3d_from_frames(planar)

    outs = {}
    for name, fn in (("preprocess_all+frames", full_path), ("decoded", lambda: sc.extract_fingerprints_3d_from_decoded(videos))):
        ms, outs[name] = timed(fn, reps, warmup=1)
        print(json.dumps({"case": "decoded", "run": name, "videos": n_videos, "frames": sum(lengths), "size": "320x240",
                          "ms": round(ms, 3), "videos_per_s": round(n_videos / ms * 1e3)}), flush=True)
    same = same_rows(outs["preprocess_all+frames"], outs["decoded"])
    print(json.dumps({"case": "decoded", "bit_identical": same}), flush=True)
    return same


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", choices=["varlen", "hwc", "scanner", "decoded"])
    ap.add_argument("--n", type=int, default=8192, help="varlen clips")
    ap.add_argument("--videos", type=int, default=1024, help="scanner videos")
    ap.add_argument("--decoded-videos", type=int, default=64)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    import torch

    import video_fingerprint_b200 as vfp

    assert torch.cuda.is_available(), "this script times the B200 path; there is nothing to time without a GPU"
    print(json.dumps(card()), flush=True)
    torch.manual_seed(0)
    m = vfp.create_model("3d", frame_stride=16).eval()
    ok = True
    if args.only in (None, "varlen"):
        ok &= varlen(m, args.n, args.reps)
        torch.cuda.empty_cache()
    if args.only in (None, "hwc"):
        ok &= hwc_case(m, args.n, args.reps)
        torch.cuda.empty_cache()
    if args.only in (None, "scanner"):
        ok &= scanner_case(vfp, m, args.videos, max(1, args.reps // 3))
        torch.cuda.empty_cache()
    if args.only in (None, "decoded"):
        ok &= decoded_case(vfp, m, args.decoded_videos, max(1, args.reps // 5))
    if not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
