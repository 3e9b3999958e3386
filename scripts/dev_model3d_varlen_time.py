"""Dev helper: throughput of the 3-D CNN model on equal-length and variable-length batches (bf16 frames resident in HBM).

    python scripts/dev_model3d_varlen_time.py                    # card, equal-length, varlen packed vs grouped by length
    python scripts/dev_model3d_varlen_time.py --equal-only --tree DIR   # equal-length case only, importing the package from DIR

Equal length: 8 192 clips x 64 frames through m(x), frame_stride 16 (the scripts/dev_model3d_time.py case).
Varlen: a seeded corpus of 8 192 clips with T ~ U[10, 128] (short videos at the scanner's default clip_length), run
  packed    - m.fingerprint_clips(clips), one packed launch sequence (includes the concatenation of the clips);
  packed*   - m.fingerprint_packed(frames, lengths) on the already concatenated frames;
  grouped   - the best possible without packing: clips pre-stacked by length, one m() call per distinct T.
Times are CUDA events around `--reps` calls after warm-up; every printed line is also a JSON object on stdout."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tree", default=ROOT, help="directory the video_fingerprint_b200 package is imported from")
    ap.add_argument("--equal-only", action="store_true")
    ap.add_argument("--n", type=int, default=8192)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    sys.path.insert(0, os.path.abspath(args.tree))
    import torch

    import video_fingerprint_b200 as vfp

    assert torch.cuda.is_available(), "this script times the B200 path; there is nothing to time without a GPU"
    fs, n = 16, args.n
    torch.manual_seed(0)
    m = vfp.create_model("3d", frame_stride=fs).eval()
    if not args.equal_only:
        print(json.dumps(card()), flush=True)

    x = torch.rand(n, 64, 3, 64, 64, device="cuda").to(torch.bfloat16)
    ms, _ = timed(lambda: m(x), args.reps)
    print(json.dumps({"case": "equal", "module": os.path.dirname(vfp.__file__), "clips": n, "frames": 64, "ms": round(ms, 3),
                      "videos_per_s": round(n / ms * 1e3), "frames_per_s": round(n * 64 / ms * 1e3)}), flush=True)
    del x
    if args.equal_only:
        return

    g = torch.Generator().manual_seed(1234)
    lengths = [int(t) for t in torch.randint(10, 129, (n,), generator=g)]
    total = sum(lengths)
    frames = torch.rand(total, 3, 64, 64, device="cuda").to(torch.bfloat16)
    starts = [0]
    for t in lengths:
        starts.append(starts[-1] + t)
    clips = [frames[starts[i] : starts[i + 1]] for i in range(n)]
    by_len = {}
    for i, t in enumerate(lengths):
        by_len.setdefault(t, []).append(i)
    groups = [(torch.tensor(idx, device="cuda"), torch.stack([clips[i] for i in idx])) for idx in by_len.values()]

    def grouped():
        out = torch.empty((n, m.embedding_dim), dtype=torch.float32, device="cuda")
        for idx, batch in groups:
            out[idx] = m(batch)
        return out

    rows = [("packed", lambda: m.fingerprint_clips(clips)), ("packed*", lambda: m.fingerprint_packed(frames, lengths)), ("grouped", grouped)]
    outs = {}
    for name, fn in rows:
        ms, outs[name] = timed(fn, args.reps)
        print(json.dumps({"case": "varlen", "run": name, "clips": n, "frames": total, "distinct_T": len(by_len), "ms": round(ms, 3),
                          "videos_per_s": round(n / ms * 1e3), "frames_per_s": round(total / ms * 1e3)}), flush=True)
    same = torch.equal(outs["packed"], outs["grouped"]) and torch.equal(outs["packed*"], outs["grouped"])
    print(json.dumps({"case": "varlen", "packed_equals_grouped": same}), flush=True)
    if not same:
        sys.exit(1)


if __name__ == "__main__":
    main()
