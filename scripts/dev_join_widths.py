"""Similarity join and top-k search across embedding widths, on one GPU.

    python scripts/dev_join_widths.py                       # width sweep: join, top-k
    python scripts/dev_join_widths.py --ab OTHER_ROOT       # width 256: this tree against another checkout, alternating
    python scripts/dev_join_widths.py --dump OUT.npz        # seeded width-256 outputs (tests/golden/search_dim256.npz)

Every timing is the median of CUDA-event-timed calls of the public device functions (`threshold_join_device`,
`topk_inner_product_device`) after one warm-up call of the same shape. The join's bf16 database at 262 144 rows is 32 MB at
width 64 and 256 MB at width 512, so the wide cases are read from HBM and the narrow ones from L2, as a user's would be.
`--ab` starts one child process per round with the other tree first on sys.path, so both builds run the same code here.
Each output line is one JSON record; the first one names the card and its power limit.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WIDTHS = (64, 128, 256, 384, 512)


def golden_inputs() -> dict:
    """Seeded width-256 inputs of the golden: planted near-duplicates on both sides of 0.9, exact copies, and a tight cluster
    of 200 rows that defeats the top-k screen bound (its rows take the exact fallback scan)."""
    rng = np.random.default_rng(256)
    E = rng.standard_normal((2000, 256)).astype(np.float32)
    E /= np.linalg.norm(E, axis=1, keepdims=True)
    for t in range(150):
        a, b = 2 * t, 1000 + 2 * t
        v = E[a] + rng.choice([0.0, 0.01, 0.02, 0.03, 0.05]) * rng.standard_normal(256).astype(np.float32)
        E[b] = v / np.linalg.norm(v)
    E[1500:1520] = E[400:420]
    E[1600:1800] = E[5] + 1e-4 * rng.standard_normal((200, 256)).astype(np.float32)
    E[1600:1800] /= np.linalg.norm(E[1600:1800], axis=1, keepdims=True)
    Q = rng.standard_normal((500, 256)).astype(np.float32)
    Q /= np.linalg.norm(Q, axis=1, keepdims=True)
    Q[::5] = E[1000:1200:2]
    return {"E": E, "Q": Q}


def inputs_sha256(inputs: dict) -> str:
    h = hashlib.sha256()
    for name in sorted(inputs):
        h.update(name.encode())
        h.update(np.ascontiguousarray(inputs[name]).tobytes())
    return h.hexdigest()


def sorted_pairs(i, j, s):
    i, j, s = (x.cpu().numpy() for x in (i, j, s))
    order = np.lexsort((j, i))
    return i[order].astype(np.int32), j[order].astype(np.int32), s[order]


def golden_outputs(vfp, inputs: dict) -> dict:
    """The outputs the golden pins, from the public device functions at their default settings."""
    import torch

    E, Q = (torch.from_numpy(inputs[k]).cuda() for k in ("E", "Q"))
    out = {}
    out["join_self_i"], out["join_self_j"], out["join_self_s"] = sorted_pairs(*vfp.threshold_join_device(E, 0.9))
    out["join_cross_i"], out["join_cross_j"], out["join_cross_s"] = sorted_pairs(*vfp.threshold_join_device(E, 0.9, q=Q, q_row0=1000))
    S, I = vfp.topk_inner_product_device(Q[:300], E, 20)
    out["topk_cross_s"], out["topk_cross_i"] = S.cpu().numpy(), I.cpu().numpy()
    S, I = vfp.topk_inner_product_device(E[1590:1700], E, 20)
    out["topk_tie_s"], out["topk_tie_i"] = S.cpu().numpy(), I.cpu().numpy()
    return out


def unit_rows(n: int, dim: int, seed: int, copies: float = 0.01):
    """n unit rows, a fraction `copies` of them noisy copies of others (duplicate pairs above 0.95)."""
    import torch

    g = torch.Generator(device="cuda").manual_seed(seed)
    X = torch.randn((n, dim), generator=g, device="cuda")
    m = int(n * copies)
    src = torch.randint(0, n, (m,), generator=g, device="cuda")
    dst = torch.randint(0, n, (m,), generator=g, device="cuda")
    X[dst] = X[src] + 0.1 / dim ** 0.5 * torch.randn((m, dim), generator=g, device="cuda")
    return X / X.norm(dim=1, keepdim=True)


def time_ms(fn, reps: int) -> list:
    import torch

    fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b))
    return out


def join_record(vfp, dim: int, n: int, reps: int) -> dict:
    X = unit_rows(n, dim, seed=dim)
    res = {}
    ms = time_ms(lambda: res.update(out=vfp.threshold_join_device(X, 0.95)), reps)
    med = float(np.median(ms))
    pairs = n * n                 # every ordered pair, the count of np.dot(E, E.T)
    screened = n * (n + 1) // 2   # a self join screens the upper triangle only
    kb = -(-dim // 64)
    return {"case": "join", "dim": dim, "rows": n, "thr": 0.95, "ms_median": round(med, 3), "ms": [round(x, 3) for x in ms],
            "result_pairs": int(res["out"][0].numel()), "gpairs_per_s": round(pairs / med / 1e6, 1),
            "executed_tflops": round(2 * screened * 64 * kb / med / 1e9, 1),
            "algorithmic_tflops": round(2 * screened * dim / med / 1e9, 1)}


def topk_record(vfp, dim: int, n_db: int, n_q: int, k: int, reps: int) -> dict:
    db = unit_rows(n_db, dim, seed=dim + 1)
    q = unit_rows(n_q, dim, seed=dim + 2)
    q[: n_q // 100] = db[: n_q // 100]
    ms = time_ms(lambda: vfp.topk_inner_product_device(q, db, k), reps)
    med = float(np.median(ms))
    pairs = n_db * n_q
    return {"case": "topk", "dim": dim, "db_rows": n_db, "queries": n_q, "k": k, "ms_median": round(med, 3),
            "ms": [round(x, 3) for x in ms], "gpairs_per_s": round(pairs / med / 1e6, 1),
            "executed_tflops": round(2 * pairs * 64 * -(-dim // 64) / med / 1e9, 1),
            "algorithmic_tflops": round(2 * pairs * dim / med / 1e9, 1)}


def card() -> dict:
    import torch

    rec = {"case": "card", "name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        rec["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        rec["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return rec


def emit(rec: dict) -> None:
    print(json.dumps(rec), flush=True)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--dump", metavar="OUT_NPZ", help="write the seeded width-256 outputs the golden test reads")
    ap.add_argument("--ab", metavar="OTHER_ROOT", help="alternate this tree and OTHER_ROOT at width 256")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--root", default=ROOT, help=argparse.SUPPRESS)   # child of --ab: the tree to import
    ap.add_argument("--time256", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--join-rows", type=int, default=262_144)
    ap.add_argument("--topk-db", type=int, default=1_000_000)
    ap.add_argument("--topk-q", type=int, default=100_000)
    args = ap.parse_args()
    sys.path.insert(0, args.root)
    import torch

    import video_fingerprint_b200 as vfp

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: every figure here is measured on the GPU")
    torch.cuda.set_device(0)

    if args.dump:
        inputs = golden_inputs()
        out = golden_outputs(vfp, inputs)
        np.savez_compressed(args.dump, inputs_sha256=np.array(inputs_sha256(inputs)), **out)
        emit({"case": "dump", "path": args.dump, "inputs_sha256": inputs_sha256(inputs), "arrays": sorted(out)})
        return
    if args.time256:   # one round of --ab, in the tree given by --root
        emit(dict(join_record(vfp, 256, args.join_rows, args.reps), root=args.root))
        emit(dict(topk_record(vfp, 256, 10_000_000, 100_000, 10, args.reps), root=args.root, sized_as="bench.py cfg5_topk"))
        return
    emit(card())
    if args.ab:
        for r in range(args.rounds):
            for root in (os.path.abspath(args.ab), ROOT):
                cmd = [sys.executable, os.path.abspath(__file__), "--time256", "--root", root, "--reps", str(args.reps),
                       "--join-rows", str(args.join_rows)]
                child = subprocess.run(cmd, capture_output=True, text=True)
                for line in child.stdout.splitlines():
                    emit(dict(json.loads(line), round=r))
                if child.returncode:
                    raise SystemExit(child.stderr)
        return
    for dim in WIDTHS:
        emit(join_record(vfp, dim, args.join_rows, args.reps))
    for dim in WIDTHS:
        emit(topk_record(vfp, dim, args.topk_db, args.topk_q, 20, args.reps))


if __name__ == "__main__":
    main()
