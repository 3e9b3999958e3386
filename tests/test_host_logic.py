"""CPU: host-side logic of the package (no device compute): grouping, JSON schema, checkpoint layout, the
C-ABI library's exported symbols, and the "fail loudly without a GPU" contract."""
import ctypes
import json
import os
import re

import numpy as np
import pytest
import torch

import video_fingerprint_b200 as vfp
from oracle import join_oracle
from oracle.weights import make_state_dict, state_dict_digest, state_spec
from video_fingerprint_b200 import _native, fingerprint
from video_fingerprint_b200.sharding import partition_clips, row_block, symmetric_block_plan

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_state_dict_layout_is_the_reference_layout():
    m = vfp.create_model("attention")
    sd = m.state_dict()
    spec = state_spec()
    assert list(sd.keys()) == [k for k, _, _ in spec]
    for k, shape, kind in spec:
        assert tuple(sd[k].shape) == tuple(shape), k
        assert sd[k].dtype == (torch.int64 if kind == "bn_count" else torch.float32), k
    m.load_state_dict(make_state_dict(3, "stress"), strict=True)


def test_default_init_reproduces_reference_init(manifest):
    """torch.manual_seed(0); create_model("attention") must give the weights the reference gives (BASELINE cfg 1)."""
    torch.manual_seed(0)
    m = vfp.create_model("attention")
    assert state_dict_digest(m.state_dict()) == manifest["cfg1_refinit"]["weights_sha256"]
    assert len(m.state_dict()) == manifest["cfg1_refinit"]["keys"]


def test_factory_error_behaviour():
    with pytest.raises(ValueError, match="Unknown model type"):
        vfp.create_model("nope")
    assert isinstance(vfp.create_model("3d"), vfp.VideoFingerprint3D)          # the reference's second model (model.py:602-607)
    m = vfp.create_model("attention", embedding_dim=128, num_attention_blocks=2, frame_stride=32)  # extra kwargs ignored
    assert m.state_dict()["final_projection.3.weight"].shape == (128, 256)
    assert not any(k.startswith("attention_blocks.2.") for k in m.state_dict())


def test_grouping_matches_oracle_on_random_pair_sets():
    rng = np.random.default_rng(0)
    for trial in range(20):
        n = int(rng.integers(2, 60))
        E = rng.standard_normal((n, 8)).astype(np.float32)
        E /= np.linalg.norm(E, axis=1, keepdims=True)
        if trial % 3 == 0:
            E *= rng.uniform(0.7, 1.0, size=(n, 1)).astype(np.float32)  # self-similarity may drop below thr
        thr = float(rng.uniform(0.2, 0.9))
        pi, pj, ps = join_oracle.threshold_pairs(E, thr)
        assert vfp.group_pairs_direct(n, pi, pj, ps) == join_oracle.group_direct(n, pi, pj, ps)
        S, I = join_oracle.topk_inner_product(E, E, min(5, n))
        assert vfp.group_pairs_topk(S, I, thr) == join_oracle.group_topk(S, I, thr)
    assert vfp.group_pairs_direct(5, np.zeros(0, np.int64), np.zeros(0, np.int64), np.zeros(0, np.float32)) == []


def test_partition_and_row_blocks():
    lengths = [300, 16, 16, 200, 100, 100, 64, 64, 64, 10]
    for world in (1, 2, 4, 8):
        parts = partition_clips(lengths, world)
        assert sorted(i for p in parts for i in p) == list(range(len(lengths)))
        loads = [sum(lengths[i] for i in p) for p in parts]
        assert max(loads) - min(loads) <= max(lengths)
        blocks = [row_block(1000, world, r) for r in range(world)]
        assert blocks[0][0] == 0 and blocks[-1][1] == 1000
        assert all(b[1] == blocks[i + 1][0] for i, b in enumerate(blocks[:-1]))
        assert all(b[0] % 128 == 0 for b in blocks)


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "vfp_b200.h")).read()
    declared = set(re.findall(r"\b(vfp(?:3d)?_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_native.EXPORTED_SYMBOLS)
    assert os.path.exists(_native.LIB_PATH), "build the library first: python -m video_fingerprint_b200.build"
    lib = ctypes.CDLL(_native.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    assert _native.load().vfp_abi_version() == _native.ABI_VERSION
    # pure host-side entry points are callable without a GPU
    assert _native.load().vfp_forward_workspace_bytes(64, 1) > 64 * 100_000
    assert _native.load().vfp_join_workspace_bytes(1000, 1000, 4096) >= 2 * 1000 * 512


def test_tuning_keys_of_removed_paths_are_rejected():
    lib = _native.load()
    # former defaults of the keys whose alternative paths are gone: the library no longer knows them
    for key, value in {0: 16384, 5: 16, 6: 0, 7: 0, 8: 0, 10: 2, 11: 1, 12: 512, 13: 0, 14: 1, 15: 1, 16: 1}.items():
        assert lib.vfp_set_tuning(key, value) == 1, key
    for key, value in {1: 2, 3: 65536, 9: 1, 17: 1}.items():   # key 2 needs a device
        assert lib.vfp_set_tuning(key, value) == 0, key


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_product_path_fails_loudly_without_gpu():
    m = vfp.create_model("attention").eval()
    with pytest.raises(_native.NativeError, match="no CUDA device"):
        m(torch.zeros(1, 10, 3, 64, 64))
    with pytest.raises(_native.NativeError, match="no CUDA device"):
        vfp.threshold_join(np.zeros((4, 256), np.float32), 0.9)
    with pytest.raises(_native.NativeError, match="no CUDA device"):
        vfp.VideoFingerprintScanner(model=m)


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "video_fingerprint_b200")
    for name in os.listdir(pkg):
        if name.endswith(".py"):
            src = open(os.path.join(pkg, name)).read()
            assert "oracle" not in src.replace("the oracle", "").replace("inject the oracle", ""), name


def test_save_results_schema(tmp_path):
    scanner = vfp.VideoFingerprintScanner.__new__(vfp.VideoFingerprintScanner)
    scanner.config, scanner.model_type = {"model_type": "attention"}, "attention"
    e = np.ones(256, np.float32) / 16
    fps = {"a.mp4": {"embedding": e, "path": "a.mp4", "name": "a.mp4", "size": 5, "file_hash": "h", "embedding_norm": np.float32(1.0)}}
    groups = [[dict(fps["a.mp4"], similarity=1.0, exact_duplicate=False)]]
    out = tmp_path / "r.json"
    scanner.save_results(fps, groups, out)  # the reference raises TypeError here (np.float32 / ndarray members)
    data = json.loads(out.read_text())
    assert set(data) == {"metadata", "fingerprints", "duplicate_groups"}
    assert set(data["metadata"]) == {"scan_date", "total_videos", "duplicate_groups", "model_config", "model_type"}
    assert isinstance(data["fingerprints"]["a.mp4"]["embedding"], list) and len(data["fingerprints"]["a.mp4"]["embedding"]) == 256
    assert data["duplicate_groups"][0][0]["similarity"] == 1.0


def test_topk_grouping_compares_in_float32_like_the_reference():
    """fingerprint.py:540 compares an np.float32 score with the Python-float threshold; NumPy 2 evaluates that in float32, so
    a score equal to np.float32(0.95) (which is < 0.95 as a double) IS a hit. Both the restatement and the product keep it."""
    thr = 0.95
    edge = np.float32(thr)
    assert float(edge) < thr and bool(edge >= thr)          # the situation the rule is about
    below = np.nextafter(edge, np.float32(0))
    S = np.array([[1.0, edge, below], [1.0, edge, 0.1], [1.0, below, 0.2]], dtype=np.float32)
    I = np.array([[0, 1, 2], [1, 0, 2], [2, 0, 1]], dtype=np.int64)
    want = join_oracle.group_topk(S, I, thr)
    got = fingerprint.group_pairs_topk(S, I, thr)
    assert [[i for i, _ in g] for g in got] == [[i for i, _ in g] for g in want] == [[0, 1]]
    # and the direct path's rule (np.where(row >= thr) on a float32 matrix, fingerprint.py:499) on the same score
    pi, pj = np.array([0, 0, 1, 1]), np.array([0, 1, 0, 1])
    ps = np.array([1.0, edge, edge, 1.0], dtype=np.float32)
    assert [[i for i, _ in g] for g in fingerprint.group_pairs_direct(2, pi, pj, ps)] == [[0, 1]]


@pytest.mark.parametrize("counts", [[5], [4, 3], [3, 4, 2], [5, 5, 4, 6], [3, 1, 4, 1, 5], [2, 3, 2, 3, 2, 3, 2, 3], [4, 0, 3, 5]])
def test_symmetric_block_plan_covers_every_ordered_pair_once(counts):
    """Sharded join: each block of the symmetric score matrix is computed by one rank and mirrored. Element-level check that
    diagonal blocks + (off-diagonal blocks and their mirror images) tile the n x n matrix exactly once."""
    world, n = len(counts), sum(counts)
    starts = np.concatenate([[0], np.cumsum(counts)])
    cover = np.zeros((n, n), dtype=int)
    for rank in range(world):
        plan = symmetric_block_plan(world, rank, counts)
        q_lo, q_hi, c_lo, c_hi = plan[0]
        assert (q_lo, q_hi, c_lo, c_hi) == (0, counts[rank], starts[rank], starts[rank + 1])
        cover[starts[rank] : starts[rank + 1], starts[rank] : starts[rank + 1]] += 1
        for q_lo, q_hi, c_lo, c_hi in plan[1:]:
            cover[starts[rank] + q_lo : starts[rank] + q_hi, c_lo:c_hi] += 1
            cover[c_lo:c_hi, starts[rank] + q_lo : starts[rank] + q_hi] += 1     # the mirrored pairs
    assert np.all(cover == 1)


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the driver runs it before our arm) times the oracle port on the host cores and prints
    one JSON line with the keys the contract names; no GPU, no extension needed."""
    import json
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--ref-budget", "1.5"],
                         capture_output=True, text=True, timeout=300, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["impl"] == "reference" and line["unit"] == "videos/s" and line["value"] > 0 and line["higher_is_better"] is True
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and line["cpu_baseline"]["value"] == line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": "videos/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["gpu_launches"] == 0 and line["steps"] == 1 and line["warmup"] == 0
