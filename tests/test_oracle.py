"""CPU: the oracle restatement against the golden vectors recorded from the unmodified reference
(tests/golden/make_golden.py): embeddings, pooled features and duplicate groups."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import join_oracle
from oracle.forward_oracle import fingerprint_clips, forward_oracle, positional_table, subsample_indices
from oracle.weights import make_clips, make_state_dict, state_dict_digest, state_spec

FORWARD_CASES = ["cfg1_default", "cfg1_stress", "varlen_stress", "t64_default"]


def _fake_fingerprints(E, n_hash_dups=0):
    return {
        f"/videos/v{i:05d}.mp4": {
            "embedding": e, "path": f"/videos/v{i:05d}.mp4", "name": f"v{i:05d}.mp4", "size": 1000 + 7 * i,
            "file_hash": f"hash{i if i >= n_hash_dups else 0:05d}", "embedding_norm": float(np.linalg.norm(e)),
        }
        for i, e in enumerate(E)
    }


def test_state_spec_shape():
    spec = state_spec()
    assert len(spec) == 144
    sd = make_state_dict(0)
    assert sum(v.numel() for v in sd.values()) == 6_521_165
    assert sum(1 for _, _, kind in spec if kind == "bn_count") == 12


@pytest.mark.parametrize("name", FORWARD_CASES)
def test_forward_oracle_matches_reference_golden(name, golden_dir, manifest):
    c = manifest[name]
    sd = make_state_dict(c["wseed"], c["wstyle"])
    assert state_dict_digest(sd) == c["weights_sha256"], "seeded weights differ from the ones the golden run used"
    clips = make_clips(c["cseed"], c["lengths"], c["cstyle"], c["quantise"])
    assert abs(float(clips[0].double().sum()) - c["clip0_sum"]) < 1e-6
    gold = np.load(os.path.join(golden_dir, f"forward_{name}.npz"))
    if len(set(c["lengths"])) > 1:
        clips, rows = clips[:6], slice(0, 6)  # keep the CPU suite short; the long clips are covered on the GPU
    else:
        rows = slice(None)
    out = torch.stack(fingerprint_clips(sd, clips)).numpy()
    np.testing.assert_allclose(out, gold["embeddings"][rows], atol=2e-6, rtol=0)


def test_min_frames_and_subsampling_rule():
    sd = make_state_dict(0)
    assert fingerprint_clips(sd, [torch.zeros(9, 3, 64, 64)]) == [None]
    assert subsample_indices(400) == list(range(400))
    assert subsample_indices(1200) == list(range(0, 1200, 2))[:500]
    assert len(subsample_indices(1499)) == 500 and subsample_indices(1499)[1] == 2
    assert subsample_indices(999)[:3] == [0, 1, 2] and len(subsample_indices(999)) == 500


def test_positional_table_is_the_checkpoint_buffer():
    sd = make_state_dict(0)
    assert torch.equal(sd["pos_encoding.pe"][0, :64], positional_table(64))


def test_layout_quirk_dim1_equals_3():
    sd = make_state_dict(0)
    x = torch.rand(1, 3, 12, 64, 64)  # (B, C=3, T, H, W) is re-interpreted (model.py:283)
    a = forward_oracle(sd, x)
    b = forward_oracle(sd, x.permute(0, 2, 1, 3, 4).contiguous())
    assert torch.allclose(a, b, atol=1e-6)


def test_join_oracle_matches_reference_golden(golden_dir):
    with open(os.path.join(golden_dir, "find_duplicates.json")) as f:
        gold = json.load(f)
    Es = np.load(os.path.join(golden_dir, "forward_cfg1_stress.npz"))["embeddings"]
    E0 = np.load(os.path.join(golden_dir, "forward_cfg1_refinit.npz"))["embeddings"]
    X = np.load(os.path.join(golden_dir, "join_planted150.npy"))
    cases = {
        "cfg1_stress_thr0.95": (_fake_fingerprints(Es, 3), 0.95, True),
        "cfg1_stress_thr0.99": (_fake_fingerprints(Es, 3), 0.99, True),
        "cfg1_refinit_thr0.95": (_fake_fingerprints(E0), 0.95, True),
        "planted150_thr0.95_direct": (_fake_fingerprints(X, 2), 0.95, False),
        "planted150_thr0.8_direct": (_fake_fingerprints(X, 2), 0.8, False),
    }
    for key, (fps, thr, use_faiss) in cases.items():
        got = join_oracle.find_duplicates(fps, thr, use_faiss)
        want = gold[key]
        assert [[it["name"] for it in g] for g in got] == [[it["name"] for it in g] for g in want], key
        for g, w in zip(got, want):
            for a, b in zip(g, w):
                assert abs(a["similarity"] - b["similarity"]) < 1e-6
                assert a["exact_duplicate"] == b["exact_duplicate"]


def test_topk_restatement_properties():
    rng = np.random.default_rng(3)
    db = rng.standard_normal((500, 256)).astype(np.float32)
    db[77] = db[5]  # exact tie -> broken by ascending index
    S, I = join_oracle.topk_inner_product(db[:40], db, 20)
    assert S.shape == (40, 20) and I.dtype == np.int64
    assert np.all(S[:, :-1] >= S[:, 1:])
    assert I[5, 0] == 5 and I[5, 1] == 77 and S[5, 0] == S[5, 1]
    full = db[:40] @ db.T
    assert np.allclose(np.sort(full, axis=1)[:, ::-1][:, :20], S)


@pytest.mark.parametrize("name", FORWARD_CASES)
def test_oracle_features_match_reference_golden(name, golden_dir, manifest):
    """B=1 forwards, clip by clip, against the embeddings and the pooled attention features (`adaptive_pooling` of the
    last block's output) the reference recorded for the same seeded weights and clips."""
    c = manifest[name]
    sd = make_state_dict(c["wseed"], c["wstyle"])
    clips = make_clips(c["cseed"], c["lengths"], c["cstyle"], c["quantise"])[:6]   # the long clips are covered on the GPU
    gold = np.load(os.path.join(golden_dir, f"forward_{name}.npz"))
    for i, clip in enumerate(clips):
        st = {}
        got = forward_oracle(sd, clip.unsqueeze(0), st)
        assert torch.allclose(got[0], torch.from_numpy(gold["embeddings"][i]), atol=2e-6), (name, i)
        assert torch.allclose(st["pooled"][0], torch.from_numpy(gold["pooled"][i]), atol=1e-4, rtol=1e-5), (name, i)


def test_tanh_gelu_is_harmless():
    """The CUDA MLP epilogue evaluates GELU in its tanh form (csrc/epilogues.cuh). Pin the claim made there: swapping
    the exact erf form for the tanh form in the fp32 oracle moves the embeddings by far less than the parity bar."""
    import torch.nn.functional as F

    import oracle.forward_oracle as fo

    sd = make_state_dict(2, "stress")
    clips = make_clips(41, [37, 64, 10, 21], "colour")
    exact = torch.stack(fo.fingerprint_clips(sd, clips)).double()
    orig = F.gelu
    try:
        fo.F.gelu = lambda h: orig(h, approximate="tanh")
        approx = torch.stack(fo.fingerprint_clips(sd, clips)).double()
    finally:
        fo.F.gelu = orig
    cos = (exact * approx).sum(-1) / (exact.norm(dim=-1) * approx.norm(dim=-1))
    assert float((1 - cos).max()) < 1e-7
