"""GPU: the similarity join and the top-k search at every embedding width the models produce (1 to 512 columns).

Bars, as in tests/test_join_gpu.py and tests/test_topk_gpu.py: the join's pair set equals the fp32 NumPy oracle's except pairs
whose score lies within 1e-6 of the threshold (summation order); top-k indices equal the oracle's after (score desc, index asc)
tie-breaking except inside near-ties of 2e-6; scores agree to 1e-5. At width 256 the outputs are bitwise those of the build
before other widths existed (tests/golden/search_dim256.npz, written by `scripts/dev_join_widths.py --dump`)."""
import ctypes as C
import importlib.util
import os

import numpy as np
import pytest
import torch

import video_fingerprint_b200 as vfp
from oracle import join_oracle
from video_fingerprint_b200 import _native
from video_fingerprint_b200 import fingerprint as fp
from video_fingerprint_b200.fingerprint import screen_margin

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GUARD = 1 << 20
PATTERN = 0xA5


def unit(n, dim, seed):
    rng = np.random.default_rng(seed)
    E = rng.standard_normal((n, dim)).astype(np.float32)
    return E / np.linalg.norm(E, axis=1, keepdims=True)


def planted(n, dim, seed, thr):
    """Unit rows with pairs planted at set similarities on both sides of `thr`, plus exact copies."""
    rng = np.random.default_rng(seed)
    E = unit(n, dim, seed)
    targets = [thr - 0.05, thr - 5e-4, thr - 1e-5, thr + 1e-5, thr + 5e-4, thr + 0.03, 1.0] * 6
    for t, target in enumerate(targets):
        a, b = 3 * t, 3 * t + 1
        r = rng.standard_normal(dim).astype(np.float32)
        r -= (r @ E[a]) * E[a]
        r /= max(np.linalg.norm(r), 1e-12)
        E[b] = target * E[a] + np.sqrt(max(0.0, 1 - target * target)) * r
    E[n - 30 : n] = E[200:230]   # exact copies
    return E


def assert_pairs_match(got, want, thr, band=1e-6):
    g = {(int(a), int(b)): float(s) for a, b, s in zip(*got)}
    w = {(int(a), int(b)): float(s) for a, b, s in zip(*want)}
    for key in set(g) ^ set(w):
        s = g.get(key, w.get(key))
        assert abs(s - thr) < band, (key, s)
    for key in set(g) & set(w):
        assert abs(g[key] - w[key]) < 1e-5, key
    return len(g)


def check_topk(S, I, Q, DB, k):
    wS, wI = join_oracle.topk_inner_product(Q, DB, k)
    assert S.shape == wS.shape and I.shape == wI.shape
    np.testing.assert_allclose(S, wS, atol=1e-5, rtol=0)
    mism = I != wI
    if mism.any():
        r, c = np.nonzero(mism)
        full = Q[r] @ DB.T
        assert np.all(np.abs(full[np.arange(len(r)), I[r, c]] - full[np.arange(len(r)), wI[r, c]]) < 2e-6)


def ptr(t):
    return C.c_void_p(t.data_ptr())


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class Guarded:
    """A device buffer of `nbytes` between 1 MiB guard zones filled with a pattern; `.t` is the usable uint8 view."""

    def __init__(self, nbytes):
        self.n = (int(nbytes) + 255) // 256 * 256
        self.raw = torch.full((self.n + 2 * GUARD,), PATTERN, dtype=torch.uint8, device="cuda")
        self.t = self.raw[GUARD : GUARD + self.n]

    def view(self, dtype, shape):
        n = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
        return self.t[:n].view(dtype).view(shape)

    def intact(self):
        return bool((self.raw[:GUARD] == PATTERN).all()) and bool((self.raw[GUARD + self.n :] == PATTERN).all())


def raw_topk(Q, DB, k, dim=None, ws_dim=None):
    """vfp_topk_ip through the ABI: (rc, S, I, flags), outputs pre-filled with a sentinel."""
    lib = _native.load()
    q, db = torch.from_numpy(Q).cuda(), torch.from_numpy(DB).cuda()
    dim = q.shape[1] if dim is None else dim
    ws = torch.empty(max(1, lib.vfp_topk_workspace_bytes_dim(len(Q), len(DB), k, ws_dim or q.shape[1])), dtype=torch.uint8, device="cuda")
    S = torch.full((len(Q), k), -7.0, device="cuda")
    I = torch.full((len(Q), k), -7, dtype=torch.int64, device="cuda")
    flags = torch.full((2,), -7, dtype=torch.int64, device="cuda")
    rc = lib.vfp_topk_ip(ptr(q), ptr(db), len(Q), len(DB), dim, k, float(screen_margin(q, db)), ptr(S), ptr(I), ptr(flags),
                         ptr(ws), ws.numel(), stream())
    torch.cuda.synchronize()
    return rc, S.cpu().numpy(), I.cpu().numpy(), flags.cpu().numpy()


# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dim", [16, 32, 64, 96, 128, 192, 240, 256, 320, 384, 448, 512])
def test_pair_join_parity_across_widths(dim):
    thr = 0.9
    E = planted(1500, dim, seed=dim, thr=thr)
    Q = np.ascontiguousarray(E[700:1100])
    want_self = join_oracle.threshold_pairs(E, thr)
    wi, wj, ws = join_oracle.threshold_pairs(E, thr, Q=Q)
    want_cross = (wi + 700, wj, ws)
    n = assert_pairs_match(vfp.threshold_join(E, thr), want_self, thr)
    assert n >= 1500 + 30
    assert_pairs_match(vfp.threshold_join(E, thr, q=Q, q_row0=700), want_cross, thr)


@pytest.mark.parametrize("dim", [32, 128, 512])
@pytest.mark.parametrize("k", [1, 10, 20, 32])
def test_topk_parity_across_widths(dim, k):
    DB = unit(3000, dim, seed=dim + k)
    Q = unit(300, dim, seed=dim + k + 1)
    Q[:150] = DB[:150]
    DB[2900:2940] = DB[10:50]    # exact copies: tied scores ranked by index
    S, I = vfp.topk_inner_product(Q, DB, k)
    check_topk(S, I, Q, DB, k)
    assert np.all(I[:10, 0] == np.arange(10))


@pytest.mark.parametrize("dim", [64, 512])
def test_topk_dense_tie_cluster_takes_the_exact_fallback(dim):
    rng = np.random.default_rng(dim)
    E = unit(5000, dim, seed=dim)
    E[1000:1300] = E[0] + 1e-4 * rng.standard_normal((300, dim)).astype(np.float32)
    E[1000:1300] /= np.linalg.norm(E[1000:1300], axis=1, keepdims=True)
    Q = np.ascontiguousarray(E[990:1310])
    rc, S, I, flags = raw_topk(Q, E, 20)
    assert rc == 0
    assert flags[0] > 0 and flags[1] == 0, flags
    check_topk(S, I, Q, E, 20)


@pytest.mark.parametrize("dim", [1, 3, 100, 129, 500])
def test_widths_off_the_multiple_of_16_are_zero_padded(dim):
    thr = 0.8 if dim > 3 else 0.999
    E = planted(700, dim, seed=dim + 7, thr=thr)
    assert_pairs_match(vfp.threshold_join(E, thr), join_oracle.threshold_pairs(E, thr), thr)
    Q = np.ascontiguousarray(E[100:300])
    wi, wj, ws = join_oracle.threshold_pairs(E, thr, Q=Q)
    assert_pairs_match(vfp.threshold_join(E, thr, q=Q, q_row0=100), (wi + 100, wj, ws), thr)
    k = 10
    S, I = vfp.topk_inner_product(Q, E, k)
    if dim > 3:
        check_topk(S, I, Q, E, k)
    else:   # a few columns: many exact ties, whose fp32 scores the oracle and the warp sum both compute exactly
        wS, _ = join_oracle.topk_inner_product(Q, E, k)
        np.testing.assert_allclose(S, wS, atol=1e-5, rtol=0)
        full = Q @ E.T
        np.testing.assert_allclose(np.take_along_axis(full, I, axis=1), wS, atol=1e-5, rtol=0)


def test_width_256_pair_join_is_bitwise_the_earlier_build(golden_dir):
    spec = importlib.util.spec_from_file_location("dev_join_widths", os.path.join(ROOT, "scripts", "dev_join_widths.py"))
    dev = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(dev)
    gold = np.load(os.path.join(golden_dir, "search_dim256.npz"))
    inputs = dev.golden_inputs()
    assert str(gold["inputs_sha256"]) == dev.inputs_sha256(inputs)
    got = dev.golden_outputs(vfp, inputs)
    for name, arr in got.items():
        assert arr.dtype == gold[name].dtype and arr.shape == gold[name].shape, name
        assert np.array_equal(arr.view(np.uint8), gold[name].view(np.uint8)), name


@pytest.mark.parametrize("dim", [128, 512])
def test_writes_stay_inside_their_buffers_and_repeat(dim):
    lib = _native.load()
    n = 3001
    E = planted(n, dim, seed=dim + 3, thr=0.95)
    dev = torch.from_numpy(E).cuda()
    margin = float(screen_margin(dev, dev))
    cap = 8 * n
    results = []
    for _ in range(2):
        ws = Guarded(lib.vfp_join_workspace_bytes_dim(n, n, 4 * cap, dim))
        oi, oj, os_, cnt = Guarded(cap * 4), Guarded(cap * 4), Guarded(cap * 4), Guarded(16)
        _native.check(lib.vfp_join_threshold(ptr(dev), ptr(dev), n, n, dim, 0, 0.95, margin, ptr(oi.t), ptr(oj.t), ptr(os_.t), cap,
                                             ptr(cnt.t), ptr(ws.t), ws.n, stream()), "vfp_join_threshold")
        kk = 20
        ws2 = Guarded(lib.vfp_topk_workspace_bytes_dim(n, n, kk, dim))
        S, I, fl = Guarded(n * kk * 4), Guarded(n * kk * 8), Guarded(16)
        _native.check(lib.vfp_topk_ip(ptr(dev), ptr(dev), n, n, dim, kk, margin, ptr(S.t), ptr(I.t), ptr(fl.t), ptr(ws2.t), ws2.n,
                                      stream()), "vfp_topk_ip")
        torch.cuda.synchronize()
        assert lib.vfp_device_error_word() == 0
        assert all(g.intact() for g in (ws, oi, oj, os_, cnt, ws2, S, I, fl))
        m = int(cnt.view(torch.int64, (2,))[0])
        gi, gj, gs = (b.view(dt, (cap,))[:m].cpu().numpy() for b, dt in ((oi, torch.int32), (oj, torch.int32), (os_, torch.float32)))
        order = np.lexsort((gj, gi))
        results.append((gi[order], gj[order], gs[order], S.view(torch.float32, (n, kk)).cpu().numpy(),
                        I.view(torch.int64, (n, kk)).cpu().numpy()))
    for a, b in zip(*results):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    wi, wj, ws_ = join_oracle.threshold_pairs(E, 0.95)
    assert_pairs_match(results[0][:3], (wi, wj, ws_), 0.95)
    check_topk(results[0][3], results[0][4], E, E, 20)


def test_abi_rejects_unsupported_widths_before_running():
    lib = _native.load()
    n = 1000
    E = unit(n, 512, seed=1)
    dev = torch.from_numpy(E).cuda()
    margin = float(screen_margin(dev, dev))
    cap = 4096

    def join(dim, ws_dim):
        ws = torch.empty(max(1, lib.vfp_join_workspace_bytes_dim(n, n, cap, ws_dim)), dtype=torch.uint8, device="cuda")
        oi, oj = (torch.full((cap,), -7, dtype=torch.int32, device="cuda") for _ in range(2))
        os_ = torch.full((cap,), -7.0, device="cuda")
        cnt = torch.full((2,), -7, dtype=torch.int64, device="cuda")
        rc = lib.vfp_join_threshold(ptr(dev), ptr(dev), n, n, dim, 0, 0.9, margin, ptr(oi), ptr(oj), ptr(os_), cap, ptr(cnt),
                                    ptr(ws), ws.numel(), stream())
        torch.cuda.synchronize()
        untouched = bool((oi == -7).all() and (oj == -7).all() and (os_ == -7.0).all() and (cnt == -7).all())
        return rc, untouched

    for dim in (0, 8, 24, 528):
        assert lib.vfp_join_workspace_bytes_dim(n, n, cap, dim) == 0 and lib.vfp_topk_workspace_bytes_dim(n, n, 10, dim) == 0
        rc, untouched = join(dim, 512)
        assert rc != 0 and untouched and f"dim {dim}" in lib.vfp_last_error().decode()
        rc, S, I, flags = raw_topk(E, E, 10, dim=dim, ws_dim=512)
        assert rc != 0 and (S == -7.0).all() and (I == -7).all() and (flags == -7).all()
        assert f"dim {dim}" in lib.vfp_last_error().decode()
    # a workspace sized for a narrower row than the call's
    rc, untouched = join(512, 128)
    assert rc != 0 and untouched and "workspace too small" in lib.vfp_last_error().decode()
    rc, S, I, flags = raw_topk(E, E, 10, dim=512, ws_dim=128)
    assert rc != 0 and (S == -7.0).all() and (I == -7).all() and (flags == -7).all()
    assert "workspace too small" in lib.vfp_last_error().decode()
    # the width-less sizes keep their meaning (256)
    assert lib.vfp_join_workspace_bytes(n, n, cap) == lib.vfp_join_workspace_bytes_dim(n, n, cap, 256)
    assert lib.vfp_topk_workspace_bytes(n, n, 10) == lib.vfp_topk_workspace_bytes_dim(n, n, 10, 256)


def test_python_rejects_bad_shapes_before_touching_the_device(monkeypatch):
    def no_device(*a, **k):
        raise AssertionError("reached the device")

    monkeypatch.setattr(fp, "_as_device_f32", no_device)
    monkeypatch.setattr(fp._native, "load", no_device)
    E = unit(50, 128, seed=2)
    for call in (lambda: fp.threshold_join_device(E, 0.9, q=unit(5, 64, 3)),
                 lambda: fp.topk_inner_product_device(unit(5, 64, 3), E, 5),
                 lambda: fp.threshold_join_device(unit(50, 513, 4), 0.9),
                 lambda: fp.topk_inner_product_device(None, unit(50, 513, 4), 5),
                 lambda: fp.duplicate_pairs(unit(50, 513, 4), 0.9),
                 lambda: fp.threshold_join_device(E[0], 0.9)):
        with pytest.raises(ValueError):
            call()


# ---------------------------------------------------------------------------------------------------------------------------
def fingerprints_of(emb):
    return {
        f"v{i:04d}": {"embedding": e, "path": f"v{i:04d}", "name": f"v{i:04d}", "size": i, "file_hash": f"h{i % 97}",
                      "embedding_norm": float(np.linalg.norm(e))}
        for i, e in enumerate(emb)
    }


def threshold_in_a_gap(emb):
    """A threshold above the 95th percentile of the pair scores, in the middle of a gap of more than 1e-5 between two of
    them (ten times the summation-order noise), so that no summation order can move a pair across it."""
    off = np.sort((emb @ emb.T)[np.triu_indices(len(emb), 1)])
    gaps = np.nonzero((np.diff(off) > 1e-5) & (off[:-1] >= np.quantile(off, 0.95)))[0]
    assert len(gaps), ("no gap in the score distribution", off[-20:])
    return float((off[gaps[0]] + off[gaps[0] + 1]) / 2)


def assert_same_groups(emb, model, width):
    fps = fingerprints_of(emb)
    thr = threshold_in_a_gap(emb)
    sc = vfp.VideoFingerprintScanner(model=model, config={"embedding_dim": width})
    n_groups = 0
    for use_faiss in (True, False):   # N > 100: top-20 path; use_faiss=False: the direct join
        got = sc.find_duplicates(fps, thr, use_faiss)
        want = join_oracle.find_duplicates(fps, thr, use_faiss)
        # same seeds and members; the order inside a top-k group is the top-k order, defined up to near-ties of 2e-6
        assert [g[0]["name"] for g in got] == [g[0]["name"] for g in want], use_faiss
        for g, w in zip(got, want):
            gm, wm = {it["name"]: it for it in g}, {it["name"]: it for it in w}
            assert set(gm) == set(wm), use_faiss
            for name, a in gm.items():
                assert abs(a["similarity"] - wm[name]["similarity"]) < 1e-5 and a["exact_duplicate"] == wm[name]["exact_duplicate"]
        n_groups = len(got)
    assert n_groups >= 10, (n_groups, thr)


def near_copies(seed, lengths, n_copies):
    """Seeded clips, the last `n_copies` of them copies of earlier ones with a few pixels changed by one level."""
    from oracle.weights import make_clips

    clips = make_clips(seed, lengths, "colour")
    g = torch.Generator().manual_seed(seed)
    src = torch.randint(0, len(clips) - n_copies, (n_copies,), generator=g)
    for c, s in enumerate(src.tolist()):
        x = clips[s].clone()
        mask = torch.rand(x.shape, generator=g) < 0.002
        x[mask] = torch.clamp(x[mask] + 1.0 / 255.0, 0.0, 1.0)
        clips[len(clips) - n_copies + c] = x
    return clips


def test_find_duplicates_with_a_128_wide_attention_model():
    m = vfp.create_model("attention", spatial_dim=64, embedding_dim=128, num_attention_blocks=2).eval()
    torch.manual_seed(5)
    for p in m.parameters():
        if p.dim() > 1:
            p.data.mul_(2.0)
    clips = near_copies(41, [10 + (i % 7) for i in range(160)], 30)
    emb = m.fingerprint_clips([c.cuda() for c in clips]).cpu().numpy()
    assert emb.shape == (160, 128)
    assert_same_groups(emb, m, 128)


def test_find_duplicates_with_a_512_wide_3d_model():
    m = vfp.create_model("3d", embedding_dim=512).eval()
    torch.manual_seed(6)
    for p in m.parameters():
        if p.dim() > 1:
            p.data.mul_(2.0)
    clips = near_copies(42, [16 + (i % 9) for i in range(150)], 30)
    emb = m.fingerprint_clips([c.cuda() for c in clips]).cpu().numpy()
    assert emb.shape == (150, 512)
    assert_same_groups(emb, m, 512)
