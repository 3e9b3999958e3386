"""Clips read in place by the attention model: VideoFingerprintAttention.fingerprint_views (vfp_forward_clips), and the
batched decoded-video scanner path (VideoFingerprintScanner.extract_fingerprints_from_decoded).

Where a clip's frames sit changes only the address the stem reads each frame from (one entry of the pass's frame address
table), so every row must have the bits fingerprint_packed gives on the same frames packed in the same order (torch.equal).
Results of different pass cuts are held to the bar of test_forward_gpu.py::test_pass_splitting_is_invisible (atol 1e-6),
and the fp32 oracle bar is cosine >= 0.9999."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import video_fingerprint_b200 as vfp
from oracle.weights import make_clips, make_state_dict
from video_fingerprint_b200 import _native
from video_fingerprint_b200 import fingerprint as fp_mod

pytestmark = pytest.mark.gpu

COS_BAR = 0.9999
GUARD = 1 << 20
PATTERN = 0xA5
FRAME = 12288   # elements of one (3, 64, 64) frame


def cosine(a, b):
    a, b = torch.as_tensor(a).double(), torch.as_tensor(b).double()
    return (a * b).sum(-1) / (a.norm(dim=-1) * b.norm(dim=-1))


@pytest.fixture(scope="module")
def model():
    m = vfp.create_model("attention").eval()
    m.load_state_dict(make_state_dict(2, "stress"))
    return m


def u8_frames(seed, n):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randint(0, 256, (n, 3, 64, 64), dtype=torch.uint8, device="cuda", generator=g)


def as_type(u8, kind):
    """u8 planar frames as one of the four frame types the model takes."""
    if kind == "u8":
        return u8
    if kind == "hwc":
        return u8.permute(0, 2, 3, 1).contiguous()
    return (u8.float() / 255).to(torch.bfloat16 if kind == "bf16" else torch.float32)


def packed_reference(m, clips, return_features=False):
    return m.fingerprint_packed(torch.cat([c.contiguous() for c in clips]), [c.shape[0] for c in clips], return_features=return_features)


def assert_same(got, want):
    if isinstance(want, tuple):
        assert all(torch.equal(g, w) for g, w in zip(got, want))
    else:
        assert torch.equal(got, want)


# ---------------------------------------------------------------------------------------------- bits = fingerprint_packed
@pytest.mark.parametrize("kind", ["u8", "bf16", "f32", "hwc"])
@pytest.mark.parametrize("features", [False, True])
def test_views_equal_packed_bitwise(model, kind, features):
    pe_len = model.pos_encoding.pe.shape[1]
    lengths = [1, 2, 63, 64, 65, 300, pe_len]
    clips = [as_type(u8_frames(100 + i, t), kind) for i, t in enumerate(lengths)]   # separate allocations
    got = model.fingerprint_views(clips, return_features=features)
    want = packed_reference(model, clips, return_features=features)
    assert_same(got, want)
    if features:
        assert got[1].shape == (sum(lengths), 256)


def test_views_in_place(model):
    buf = u8_frames(7, 600)
    clips = [
        u8_frames(8, 37),           # a separate allocation
        buf[0:130],                 # overlapping windows of one buffer
        buf[90:300],
        buf[90:300],                # the same view twice
        buf[::3],                   # every 3rd frame (200 frames)
        buf[1::3][:45],
        buf[5:6],
        buf[::7][:80],
    ]
    assert clips[4].stride(0) == 3 * FRAME
    emb, feats = model.fingerprint_views(clips, return_features=True)
    want_emb, want_feats = packed_reference(model, clips, return_features=True)
    assert torch.equal(emb, want_emb) and torch.equal(feats, want_feats)
    assert torch.equal(emb[2], emb[3])
    # HWC views with a frame stride too
    hwc = buf.permute(0, 2, 3, 1).contiguous()
    hclips = [hwc[::2][:100], hwc[10:75], hwc[3::5]]
    assert torch.equal(model.fingerprint_views(hclips), packed_reference(model, hclips))
    assert torch.equal(model.fingerprint_views(hclips), model.fingerprint_views([buf[::2][:100], buf[10:75], buf[3::5]]))


def test_clip_isolation(model):
    clip = u8_frames(11, 50)
    buf = torch.full((130, 3, 64, 64), 255, dtype=torch.uint8, device="cuda")
    buf[40:90] = clip
    alone = model.fingerprint_views([clip])
    assert torch.equal(model.fingerprint_views([buf[40:90]]), alone)
    assert torch.equal(model.fingerprint_views([buf[:40], buf[40:90], buf[90:]])[1], alone[0])
    assert torch.equal(alone, model.fingerprint_packed(clip, [50]))


def test_oracle_bar_varlen_golden(golden_dir, manifest):
    c = manifest["varlen_stress"]
    m = vfp.create_model("attention").eval()
    m.load_state_dict(make_state_dict(c["wseed"], c["wstyle"]))
    clips = [x.cuda() for x in make_clips(c["cseed"], c["lengths"], c["cstyle"], c["quantise"])]
    gold = np.load(os.path.join(golden_dir, "forward_varlen_stress.npz"))["embeddings"]
    emb = m.fingerprint_views(clips).cpu()
    assert cosine(emb, gold).min() >= COS_BAR


# ---------------------------------------------------------------------------------------------- raw ABI: passes, guards
class Guarded:
    """A device buffer of `nbytes` between two 1 MiB guard zones filled with a pattern; `.t` is the usable uint8 view."""

    def __init__(self, nbytes):
        self.n = (int(nbytes) + 255) // 256 * 256
        self.raw = torch.full((self.n + 2 * GUARD,), PATTERN, dtype=torch.uint8, device="cuda")
        self.t = self.raw[GUARD : GUARD + self.n]

    def intact(self):
        return bool((self.raw[:GUARD] == PATTERN).all()) and bool((self.raw[GUARD + self.n :] == PATTERN).all())

    def untouched(self):
        return bool((self.raw == PATTERN).all())


def abi_clips(lib, m, clips, ws_bytes, code=_native.FRAME_U8, ptrs=None, pitches=None, lengths=None):
    """vfp_forward_clips on `clips` into guarded buffers -> (rc, emb, feats, guards)."""
    n = len(clips)
    lengths = lengths if lengths is not None else [int(c.shape[0]) for c in clips]
    total = max(1, sum(max(t, 0) for t in lengths))
    ptrs = ptrs if ptrs is not None else [c.data_ptr() for c in clips]
    pitches = pitches if pitches is not None else [c.stride(0) * c.element_size() if c.shape[0] > 1 else FRAME * c.element_size() for c in clips]
    weights = m._ensure_native(torch.cuda.current_device())
    ws, emb, feats = Guarded(ws_bytes), Guarded(n * 256 * 4), Guarded(total * 256 * 4)
    rc = lib.vfp_forward_clips(C.c_void_p(weights), (C.c_void_p * n)(*ptrs), (C.c_int64 * n)(*pitches), (C.c_int32 * n)(*lengths), n, code,
                               C.c_void_p(emb.t.data_ptr()), C.c_void_p(feats.t.data_ptr()), C.c_void_p(ws.t.data_ptr()), ws.n,
                               C.c_void_p(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return rc, emb.t[: n * 1024].view(torch.float32).view(n, 256).clone(), feats.t[: total * 1024].view(torch.float32).view(total, 256).clone(), (ws, emb, feats)


def test_pass_splitting_through_the_abi(model):
    lib = _native.load()
    buf = u8_frames(21, 900)
    clips = [buf[0:300], buf[::4][:120], buf[200:201], buf[100:400], u8_frames(22, 77), buf[3::2][:250], buf[0:300]]
    lengths = [int(c.shape[0]) for c in clips]
    n, total, max_t = len(clips), sum(lengths), max(lengths)
    one_pass, _ = model.fingerprint_views(clips, return_features=True)   # everything in one pass
    try:
        for conv_pass, pipes in [(None, 1), (64, 1), (64, 2), (128, 3), (64, 4)]:
            if conv_pass is not None:
                assert lib.vfp_set_tuning(3, conv_pass) == 0 and lib.vfp_set_tuning(0, conv_pass) == 0
            assert lib.vfp_set_tuning(9, pipes) == 0
            # just large enough for the longest clip (a pass of max_t frames may hold min(max_t, n) clips)
            tight = lib.vfp_forward_workspace_bytes(max_t, min(max_t, n))
            for ws_bytes in (tight, lib.vfp_forward_workspace_bytes(total, n)):
                rc, emb, feats, guards = abi_clips(lib, model, clips, ws_bytes)
                _native.check(rc, "vfp_forward_clips")
                assert lib.vfp_device_error_word() == 0
                assert all(g.intact() for g in guards)
                assert torch.allclose(emb, one_pass, atol=1e-6)
                # same pass cuts: vfp_forward on the packed copy under the same settings gives the same bits
                packed = torch.cat([c.contiguous() for c in clips])
                cu = (C.c_int32 * (n + 1))(*np.concatenate([[0], np.cumsum(lengths)]).tolist())
                ws2, emb2, feats2 = Guarded(ws_bytes), Guarded(n * 1024), Guarded(total * 1024)
                weights = model._ensure_native(torch.cuda.current_device())
                _native.check(lib.vfp_forward(C.c_void_p(weights), C.c_void_p(packed.data_ptr()), _native.FRAME_U8, C.cast(cu, C.c_void_p), n,
                                              C.c_void_p(emb2.t.data_ptr()), C.c_void_p(feats2.t.data_ptr()), C.c_void_p(ws2.t.data_ptr()), ws2.n,
                                              C.c_void_p(torch.cuda.current_stream().cuda_stream)), "vfp_forward")
                torch.cuda.synchronize()
                assert torch.equal(emb, emb2.t[: n * 1024].view(torch.float32).view(n, 256))
                assert torch.equal(feats, feats2.t[: total * 1024].view(torch.float32).view(total, 256))
    finally:
        lib.vfp_set_tuning(3, 65536)
        lib.vfp_set_tuning(0, 16384)
        lib.vfp_set_tuning(9, 1)


def test_pipelines_over_many_views(model):
    """Enough frames (> 2 x 262 144) for the library to really run several pipelines, all of them views of one 4 096-frame
    buffer, so the frames themselves take 50 MB."""
    buf = u8_frames(31, 4096)
    g = torch.Generator().manual_seed(3)
    starts = torch.randint(0, 4096 - 300, (2200,), generator=g).tolist()
    lens = torch.randint(200, 300, (2200,), generator=g).tolist()
    clips = [buf[s : s + t] for s, t in zip(starts, lens)]
    total = sum(lens)
    assert total > 2 * 262144
    pipelines, per_pass = model.pipelines, model.frames_per_pass
    try:
        one = model.fingerprint_views(clips)
        for k in (2, 3, 4):
            model.pipelines, model.frames_per_pass = k, total // k + 300
            model._workspaces.clear()
            views = model.fingerprint_views(clips)
            assert torch.allclose(views, one, atol=1e-6)
            if k == 2:
                assert torch.equal(views, packed_reference(model, clips))
        assert _native.load().vfp_device_error_word() == 0
    finally:
        model.pipelines, model.frames_per_pass = pipelines, per_pass
        model._workspaces.clear()
        _native.load().vfp_set_tuning(9, 1)


# ---------------------------------------------------------------------------------------------- rejections
def test_abi_rejections_name_the_clip_and_run_nothing(model):
    lib = _native.load()
    buf = u8_frames(41, 40)
    clips = [buf[0:10], buf[10:30], buf[30:40]]
    big = lib.vfp_forward_workspace_bytes(40, 3)
    pe_len = model.pos_encoding.pe.shape[1]
    p = [c.data_ptr() for c in clips]
    cases = [
        (dict(ptrs=[p[0], None, p[2]]), "clip 1 has a null frame pointer"),
        (dict(ptrs=[p[0], p[1], p[2] + 8]), "clip 2's frame pointer is not 16-byte aligned"),
        (dict(pitches=[FRAME, FRAME - 16, FRAME]), "clip 1 has a frame pitch of 12272"),
        (dict(pitches=[FRAME, FRAME, FRAME + 8]), "clip 2 has a frame pitch of 12296"),
        (dict(lengths=[10, 0, 10]), "clip 1 has no frames"),
        (dict(lengths=[10, -3, 10]), "clip 1 has no frames"),
        (dict(lengths=[10, 20, pe_len + 1]), f"clip 2 has {pe_len + 1} frames; the positional table"),
        (dict(code=7), "unknown frame_dtype 7"),
    ]
    for kw, msg in cases:
        rc, _, _, guards = abi_clips(lib, model, clips, big, **kw)
        assert rc != 0
        assert msg in lib.vfp_last_error().decode(), (msg, lib.vfp_last_error())
        assert all(g.untouched() for g in guards), msg   # nothing was enqueued: output and workspace keep their pattern
    small = lib.vfp_forward_workspace_bytes(15, 3)
    rc, _, _, guards = abi_clips(lib, model, clips, small)
    assert rc != 0 and "cannot hold the longest clip (clip 1: 20 frames" in lib.vfp_last_error().decode()
    assert all(g.untouched() for g in guards)
    assert lib.vfp_device_error_word() == 0


def test_python_rejections(model):
    buf = u8_frames(51, 30)
    hwc = buf.permute(0, 2, 3, 1).contiguous()
    bad = [
        ([buf[:10], buf[10:20].cpu()], "clip 1 is not a CUDA tensor"),
        ([buf[:10], buf[10:20].float()], "clip 1 is torch.float32"),
        ([buf[:10], hwc[:10]], "clip 1 has shape"),
        ([hwc[:10], buf[:10]], "clip 1 has shape"),
        ([buf[:10], hwc[:10].permute(0, 3, 1, 2)], "clip 1 has strides"),          # planar shape, frames not contiguous
        ([buf[:10], buf[:10].transpose(2, 3)], "clip 1 has strides"),
        ([buf[:10], buf[0].unsqueeze(0).expand(4, 3, 64, 64)], "clip 1 has a frame stride of 0"),
        ([buf[:10], buf[:5].double()], "clip 1 is torch.float64"),
        ([buf[:10].half()], "float16 clips"),
        ([], "at least one clip"),
    ]
    for clips, msg in bad:
        with pytest.raises(ValueError, match=msg):
            model.fingerprint_views(clips)
    with pytest.raises(ValueError, match="clip 1 has no frames"):
        model.fingerprint_views([buf[:10], buf[10:10]])
    with pytest.raises(_native.NativeError, match="clip 0 has 10001 frames"):
        big = torch.zeros((10001, 3, 64, 64), dtype=torch.uint8, device="cuda")
        model.fingerprint_views([big])
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError, match="clip 1 is on cuda:1"):
            model.fingerprint_views([buf[:10], buf[:10].to("cuda:1")])
    assert _native.load().vfp_device_error_word() == 0


# ---------------------------------------------------------------------------------------------- decoded-video scanner
def decoded_video(seed, t, h, w):
    rng = np.random.default_rng(seed)
    base = rng.integers(0, 256, (1, h, w, 3), dtype=np.uint8)
    noise = rng.integers(0, 64, (t, h, w, 3), dtype=np.uint8)
    return (base // 2 + noise).astype(np.uint8)


def test_scanner_decoded_batch_matches_per_video(model, monkeypatch):
    sc = vfp.VideoFingerprintScanner(model=model, config={"model_type": "attention"})
    specs = [(5, 90, 120), (9, 64, 64), (10, 48, 40), (400, 120, 160), (1200, 72, 96), (37, 64, 100)]
    videos = [decoded_video(60 + i, t, h, w) for i, (t, h, w) in enumerate(specs)]
    videos[5] = list(videos[5])   # a list of frames is accepted too
    want = [sc.extract_fingerprint_from_decoded(v) for v in videos]

    calls, frames_seen = [], []
    real_views, real_pre = model.fingerprint_views, fp_mod.preprocess_frames_device

    def views(clips, *a, **k):
        calls.append(len(clips))
        return real_views(clips, *a, **k)

    def pre(frames, *a, **k):
        frames_seen.append(len(frames))
        return real_pre(frames, *a, **k)

    monkeypatch.setattr(model, "fingerprint_views", views)
    monkeypatch.setattr(fp_mod, "preprocess_frames_device", pre)
    got = sc.extract_fingerprints_from_decoded(videos)
    assert calls == [4]
    kept = [len(sc.subsample(len(v))) for v in videos]
    assert kept == [5, 9, 10, 400, 500, 37]
    assert sorted(frames_seen) == sorted(k for k in kept if k >= 10)
    bitwise = True
    for g, w in zip(got, want):
        assert (g is None) == (w is None)
        if w is not None:
            assert g.shape == (256,) and np.allclose(g, w, atol=1e-6)
            bitwise &= np.array_equal(g, w)
    assert bitwise   # same frames, same kernels: the batch gives the per-video bits
    assert sc.extract_fingerprints_from_decoded([videos[0], videos[1]]) == [None, None]
