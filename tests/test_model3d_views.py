"""Clips read in place by the 3-D CNN model: VideoFingerprint3D.fingerprint_views (vfp3d_forward_clips), decoder-layout
(T, 64, 64, 3) uint8 frames, and the decoded-video 3-D scanner path (extract_fingerprints_3d_from_decoded).

Where a clip's frames sit changes only the address its layer-1 groups read from, and decoder-layout uint8 frames are scaled
exactly like planar uint8 ones, so every row must have the bits of fingerprint_packed / a B=1 forward on the same frames
(torch.equal). Against the fp32 oracle the bar is that of test_model3d.py: cosine >= 0.9999."""
import ctypes as C
import os
import random
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import forward3d_oracle as fo  # noqa: E402

import video_fingerprint_b200 as vfp  # noqa: E402
from video_fingerprint_b200 import _native  # noqa: E402
from video_fingerprint_b200 import fingerprint as fp_mod  # noqa: E402

COS_BAR = 0.9999
GUARD = 1 << 20
PATTERN = 0xA5


def cosine(a, b):
    a, b = torch.as_tensor(a).double(), torch.as_tensor(b).double()
    return (a * b).sum(-1) / (a.norm(dim=-1) * b.norm(dim=-1))


def make_model(fs, seed=31):
    sd = fo.make_state_dict_3d(seed, fs, stress=True)
    m = vfp.create_model("3d", frame_stride=fs).eval()
    m.load_state_dict(sd)
    return m, sd


def edge_lengths(fs):
    """The edge lengths of test_model3d_packed.py: 1, fs-1, fs, fs+1, 2fs, 2fs+1, 10, 150 and 64*fs (T3 = 32)."""
    return [t for t in [1, fs - 1, fs, fs + 1, 2 * fs, 2 * fs + 1, 10, 150, 64 * fs] if t > 0]


def u8_clip(seed, t):
    return torch.round(fo.make_clips_3d(seed, 1, t)[0] * 255).to(torch.uint8)


def as_dtype(u8, dtype):
    return u8 if dtype == torch.uint8 else (u8.float() / 255).to(dtype)


def hwc(planar):
    return planar.permute(0, 2, 3, 1).contiguous()


class Guarded:
    """A device buffer of `nbytes` between two 1 MiB guard zones filled with a pattern; `.t` is the usable uint8 view."""

    def __init__(self, nbytes):
        self.n = int(nbytes)
        self.raw = torch.full((self.n + 2 * GUARD,), PATTERN, dtype=torch.uint8, device="cuda")
        self.t = self.raw[GUARD : GUARD + self.n]

    def intact(self):
        return bool((self.raw[:GUARD] == PATTERN).all()) and bool((self.raw[GUARD + self.n :] == PATTERN).all())


def raw_clips(m, ptrs, lengths, code, ws_bytes, n_out=None):
    """vfp3d_forward_clips through the raw ABI -> (rc, error message, embeddings, guarded buffers)."""
    lib = _native.load()
    w = m._ensure_native()
    n = len(lengths)
    ws, emb = Guarded(ws_bytes), Guarded((n_out or n) * m.embedding_dim * 4)
    rc = lib.vfp3d_forward_clips(C.c_void_p(w), (C.c_void_p * n)(*ptrs), (C.c_int32 * n)(*lengths), n, code,
                                 C.c_void_p(emb.t.data_ptr()), C.c_void_p(ws.t.data_ptr()), ws_bytes,
                                 C.c_void_p(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    out = emb.t[: n * m.embedding_dim * 4].view(torch.float32).view(n, m.embedding_dim).clone()
    return rc, (lib.vfp_last_error().decode() if rc else ""), out, (ws, emb)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_views_and_decoded_scanner_fail_loudly_without_gpu():
    m = vfp.create_model("3d").eval()
    with pytest.raises(_native.NativeError, match="no CUDA device"):
        m.fingerprint_views([torch.zeros(20, 3, 64, 64)])
    scanner = vfp.VideoFingerprintScanner.__new__(vfp.VideoFingerprintScanner)
    scanner.model, scanner.config, scanner.model_type = m, {"model_type": "3d"}, "3d"
    with pytest.raises(_native.NativeError, match="no CUDA device"):
        scanner.extract_fingerprints_3d_from_decoded([np.zeros((20, 80, 100, 3), np.uint8)])
    with pytest.raises(_native.NativeError, match="no CUDA device"):
        scanner.extract_fingerprint_3d_from_decoded(np.zeros((20, 80, 100, 3), np.uint8))


@pytest.mark.gpu
@pytest.mark.parametrize("fs", [16, 32, 5])
@pytest.mark.parametrize("dtype", [torch.uint8, torch.bfloat16, torch.float32])
def test_views_equal_packed_bitwise(fs, dtype):
    """Clips as separate allocations, in shuffled order: the same bits as fingerprint_packed on their concatenation."""
    m, _ = make_model(fs)
    lengths = edge_lengths(fs)
    clips = [as_dtype(u8_clip(100 + i, t), dtype).cuda() for i, t in enumerate(lengths)]
    random.Random(fs).shuffle(clips)
    got = m.fingerprint_views(clips)
    assert got.shape == (len(clips), 256) and got.dtype == torch.float32 and got.is_cuda
    want = m.fingerprint_packed(torch.cat(clips), [c.shape[0] for c in clips])
    assert torch.equal(got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("fs", [16, 5])
def test_hwc_views_give_the_planar_bits(fs):
    m, _ = make_model(fs)
    lengths = edge_lengths(fs)
    planar = torch.cat([u8_clip(200 + i, t) for i, t in enumerate(lengths)]).cuda()
    dec = hwc(planar)
    cu = np.concatenate([[0], np.cumsum(lengths)]).tolist()
    got = m.fingerprint_views([dec[cu[i] : cu[i + 1]] for i in range(len(lengths))])
    assert torch.equal(got, m.fingerprint_views([planar[cu[i] : cu[i + 1]] for i in range(len(lengths))]))
    assert torch.equal(got, m.fingerprint_packed(planar, lengths))


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["planar", "hwc"])
def test_overlapping_and_repeated_views(layout):
    """Windows of one buffer that overlap by all but one frame, one view listed twice, a window ending at the last frame."""
    fs = 16
    m, _ = make_model(fs)
    buf = u8_clip(301, 100).cuda()
    src = hwc(buf) if layout == "hwc" else buf
    spans = [(0, 99), (1, 100), (30, 60), (30, 60), (70, 100), (99, 100), (0, 100)]
    got = m.fingerprint_views([src[a:b] for a, b in spans])
    for i, (a, b) in enumerate(spans):
        assert torch.equal(got[i], m(buf[a:b].clone()[None])[0]), (a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["planar", "hwc"])
def test_padding_reads_zero_not_the_next_frames(layout):
    """A window of 40 frames (40 % 16 = 8: its last group is half padding) followed in memory by all-255 frames."""
    fs = 16
    m, _ = make_model(fs)
    buf = torch.cat([u8_clip(302, 40), torch.full((32, 3, 64, 64), 255, dtype=torch.uint8)]).cuda()
    src = hwc(buf) if layout == "hwc" else buf
    got = m.fingerprint_views([src[:40], src[:21]])
    assert torch.equal(got[0], m(buf[:40].clone()[None])[0])
    assert torch.equal(got[1], m(buf[:21].clone()[None])[0])


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["planar", "hwc"])
def test_raw_abi_pass_split_and_guard_zones(layout):
    """Workspace just large enough for the longest clip (many passes), then the whole-batch bound: same bits, no write
    outside the workspace or the output, no device error."""
    fs = 16
    m, _ = make_model(fs)
    lengths = [37, 10, 150, 16, 1, 333, 64, 17, 100, 15, 48, 200, 33, 5, 129]
    planar = [u8_clip(500 + i, t).cuda() for i, t in enumerate(lengths)]
    clips = [hwc(c) for c in planar] if layout == "hwc" else planar
    want = m.fingerprint_packed(torch.cat(planar), lengths)
    code = _native.FRAME_U8_HWC if layout == "hwc" else _native.FRAME_U8
    lib = _native.load()
    w = C.c_void_p(m._ensure_native())
    small = lib.vfp3d_forward_packed_workspace_bytes(w, max(lengths), 1)
    whole = lib.vfp3d_forward_packed_workspace_bytes(w, sum(lengths), len(lengths))
    assert 0 < small < whole
    for ws_bytes in (small, whole):
        rc, msg, got, guards = raw_clips(m, [c.data_ptr() for c in clips], lengths, code, ws_bytes)
        assert rc == 0, msg
        assert lib.vfp_device_error_word() == 0
        assert all(g.intact() for g in guards)
        assert torch.equal(got, want)


@pytest.mark.gpu
def test_bad_input_is_rejected():
    fs = 16
    m, _ = make_model(fs)
    x = u8_clip(600, 64).cuda()
    lib = _native.load()
    w = C.c_void_p(m._ensure_native())
    ws_bytes = lib.vfp3d_forward_packed_workspace_bytes(w, 64 * fs * 3, 3)
    ok = [x.data_ptr(), x[16:].data_ptr(), x[32:].data_ptr()]

    def rejected(ptrs, lengths, match, code=_native.FRAME_U8, nbytes=ws_bytes):
        rc, msg, _, _ = raw_clips(m, ptrs, lengths, code, nbytes)
        assert rc != 0 and match in msg, msg

    rejected([ok[0], None, ok[2]], [16, 16, 16], "clip 1 has a null frame pointer")
    rejected([ok[0], ok[1], x.data_ptr() + 1], [16, 16, 16], "clip 2's frame pointer is not 16-byte aligned")
    rejected(ok, [16, 0, 16], "clip 1 has length 0")
    rejected(ok, [16, 16, -3], "clip 2 has length -3")
    rejected(ok, [16, 64 * fs + 1, 16], "clip 1 too long")
    rejected(ok, [16, 16, 16], "too small for clip 0", nbytes=4096)
    rejected(ok, [16, 16, 16], "unknown frame_dtype 7", code=7)
    rc, msg, _, _ = raw_clips(m, ok, [16, 16, 16], _native.FRAME_U8, ws_bytes)
    assert rc == 0, msg

    with pytest.raises(ValueError, match="one dtype"):
        m.fingerprint_views([x[:10], x[:10].float()])
    with pytest.raises(ValueError, match="shape"):
        m.fingerprint_views([x[:10], hwc(x[:10])])
    with pytest.raises(ValueError, match="not contiguous"):
        m.fingerprint_views([x[:10], x[::2]])
    with pytest.raises(ValueError, match="not a CUDA tensor"):
        m.fingerprint_views([x[:10], x[:10].cpu()])
    with pytest.raises(ValueError):
        m.fingerprint_views([hwc(x[:10]).float()])
    with pytest.raises(ValueError):
        m.fingerprint_views([])
    with pytest.raises(_native.NativeError, match="clip 1 has length 0"):
        m.fingerprint_views([x[:10], x[:0]])


# decoded videos (T, H, W, 3) uint8 at several resolutions, one below 64 px: (T, H, W)
DECODED = [(9, 120, 160), (20, 48, 80), (32, 240, 320), (129, 90, 100), (400, 100, 72), (1000, 72, 96)]


def decoded_video(seed, t, h, w):
    x = fo.make_clips_3d(seed, 1, t)[0]   # (t, 3, 64, 64) on the uint8 grid
    x = F.interpolate(x, size=(h, w), mode="bilinear", align_corners=False)
    return torch.round(x.clamp(0, 1) * 255).to(torch.uint8).permute(0, 2, 3, 1).contiguous().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("clip_length", [32, None])
def test_decoded_scanner(clip_length, monkeypatch):
    fs = 16
    m, sd = make_model(fs, seed=21)
    config = {"model_type": "3d", "frame_stride": fs}
    if clip_length is not None:
        config["clip_length"] = clip_length
    L = clip_length or 128
    scanner = vfp.VideoFingerprintScanner(model=m, config=config)
    videos = [decoded_video(700 + i, t, h, w) for i, (t, h, w) in enumerate(DECODED)]
    # the same frames the long way: every frame preprocessed, permuted to planar uint8, the batched frames path
    planar = [fp_mod.preprocess_frames_device(v).permute(0, 3, 1, 2).contiguous() for v in videos]
    want = scanner.extract_fingerprints_3d_from_frames(planar)

    views_calls, preprocessed = [], []
    inner_views, inner_pre = m.fingerprint_views, fp_mod.preprocess_frames_device

    def counting_views(clips):
        views_calls.append([int(c.shape[0]) for c in clips])
        return inner_views(clips)

    def counting_pre(frames, device=None):
        preprocessed.append(len(frames))
        return inner_pre(frames, device)

    monkeypatch.setattr(m, "fingerprint_views", counting_views)
    monkeypatch.setattr(fp_mod, "preprocess_frames_device", counting_pre)
    got = scanner.extract_fingerprints_3d_from_decoded(videos)
    monkeypatch.undo()

    assert len(views_calls) == 1
    windowed = sum(len(set().union(*(range(s, s + min(t, L)) for s in scanner.window_starts_3d(t)))) for t, _, _ in DECODED if t >= 10)
    assert sum(preprocessed) == windowed   # every windowed frame once, no other frame
    assert max(preprocessed) <= 5 * L
    assert got[0] is None and want[0] is None
    for i in range(1, len(videos)):
        assert got[i].dtype == want[i].dtype and np.array_equal(got[i], want[i]), i

    # the fp32 oracle with the same window rule on the reference's float frames
    for i, v in enumerate(videos[1:], start=1):
        frames = scanner._preprocess_frames(v).cpu()
        t = frames.shape[0]
        span = min(t, L)
        embs = torch.cat([fo.forward3d_oracle(sd, frames[s : s + span][None], fs) for s in scanner.window_starts_3d(t)])
        ref = embs[0] if t <= L else embs.mean(0) / embs.mean(0).norm()
        assert float(cosine(got[i], ref)) >= COS_BAR, (i, float(cosine(got[i], ref)))

    # the one-video form is a row of the batched form; frames as a tensor and as a list give the same bits
    assert np.array_equal(scanner.extract_fingerprint_3d_from_decoded(videos[4]), got[4])
    assert np.array_equal(scanner.extract_fingerprint_3d_from_decoded(torch.from_numpy(videos[3])), got[3])
    assert np.array_equal(scanner.extract_fingerprint_3d_from_decoded(list(videos[5])), got[5])
    assert scanner.extract_fingerprint_3d_from_decoded(videos[0]) is None
