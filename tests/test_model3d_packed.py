"""Variable-length batches of the 3-D CNN model: VideoFingerprint3D.fingerprint_packed / fingerprint_clips
(vfp3d_forward_packed), the batched 3-D scanner path and sharded_fingerprint on the 3-D model.

Packing changes how a row or CTA finds its clip, not the arithmetic, so every packed row must have exactly the bits of a
B=1 forward on that clip alone (torch.equal), whatever the clip's neighbours, the pass split or the frame type. Against the
fp32 oracle the bar is that of test_model3d.py: cosine >= 0.9999 per clip."""
import ctypes as C
import os
import random
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import forward3d_oracle as fo  # noqa: E402

import video_fingerprint_b200 as vfp  # noqa: E402
from video_fingerprint_b200 import _native  # noqa: E402

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
    """1, fs-1, fs, fs+1, 2fs, an odd G (2fs+1: G = 3, T3 rounds up to 2), 10, 150 and 64*fs (T3 = 32), in mixed order."""
    lengths = [1, fs - 1, fs, fs + 1, 2 * fs, 2 * fs + 1, 10, 150, 64 * fs]
    lengths = [t for t in lengths if t > 0]
    random.Random(fs).shuffle(lengths)
    return lengths


def as_dtype(x, dtype):
    """x: fp32 frames on the uint8/255 grid -> frames of `dtype` and the fp32 values the device sees."""
    if dtype == torch.uint8:
        u8 = torch.round(x * 255).to(torch.uint8)
        return u8, u8.float() / 255
    if dtype == torch.bfloat16:
        b = x.to(torch.bfloat16)
        return b, b.float()
    return x, x


def clip(seed, t):
    return fo.make_clips_3d(seed, 1, t)[0]


def native_packed(m, frames, lengths, ws_bytes):
    """vfp3d_forward_packed through the raw ABI; the workspace (exactly ws_bytes) and the output sit between guard zones."""
    lib = _native.load()
    w = m._ensure_native()
    n = len(lengths)
    cu = (C.c_int32 * (n + 1))(*np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64).tolist())
    code = {torch.uint8: _native.FRAME_U8, torch.bfloat16: _native.FRAME_BF16, torch.float32: _native.FRAME_F32}[frames.dtype]
    ws, emb = Guarded(ws_bytes), Guarded(n * m.embedding_dim * 4)
    rc = lib.vfp3d_forward_packed(C.c_void_p(w), C.c_void_p(frames.data_ptr()), code, C.cast(cu, C.c_void_p), n, C.c_void_p(emb.t.data_ptr()),
                                  C.c_void_p(ws.t.data_ptr()), ws_bytes, C.c_void_p(torch.cuda.current_stream().cuda_stream))
    _native.check(rc, "vfp3d_forward_packed")
    torch.cuda.synchronize()
    return emb.view(torch.float32, (n, m.embedding_dim)).clone(), (ws, emb)


class Guarded:
    """A device buffer of `nbytes` between two 1 MiB guard zones filled with a pattern; `.t` is the usable uint8 view."""

    def __init__(self, nbytes):
        self.n = int(nbytes)
        self.raw = torch.full((self.n + 2 * GUARD,), PATTERN, dtype=torch.uint8, device="cuda")
        self.t = self.raw[GUARD : GUARD + self.n]

    def view(self, dtype, shape):
        n = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
        return self.t[:n].view(dtype).view(shape)

    def intact(self):
        return bool((self.raw[:GUARD] == PATTERN).all()) and bool((self.raw[GUARD + self.n :] == PATTERN).all())


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_packed_path_fails_loudly_without_gpu():
    m = vfp.create_model("3d").eval()
    with pytest.raises(_native.NativeError, match="no CUDA device"):
        m.fingerprint_packed(torch.zeros(20, 3, 64, 64), [10, 10])


@pytest.mark.gpu
@pytest.mark.parametrize("fs", [16, 32, 5])
@pytest.mark.parametrize("dtype", [torch.uint8, torch.bfloat16, torch.float32])
def test_packed_equals_b1_forward_bitwise(fs, dtype):
    m, _ = make_model(fs)
    clips = [as_dtype(clip(100 + i, t), dtype)[0].cuda() for i, t in enumerate(edge_lengths(fs))]
    got = m.fingerprint_clips(clips)
    assert got.shape == (len(clips), 256) and got.dtype == torch.float32 and got.is_cuda
    for i, c in enumerate(clips):
        assert torch.equal(got[i], m(c[None])[0]), (i, c.shape[0])


@pytest.mark.gpu
@pytest.mark.parametrize("fs", [16, 32, 5])
@pytest.mark.parametrize("dtype", [torch.uint8, torch.bfloat16, torch.float32])
def test_packed_matches_oracle(fs, dtype):
    m, sd = make_model(fs)
    lengths = edge_lengths(fs)
    pairs = [as_dtype(clip(200 + i, t), dtype) for i, t in enumerate(lengths)]
    got = m.fingerprint_packed(torch.cat([p[0] for p in pairs]), lengths).cpu()
    assert torch.allclose(got.norm(dim=1), torch.ones(len(lengths)), atol=1e-5)
    for i, (_, seen) in enumerate(pairs):
        want = fo.forward3d_oracle(sd, seen[None], fs)[0]
        assert float(cosine(got[i], want)) >= COS_BAR, (i, lengths[i], float(cosine(got[i], want)))


@pytest.mark.gpu
def test_clip_bits_do_not_depend_on_neighbours():
    """A clip whose length is not a multiple of fs, before a clip of all-255 frames: its padded last group must read zeros,
    never the next clip's frames. Same bits in every order."""
    fs = 16
    m, _ = make_model(fs)
    a = as_dtype(clip(301, 40), torch.uint8)[0].cuda()                 # 40 % 16 = 8: the last group is half padding
    b = torch.full((32, 3, 64, 64), 255, dtype=torch.uint8, device="cuda")
    c = as_dtype(clip(302, 21), torch.uint8)[0].cuda()
    alone = {k: m(v[None])[0] for k, v in (("a", a), ("b", b), ("c", c))}
    named = {"a": a, "b": b, "c": c}
    orders = [["a", "b"], ["b", "a"], ["c", "b", "a", "b"], ["b", "c", "b", "a", "c"]]
    for order in orders + [random.Random(7).sample(order, len(order)) for order in orders]:
        got = m.fingerprint_clips([named[k] for k in order])
        for i, k in enumerate(order):
            assert torch.equal(got[i], alone[k]), (order, i)


@pytest.mark.gpu
@pytest.mark.parametrize("t", [64, 150])
def test_equal_lengths_match_forward(t):
    m, _ = make_model(16)
    x = fo.make_clips_3d(401, 37, t).to(torch.bfloat16).cuda()
    assert torch.equal(m.fingerprint_clips(list(x)), m(x))
    assert torch.equal(m.fingerprint_packed(x.reshape(-1, 3, 64, 64), [t] * 37), m(x))


@pytest.mark.gpu
def test_pass_split_does_not_change_bits_and_writes_stay_inside_buffers():
    """Workspace just large enough for the longest clip: many passes, guard zones around the workspace and the output."""
    fs = 16
    m, _ = make_model(fs)
    lengths = [37, 10, 150, 16, 1, 333, 64, 17, 100, 15, 48, 200, 33, 5, 129]
    frames = torch.cat([as_dtype(clip(500 + i, t), torch.uint8)[0] for i, t in enumerate(lengths)]).cuda()
    one_pass = m.fingerprint_packed(frames, lengths)
    lib = _native.load()
    w = C.c_void_p(m._ensure_native())
    small = lib.vfp3d_forward_packed_workspace_bytes(w, max(lengths), 1)
    assert 0 < small < lib.vfp3d_forward_packed_workspace_bytes(w, sum(lengths), len(lengths))
    got, guards = native_packed(m, frames, lengths, small)
    assert lib.vfp_device_error_word() == 0
    assert all(g.intact() for g in guards)
    assert torch.equal(got, one_pass)
    # a workspace of exactly the bound for the whole batch: one pass, same bits, guards intact
    whole = lib.vfp3d_forward_packed_workspace_bytes(w, sum(lengths), len(lengths))
    got, guards = native_packed(m, frames, lengths, whole)
    assert lib.vfp_device_error_word() == 0
    assert all(g.intact() for g in guards)
    assert torch.equal(got, one_pass)


@pytest.mark.gpu
def test_bad_input_is_rejected():
    fs = 16
    m, _ = make_model(fs)
    x = torch.rand(40, 3, 64, 64, device="cuda")
    with pytest.raises(_native.NativeError, match="clip 1 has length 0"):
        m.fingerprint_packed(x, [20, 0, 20])
    with pytest.raises(_native.NativeError, match="clip 1 too long"):
        m.fingerprint_packed(torch.rand(10 + 64 * fs + 1, 3, 64, 64, device="cuda"), [10, 64 * fs + 1])
    with pytest.raises(_native.NativeError, match="not monotone"):
        m.fingerprint_packed(x, [30, -10, 20])
    with pytest.raises(ValueError):
        m.fingerprint_packed(x, [20, 19])
    with pytest.raises(ValueError):
        m.fingerprint_clips([x[:10], x[:10].to(torch.uint8)])
    lib = _native.load()
    w = C.c_void_p(m._ensure_native())
    cu = (C.c_int32 * 3)(0, 20, 40)
    emb = torch.empty(2, 256, device="cuda")
    ws = torch.empty(lib.vfp3d_forward_packed_workspace_bytes(w, 40, 2), dtype=torch.uint8, device="cuda")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    rc = lib.vfp3d_forward_packed(w, C.c_void_p(x.data_ptr()), _native.FRAME_U8_HWC, C.cast(cu, C.c_void_p), 2, C.c_void_p(emb.data_ptr()),
                                  C.c_void_p(ws.data_ptr()), ws.numel(), st)
    assert rc != 0 and "HWC" in lib.vfp_last_error().decode()
    rc = lib.vfp3d_forward_packed(w, C.c_void_p(x.data_ptr()), _native.FRAME_F32, C.cast(cu, C.c_void_p), 2, C.c_void_p(emb.data_ptr()),
                                  C.c_void_p(ws.data_ptr()), 4096, st)
    assert rc != 0 and "too small for clip 0" in lib.vfp_last_error().decode()


@pytest.mark.gpu
def test_batched_scanner_matches_per_video_scanner_in_one_call():
    fs = 16
    m, _ = make_model(fs, seed=21)
    scanner = vfp.VideoFingerprintScanner(model=m, config={"model_type": "3d", "clip_length": 32, "frame_stride": fs})
    videos = [clip(600 + i, t).cuda() for i, t in enumerate([9, 20, 32, 100, 400])]
    calls = []
    inner = m.fingerprint_packed

    def counting(*a, **k):
        calls.append(a[1] if len(a) > 1 else k["lengths"])
        return inner(*a, **k)

    m.fingerprint_packed = counting
    try:
        got = scanner.extract_fingerprints_3d_from_frames(videos)
    finally:
        del m.fingerprint_packed
    assert len(calls) == 1 and list(calls[0]) == [20, 32] + [32] * 3 + [32] * 5
    want = [scanner.extract_fingerprint_3d_from_frames(v) for v in videos]
    assert got[0] is None and want[0] is None
    for g, w_ in zip(got[1:], want[1:]):
        assert g.dtype == w_.dtype and np.array_equal(g, w_)
    assert scanner.extract_fingerprints_3d_from_frames([videos[0]]) == [None]


@pytest.mark.gpu
def test_sharded_fingerprint_runs_the_3d_model():
    from video_fingerprint_b200.sharding import sharded_fingerprint

    m, _ = make_model(16)
    clips = [clip(700 + i, t) for i, t in enumerate([12, 64, 150, 33, 1, 90])]
    assert torch.equal(sharded_fingerprint(m, clips), m.fingerprint_clips(clips))
