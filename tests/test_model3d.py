"""3-D CNN fingerprint model (SURVEY.md section 8f rank 4; /root/reference/model.py:406-512).

CPU: the fp32 oracle against the golden embeddings of the UNMODIFIED reference module (tests/golden/forward3d.npz); the
host mirror's default initialisation against the reference through the refinit case of that file, and its state_dict layout
against the oracle's and against the recorded layout and initial values of a non-default configuration
(tests/golden/host_mirror_3d.json). GPU (-m gpu): vfp3d_forward through the C ABI against the
golden file and the oracle. Tolerance: cosine >= 0.9999 per embedding (bf16 operands, fp32 accumulation), like the attention model.
"""
import json
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import forward3d_oracle as fo  # noqa: E402
from oracle.weights import state_dict_digest  # noqa: E402

GOLD = np.load(os.path.join(ROOT, "tests", "golden", "forward3d.npz"))
COS_BAR = 0.9999


def cosine(a, b):
    a, b = torch.as_tensor(a).double(), torch.as_tensor(b).double()
    return (a * b).sum(-1) / (a.norm(dim=-1) * b.norm(dim=-1))


def case_inputs(name):
    wseed, fs, cseed, n, t, stress = fo.CASES_3D[name]
    if name.endswith("refinit"):
        import video_fingerprint_b200 as vfp

        torch.manual_seed(wseed)
        sd = {k: v.clone() for k, v in vfp.create_model("3d", frame_stride=fs).state_dict().items()}
    else:
        sd = fo.make_state_dict_3d(wseed, fs, stress=stress)
    return sd, fs, fo.make_clips_3d(cseed, n, t)


@pytest.mark.parametrize("name", sorted(fo.CASES_3D))
def test_oracle_matches_reference_golden(name):
    sd, fs, clips = case_inputs(name)       # the refinit case also proves the host mirror reproduces the reference's default init
    got = fo.forward3d_oracle(sd, clips, fs)
    assert torch.allclose(got, torch.from_numpy(GOLD[name]), atol=2e-6), float((got - torch.from_numpy(GOLD[name])).abs().max())


def test_host_mirror_layout():
    import video_fingerprint_b200 as vfp

    m = vfp.create_model("cnn3d")
    assert isinstance(m, vfp.VideoFingerprint3D) and m.frame_stride == 16 and m.embedding_dim == 256    # factory defaults, model.py:602-607
    sd = m.state_dict()
    assert len(sd) == 37 and sd["encoder.0.conv.weight"].shape == (16, 3, 16, 5, 5) and sd["projector.3.weight"].shape == (256, 128)
    want = fo.make_state_dict_3d(1, 16)
    assert set(sd) == set(want) and all(sd[k].shape == want[k].shape for k in sd)
    m.load_state_dict(want, strict=True)
    # non-default factory arguments: key order, shapes and initial values as recorded in tests/golden/host_mirror_3d.json
    with open(os.path.join(ROOT, "tests", "golden", "host_mirror_3d.json")) as f:
        rec = json.load(f)
    torch.manual_seed(3)
    o = vfp.create_model("3d", frame_stride=32, embedding_dim=128).state_dict()
    assert list(o) == rec["keys"] and [list(v.shape) for v in o.values()] == rec["shapes"]
    assert state_dict_digest(o) == rec["weights_sha256"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(fo.CASES_3D))
def test_device_forward_matches_reference_golden(name):
    import video_fingerprint_b200 as vfp

    sd, fs, clips = case_inputs(name)
    m = vfp.create_model("3d", frame_stride=fs).eval()
    m.load_state_dict(sd)
    emb = m(clips.cuda()).cpu()
    assert emb.shape == GOLD[name].shape
    assert torch.allclose(emb.norm(dim=1), torch.ones(len(emb)), atol=1e-5)
    assert float(cosine(emb, GOLD[name]).min()) >= COS_BAR, float(cosine(emb, GOLD[name]).min())


@pytest.mark.gpu
def test_device_forward_dtypes_layouts_and_passes():
    import video_fingerprint_b200 as vfp
    from video_fingerprint_b200 import _native

    sd, fs, clips = case_inputs("fs16_t150")
    m = vfp.create_model("3d", frame_stride=fs).eval()
    m.load_state_dict(sd)
    want = fo.forward3d_oracle(sd, clips, fs)
    e_f32 = m(clips.cuda()).cpu()
    e_u8 = m(torch.round(clips * 255).to(torch.uint8).cuda()).cpu()
    e_bf16 = m(clips.to(torch.bfloat16).cuda()).cpu()
    e_cthw = m(clips.permute(0, 2, 1, 3, 4).contiguous().cuda()).cpu()          # (B, 3, T, H, W)
    for e in (e_f32, e_u8, e_bf16):
        assert float(cosine(e, want).min()) >= COS_BAR
    assert torch.equal(e_f32, e_cthw)
    m.clips_per_pass = 1                                                       # one clip per pass: same results
    assert torch.equal(m(clips.cuda()).cpu(), e_f32)
    with pytest.raises(_native.NativeError):
        m(torch.zeros(1, 16 * 2 * 33, 3, 64, 64))                              # more than 32 temporal positions


@pytest.mark.gpu
def test_scanner_3d_window_semantics():
    """fingerprint.py:272-320: short video = one clip; long video = 3..5 windows of clip_length frames, mean, re-normalise."""
    import video_fingerprint_b200 as vfp

    fs = 16
    sd = fo.make_state_dict_3d(21, fs)
    m = vfp.create_model("3d", frame_stride=fs).eval()
    m.load_state_dict(sd)
    scanner = vfp.VideoFingerprintScanner(model=m, config={"model_type": "3d", "clip_length": 32, "frame_stride": fs})
    assert scanner.window_starts_3d(30) == [0] and scanner.window_starts_3d(100) == [0, 34, 68] and len(scanner.window_starts_3d(400)) == 5
    video = fo.make_clips_3d(7, 1, 100)[0]                  # (100, 3, 64, 64)
    got = scanner.extract_fingerprint_3d_from_frames(video.cuda())
    embs = torch.cat([fo.forward3d_oracle(sd, video[s : s + 32].unsqueeze(0), fs) for s in (0, 34, 68)]).numpy()
    want = embs.mean(axis=0)
    want = want / np.linalg.norm(want)
    assert float(cosine(got, want)) >= COS_BAR
    short = scanner.extract_fingerprint_3d_from_frames(video[:20].cuda())
    assert float(cosine(short, fo.forward3d_oracle(sd, video[:20].unsqueeze(0), fs)[0])) >= COS_BAR
    assert scanner.extract_fingerprint_3d_from_frames(video[:9].cuda()) is None
