"""GPU: the sm_100a forward (through the C ABI) against the reference's golden outputs and the oracle.
Bar (BASELINE.json north_star): every embedding reaches cosine >= 0.9999 against the reference fp32 output."""
import os

import numpy as np
import pytest
import torch

import video_fingerprint_b200 as vfp
from oracle.forward_oracle import fingerprint_clips, forward_oracle
from oracle.weights import make_clips, make_state_dict
from video_fingerprint_b200 import _native

pytestmark = pytest.mark.gpu

COS_BAR = 0.9999          # stated tolerance (north_star)
CENTRED_COS_BAR = 0.995   # extra gate on the stress init (SURVEY.md section 7, hard part 1)
FEATURE_BAR = 1.6e-2      # per-token relative error of return_features: BETA of test_model_shapes_gpu.py


def cosine(a, b):
    a, b = torch.as_tensor(a).double(), torch.as_tensor(b).double()
    return (a * b).sum(-1) / (a.norm(dim=-1) * b.norm(dim=-1))


def model_for(wseed, wstyle, **kw):
    m = vfp.create_model("attention", **kw).eval()
    if not kw:
        m.load_state_dict(make_state_dict(wseed, wstyle))
    return m


@pytest.mark.parametrize("name", ["cfg1_default", "cfg1_stress", "varlen_stress", "t64_default"])
def test_golden_parity(name, golden_dir, manifest):
    c = manifest[name]
    m = model_for(c["wseed"], c["wstyle"])
    clips = make_clips(c["cseed"], c["lengths"], c["cstyle"], c["quantise"])
    gold = np.load(os.path.join(golden_dir, f"forward_{name}.npz"))["embeddings"]
    emb = m.fingerprint_clips(clips).cpu()
    assert emb.shape == gold.shape
    assert torch.allclose(emb.norm(dim=1), torch.ones(len(clips)), atol=1e-5)
    cs = cosine(emb, gold)
    assert cs.min() >= COS_BAR, f"{name}: min cosine {cs.min():.6f}"
    if c["wstyle"] == "stress":
        g = torch.from_numpy(gold)
        cc = cosine(emb - emb.mean(0, keepdim=True), g - g.mean(0, keepdim=True))
        assert cc.min() >= CENTRED_COS_BAR, f"{name}: centred cosine {cc.min():.5f}"
        # the duplicate pair set at 0.95 is identical apart from pairs within 1e-3 of the threshold
        S_ref, S_new = g @ g.T, emb @ emb.T
        decided = (S_ref - 0.95).abs() >= 1e-3
        assert torch.equal((S_new >= 0.95)[decided], (S_ref >= 0.95)[decided])


def test_reference_default_init_cfg1(golden_dir):
    """BASELINE configs[0]: torch.manual_seed(0) default-init model, torch.rand(16,32,3,64,64) seed 1234."""
    torch.manual_seed(0)
    m = vfp.create_model("attention").eval()
    x = torch.rand(16, 32, 3, 64, 64, generator=torch.Generator().manual_seed(1234))
    gold = np.load(os.path.join(golden_dir, "forward_cfg1_refinit.npz"))["embeddings"]
    emb = m(x.cuda()).cpu()
    assert cosine(emb, gold).min() >= COS_BAR


def test_input_dtypes_and_batched_forward():
    sd = make_state_dict(2, "stress")
    m = model_for(2, "stress")
    clips = make_clips(9, [24] * 6, "colour")            # on the uint8/255 grid
    x = torch.stack(clips)                                # (6, 24, 3, 64, 64) fp32
    want = forward_oracle(sd, x)
    e_f32 = m(x.cuda()).cpu()
    e_u8 = m(torch.round(x * 255).to(torch.uint8).cuda()).cpu()
    e_bf16 = m(x.to(torch.bfloat16).cuda()).cpu()
    e_cpu_in = m(x).cpu()                                 # host tensor is copied to the GPU, not computed on the CPU
    # decoder layout (T, H, W, 3) uint8: the /255 + HWC->CHW of _preprocess_frames (fingerprint.py:210-212) fused in
    hwc = torch.round(x * 255).to(torch.uint8).permute(0, 1, 3, 4, 2).reshape(-1, 64, 64, 3).contiguous()
    e_hwc = m.fingerprint_packed(hwc.cuda(), [24] * 6).cpu()
    assert torch.equal(e_hwc, e_u8)
    for e in (e_f32, e_u8, e_bf16, e_cpu_in):
        assert cosine(e, want).min() >= COS_BAR
    assert torch.equal(e_f32, e_cpu_in)
    # two different conv-stem paths (fp32 frames: two kernels; u8 frames: fused TS-mode stem), both within COS_BAR of the
    # oracle; against each other they differ by the summation order of bf16 products (measured 0.999989)
    assert cosine(e_f32, e_u8).min() > 0.99998


def test_varlen_packed_equals_per_clip_b1():
    """A clip inside a packed batch gets the embedding a B=1 forward on that clip alone gives (fingerprint.py:247)."""
    m = model_for(2, "stress")
    sd = make_state_dict(2, "stress")
    clips = make_clips(31, [10, 47, 16, 128, 33, 11], "colour")
    packed = m.fingerprint_clips(clips).cpu()
    for i, clip in enumerate(clips):
        alone = m(clip.unsqueeze(0).cuda()).cpu()[0]
        assert torch.allclose(packed[i], alone, atol=1e-6), i   # same kernels, same arithmetic: no cross-clip leakage
    want = torch.stack(fingerprint_clips(sd, clips))
    assert cosine(packed, want).min() >= COS_BAR


def test_pass_splitting_is_invisible():
    m = model_for(2, "stress")
    clips = make_clips(32, [40, 12, 64, 19, 50, 25, 31], "colour")
    whole = m.fingerprint_clips(clips).cpu()
    m.frames_per_pass = 70          # forces several internal passes
    m._workspaces.clear()
    split = m.fingerprint_clips(clips).cpu()
    assert torch.allclose(whole, split, atol=1e-6)


def test_pipelined_passes_and_host_upload_are_invisible():
    """Token passes dealt onto two internal streams (model.pipelines = 2, the default) and the chunked double-buffered host
    upload (fingerprint_host) must give what ONE pass on the caller's stream gives. 40 000 frames so that the library really
    runs two pipelines (it needs at least two conv passes of 16 384 frames)."""
    m = model_for(2, "stress")
    g = torch.Generator().manual_seed(77)
    lengths = [int(t) for t in torch.randint(10, 120, (620,), generator=g)]
    total = sum(lengths)
    assert total >= 2 * 16384
    frames = torch.randint(0, 256, (total, 3, 64, 64), dtype=torch.uint8, generator=g)
    dev = frames.cuda()
    m.pipelines, m.frames_per_pass = 1, 1 << 20
    one = m.fingerprint_packed(dev, lengths).cpu()
    m.pipelines, m.frames_per_pass = 2, 9000
    m._workspaces.clear()
    two = m.fingerprint_packed(dev, lengths).cpu()
    assert _native.load().vfp_device_error_word() == 0
    close = lambda a, b: torch.allclose(a, b, atol=1e-6)   # noqa: E731 (a clip's result does not depend on how it is packed)
    assert close(one, two)
    host = m.fingerprint_host(frames.pin_memory(), lengths, chunk_frames=7000).cpu()
    assert close(one, host)
    out = torch.empty((len(lengths), 256), dtype=torch.float32).pin_memory()
    assert m.fingerprint_host(frames, lengths, chunk_frames=50_000, out=out) is out      # pageable source works too
    assert close(one, out)
    assert close(m.fingerprint_packed(frames, lengths).cpu(), one)  # host tensor through the generic entry
    # spot check against the oracle (the bar of every other test here)
    sd = make_state_dict(2, "stress")
    cu = np.concatenate([[0], np.cumsum(lengths)])
    for c in (0, 311, 619):
        want = forward_oracle(sd, frames[cu[c] : cu[c + 1]].float().div(255).unsqueeze(0))
        assert cosine(two[c], want[0]) >= COS_BAR


def test_attention_key_block_boundaries():
    """Clip lengths on both sides of the attention kernel's 64-token query / key blocks (one block, exactly two, a one-token
    tail, several blocks with a masked tail). Each clip must reach the bar against the oracle, must not depend on its
    neighbours in the packed batch, and the tcgen05 kernel (default) must agree with the mma.sync kernel
    (vfp_set_tuning(17, 0)) to the rounding of their different P / summation orders."""
    lib = _native.load()
    sd = make_state_dict(2, "stress")
    m = model_for(2, "stress")
    lengths = [10, 63, 64, 65, 127, 128, 129, 191, 192, 193, 300, 11]
    clips = make_clips(71, lengths, "colour")
    want = torch.stack(fingerprint_clips(sd, clips))
    got = m.fingerprint_clips(clips).cpu()
    assert lib.vfp_device_error_word() == 0
    assert cosine(got, want).min() >= COS_BAR
    rev = m.fingerprint_clips(clips[::-1]).cpu().flip(0)              # other neighbours, other work-item order
    assert torch.allclose(got, rev, atol=1e-6)
    try:
        lib.vfp_set_tuning(17, 0)
        legacy = m.fingerprint_clips(clips).cpu()
    finally:
        lib.vfp_set_tuning(17, 1)
    assert cosine(legacy, want).min() >= COS_BAR
    assert cosine(got, legacy).min() > 0.99999


def test_clip_longer_than_1024_frames():
    """The positional table of the checkpoint (10 000 rows, model.py:77) is the only length limit."""
    sd = make_state_dict(2, "stress")
    m = model_for(2, "stress")
    clips = make_clips(61, [1500, 23], "colour")
    want = torch.stack(fingerprint_clips(sd, clips))
    got = m.fingerprint_clips(clips).cpu()
    assert cosine(got, want).min() >= COS_BAR


def test_return_features_and_layout_quirk():
    sd = make_state_dict(2, "stress")
    m = model_for(2, "stress")
    x = torch.stack(make_clips(33, [20, 20], "colour"))
    st = {}
    want = forward_oracle(sd, x, st)
    emb, feats = m(x.cuda(), return_features=True)
    assert feats.shape == (2, 20, 256)
    rel = (feats.cpu().double() - st["attn3"].double()).norm(dim=-1) / st["attn3"].double().norm(dim=-1)
    assert rel.max() <= FEATURE_BAR     # per token
    assert cosine(emb.cpu(), want).min() >= COS_BAR
    # (B, C=3, T, H, W) input is re-interpreted like the reference does (model.py:283)
    emb2 = m(x.permute(0, 2, 1, 3, 4).contiguous().cuda())
    assert torch.allclose(emb2, emb, atol=1e-6)


def test_fused_stem_matches():
    """The fused conv1+conv2 stem kernel (conv1 as a TS-mode tcgen05 UMMA with its im2col rows in tensor memory) against the
    two-kernel path (vfp_set_tuning(1, 0)) and the oracle, for every frame format it takes (planar bf16 / planar uint8 /
    decoder-layout uint8; fp32 frames stay on the two-kernel path).
    More frames than SMs so every CTA walks several frames and the rings / double buffers wrap."""
    lib = _native.load()
    sd = make_state_dict(2, "stress")
    m = model_for(2, "stress")
    lengths = [37, 64, 10, 150, 21, 300, 47]
    clips = make_clips(41, lengths, "colour")             # on the uint8/255 grid
    want = torch.stack(fingerprint_clips(sd, clips))
    x = torch.cat(clips)                                   # (sum T, 3, 64, 64) fp32
    u8 = torch.round(x * 255).to(torch.uint8)
    inputs = {"bf16": x.to(torch.bfloat16), "u8": u8, "u8_hwc": u8.permute(0, 2, 3, 1).contiguous()}
    for name, frames in inputs.items():
        frames = frames.cuda()
        try:
            lib.vfp_set_tuning(1, 0)
            ref = m.fingerprint_packed(frames, lengths).cpu()
            for mode in (2,):
                lib.vfp_set_tuning(1, mode)
                fused = m.fingerprint_packed(frames, lengths).cpu()
                assert lib.vfp_device_error_word() == 0, (name, mode)
                assert cosine(fused, want).min() >= COS_BAR, (name, mode)     # same bar as the default path
                assert cosine(fused, ref).min() > 0.99995, (name, mode)       # same bf16 operands, different summation order
        finally:
            lib.vfp_set_tuning(1, 2)


def test_weights_are_refreshed_after_load_state_dict():
    m = model_for(0, "default")
    x = torch.stack(make_clips(35, [12] * 2, "colour")).cuda()
    a = m(x).cpu()
    m.load_state_dict(make_state_dict(2, "stress"))
    b = m(x).cpu()
    want = forward_oracle(make_state_dict(2, "stress"), x.cpu())
    assert not torch.allclose(a, b, atol=1e-3)
    assert cosine(b, want).min() >= COS_BAR


def test_error_behaviour():
    m = model_for(0, "default")
    with pytest.raises(ValueError):
        m(torch.zeros(4, 3, 64, 64).cuda())
    with pytest.raises(ValueError):
        m.fingerprint_packed(torch.zeros(10, 3, 64, 64).cuda(), [4, 5])
    with pytest.raises(_native.NativeError, match="no frames"):
        m.fingerprint_packed(torch.zeros(10, 3, 64, 64).cuda(), [10, 0])
    with pytest.raises(_native.NativeError, match="positional table"):
        m.fingerprint_packed(torch.zeros(10001, 3, 64, 64, dtype=torch.uint8).cuda(), [10001])
    with pytest.raises(_native.NativeError, match="CUDA devices only"):
        vfp.VideoFingerprintScanner(model=m, device="cpu")
    m.train()
    with pytest.raises(RuntimeError, match="inference only"):
        m(torch.zeros(1, 10, 3, 64, 64).cuda())
    assert _native.load().vfp_device_error_word() == 0


def test_scanner_semantics(tmp_path):
    sd = make_state_dict(2, "stress")
    ckpt = tmp_path / "m.pth"
    torch.save({"model_state_dict": sd, "config": {"model_type": "attention", "max_frames": 40}, "metrics": None}, ckpt)
    sc = vfp.VideoFingerprintScanner(str(ckpt), device="cuda")
    clips = make_clips(36, [9, 30, 55], "colour")
    out = sc.extract_fingerprints_from_frames(clips)
    assert out[0] is None                                   # < 10 frames (fingerprint.py:238-240)
    want = fingerprint_clips(sd, [clips[1], clips[2][:40]])  # max_frames cap
    assert cosine(out[1], want[0]) >= COS_BAR and cosine(out[2], want[1]) >= COS_BAR
    assert out[1].dtype == np.float32 and out[1].shape == (256,)
    assert sc.subsample(1200) == list(range(0, 1200, 30))[:40]
