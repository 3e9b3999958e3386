"""Every model shape the weight loaders accept, against a float64 reference.

Each axis the loaders accept picks a kernel path or moves a loop bound inside one: the attention model's embedding width D
(tcgen05 head with a fused bias + L2 norm for D <= 256 and D % 32 == 0, the fp32 head with one or two 256-column stripes
otherwise), its number of attention blocks (none: the block loop is skipped and the residual stream is closed without a
delta), its spatial width S (folded on the host), its clip length (one-token attention up to 157 key blocks and the last
rows of the positional table), and the 3-D model's frame stride (5 * fs K runs and up to 139 KB of shared memory in the
first conv) and width (four 128-wide head stripes). Every row below is one packed device call, compared clip by clip with
a float64 B = 1 forward of the oracle on stress weights (non-trivial BatchNorm and LayerNorm statistics).

Bars (y: device embedding, e: float64 pre-normalisation output, h: the head's ReLU hidden, W3 / b3: its last layer):
* embeddings of width >= 16: cosine(y, e) >= COS_BAR, the suite's bar;
* every width, 1 included: |y_d - e_d / |e|| <= TAU * max_d(sum_k |W3[d,k]| h_k + |b3_d|) / |e| for every d. The bound
  scales with how much cancellation the reference's own output carries, so it means the same at D = 1 (a sign with a
  margin) as at D = 512. A row whose bound reaches 0.5 would pass anything, so that is an error too;
* attention features (return_features): the largest per-token relative L2 error against the float64 residual stream after
  the last block is at most BETA. A kernel that drops the last key of a 300-token clip moves the embedding by 3.6e-5 in
  1 - cos, inside COS_BAR, but moves the features of every token by about 1e-2.

The negative controls at the end (CPU only) run the same assertions on the float64 reference with one defect planted at a
time, and require each to miss its bar by at least a factor of 2.
"""
import ctypes as C
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import video_fingerprint_b200 as vfp
from oracle import forward3d_oracle as f3
from oracle import forward_oracle as fo
from oracle import join_oracle
from oracle import metrics_oracle as mo
from oracle.weights import PE_LEN, make_clips, make_state_dict
from video_fingerprint_b200 import _native

COS_BAR = 0.9999
# Calibrated on a B200 (1000 W power limit). TAU: the worst err / cond at the default shape is 2.52e-3 (over every row here
# 4.69e-3, at the 3-D model's fs = 2). BETA: the worst per-token feature error at the default shape is 6.41e-3 (over every
# row 1.29e-2, at spatial_dim = 1, where the folded token projection has rank one).
TAU = 1e-2
BETA = 1.6e-2
CONTROL_MISS = 2.0    # a planted defect must exceed its bar by this factor

WSEED = 2                                          # attention weights (stress style)
LENGTHS = [1, 2, 3, 9, 10, 63, 64, 65, 129, 300]   # one-token attention .. several 64-token key blocks with a tail
F64 = torch.float64

GUARD = 1 << 20
PATTERN = 0xA5


# ---------------------------------------------------------------------------------------------------------------------------
# assertions shared by the device tests and the negative controls
def embedding_errors(y, st, w3, b3):
    """Per clip: (1 - cos(y, e), the largest |y_d - e_d/|e|| over the conditioning bound without TAU, that bound)."""
    y = torch.as_tensor(y).to(F64).reshape(st["head_e"].shape)
    e, h = st["head_e"].to(F64), st["head_h"].to(F64)
    norm = e.norm(dim=1)
    cond = (h @ w3.to(F64).abs().T + b3.to(F64).abs()).max(dim=1).values / norm
    err = (y - e / norm[:, None]).abs().max(dim=1).values
    cos = (y * e).sum(1) / (y.norm(dim=1) * norm)
    return 1 - cos, err / cond, cond


def embedding_margin(y, st, w3, b3):
    """How far the worst clip is from failing: the largest of err / (TAU * cond) and, for widths >= 16,
    (1 - cos) / (1 - COS_BAR). <= 1 passes."""
    one_minus_cos, ratio, cond = embedding_errors(y, st, w3, b3)
    assert float((TAU * cond).max()) < 0.5, ("bound too loose to mean anything", float(cond.max()))
    margin = float(ratio.max()) / TAU
    if st["head_e"].shape[1] >= 16:
        margin = max(margin, float(one_minus_cos.max()) / (1 - COS_BAR))
    return margin


def feature_error(f, ref):
    """Largest per-token relative L2 error of features (T, 256) against the reference residual stream."""
    f, ref = torch.as_tensor(f).to(F64).reshape(ref.shape), ref.to(F64)
    return float(((f - ref).norm(dim=-1) / ref.norm(dim=-1)).max())


def last_stream(st):
    """The residual stream the features are: after the last attention block, or after the second temporal conv."""
    n = len([k for k in st if k.startswith("attn")])
    return st[f"attn{n - 1}"] if n else st["tconv1"]


def attention_f64(sd, clip):
    """float64 B = 1 forward of one clip -> (embedding, the stages the bars read: head_h, head_e, features)."""
    st = {}
    video = clip[None]
    if clip.shape[0] == 3:   # the oracle keeps the reference's (B, 3, T, H, W) sniff on shape[1] == 3: hand it that layout
        video = video.transpose(1, 2)
    y = fo.forward_oracle(sd, video, st, dtype=F64)
    return y, {"head_h": st["head_h"], "head_e": st["head_e"], "features": last_stream(st)}


def u8_of(x):
    return torch.round(x * 255).to(torch.uint8)


# ---------------------------------------------------------------------------------------------------------------------------
# attention model
ATTN_ROWS = (
    [{}]
    + [{"embedding_dim": d} for d in (1, 2, 16, 31, 32, 33, 96, 100, 224, 255, 257, 384, 511, 512)]
    + [{"num_attention_blocks": n} for n in (0, 1, 2, 8)]
    + [{"num_attention_blocks": 0, "embedding_dim": 100}]        # the fp32 head after the close without a delta
    + [{"spatial_dim": s} for s in (1, 16, 512)]
    + [{"spatial_dim": 64, "num_attention_blocks": 2, "embedding_dim": 128}]
)


def row_id(arch):
    return "_".join(f"{k[0]}{v}" for k, v in sorted(arch.items())) or "default"


def attention_checkpoint(arch):
    """Stress weights of the given shape, with the head's output bias scaled to the size of the head's output (entries of
    about 30): at the stress init's +-0.05 it is 1e-3 of the output, and a kernel that dropped it would go unseen."""
    sd = make_state_dict(WSEED, "stress", **arch)
    sd["final_projection.3.bias"] = sd["final_projection.3.bias"] * 400
    if sd["final_projection.3.bias"].numel() == 1:
        # one output: a sum of 256 terms of about 1 that cancels to about 5, down to 0.2 for some clips, where no kernel can
        # be held to its sign. A bias of 50 keeps it to within a factor of 6 of the sum of |terms|, so the bound means something.
        sd["final_projection.3.bias"] = torch.full((1,), 50.0)
    return sd


def attention_model(arch):
    sd = attention_checkpoint(arch)
    m = vfp.create_model("attention", **arch).eval()
    m.load_state_dict(sd)
    return m, sd


@pytest.mark.gpu
@pytest.mark.parametrize("arch", ATTN_ROWS, ids=row_id)
def test_attention_shape_against_float64(arch):
    m, sd = attention_model(arch)
    D = sd["final_projection.3.bias"].numel()
    lengths = LENGTHS + ([PE_LEN] if not arch else [])      # the default row also runs the whole positional table
    clips = [u8_of(c) for c in make_clips(71, lengths, "colour")]
    emb, feats = m.fingerprint_packed(torch.cat(clips).cuda(), lengths, return_features=True)
    assert emb.shape == (len(lengths), D) and feats.shape == (sum(lengths), 256)
    assert _native.load().vfp_device_error_word() == 0
    emb, feats = emb.cpu(), feats.cpu()
    w3, b3 = sd["final_projection.3.weight"], sd["final_projection.3.bias"]
    rows, f0 = [], 0
    for i, (x, T) in enumerate(zip(clips, lengths)):
        _, st = attention_f64(sd, x.to(F64) / 255)
        rows.append((i, embedding_errors(emb[i], st, w3, b3), feature_error(feats[f0 : f0 + T], st["features"][0]), st))
        f0 += T
    report("attention " + row_id(arch), D, rows)
    for i, _, fe, st in rows:
        assert embedding_margin(emb[i], st, w3, b3) <= 1, (row_id(arch), lengths[i])
        assert fe <= BETA, (row_id(arch), lengths[i], fe)


def report(name, D, rows):
    """The measured worst of each bar's quantity over the row (pytest -s shows it): what TAU and BETA are calibrated on."""
    cos = max(float(r[1][0].max()) for r in rows) if D >= 16 else float("nan")
    tau = max(float(r[1][1].max()) for r in rows)
    cond = max(float(r[1][2].max()) for r in rows)
    beta = max((r[2] for r in rows if r[2] is not None), default=float("nan"))
    print(f"\n[measured] {name}: 1-cos {cos:.3e}  err/cond {tau:.3e}  feature err {beta:.3e}  max cond {cond:.3e}")


# ---------------------------------------------------------------------------------------------------------------------------
# 3-D model
W3D_SEED = 31
FS_ROWS = [(fs, 256, torch.uint8) for fs in (1, 2, 3, 4, 8, 63, 64)]
D3_ROWS = [(16, d, torch.uint8) for d in (1, 16, 100, 127, 128, 129, 255, 257, 384, 511, 512)] + [(1, 512, torch.uint8), (64, 1, torch.uint8)]
DTYPE_ROWS = [(fs, 256, dt) for fs in (1, 64) for dt in (torch.bfloat16, torch.float32)]


def edge_lengths(fs):
    """1, fs-1, fs, fs+1, 2fs, 2fs+1 (an odd number of groups), 10, 150 and 64*fs (T3 = 32): the lengths of
    test_model3d_packed.py that the stride admits (at most 64 * fs frames), in a fixed mixed order."""
    lengths = [t for t in (1, fs - 1, fs, fs + 1, 2 * fs, 2 * fs + 1, 10, 150, 64 * fs) if 0 < t <= 64 * fs]
    return lengths[1::2] + lengths[::2]


def frames_as(x, dtype):
    """fp32 frames on the uint8/255 grid -> (frames of `dtype`, the float64 values the device sees)."""
    if dtype == torch.uint8:
        u8 = u8_of(x)
        return u8, u8.to(F64) / 255
    y = x.to(dtype)
    return y, y.to(F64)


def model3d(fs, D):
    sd = f3.make_state_dict_3d(W3D_SEED, fs, embedding_dim=D, stress=True)
    m = vfp.create_model("3d", frame_stride=fs, embedding_dim=D).eval()
    m.load_state_dict(sd)
    return m, sd


@pytest.mark.gpu
@pytest.mark.parametrize("fs,D,dtype", FS_ROWS + D3_ROWS + DTYPE_ROWS, ids=lambda v: str(v).replace("torch.", ""))
def test_3d_shape_against_float64(fs, D, dtype):
    m, sd = model3d(fs, D)
    lengths = edge_lengths(fs)
    pairs = [frames_as(f3.make_clips_3d(800 + i, 1, t)[0], dtype) for i, t in enumerate(lengths)]
    emb = m.fingerprint_packed(torch.cat([p[0] for p in pairs]).cuda(), lengths)
    assert emb.shape == (len(lengths), D)
    assert _native.load().vfp_device_error_word() == 0
    emb = emb.cpu()
    w3, b3 = sd["projector.3.weight"], sd["projector.3.bias"]
    rows = []
    for i, (_, seen) in enumerate(pairs):
        st = {}
        f3.forward3d_oracle(sd, seen[None], fs, st, dtype=F64)
        rows.append((i, embedding_errors(emb[i], st, w3, b3), None, st))
    report(f"3-D fs {fs} D {D} {dtype}", D, rows)
    for i, _, _, st in rows:
        assert embedding_margin(emb[i], st, w3, b3) <= 1, (fs, D, lengths[i])


# ---------------------------------------------------------------------------------------------------------------------------
# where rows land in the output at widths other than 256
class Guarded:
    """A device buffer of exactly `nbytes` between two 1 MiB guard zones filled with a pattern."""

    def __init__(self, nbytes):
        self.n = int(nbytes)
        self.raw = torch.full((self.n + 2 * GUARD,), PATTERN, dtype=torch.uint8, device="cuda")
        self.t = self.raw[GUARD : GUARD + self.n]

    def intact(self):
        return bool((self.raw[:GUARD] == PATTERN).all()) and bool((self.raw[GUARD + self.n :] == PATTERN).all())


def cu_seqlens(lengths):
    return (C.c_int32 * (len(lengths) + 1))(*np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64).tolist())


@pytest.mark.gpu
@pytest.mark.parametrize("D", [1, 100, 128, 384])
def test_attention_passes_place_rows_by_width(D):
    """A workspace of 70 frames splits the batch into several passes; each pass writes its rows at c0 * D of an output of
    exactly n * D floats. Same bits as one pass."""
    m, _ = attention_model({"embedding_dim": D})
    lengths = [40, 12, 64, 19, 50, 25, 31, 3, 70]
    frames = torch.cat([u8_of(c) for c in make_clips(72, lengths, "colour")]).cuda()
    one_pass = m.fingerprint_packed(frames, lengths)
    lib = _native.load()
    w = m._ensure_native(frames.device.index)
    n = len(lengths)
    ws_bytes = lib.vfp_forward_workspace_bytes(max(lengths), min(max(lengths), n)) + 1024
    assert ws_bytes < lib.vfp_forward_workspace_bytes(sum(lengths), n)
    ws, out = Guarded(ws_bytes), Guarded(n * D * 4)
    rc = lib.vfp_forward(C.c_void_p(w), C.c_void_p(frames.data_ptr()), _native.FRAME_U8, C.cast(cu_seqlens(lengths), C.c_void_p), n,
                         C.c_void_p(out.t.data_ptr()), None, C.c_void_p(ws.t.data_ptr()), ws_bytes,
                         C.c_void_p(torch.cuda.current_stream().cuda_stream))
    _native.check(rc, "vfp_forward")
    torch.cuda.synchronize()
    assert lib.vfp_device_error_word() == 0
    assert ws.intact() and out.intact()
    assert torch.equal(out.t.view(torch.float32).view(n, D), one_pass)


@pytest.mark.gpu
@pytest.mark.parametrize("D", [1, 100, 384, 512])
def test_3d_passes_place_rows_by_width(D):
    """A workspace for two clips: several passes, rows at c0 * D of an output of exactly n * D floats, same bits."""
    fs = 16
    m, _ = model3d(fs, D)
    lengths = [37, 10, 150, 16, 1, 333, 64, 17]
    frames = torch.cat([u8_of(f3.make_clips_3d(900 + i, 1, t)[0]) for i, t in enumerate(lengths)]).cuda()
    one_pass = m.fingerprint_packed(frames, lengths)
    lib = _native.load()
    w = C.c_void_p(m._ensure_native())
    n = len(lengths)
    ws_bytes = lib.vfp3d_forward_packed_workspace_bytes(w, sum(sorted(lengths)[-2:]), 2)
    ws, out = Guarded(ws_bytes), Guarded(n * D * 4)
    rc = lib.vfp3d_forward_packed(w, C.c_void_p(frames.data_ptr()), _native.FRAME_U8, C.cast(cu_seqlens(lengths), C.c_void_p), n,
                                  C.c_void_p(out.t.data_ptr()), C.c_void_p(ws.t.data_ptr()), ws_bytes,
                                  C.c_void_p(torch.cuda.current_stream().cuda_stream))
    _native.check(rc, "vfp3d_forward_packed")
    torch.cuda.synchronize()
    assert lib.vfp_device_error_word() == 0
    assert ws.intact() and out.intact()
    assert torch.equal(out.t.view(torch.float32).view(n, D), one_pass)


# ---------------------------------------------------------------------------------------------------------------------------
# a D = 100 checkpoint through the scanner, the duplicate search and the metrics
@pytest.mark.gpu
def test_scanner_search_and_metrics_with_a_100_wide_checkpoint(tmp_path):
    arch = {"spatial_dim": 64, "embedding_dim": 100, "num_attention_blocks": 1}
    sd = attention_checkpoint(arch)
    ckpt = tmp_path / "d100.pth"
    torch.save({"model_state_dict": sd, "config": dict(model_type="attention", **arch), "metrics": None}, ckpt)
    sc = vfp.VideoFingerprintScanner(str(ckpt), device="cuda")
    # 120 clips: 90 videos, 30 of them with a second clip (the first few frames dropped); one clip too short
    g = torch.Generator().manual_seed(73)
    lengths = [int(t) for t in torch.randint(12, 40, (90,), generator=g)]
    clips = make_clips(74, lengths, "colour")
    src = list(range(0, 90, 3))
    clips += [clips[s][2:] for s in src] + [clips[0][:9]]
    ids = np.array(list(range(90)) + src)
    out = sc.extract_fingerprints_from_frames(clips)
    assert out[-1] is None and all(e is not None and e.shape == (100,) and e.dtype == np.float32 for e in out[:-1])
    emb = np.stack(out[:-1])
    w3, b3 = sd["final_projection.3.weight"], sd["final_projection.3.bias"]
    for i, x in enumerate(clips[:-1]):
        _, st = attention_f64(sd, x.to(F64))
        assert embedding_margin(torch.from_numpy(emb[i]), st, w3, b3) <= 1, i
    # the search: the scanner's find_duplicates against the oracle's on the same embeddings, at a threshold in a gap of the
    # pair scores wider than their summation-order noise
    fps = {f"v{i:03d}": {"embedding": e, "path": f"v{i:03d}", "name": f"v{i:03d}", "size": i, "file_hash": f"h{i % 50}",
                         "embedding_norm": float(np.linalg.norm(e))} for i, e in enumerate(emb)}
    off = np.sort((emb @ emb.T)[np.triu_indices(len(emb), 1)])
    gaps = np.nonzero((np.diff(off) > 1e-5) & (off[:-1] >= np.quantile(off, 0.99)))[0]
    thr = float((off[gaps[0]] + off[gaps[0] + 1]) / 2)
    for use_faiss in (True, False):          # 119 embeddings: the top-20 path, then the direct join
        got = sc.find_duplicates(fps, thr, use_faiss)
        want = join_oracle.find_duplicates(fps, thr, use_faiss)
        assert len(got) >= 5 and [sorted(it["name"] for it in g_) for g_ in got] == [sorted(it["name"] for it in w_) for w_ in want]
    # the metrics at width 100 (device pass on zero-padded rows) against the oracle on the same embeddings
    from video_fingerprint_b200 import metrics

    for got, want in ((metrics.compute_retrieval_metrics(emb, ids), mo.retrieval_metrics(emb, ids)),
                      (metrics.compute_discrimination_metrics(emb, ids), mo.discrimination_metrics(emb, ids))):
        assert set(got) == set(want)
        for k, v in want.items():
            assert abs(got[k] - v) <= 2e-6, (k, got[k], v)


# ---------------------------------------------------------------------------------------------------------------------------
# negative controls: the float64 reference with one defect planted, in place of the device output, must miss the bars
def attention_ignoring_last_key(sd, prefix, x):
    """oracle.forward_oracle.attention_block with the clip's last key masked out of every query's softmax."""
    B, T, C = x.shape
    hd = C // fo.NUM_HEADS
    h = F.layer_norm(x, (C,), sd[prefix + ".norm1.weight"], sd[prefix + ".norm1.bias"], fo.LN_EPS)
    qkv = F.linear(h, sd[prefix + ".attn.in_proj_weight"], sd[prefix + ".attn.in_proj_bias"])
    q, k, v = (t.view(B, T, fo.NUM_HEADS, hd).transpose(1, 2) for t in qkv.split(C, dim=-1))
    scores = (q @ k.transpose(-1, -2)) / math.sqrt(hd)
    scores[..., -1] = -math.inf
    x = x + F.linear((torch.softmax(scores, dim=-1) @ v).transpose(1, 2).reshape(B, T, C), sd[prefix + ".attn.out_proj.weight"],
                     sd[prefix + ".attn.out_proj.bias"])
    h = F.layer_norm(x, (C,), sd[prefix + ".norm2.weight"], sd[prefix + ".norm2.bias"], fo.LN_EPS)
    h = F.conv1d(F.gelu(F.conv1d(h.transpose(1, 2), sd[prefix + ".conv1.weight"], sd[prefix + ".conv1.bias"])),
                 sd[prefix + ".conv2.weight"], sd[prefix + ".conv2.bias"])
    return x + h.transpose(1, 2)


def pooling_missing_last_token(sd, x, _pool=fo.adaptive_pooling):
    p = _pool(sd, x).clone()
    C = x.shape[2]
    p[:, C : 2 * C] = x[:, :-1].max(dim=1).values
    return p


def tconv1_dropping_last_update(sd, prefix, x_bct, _block=fo.temporal_conv_block):
    y = _block(sd, prefix, x_bct)
    if prefix == "temporal_conv_blocks.1":
        y = y.clone()
        y[:, :, -1] = 0
    return y


def pe_off_by_one(sd):
    pe = sd["pos_encoding.pe"]
    return dict(sd, **{"pos_encoding.pe": torch.cat([pe[:, 1:], pe[:, -1:]], dim=1)})


def attention_control(monkeypatch, T, arch=None, patch=None, edit_sd=None, edit_out=None, features=True):
    """Margin (worst bar's error over the bar) of a defective float64 forward of one T-frame clip against the true one."""
    sd = attention_checkpoint(arch or {})
    x = make_clips(75, [T], "colour")[0].to(F64)
    _, st = attention_f64(sd, x)
    if patch is not None:
        monkeypatch.setattr(fo, *patch)
    y_bad, st_bad = attention_f64(edit_sd(sd) if edit_sd else sd, x)
    monkeypatch.undo()
    if edit_out is not None:
        y_bad = edit_out(st_bad["head_e"])
    margin = embedding_margin(y_bad, st, sd["final_projection.3.weight"], sd["final_projection.3.bias"])
    if features:
        margin = max(margin, feature_error(st_bad["features"][0], st["features"][0]) / BETA)
    return margin


def bias_lost_on_96_to_99(sd):
    return dict(sd, **{"final_projection.3.bias": torch.cat([sd["final_projection.3.bias"][:96], torch.zeros(4)])})


def second_stripe_out_of_norm(e):
    return e / e[:, :256].norm(dim=1, keepdim=True)


ATTENTION_CONTROLS = {
    # name: (clip lengths where the defect is planted, keyword arguments of attention_control)
    # at T = 300 this defect moves the features by at most 1.14e-2, 0.71 x BETA: inside what S = 1 needs, not separable there
    "attention ignores the last key": ([65], dict(patch=("attention_block", attention_ignoring_last_key))),
    "positional table off by one": ([10, 64, 300], dict(edit_sd=pe_off_by_one)),
    "max-pool misses the last token": ([10, 64, 300], dict(patch=("adaptive_pooling", pooling_missing_last_token))),
    "second temporal conv drops the last token's update": ([10, 64, 300], dict(patch=("temporal_conv_block", tconv1_dropping_last_update))),
    "last attention block skipped": ([10, 300], dict(edit_sd=lambda sd: {k: v for k, v in sd.items() if not k.startswith("attention_blocks.3.")})),
    "fp32 head loses its bias on columns 96-99": ([64], dict(arch={"embedding_dim": 100}, edit_sd=bias_lost_on_96_to_99)),
    "fp32 head leaves its second stripe out of the norm": ([64], dict(arch={"embedding_dim": 384}, edit_out=second_stripe_out_of_norm)),
}


@pytest.mark.parametrize("name", sorted(ATTENTION_CONTROLS))
def test_negative_control_attention(name, monkeypatch):
    lengths, kw = ATTENTION_CONTROLS[name]
    for T in lengths:
        margin = attention_control(monkeypatch, T, **kw)
        print(f"\n[control] {name}, T = {T}: {margin:.2f} x the bar")
        assert margin >= CONTROL_MISS, (name, T, margin)


def pad_with_white(x, fs):
    """Frames past the clip end read as 255 instead of the reference's zero padding."""
    return torch.cat([x, torch.ones((-x.shape[0] % fs,) + tuple(x.shape[1:]), dtype=x.dtype)])


def last_stripe_dropped(e):
    e = e.clone()
    e[:, 384:] = 0
    return e / e.norm(dim=1, keepdim=True)


@pytest.mark.parametrize("name,fs,D,lengths", [
    ("frames past the clip end read as 255", 16, 256, [1, 15, 17, 33, 40, 150]),
    ("frames past the clip end read as 255", 64, 256, [1, 63, 65, 129, 150]),
    ("head3d drops the stripe d >= 384", 16, 512, [16, 64, 150]),
])
def test_negative_control_3d(name, fs, D, lengths):
    sd = f3.make_state_dict_3d(W3D_SEED, fs, embedding_dim=D, stress=True)
    for i, T in enumerate(lengths):
        x = u8_of(f3.make_clips_3d(800 + i, 1, T)[0]).to(F64) / 255
        st, st_bad = {}, {}
        f3.forward3d_oracle(sd, x[None], fs, st, dtype=F64)
        if "255" in name:
            y_bad = f3.forward3d_oracle(sd, pad_with_white(x, fs)[None], fs, dtype=F64)
        else:
            y_bad = last_stripe_dropped(st["head_e"])
        margin = embedding_margin(y_bad, st, sd["projector.3.weight"], sd["projector.3.bias"])
        print(f"\n[control] 3-D {name}, fs = {fs}, D = {D}, T = {T}: {margin:.2f} x the bar")
        assert margin >= CONTROL_MISS, (name, T, margin)
