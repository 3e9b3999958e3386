"""CPU oracle for the fingerprint forward  --  TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline / ``--impl reference``
legs may import this module; the shipped path (``video_fingerprint_b200``) never does.

This is a plain fp32 restatement, in ``torch.nn.functional`` calls on a bare ``state_dict``, of the
reference's attention-model inference forward:

    /root/reference/model.py:272-298   VideoFingerprintAttention.forward
    /root/reference/model.py:92-121    SpatialEncoder            -> ``spatial_encoder``
    /root/reference/model.py:74-89     PositionalEncoding        -> ``positional_table`` / ``embed_tokens``
    /root/reference/model.py:155-179   TemporalConvBlock         -> ``temporal_conv_block``
    /root/reference/model.py:124-152   TemporalAttentionBlock    -> ``attention_block``
    /root/reference/model.py:256-270   adaptive_pooling          -> ``adaptive_pooling``
    /root/reference/model.py:219-224   final_projection + F.normalize (:292-294) -> ``project_and_normalise``
    /root/reference/fingerprint.py:232-270  per-video B=1 semantics -> ``fingerprint_clips``
    /root/reference/fingerprint.py:90-101   frame subsampling rule   -> ``subsample_indices``

Parity pin: ``tests/golden/make_golden.py`` runs the UNMODIFIED reference module on seeded weights/inputs
and stores its outputs (embeddings and pooled features) under ``tests/golden/``; ``tests/test_oracle.py``
checks this restatement against those files.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence

import torch
import torch.nn.functional as F

BN_EPS = 1e-5
LN_EPS = 1e-5
NUM_HEADS = 8
TEMPORAL_KERNELS = (3, 5, 7, 11)


def _bn(sd: Dict[str, torch.Tensor], prefix: str, x: torch.Tensor) -> torch.Tensor:
    """Inference-mode batch norm with the stored running statistics (model.py:100,104,108,112,170)."""
    return F.batch_norm(
        x,
        sd[prefix + ".running_mean"],
        sd[prefix + ".running_var"],
        sd[prefix + ".weight"],
        sd[prefix + ".bias"],
        training=False,
        eps=BN_EPS,
    )


def spatial_encoder(sd, frames: torch.Tensor, stages: Optional[dict] = None) -> torch.Tensor:
    """(F,3,64,64) -> (F,spatial_dim).  model.py:97-118."""
    p = "spatial_encoder.encoder."
    x = frames
    for conv_i, bn_i, stride_pad in ((0, 1, (2, 2)), (3, 4, (2, 1)), (6, 7, (2, 1)), (9, 10, (2, 1))):
        x = F.conv2d(x, sd[f"{p}{conv_i}.weight"], sd[f"{p}{conv_i}.bias"], stride=stride_pad[0], padding=stride_pad[1])
        x = F.relu(_bn(sd, f"{p}{bn_i}", x))
        if stages is not None:
            stages[f"conv{conv_i // 3 + 1}"] = x
    x = x.mean(dim=(2, 3))  # AdaptiveAvgPool2d(1) + Flatten
    if stages is not None:
        stages["pooled_conv4"] = x
    return F.linear(x, sd[p + "14.weight"], sd[p + "14.bias"])


def positional_table(length: int, dim: int = 256) -> torch.Tensor:
    """The sinusoidal table the reference registers as a buffer (model.py:79-86)."""
    pos = torch.arange(0, length, dtype=torch.float).unsqueeze(1)
    div = torch.exp(torch.arange(0, dim, 2).float() * (-math.log(10000.0) / dim))
    pe = torch.zeros(length, dim)
    pe[:, 0::2] = torch.sin(pos * div)
    pe[:, 1::2] = torch.cos(pos * div)
    return pe


def temporal_conv_block(sd, prefix: str, x_bct: torch.Tensor) -> torch.Tensor:
    """(B,C,T) -> (B,C,T): four grouped convs (k=3,5,7,11) + BN + ReLU, concatenated.  model.py:160-179."""
    outs = []
    for j, k in enumerate(TEMPORAL_KERNELS):
        w = sd[f"{prefix}.convs.{j}.0.weight"]
        y = F.conv1d(x_bct, w, sd[f"{prefix}.convs.{j}.0.bias"], padding=k // 2, groups=w.shape[0])
        outs.append(F.relu(_bn(sd, f"{prefix}.convs.{j}.1", y)))
    return torch.cat(outs, dim=1)


def attention_block(sd, prefix: str, x: torch.Tensor) -> torch.Tensor:
    """(B,T,C) -> (B,T,C): pre-LN multi-head self-attention + pre-LN 1x1-conv MLP.  model.py:140-152."""
    B, T, C = x.shape
    hd = C // NUM_HEADS
    h = F.layer_norm(x, (C,), sd[prefix + ".norm1.weight"], sd[prefix + ".norm1.bias"], LN_EPS)
    qkv = F.linear(h, sd[prefix + ".attn.in_proj_weight"], sd[prefix + ".attn.in_proj_bias"])
    q, k, v = qkv.split(C, dim=-1)
    q = q.view(B, T, NUM_HEADS, hd).transpose(1, 2)
    k = k.view(B, T, NUM_HEADS, hd).transpose(1, 2)
    v = v.view(B, T, NUM_HEADS, hd).transpose(1, 2)
    scores = (q @ k.transpose(-1, -2)) / math.sqrt(hd)
    ctx = torch.softmax(scores, dim=-1) @ v
    ctx = ctx.transpose(1, 2).reshape(B, T, C)
    x = x + F.linear(ctx, sd[prefix + ".attn.out_proj.weight"], sd[prefix + ".attn.out_proj.bias"])

    h = F.layer_norm(x, (C,), sd[prefix + ".norm2.weight"], sd[prefix + ".norm2.bias"], LN_EPS)
    h = F.conv1d(h.transpose(1, 2), sd[prefix + ".conv1.weight"], sd[prefix + ".conv1.bias"])
    h = F.gelu(h)  # exact erf form, nn.GELU() default
    h = F.conv1d(h, sd[prefix + ".conv2.weight"], sd[prefix + ".conv2.bias"]).transpose(1, 2)
    return x + h


def adaptive_pooling(sd, x: torch.Tensor) -> torch.Tensor:
    """(B,T,C) -> (B,3C) = [mean_T | max_T | softmax_T-weighted sum].  model.py:256-270."""
    avg = x.mean(dim=1)
    mx = x.max(dim=1).values
    xc = x.transpose(1, 2)
    logits = F.relu(F.conv1d(xc, sd["temporal_pool.0.weight"], sd["temporal_pool.0.bias"]))
    w = torch.softmax(logits, dim=2)
    weighted = (xc * w).sum(dim=2)
    return torch.cat([avg, mx, weighted], dim=1)


def project_and_normalise(sd, pooled: torch.Tensor, stages: Optional[dict] = None) -> torch.Tensor:
    """(B,3C) -> unit-norm (B,D).  model.py:219-224, 292-294. Records the ReLU hidden `head_h` and the pre-normalisation
    output `head_e` in `stages`."""
    h = F.relu(F.linear(pooled, sd["final_projection.0.weight"], sd["final_projection.0.bias"]))
    e = F.linear(h, sd["final_projection.3.weight"], sd["final_projection.3.bias"])
    if stages is not None:
        stages["head_h"], stages["head_e"] = h, e
    return e / e.norm(dim=1, keepdim=True).clamp_min(1e-12)


@torch.no_grad()
def forward_oracle(sd: Dict[str, torch.Tensor], video: torch.Tensor, stages: Optional[dict] = None,
                   dtype: torch.dtype = torch.float32) -> torch.Tensor:
    """Reference forward on a dense batch (B,T,3,64,64) (or (B,3,T,H,W), see model.py:283). `dtype`: the precision of every
    weight, frame, the checkpoint's positional table and all arithmetic (fp32 is the reference's own; float64 gives the
    high-precision reference the kernels are measured against)."""
    sd = {k: (v.to(dtype) if v.is_floating_point() else v) for k, v in sd.items()}
    video = video.to(dtype)
    if video.dim() == 5 and video.shape[1] == 3:  # the reference's layout sniff, quirk included
        video = video.permute(0, 2, 1, 3, 4)
    B, T = video.shape[:2]
    feats = spatial_encoder(sd, video.reshape(B * T, *video.shape[2:]), stages).view(B, T, -1)
    x = F.linear(feats, sd["temporal_projection.weight"], sd["temporal_projection.bias"])
    x = x + sd["pos_encoding.pe"][:, :T]
    if stages is not None:
        stages["tokens"] = x
    n_tconv = len({k.split(".")[1] for k in sd if k.startswith("temporal_conv_blocks.")})
    for i in range(n_tconv):
        x = x + temporal_conv_block(sd, f"temporal_conv_blocks.{i}", x.transpose(1, 2)).transpose(1, 2)
        if stages is not None:
            stages[f"tconv{i}"] = x
    n_attn = len({k.split(".")[1] for k in sd if k.startswith("attention_blocks.")})
    for i in range(n_attn):
        x = attention_block(sd, f"attention_blocks.{i}", x)
        if stages is not None:
            stages[f"attn{i}"] = x
    pooled = adaptive_pooling(sd, x)
    if stages is not None:
        stages["pooled"] = pooled
    return project_and_normalise(sd, pooled, stages)


def subsample_indices(total_frames: int, max_frames: int = 500) -> List[int]:
    """Which decoded frame indices the scanner keeps (fingerprint.py:90-101)."""
    skip = 1
    if total_frames > max_frames:
        skip = max(skip, total_frames // max_frames)
    keep = []
    for i in range(total_frames):
        if i % skip == 0:
            keep.append(i)
            if len(keep) >= max_frames:
                break
    return keep


@torch.no_grad()
def fingerprint_clips(sd, clips: Sequence[torch.Tensor], min_frames: int = 10) -> List[Optional[torch.Tensor]]:
    """Scanner semantics: one B=1 forward per clip (T_i,3,64,64); clips shorter than 10 frames give None
    (fingerprint.py:238-249, 268-270)."""
    out: List[Optional[torch.Tensor]] = []
    for clip in clips:
        if clip.shape[0] < min_frames:
            out.append(None)
            continue
        out.append(forward_oracle(sd, clip.unsqueeze(0))[0])
    return out
