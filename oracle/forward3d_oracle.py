"""CPU oracle for the 3-D CNN fingerprint model  --  TEST INFRASTRUCTURE, NOT PRODUCT CODE.

fp32 ``torch.nn.functional`` restatement of /root/reference/model.py:406-512 (``VideoFingerprint3D.forward``, eval mode) on a
bare state_dict, plus the window / mean / renormalise rule of the scanner's 3-D path (/root/reference/fingerprint.py:272-320).
Kept as a torch fp32 reference because the path is floating point. Pinned by tests/golden/forward3d_*.npz, which
tests/golden/make_golden_3d.py produces by running the UNMODIFIED reference module on the same seeded weights and clips.
"""
from __future__ import annotations

from typing import Dict, List, Optional

import torch
import torch.nn.functional as F


def make_state_dict_3d(seed: int, frame_stride: int = 16, embedding_dim: int = 256, stress: bool = True) -> Dict[str, torch.Tensor]:
    """Seeded weights with the reference's key layout. `stress`: non-trivial BatchNorm statistics and larger projector weights
    (the reference's default init gives BN = identity and a 0.01-std projector, which would hide folding mistakes)."""
    g = torch.Generator().manual_seed(seed)
    sd: Dict[str, torch.Tensor] = {}
    spec = [(3, 16, (frame_stride, 5, 5)), (16, 32, (3, 3, 3)), (32, 64, (3, 3, 3)), (64, 128, (3, 3, 3))]
    for i, (cin, cout, k) in enumerate(spec):
        fan_out = cout * k[0] * k[1] * k[2]
        sd[f"encoder.{i}.conv.weight"] = torch.randn((cout, cin, *k), generator=g) * (2.0 / fan_out) ** 0.5 * (3.0 if stress else 1.0)
        sd[f"encoder.{i}.conv.bias"] = torch.randn(cout, generator=g) * (0.1 if stress else 0.0)
        sd[f"encoder.{i}.bn.weight"] = torch.rand(cout, generator=g) + 0.5 if stress else torch.ones(cout)
        sd[f"encoder.{i}.bn.bias"] = torch.randn(cout, generator=g) * 0.2 if stress else torch.zeros(cout)
        sd[f"encoder.{i}.bn.running_mean"] = torch.randn(cout, generator=g) * 0.3 if stress else torch.zeros(cout)
        sd[f"encoder.{i}.bn.running_var"] = torch.rand(cout, generator=g) * 1.5 + 0.5 if stress else torch.ones(cout)
        sd[f"encoder.{i}.bn.num_batches_tracked"] = torch.tensor(0, dtype=torch.long)
    sd["temporal_conv.weight"] = torch.randn((128, 128, 3), generator=g) * 0.08
    sd["temporal_conv.bias"] = torch.randn(128, generator=g) * 0.05
    sd["temporal_attention.weight"] = torch.randn((1, 128, 1), generator=g) * 0.3
    sd["temporal_attention.bias"] = torch.randn(1, generator=g) * 0.1
    sd["projector.0.weight"] = torch.randn((128, 128), generator=g) * (0.12 if stress else 0.01)
    sd["projector.0.bias"] = torch.randn(128, generator=g) * (0.05 if stress else 0.0)
    sd["projector.3.weight"] = torch.randn((embedding_dim, 128), generator=g) * (0.12 if stress else 0.01)
    sd["projector.3.bias"] = torch.randn(embedding_dim, generator=g) * (0.05 if stress else 0.0)
    sd["temperature"] = torch.ones(1) * 0.07
    return sd


def forward3d_oracle(sd: Dict[str, torch.Tensor], video: torch.Tensor, frame_stride: int, stages: Optional[dict] = None,
                     dtype: torch.dtype = torch.float32) -> torch.Tensor:
    """model.py:468-509 in eval mode. video: (B, T, 3, H, W) or (B, 3, T, H, W) in [0, 1]. `dtype`: the precision of the
    weights, frames and arithmetic (float64 for the high-precision reference). `stages` receives the projector's ReLU hidden
    `head_h` and its pre-normalisation output `head_e`."""
    sd = {k: (v.to(dtype) if v.is_floating_point() else v) for k, v in sd.items()}
    x = video.to(dtype)
    if x.dim() == 5 and x.shape[2] == 3:
        x = x.permute(0, 2, 1, 3, 4)
    T = x.shape[2]
    pad = (frame_stride - T % frame_stride) % frame_stride
    if pad:
        x = F.pad(x, (0, 0, 0, 0, 0, pad))
    strides = [(frame_stride, 2, 2), (1, 2, 2), (2, 2, 2), (1, 2, 2)]
    pads = [(0, 2, 2), (1, 1, 1), (1, 1, 1), (1, 1, 1)]
    for i in range(4):
        x = F.conv3d(x, sd[f"encoder.{i}.conv.weight"], sd[f"encoder.{i}.conv.bias"], stride=strides[i], padding=pads[i])
        x = F.batch_norm(x, sd[f"encoder.{i}.bn.running_mean"], sd[f"encoder.{i}.bn.running_var"], sd[f"encoder.{i}.bn.weight"],
                         sd[f"encoder.{i}.bn.bias"], training=False, eps=1e-5)
        x = F.relu(x)
    feat = x.mean(dim=(3, 4))                                     # AdaptiveAvgPool3d((None, 1, 1)) + squeeze
    tf = F.conv1d(feat, sd["temporal_conv.weight"], sd["temporal_conv.bias"], padding=1)
    attn = F.softmax(F.conv1d(tf, sd["temporal_attention.weight"], sd["temporal_attention.bias"]), dim=2)
    combined = (tf * attn).sum(dim=2) + tf.mean(dim=2)
    h = F.relu(F.linear(combined, sd["projector.0.weight"], sd["projector.0.bias"]))   # Dropout inactive in eval
    e = F.linear(h, sd["projector.3.weight"], sd["projector.3.bias"])
    if stages is not None:
        stages["head_h"], stages["head_e"] = h, e
    return F.normalize(e, p=2, dim=1)


def make_clips_3d(seed: int, n: int, t: int) -> torch.Tensor:
    """(n, t, 3, 64, 64) fp32 on the uint8/255 grid: a per-clip colour cast + moving gradient + noise (so embeddings differ)."""
    g = torch.Generator().manual_seed(seed)
    base = torch.rand((n, 1, 3, 1, 1), generator=g)
    yy = torch.linspace(0, 1, 64).view(1, 1, 1, 64, 1)
    tt = torch.linspace(0, 1, t).view(1, t, 1, 1, 1)
    phase = torch.rand((n, 1, 1, 1, 1), generator=g)
    x = 0.45 * base + 0.25 * ((yy + tt * phase) % 1.0) + 0.3 * torch.rand((n, t, 3, 64, 64), generator=g)
    return torch.round(x.clamp(0, 1) * 255) / 255


CASES_3D = {
    # name: (weight seed, frame_stride, clip seed, n clips, frames per clip, stress weights)
    "fs16_t64": (11, 16, 101, 6, 64, True),
    "fs16_t150": (12, 16, 102, 4, 150, True),      # T not a multiple of the stride -> zero padding; T3 = 5
    "fs32_t64": (13, 32, 103, 4, 64, True),        # the class default stride
    "fs16_t16_refinit": (0, 16, 104, 4, 16, False),   # single group, reference default initialisation (via the module itself)
}
