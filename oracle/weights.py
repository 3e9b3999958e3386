"""Seeded checkpoints and synthetic clips for the parity tests  --  TEST INFRASTRUCTURE, NOT PRODUCT CODE.

``state_spec()`` restates the reference checkpoint layout (144 entries; /root/reference/model.py:97-118,
129-138, 160-175, 195-226 and SURVEY.md section 8b). ``make_state_dict`` fills it from a seeded
``torch.Generator`` so the build container (where the reference can be imported) and the GPU box (where
it cannot) see bit-identical weights without shipping a 26 MB checkpoint:

* style "default": PyTorch-default-like statistics (uniform(+-1/sqrt(fan_in)) weights, identity norms).
  With this init all embeddings of noise clips are nearly collinear (SURVEY.md section 4), so it mainly
  pins the "cos >= 0.9999" bar the task states.
* style "stress": randomised BN/LN statistics and 3x larger matrices (SURVEY.md section 8d) - embeddings
  spread out (pairwise cos 0.89..0.999), which makes the duplicate-set parity check discriminating.
"""
from __future__ import annotations

import hashlib
import math
from typing import Dict, List, Tuple

import torch

from .forward_oracle import TEMPORAL_KERNELS, positional_table

PE_LEN = 10000


def state_spec(spatial_dim=128, temporal_dim=256, embedding_dim=256, num_attention_blocks=4) -> List[Tuple[str, tuple, str]]:
    """[(key, shape, kind)] in checkpoint order. kind: w (weight matrix/filter), b (bias), bn_w, bn_b, bn_mean,
    bn_var, bn_count, ln_w, ln_b, temp, pe."""
    spec: List[Tuple[str, tuple, str]] = []

    def bn(prefix, c):
        spec.extend(
            [
                (prefix + ".weight", (c,), "bn_w"),
                (prefix + ".bias", (c,), "bn_b"),
                (prefix + ".running_mean", (c,), "bn_mean"),
                (prefix + ".running_var", (c,), "bn_var"),
                (prefix + ".num_batches_tracked", (), "bn_count"),
            ]
        )

    spec.append(("temperature", (1,), "temp"))
    chans = [(3, 32, 5), (32, 64, 3), (64, 128, 3), (128, 256, 3)]
    for i, (cin, cout, k) in enumerate(chans):
        p = f"spatial_encoder.encoder.{3 * i}"
        spec.append((p + ".weight", (cout, cin, k, k), "w"))
        spec.append((p + ".bias", (cout,), "b"))
        bn(f"spatial_encoder.encoder.{3 * i + 1}", cout)
    spec.append(("spatial_encoder.encoder.14.weight", (spatial_dim, 256), "w"))
    spec.append(("spatial_encoder.encoder.14.bias", (spatial_dim,), "b"))
    spec.append(("temporal_projection.weight", (temporal_dim, spatial_dim), "w"))
    spec.append(("temporal_projection.bias", (temporal_dim,), "b"))
    spec.append(("pos_encoding.pe", (1, PE_LEN, temporal_dim), "pe"))
    branch = temporal_dim // len(TEMPORAL_KERNELS)
    for blk in range(2):
        for j, k in enumerate(TEMPORAL_KERNELS):
            p = f"temporal_conv_blocks.{blk}.convs.{j}"
            spec.append((p + ".0.weight", (branch, temporal_dim // branch, k), "w"))
            spec.append((p + ".0.bias", (branch,), "b"))
            bn(p + ".1", branch)
    for blk in range(num_attention_blocks):
        p = f"attention_blocks.{blk}"
        spec.append((p + ".norm1.weight", (temporal_dim,), "ln_w"))
        spec.append((p + ".norm1.bias", (temporal_dim,), "ln_b"))
        spec.append((p + ".attn.in_proj_weight", (3 * temporal_dim, temporal_dim), "w"))
        spec.append((p + ".attn.in_proj_bias", (3 * temporal_dim,), "b"))
        spec.append((p + ".attn.out_proj.weight", (temporal_dim, temporal_dim), "w"))
        spec.append((p + ".attn.out_proj.bias", (temporal_dim,), "b"))
        spec.append((p + ".norm2.weight", (temporal_dim,), "ln_w"))
        spec.append((p + ".norm2.bias", (temporal_dim,), "ln_b"))
        spec.append((p + ".conv1.weight", (4 * temporal_dim, temporal_dim, 1), "w"))
        spec.append((p + ".conv1.bias", (4 * temporal_dim,), "b"))
        spec.append((p + ".conv2.weight", (temporal_dim, 4 * temporal_dim, 1), "w"))
        spec.append((p + ".conv2.bias", (temporal_dim,), "b"))
    spec.append(("temporal_pool.0.weight", (temporal_dim, temporal_dim, 1), "w"))
    spec.append(("temporal_pool.0.bias", (temporal_dim,), "b"))
    spec.append(("final_projection.0.weight", (temporal_dim, 3 * temporal_dim), "w"))
    spec.append(("final_projection.0.bias", (temporal_dim,), "b"))
    spec.append(("final_projection.3.weight", (embedding_dim, temporal_dim), "w"))
    spec.append(("final_projection.3.bias", (embedding_dim,), "b"))
    return spec


def make_state_dict(seed: int, style: str = "default", **arch) -> Dict[str, torch.Tensor]:
    """Seeded checkpoint of `state_spec(**arch)`: `arch` may set spatial_dim, embedding_dim and num_attention_blocks."""
    assert style in ("default", "stress")
    assert set(arch) <= {"spatial_dim", "embedding_dim", "num_attention_blocks"}, sorted(arch)
    g = torch.Generator().manual_seed(seed)
    stress = style == "stress"
    sd: Dict[str, torch.Tensor] = {}

    def uni(shape, lo, hi):
        return torch.rand(shape, generator=g) * (hi - lo) + lo

    for key, shape, kind in state_spec(**arch):
        if kind == "w":
            fan_in = 1
            for d in shape[1:]:
                fan_in *= d
            bound = 1.0 / math.sqrt(fan_in)
            t = uni(shape, -bound, bound)
            if stress:
                t = t * 3.0
        elif kind == "b":
            t = uni(shape, -0.05, 0.05)
        elif kind in ("bn_w", "ln_w"):
            t = uni(shape, 0.5, 1.5) if stress else torch.ones(shape)
        elif kind in ("bn_b", "ln_b"):
            t = torch.randn(shape, generator=g) * 0.2 if stress else torch.zeros(shape)
        elif kind == "bn_mean":
            t = torch.randn(shape, generator=g) * 0.5 if stress else torch.zeros(shape)
        elif kind == "bn_var":
            t = uni(shape, 0.5, 2.0) if stress else torch.ones(shape)
        elif kind == "bn_count":
            t = torch.tensor(0, dtype=torch.int64)
        elif kind == "temp":
            t = torch.ones(1) * 0.07
        elif kind == "pe":
            t = positional_table(shape[1], shape[2]).unsqueeze(0)
        else:  # pragma: no cover
            raise AssertionError(kind)
        sd[key] = t.contiguous()
    return sd


def state_dict_digest(sd: Dict[str, torch.Tensor]) -> str:
    """sha256 over all parameter bytes except the (formula-defined, libm-dependent) pe buffer."""
    h = hashlib.sha256()
    for key in sorted(sd):
        if key == "pos_encoding.pe":
            continue
        h.update(key.encode())
        h.update(sd[key].detach().cpu().contiguous().numpy().tobytes())
    return h.hexdigest()


def make_clips(seed: int, lengths, style: str = "noise", quantise: bool = True) -> List[torch.Tensor]:
    """Synthetic pre-decoded clips (T,3,64,64) in [0,1], quantised to the uint8/255 grid the scanner's
    preprocessing produces (fingerprint.py:210). "noise": i.i.d. uniform pixels (BASELINE cfg 1);
    "colour": 0.8*per-video colour + 0.2*noise (SURVEY.md section 8d stress inputs)."""
    g = torch.Generator().manual_seed(seed)
    clips = []
    for T in lengths:
        x = torch.rand((T, 3, 64, 64), generator=g)
        if style == "colour":
            c = torch.rand((1, 3, 1, 1), generator=g)
            x = 0.8 * c + 0.2 * x
        clips.append(torch.round(x * 255.0) / 255.0 if quantise else x)
    return clips
