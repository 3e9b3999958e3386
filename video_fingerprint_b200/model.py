"""Drop-in for the reference model factory (/root/reference/model.py:585-610) and attention model
(/root/reference/model.py:182-298), inference only.

`create_model("attention", ...)` returns an ``nn.Module`` whose ``state_dict()`` has the reference's 144 keys,
shapes and dtypes (so ``load_state_dict(checkpoint["model_state_dict"])`` from fingerprint.py:70 works
unchanged, and default construction under a fixed ``torch.manual_seed`` yields the reference's initial
weights), but whose ``forward`` does not run any PyTorch operator: it hands raw device pointers to
``vfp_forward`` in libvfp_b200.so (hand-written sm_100a kernels). The parameter-holding submodules exist only
to own tensors under the right names.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import List, Optional, Sequence, Tuple

import torch
import torch.nn as nn

from . import _native

_TEMPORAL_KERNELS = (3, 5, 7, 11)
_NUM_HEADS = 8


class _ParamsOnly(nn.Module):
    """Base for containers that own parameters but are never called."""

    def forward(self, *a, **k):  # pragma: no cover
        raise RuntimeError("parameter container: compute happens in libvfp_b200.so, not in PyTorch modules")


class PositionalEncoding(_ParamsOnly):
    """Owns the persistent sinusoidal buffer `pe` (1, max_len, d) of model.py:74-89."""

    def __init__(self, d_model: int, max_len: int = 10000):
        super().__init__()
        angle = torch.arange(0, max_len, dtype=torch.float).unsqueeze(1) * torch.exp(
            torch.arange(0, d_model, 2).float() * (-math.log(10000.0) / d_model)
        )
        table = torch.zeros(max_len, d_model)
        table[:, 0::2] = torch.sin(angle)
        table[:, 1::2] = torch.cos(angle)
        self.register_buffer("pe", table.unsqueeze(0))


class SpatialEncoder(_ParamsOnly):
    """Parameter layout of model.py:92-121: `encoder.{0,3,6,9}` convs, `{1,4,7,10}` batch norms, `14` linear."""

    STAGES = ((3, 32, 5, 2), (32, 64, 3, 1), (64, 128, 3, 1), (128, 256, 3, 1))  # cin, cout, kernel, padding

    def __init__(self, in_channels: int = 3, out_dim: int = 128):
        super().__init__()
        layers: List[nn.Module] = []
        for cin, cout, k, pad in self.STAGES:
            layers += [nn.Conv2d(in_channels if cin == 3 else cin, cout, k, stride=2, padding=pad), nn.BatchNorm2d(cout), nn.ReLU(inplace=True)]
        layers += [nn.AdaptiveAvgPool2d(1), nn.Flatten(), nn.Linear(256, out_dim)]
        self.encoder = nn.Sequential(*layers)


class TemporalConvBlock(_ParamsOnly):
    """model.py:155-179: `convs.{j}.0` grouped Conv1d(dim -> dim/n, k_j, groups=dim/n), `convs.{j}.1` BatchNorm1d."""

    def __init__(self, dim: int, kernel_sizes: Sequence[int] = _TEMPORAL_KERNELS):
        super().__init__()
        width = dim // len(kernel_sizes)
        self.convs = nn.ModuleList(
            nn.Sequential(nn.Conv1d(dim, width, k, padding=k // 2, groups=width), nn.BatchNorm1d(width), nn.ReLU(inplace=True))
            for k in kernel_sizes
        )


class TemporalAttentionBlock(_ParamsOnly):
    """model.py:124-152: norm1, attn (packed in_proj + out_proj), norm2, conv1 (1x1, dim->4dim), conv2 (1x1)."""

    def __init__(self, dim: int, num_heads: int = _NUM_HEADS, mlp_ratio: int = 4, drop: float = 0.1):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim)
        self.attn = nn.MultiheadAttention(dim, num_heads, dropout=drop, batch_first=True)
        self.norm2 = nn.LayerNorm(dim)
        self.conv1 = nn.Conv1d(dim, dim * mlp_ratio, 1)
        self.act = nn.GELU()
        self.conv2 = nn.Conv1d(dim * mlp_ratio, dim, 1)
        self.drop = nn.Dropout(drop)


class VideoFingerprintAttention(nn.Module):
    """Fingerprint model: (B,T,3,64,64) frames in [0,1] -> unit-norm (B, embedding_dim) embeddings."""

    def __init__(self, spatial_dim=128, temporal_dim=256, embedding_dim=256, num_attention_blocks=4, num_heads=_NUM_HEADS):
        super().__init__()
        if temporal_dim != 256 or num_heads != 8:
            raise ValueError("the sm_100a kernels are specialised for temporal_dim=256 with 8 heads (reference defaults)")
        self.spatial_encoder = SpatialEncoder(out_dim=spatial_dim)
        self.temporal_projection = nn.Linear(spatial_dim, temporal_dim)
        self.pos_encoding = PositionalEncoding(temporal_dim)
        self.temporal_conv_blocks = nn.ModuleList(TemporalConvBlock(temporal_dim) for _ in range(2))
        self.attention_blocks = nn.ModuleList(TemporalAttentionBlock(temporal_dim, num_heads) for _ in range(num_attention_blocks))
        self.temporal_pool = nn.Sequential(nn.Conv1d(temporal_dim, temporal_dim, 1), nn.ReLU(inplace=True))
        self.final_projection = nn.Sequential(
            nn.Linear(temporal_dim * 3, temporal_dim), nn.ReLU(inplace=True), nn.Dropout(0.1), nn.Linear(temporal_dim, embedding_dim)
        )
        self.temperature = nn.Parameter(torch.ones(1) * 0.07)
        self.embedding_dim = embedding_dim
        # frames per token pass (workspace per pass: 8.5 KB/frame + 1.8 GB for the conv pass) and the number of passes kept in
        # flight on internal streams of the library (vfp_forward deals the passes round-robin onto `pipelines` streams)
        # Measured on B200: one pass over everything on the caller's stream is as fast as two or three passes in flight
        # (38.6-38.9 vs 38.6-39.9 ms per 10 000 clips), so that is the default; `pipelines` > 1 remains for callers whose
        # batches are too small to fill the GPU on their own.
        self.frames_per_pass = 1 << 20
        self.pipelines = 1
        self._native: dict = {}          # device index -> (weights handle, key): one native handle per GPU
        self._workspaces: dict = {}      # device index -> uint8 tensor
        self._upload: dict = {}          # fingerprint_host: (device, dtype, frame shape) -> (two device buffers, copy stream)

    # ------------------------------------------------------------------ native weight handle
    def _weights_key(self) -> tuple:
        return tuple((t.data_ptr(), t._version) for t in self.state_dict(keep_vars=True).values())

    def _release_native(self, device_index: Optional[int] = None) -> None:
        for idx in list(self._native) if device_index is None else [device_index]:
            handle, _ = self._native.pop(idx, (None, None))
            if handle is not None:
                try:
                    with torch.cuda.device(idx):
                        _native.load().vfp_weights_destroy(C.c_void_p(handle))
                except Exception:  # pragma: no cover - interpreter teardown
                    pass

    def __del__(self):  # pragma: no cover
        try:
            self._release_native()
        except Exception:  # interpreter teardown: torch internals may already be gone
            pass

    def _ensure_native(self, device_index: int) -> int:
        """(Re)build the folded / packed device weights of the CURRENT device whenever a parameter or buffer changed.
        Handles are per device: the packed weights live in the memory of the GPU they were created on."""
        key = self._weights_key()
        handle, have = self._native.get(device_index, (None, None))
        if handle is not None and key == have:
            return handle
        self._release_native(device_index)
        lib = _native.load()
        host = {k: v.detach().to("cpu").contiguous() for k, v in self.state_dict().items()}
        host = {k: (v.float() if v.is_floating_point() else v) for k, v in host.items()}
        descs = (_native.TensorDesc * len(host))()
        for i, (k, v) in enumerate(host.items()):
            descs[i] = _native.TensorDesc(k.encode(), v.data_ptr(), v.numel())
        out = C.c_void_p()
        _native.check(lib.vfp_weights_create(descs, len(host), C.byref(out)), "vfp_weights_create")
        self._native[device_index] = (out.value, key)
        return out.value

    def _get_workspace(self, nbytes: int, device) -> torch.Tensor:
        ws = self._workspaces.get(device.index)
        if ws is None or ws.numel() < nbytes:
            self._workspaces.pop(device.index, None)
            ws = torch.empty(nbytes, dtype=torch.uint8, device=device)
            self._workspaces[device.index] = ws
        return ws

    # ------------------------------------------------------------------ packed (variable-length) entry
    @torch.no_grad()
    def fingerprint_packed(self, frames: torch.Tensor, lengths: Sequence[int], return_features: bool = False):
        """frames: (sum T, 3, 64, 64) uint8 / bf16 / fp32, or decoder-layout (sum T, 64, 64, 3) uint8, clips back to back;
        lengths: frames per clip.
        Every clip gets exactly the embedding a B=1 reference forward on that clip alone would give."""
        _native.require_cuda()
        if self.training:
            raise RuntimeError("inference only: call .eval() first (the reference scanner does, fingerprint.py:33)")
        lengths = [int(t) for t in lengths]
        total = sum(lengths)
        hwc = frames.dim() == 4 and tuple(frames.shape[1:]) == (64, 64, 3) and frames.dtype == torch.uint8
        if frames.dim() != 4 or not (hwc or tuple(frames.shape[1:]) == (3, 64, 64)) or frames.shape[0] != total:
            raise ValueError(f"frames must be (sum(lengths)={total}, 3, 64, 64) or uint8 (.., 64, 64, 3), got {tuple(frames.shape)}")
        if not frames.is_cuda:  # host frames: chunked, double-buffered upload overlapped with the forward (fingerprint.py:246-249)
            out = self.fingerprint_host(frames, lengths, return_features=return_features)
            return out
        if hwc:
            code = _native.FRAME_U8_HWC  # decoder layout: /255 and HWC->CHW (fingerprint.py:210-212) happen in conv1's loader
        elif frames.dtype == torch.uint8:
            code = _native.FRAME_U8
        elif frames.dtype == torch.bfloat16:
            code = _native.FRAME_BF16
        else:
            code = _native.FRAME_F32
            frames = frames.float()
        frames = frames.contiguous()
        dev = frames.device
        lib = _native.load()
        with torch.cuda.device(dev):
            weights = self._ensure_native(dev.index)
            n = len(lengths)
            cu = (C.c_int32 * (n + 1))()
            acc = 0
            for i, t in enumerate(lengths):
                cu[i] = acc
                acc += t
            cu[n] = acc
            pass_frames = max(min(total, self.frames_per_pass), max(lengths))
            slices = max(1, min(int(self.pipelines), 4, -(-total // pass_frames)))   # one workspace slice per pass in flight
            ws = self._get_workspace(slices * (lib.vfp_forward_workspace_bytes(pass_frames, min(pass_frames, n)) + 1024), dev)
            emb = torch.empty((n, self.embedding_dim), dtype=torch.float32, device=dev)
            feats = torch.empty((total, 256), dtype=torch.float32, device=dev) if return_features else None
            stream = torch.cuda.current_stream(dev).cuda_stream
            lib.vfp_set_tuning(9, slices)   # passes in flight = workspace slices (library-wide setting, re-stated per call)
            rc = lib.vfp_forward(
                C.c_void_p(weights), C.c_void_p(frames.data_ptr()), code, C.cast(cu, C.c_void_p), n,
                C.c_void_p(emb.data_ptr()), C.c_void_p(feats.data_ptr() if feats is not None else None),
                C.c_void_p(ws.data_ptr()), ws.numel(), C.c_void_p(stream),
            )
            _native.check(rc, "vfp_forward")
        return (emb, feats) if return_features else emb

    @torch.no_grad()
    def fingerprint_host(self, frames: torch.Tensor, lengths: Sequence[int], chunk_frames: int = 32768, device=None,
                         out: Optional[torch.Tensor] = None, return_features: bool = False):
        """Host-resident frames -> embeddings, the scanner's `clip.to(device); model(clip)` (fingerprint.py:246-249) for a
        whole corpus: `frames` is a HOST tensor (pinned memory gives asynchronous copies) laid out like `fingerprint_packed`
        expects. Clips are grouped into chunks of about `chunk_frames` frames; chunk i+1 is uploaded on a copy stream into
        the second of two device buffers while chunk i runs through the network, so the PCIe transfer and the forward
        overlap. Returns the (n, D) embeddings on the device, or - when `out` (a host tensor, ideally pinned) is given -
        copies them into it, synchronises and returns `out`."""
        _native.require_cuda()
        if frames.is_cuda:
            raise ValueError("fingerprint_host takes host frames; use fingerprint_packed for device tensors")
        lengths = [int(t) for t in lengths]
        n, total = len(lengths), sum(lengths)
        if frames.dim() != 4 or frames.shape[0] != total:
            raise ValueError(f"frames must be (sum(lengths)={total}, ...), got {tuple(frames.shape)}")
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        frames = frames.contiguous()
        # chunk boundaries on clip boundaries
        chunks, c0, f0 = [], 0, 0
        while c0 < n:
            c1, f1 = c0, f0
            while c1 < n and (c1 == c0 or f1 - f0 + lengths[c1] <= chunk_frames):
                f1 += lengths[c1]
                c1 += 1
            chunks.append((c0, c1, f0, f1))
            c0, f0 = c1, f1
        cap = max(f1 - f0 for _, _, f0, f1 in chunks)
        key = (dev.index, frames.dtype, tuple(frames.shape[1:]))
        state = self._upload.get(key)
        if state is None or state[0][0].shape[0] < cap:
            bufs = [torch.empty((cap,) + tuple(frames.shape[1:]), dtype=frames.dtype, device=dev) for _ in range(2)]
            state = (bufs, torch.cuda.Stream(dev))
            self._upload = {key: state}   # one cached pair: the buffers are as large as a chunk
        bufs, copy_stream = state
        with torch.cuda.device(dev):
            main = torch.cuda.current_stream(dev)
            emb = torch.empty((n, self.embedding_dim), dtype=torch.float32, device=dev)
            feats = torch.empty((total, 256), dtype=torch.float32, device=dev) if return_features else None
            ready = [torch.cuda.Event(), torch.cuda.Event()]
            free = [torch.cuda.Event(), torch.cuda.Event()]
            for ev in free:
                ev.record(main)
            for i, (a, b, fa, fb) in enumerate(chunks):
                k = i & 1
                with torch.cuda.stream(copy_stream):
                    copy_stream.wait_event(free[k])   # the forward that last read this buffer has finished
                    bufs[k][: fb - fa].copy_(frames[fa:fb], non_blocking=True)
                    ready[k].record(copy_stream)
                main.wait_event(ready[k])
                res = self.fingerprint_packed(bufs[k][: fb - fa], lengths[a:b], return_features=return_features)
                if return_features:
                    emb[a:b], feats[fa:fb] = res
                else:
                    emb[a:b] = res
                free[k].record(main)
            if out is not None:
                out.copy_(emb, non_blocking=True)
                main.synchronize()
                return (out, feats) if return_features else out
        return (emb, feats) if return_features else emb

    def fingerprint_clips(self, clips: Sequence[torch.Tensor]) -> torch.Tensor:
        """List of (T_i,3,64,64) clips -> (n, D) embeddings, one packed launch sequence (no padding, no masks)."""
        lengths = [int(c.shape[0]) for c in clips]
        return self.fingerprint_packed(torch.cat([c.cuda() for c in clips], dim=0), lengths)

    @torch.no_grad()
    def fingerprint_views(self, clips: Sequence[torch.Tensor], return_features: bool = False):
        """Device clips wherever they sit -> (n, embedding_dim) fp32 on their device, without copying a frame: each clip is a
        CUDA tensor (T_i, 3, 64, 64) uint8 / bf16 / fp32, or decoder-layout (T_i, 64, 64, 3) uint8 (what
        `preprocess_frames_device` returns), all of one dtype and layout on one device. Every frame must be contiguous; the
        frames of a clip may be any positive stride apart, so `frames[s:s + L]`, `frames[::skip][:max_frames]` and
        overlapping or repeated windows of one buffer all qualify. Row i has exactly the bits `fingerprint_packed` gives for
        the same frames packed; with return_features=True the per-frame features (sum T_i, 256) follow, in clip order.
        Raises ValueError rather than copying anything."""
        _native.require_cuda()
        if self.training:
            raise RuntimeError("inference only: call .eval() first (the reference scanner does, fingerprint.py:33)")
        clips = list(clips)
        if not clips:
            raise ValueError("fingerprint_views needs at least one clip")
        for i, c in enumerate(clips):
            if not isinstance(c, torch.Tensor) or not c.is_cuda:
                raise ValueError(f"clip {i} is not a CUDA tensor (fingerprint_views copies nothing; use fingerprint_clips for host clips)")
        hwc = tuple(clips[0].shape[1:]) == (64, 64, 3)
        frame_shape = (64, 64, 3) if hwc else (3, 64, 64)
        frame_strides = (192, 3, 1) if hwc else (4096, 64, 1)
        dtype, dev = clips[0].dtype, clips[0].device
        for i, c in enumerate(clips):
            if c.dim() != 4 or tuple(c.shape[1:]) != frame_shape:
                raise ValueError(f"clip {i} has shape {tuple(c.shape)}; all clips must be (T, 3, 64, 64), or all (T, 64, 64, 3)")
            if c.dtype != dtype:
                raise ValueError(f"clip {i} is {c.dtype}, clip 0 is {dtype}: clips must share one dtype")
            if c.device != dev:
                raise ValueError(f"clip {i} is on {c.device}, clip 0 on {dev}: clips must be on one device")
            if c.shape[0] < 1:
                raise ValueError(f"clip {i} has no frames")
            if tuple(c.stride()[1:]) != frame_strides:
                raise ValueError(f"clip {i} has strides {tuple(c.stride())}: each of its frames must be contiguous")
            if c.shape[0] > 1 and c.stride(0) < 12288:
                raise ValueError(f"clip {i} has a frame stride of {c.stride(0)} elements: frames must be a positive stride of "
                                 "at least one frame (12288 elements) apart")
        codes = {torch.uint8: _native.FRAME_U8, torch.bfloat16: _native.FRAME_BF16, torch.float32: _native.FRAME_F32}
        if dtype not in codes or (hwc and dtype != torch.uint8):
            raise ValueError(f"{dtype} clips: planar clips are uint8 / bfloat16 / float32, decoder-layout clips uint8")
        code = _native.FRAME_U8_HWC if hwc else codes[dtype]
        n = len(clips)
        lengths = [int(c.shape[0]) for c in clips]
        total = sum(lengths)
        esize = clips[0].element_size()
        # a one-frame clip has no frame stride to speak of (torch may report any value for it): dense
        pitches = [c.stride(0) * esize if c.shape[0] > 1 else 12288 * esize for c in clips]
        ptrs = (C.c_void_p * n)(*[c.data_ptr() for c in clips])
        pitch = (C.c_int64 * n)(*pitches)
        lens = (C.c_int32 * n)(*lengths)
        lib = _native.load()
        with torch.cuda.device(dev):
            weights = self._ensure_native(dev.index)
            # workspace and pipelines sized as in fingerprint_packed
            pass_frames = max(min(total, self.frames_per_pass), max(lengths))
            slices = max(1, min(int(self.pipelines), 4, -(-total // pass_frames)))
            ws = self._get_workspace(slices * (lib.vfp_forward_workspace_bytes(pass_frames, min(pass_frames, n)) + 1024), dev)
            emb = torch.empty((n, self.embedding_dim), dtype=torch.float32, device=dev)
            feats = torch.empty((total, 256), dtype=torch.float32, device=dev) if return_features else None
            stream = torch.cuda.current_stream(dev).cuda_stream
            lib.vfp_set_tuning(9, slices)
            rc = lib.vfp_forward_clips(
                C.c_void_p(weights), ptrs, pitch, lens, n, code, C.c_void_p(emb.data_ptr()),
                C.c_void_p(feats.data_ptr() if feats is not None else None), C.c_void_p(ws.data_ptr()), ws.numel(), C.c_void_p(stream),
            )
            _native.check(rc, "vfp_forward_clips")
        return (emb, feats) if return_features else emb

    # ------------------------------------------------------------------ reference-compatible forward
    def forward(self, video: torch.Tensor, return_features: bool = False):
        """Same contract as model.py:272-298, including the `(B,3,T,H,W)` layout sniff on `shape[1] == 3`."""
        if video.dim() != 5:
            raise ValueError(f"expected a 5-D video tensor, got shape {tuple(video.shape)}")
        if video.shape[1] == 3:  # reference quirk: a (B,T=3,3,H,W) input is also re-interpreted (model.py:283)
            video = video.permute(0, 2, 1, 3, 4)
        B, T = int(video.shape[0]), int(video.shape[1])
        frames = video.reshape(B * T, *video.shape[2:])
        out = self.fingerprint_packed(frames, [T] * B, return_features=return_features)
        if return_features:
            emb, feats = out
            return emb, feats.view(B, T, 256)
        return out

    def compute_loss(self, *a, **k):
        raise NotImplementedError("training (model.py:300-390) is outside the B200 inference hot path")


class Conv3DBlock(_ParamsOnly):
    """Parameter layout of model.py:393-403: `conv` (Conv3d), `bn` (BatchNorm3d)."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0):
        super().__init__()
        self.conv = nn.Conv3d(in_channels, out_channels, kernel_size, stride, padding)
        self.bn = nn.BatchNorm3d(out_channels)
        self.relu = nn.ReLU(inplace=True)


def _frame_code(frames: torch.Tensor) -> Tuple[int, torch.Tensor]:
    """Native frame type of planar (.., 3, 64, 64) frames: uint8 (0..255, scaled on the device), bf16, anything else as fp32."""
    if frames.dtype == torch.uint8:
        return _native.FRAME_U8, frames
    if frames.dtype == torch.bfloat16:
        return _native.FRAME_BF16, frames
    return _native.FRAME_F32, frames.float()


class VideoFingerprint3D(nn.Module):
    """The reference's 3-D CNN fingerprint model (model.py:406-512), inference only: same constructor arguments, same
    state_dict keys / shapes / default initialisation, same forward contract ((B,T,3,64,64) or (B,3,T,64,64) in [0,1] ->
    unit-norm (B, embedding_dim)); the compute is `vfp3d_forward` in libvfp_b200.so (im2col + tcgen05 GEMMs + a fused tail).
    `fingerprint_packed` / `fingerprint_clips` take clips of different lengths in one call (`vfp3d_forward_packed`);
    `fingerprint_views` takes device clips wherever they sit, including decoder-layout uint8 frames (`vfp3d_forward_clips`)."""

    def __init__(self, embedding_dim=256, frame_stride=32, dropout=0.2):
        super().__init__()
        self.frame_stride = frame_stride
        self.embedding_dim = embedding_dim
        self.encoder = nn.Sequential(
            Conv3DBlock(3, 16, kernel_size=(frame_stride, 5, 5), stride=(frame_stride, 2, 2), padding=(0, 2, 2)),
            Conv3DBlock(16, 32, kernel_size=(3, 3, 3), stride=(1, 2, 2), padding=(1, 1, 1)),
            Conv3DBlock(32, 64, kernel_size=(3, 3, 3), stride=(2, 2, 2), padding=(1, 1, 1)),
            Conv3DBlock(64, 128, kernel_size=(3, 3, 3), stride=(1, 2, 2), padding=(1, 1, 1)),
            nn.AdaptiveAvgPool3d((None, 1, 1)),
        )
        self.temporal_conv = nn.Conv1d(128, 128, kernel_size=3, padding=1)
        self.temporal_attention = nn.Conv1d(128, 1, kernel_size=1)
        self.projector = nn.Sequential(nn.Linear(128, 128), nn.ReLU(inplace=True), nn.Dropout(dropout), nn.Linear(128, embedding_dim))
        self.temperature = nn.Parameter(torch.ones(1) * 0.07)
        self._initialize_weights()
        self.clips_per_pass = 1024   # workspace: ~0.6 MB per 64-frame clip (layer-2 im2col + activations)
        self._native_weights: Optional[int] = None
        self._native_key: Optional[tuple] = None
        self._workspace: Optional[torch.Tensor] = None

    def _initialize_weights(self):
        """model.py:454-466 (same module order, so a fixed torch.manual_seed gives the reference's initial weights)."""
        for m in self.modules():
            if isinstance(m, nn.Conv3d):
                nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")
                if m.bias is not None:
                    nn.init.constant_(m.bias, 0)
            elif isinstance(m, nn.BatchNorm3d):
                nn.init.constant_(m.weight, 1)
                nn.init.constant_(m.bias, 0)
            elif isinstance(m, nn.Linear):
                nn.init.normal_(m.weight, 0, 0.01)
                nn.init.constant_(m.bias, 0)

    def _weights_key(self) -> tuple:
        return tuple((t.data_ptr(), t._version) for t in self.state_dict(keep_vars=True).values())

    def _release_native(self) -> None:
        if self._native_weights is not None:
            try:
                _native.load().vfp3d_weights_destroy(C.c_void_p(self._native_weights))
            except Exception:  # pragma: no cover - interpreter teardown
                pass
            self._native_weights = None
            self._native_key = None

    def __del__(self):  # pragma: no cover
        try:
            self._release_native()
        except Exception:
            pass

    def _ensure_native(self) -> int:
        key = (torch.cuda.current_device(),) + self._weights_key()   # the packed weights belong to one GPU
        if self._native_weights is not None and key == self._native_key:
            return self._native_weights
        self._release_native()
        lib = _native.load()
        host = {k: v.detach().to("cpu").contiguous() for k, v in self.state_dict().items()}
        host = {k: (v.float() if v.is_floating_point() else v) for k, v in host.items()}
        descs = (_native.TensorDesc * len(host))()
        for i, (k, v) in enumerate(host.items()):
            descs[i] = _native.TensorDesc(k.encode(), v.data_ptr(), v.numel())
        handle = C.c_void_p()
        _native.check(lib.vfp3d_weights_create(descs, len(host), int(self.frame_stride), C.byref(handle)), "vfp3d_weights_create")
        self._native_weights = handle.value
        self._native_key = key
        return self._native_weights

    @torch.no_grad()
    def forward(self, video: torch.Tensor):
        """model.py:468-509: (B,T,3,H,W) is detected by `shape[2] == 3`, anything else is taken as (B,3,T,H,W)."""
        _native.require_cuda()
        if self.training:
            raise RuntimeError("inference only: call .eval() first")
        if video.dim() != 5:
            raise ValueError(f"expected a 5-D video tensor, got shape {tuple(video.shape)}")
        if video.shape[2] != 3:      # (B, C, T, H, W) -> (B, T, C, H, W): the kernels read per-frame planar images
            video = video.permute(0, 2, 1, 3, 4)
        B, T = int(video.shape[0]), int(video.shape[1])
        if tuple(video.shape[2:]) != (3, 64, 64):
            raise ValueError("the sm_100a kernels are specialised for 3 x 64 x 64 frames")
        if not video.is_cuda:
            video = video.cuda()
        code, video = _frame_code(video)
        frames = video.contiguous()
        dev = frames.device
        lib = _native.load()
        with torch.cuda.device(dev):
            weights = self._ensure_native()
            per = max(1, min(B, self.clips_per_pass))
            ws = self._get_workspace(lib.vfp3d_forward_workspace_bytes(C.c_void_p(weights), per, T), dev)
            emb = torch.empty((B, self.embedding_dim), dtype=torch.float32, device=dev)
            rc = lib.vfp3d_forward(C.c_void_p(weights), C.c_void_p(frames.data_ptr()), code, B, T, C.c_void_p(emb.data_ptr()),
                                   C.c_void_p(ws.data_ptr()), ws.numel(), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
            _native.check(rc, "vfp3d_forward")
        return emb

    def _get_workspace(self, nbytes: int, dev) -> torch.Tensor:
        """One cached device workspace, grown on demand and shared by `forward` and `fingerprint_packed`."""
        if self._workspace is None or self._workspace.numel() < nbytes or self._workspace.device != dev:
            self._workspace = None
            self._workspace = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        return self._workspace

    # ------------------------------------------------------------------ packed (variable-length) entry
    @torch.no_grad()
    def fingerprint_packed(self, frames: torch.Tensor, lengths: Sequence[int]) -> torch.Tensor:
        """frames: (sum T, 3, 64, 64) uint8 / bf16 / fp32, clips back to back (host frames are uploaded once); lengths: frames
        per clip, each 1 .. 64 * frame_stride. Returns (n, embedding_dim) fp32 on the device; row i has exactly the bits
        `forward` gives for clip i alone. Passes hold about `clips_per_pass` clips."""
        _native.require_cuda()
        if self.training:
            raise RuntimeError("inference only: call .eval() first")
        lengths = [int(t) for t in lengths]
        n, total = len(lengths), sum(lengths)
        if frames.dim() != 4 or tuple(frames.shape[1:]) != (3, 64, 64) or frames.shape[0] != total:
            raise ValueError(f"frames must be (sum(lengths)={total}, 3, 64, 64), got {tuple(frames.shape)}")
        if not frames.is_cuda:
            frames = frames.cuda()
        code, frames = _frame_code(frames)
        frames = frames.contiguous()
        dev = frames.device
        lib = _native.load()
        with torch.cuda.device(dev):
            weights = self._ensure_native()
            cu = (C.c_int32 * (n + 1))()
            acc = 0
            for i, t in enumerate(lengths):
                cu[i] = acc
                acc += t
            cu[n] = acc
            ws = self._packed_workspace(lib, weights, lengths, dev)
            emb = torch.empty((n, self.embedding_dim), dtype=torch.float32, device=dev)
            rc = lib.vfp3d_forward_packed(C.c_void_p(weights), C.c_void_p(frames.data_ptr()), code, C.cast(cu, C.c_void_p), n,
                                          C.c_void_p(emb.data_ptr()), C.c_void_p(ws.data_ptr()), ws.numel(),
                                          C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
            _native.check(rc, "vfp3d_forward_packed")
        return emb

    def _packed_workspace(self, lib, weights: int, lengths: List[int], dev) -> torch.Tensor:
        """Workspace for passes of clips_per_pass clips of the batch's mean length (at least the longest clip)."""
        n, total = len(lengths), sum(lengths)
        per = max(1, min(n, self.clips_per_pass))
        pass_frames = total if per == n else max(max(lengths), -(-total * per // n))
        return self._get_workspace(lib.vfp3d_forward_packed_workspace_bytes(C.c_void_p(weights), max(1, pass_frames), per), dev)

    def fingerprint_clips(self, clips: Sequence[torch.Tensor]) -> torch.Tensor:
        """List of (T_i, 3, 64, 64) clips of one dtype -> (n, D) embeddings, one packed launch sequence (no padding, no masks).
        Clips that are all on one device (or all on the host, then uploaded once) are concatenated there; for clips already
        on the device, `fingerprint_views` gives the same bits without that copy."""
        if len({c.dtype for c in clips}) > 1:
            raise ValueError("clips must share one dtype (uint8 frames are scaled by 1/255, float frames are not)")
        lengths = [int(c.shape[0]) for c in clips]
        devices = {c.device for c in clips}
        if len(devices) > 1:
            dev = next(d for d in devices if d.type == "cuda")
            clips = [c.to(dev) for c in clips]
        return self.fingerprint_packed(torch.cat(list(clips), dim=0), lengths)

    @torch.no_grad()
    def fingerprint_views(self, clips: Sequence[torch.Tensor]) -> torch.Tensor:
        """Device clips wherever they sit -> (n, embedding_dim) fp32 on their device, without copying a frame: each clip is a
        contiguous CUDA tensor (T_i, 3, 64, 64) uint8 / bf16 / fp32, or decoder-layout (T_i, 64, 64, 3) uint8 (what
        `preprocess_frames_device` returns), all of one dtype and layout on one device. Views such as `frames[s:s + L]` of
        one buffer qualify, overlapping or repeated ones too. Row i has exactly the bits `forward` gives for clip i alone
        (HWC and planar uint8 frames give the same bits). Raises ValueError rather than copying anything."""
        _native.require_cuda()
        if self.training:
            raise RuntimeError("inference only: call .eval() first")
        clips = list(clips)
        if not clips:
            raise ValueError("fingerprint_views needs at least one clip")
        for i, c in enumerate(clips):
            if not isinstance(c, torch.Tensor) or not c.is_cuda:
                raise ValueError(f"clip {i} is not a CUDA tensor (fingerprint_views copies nothing; use fingerprint_clips for host clips)")
            if not c.is_contiguous():
                raise ValueError(f"clip {i} is not contiguous (its frames must be consecutive in memory)")
        hwc = tuple(clips[0].shape[1:]) == (64, 64, 3)
        dtype, dev = clips[0].dtype, clips[0].device
        for i, c in enumerate(clips):
            if c.dim() != 4 or tuple(c.shape[1:]) != ((64, 64, 3) if hwc else (3, 64, 64)):
                raise ValueError(f"clip {i} has shape {tuple(c.shape)}; all clips must be (T, 3, 64, 64), or all (T, 64, 64, 3)")
            if c.dtype != dtype:
                raise ValueError(f"clip {i} is {c.dtype}, clip 0 is {dtype}: clips must share one dtype")
            if c.device != dev:
                raise ValueError(f"clip {i} is on {c.device}, clip 0 on {dev}: clips must be on one device")
        codes = {torch.uint8: _native.FRAME_U8, torch.bfloat16: _native.FRAME_BF16, torch.float32: _native.FRAME_F32}
        if dtype not in codes or (hwc and dtype != torch.uint8):
            raise ValueError(f"{dtype} clips: planar clips are uint8 / bfloat16 / float32, decoder-layout clips uint8")
        code = _native.FRAME_U8_HWC if hwc else codes[dtype]
        n = len(clips)
        lengths = [int(c.shape[0]) for c in clips]
        ptrs = (C.c_void_p * n)(*[c.data_ptr() for c in clips])
        lens = (C.c_int32 * n)(*lengths)
        lib = _native.load()
        with torch.cuda.device(dev):
            weights = self._ensure_native()
            ws = self._packed_workspace(lib, weights, lengths, dev)
            emb = torch.empty((n, self.embedding_dim), dtype=torch.float32, device=dev)
            rc = lib.vfp3d_forward_clips(C.c_void_p(weights), ptrs, lens, n, code, C.c_void_p(emb.data_ptr()), C.c_void_p(ws.data_ptr()),
                                         ws.numel(), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
            _native.check(rc, "vfp3d_forward_clips")
        return emb

    def compute_loss(self, *a, **k):
        raise NotImplementedError("training (model.py:514-582) is outside the B200 inference hot path")


def create_model(model_type: str = "attention", **kwargs) -> nn.Module:
    """Factory with the reference's signature and error behaviour (model.py:585-610)."""
    if model_type == "attention":
        return VideoFingerprintAttention(
            spatial_dim=kwargs.get("spatial_dim", 128),
            temporal_dim=kwargs.get("temporal_dim", 256),
            embedding_dim=kwargs.get("embedding_dim", 256),
            num_attention_blocks=kwargs.get("num_attention_blocks", 4),
        )
    if model_type in ("3d", "cnn3d"):
        return VideoFingerprint3D(
            embedding_dim=kwargs.get("embedding_dim", 256),
            frame_stride=kwargs.get("frame_stride", 16),
            dropout=kwargs.get("dropout", 0.2),
        )
    raise ValueError(f"Unknown model type: {model_type}")
