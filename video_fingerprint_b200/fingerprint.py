"""Host-side mirror of the reference scanner's hot-path methods (/root/reference/fingerprint.py:15-577),
with the device work delegated to libvfp_b200.so.

Same names, argument meaning and return structures as the reference:

* ``VideoFingerprintScanner(model_path, device="cuda")``          fingerprint.py:20-72  (checkpoint -> model)
* ``scanner.extract_fingerprint_from_frames(frames)``             fingerprint.py:232-270 minus PyAV decode
* ``scanner.find_duplicates(fingerprints, similarity_threshold=0.95, use_faiss=True)``   :450-480
* ``scanner._find_duplicates_direct`` / ``_find_duplicates_faiss``                       :482-548
* ``scanner.save_results(fingerprints, duplicate_groups, output_path)``                  :550-577

Video decode (PyAV), directory walking and report printing are out of scope (SURVEY.md section 2); frames
arrive pre-decoded. There is no CPU fallback: without a CUDA device these methods raise.
"""
from __future__ import annotations

import ctypes as C
import json
from datetime import datetime
from pathlib import Path
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _native
from .model import create_model

MAX_SEARCH_DIM = 512
_BF16_DOT_BOUND = 2.0 ** -8  # |<q,d> - <bf16(q),bf16(d)>| <= 2^-8 |q||d| (two roundings of 2^-9 each, Cauchy-Schwarz)


# ----------------------------------------------------------------------------------------------
# device primitives
# ----------------------------------------------------------------------------------------------
def _as_device_f32(x, device=None) -> torch.Tensor:
    _native.require_cuda()
    if isinstance(x, np.ndarray):
        x = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32))
    if not x.is_cuda:
        x = x.cuda(device) if device is not None else x.cuda()
    return x.float().contiguous()


def _search_operands(db, q=None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Device fp32 operands of the join and the top-k search: `db` (n_db, dim) and `q` (n_q, dim), `q` is `db` when None.
    Raises ValueError, before anything is copied or launched, unless both are 2-D with the same width of 1 to 512 columns.
    The library takes widths that are multiples of 16; any other width is zero-padded to the next one in the device copy.
    Every added product is +0, so scores are those of the unpadded rows up to summation order, and so is the screen bound
    (padding changes no norm)."""
    shapes = [("db", tuple(db.shape))] + ([] if q is None else [("q", tuple(q.shape))])
    for name, shape in shapes:
        if len(shape) != 2:
            raise ValueError(f"{name} must be a 2-D (rows, dim) array, got shape {shape}")
    dim = shapes[0][1][1]
    if q is not None and shapes[1][1][1] != dim:
        raise ValueError(f"q and db must have the same width, got {shapes[1][1][1]} and {dim}")
    if not 1 <= dim <= MAX_SEARCH_DIM:
        raise ValueError(f"embedding width {dim} is not supported (1 to {MAX_SEARCH_DIM} columns)")
    db = _as_device_f32(db)
    q = db if q is None else _as_device_f32(q, db.device)
    pad = -dim % 16
    if pad:
        self_search = q is db
        db = torch.nn.functional.pad(db, (0, pad))
        q = db if self_search else torch.nn.functional.pad(q, (0, pad))
    return db, q


def screen_margin(q: torch.Tensor, db: torch.Tensor) -> float:
    """Bound on the bf16 tensor-core screen error for these operands (see include/vfp_b200.h)."""
    nq = float(torch.linalg.vector_norm(q, dim=1).max())
    nd = nq if db is q else float(torch.linalg.vector_norm(db, dim=1).max())
    return _BF16_DOT_BOUND * nq * nd * 1.02 + 1e-6


_MAX_CANDIDATES = 1 << 26  # screen candidates buffered per native call (12 bytes each); larger joins are split by query rows


def threshold_join_device(
    db: torch.Tensor, thr: float, q: Optional[torch.Tensor] = None, q_row0: int = 0, capacity: Optional[int] = None
) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """All (i, j, s) with <q_i, db_j> >= thr (fp32), as device tensors in no particular order. `db` is (n_db, dim) and `q`
    (n_q, dim), `q` = `db` when None, for any width dim of 1 to 512 (see `_search_operands`).
    i is offset by q_row0 (global row index of a row-block shard). Retries with a larger buffer on overflow; when a
    low threshold or a heavily duplicated corpus produces more candidates than `_MAX_CANDIDATES`, the query rows are
    split into blocks (the reference degrades the same way, one row at a time, fingerprint.py:497-499)."""
    db, q = _search_operands(db, q)
    lib = _native.load()
    dim = db.shape[1]
    margin = screen_margin(q, db)
    dev = db.device

    def run(qb: torch.Tensor, row0: int, cap: int):
        n_q, n_db = qb.shape[0], db.shape[0]
        cand_cap = min(4 * cap, _MAX_CANDIDATES)
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            while True:
                ws = torch.empty(lib.vfp_join_workspace_bytes_dim(n_q, n_db, cand_cap, dim), dtype=torch.uint8, device=dev)
                out_i = torch.empty(cap, dtype=torch.int32, device=dev)
                out_j = torch.empty(cap, dtype=torch.int32, device=dev)
                out_s = torch.empty(cap, dtype=torch.float32, device=dev)
                counts = torch.zeros(2, dtype=torch.int64, device=dev)
                rc = lib.vfp_join_threshold(
                    C.c_void_p(qb.data_ptr()), C.c_void_p(db.data_ptr()), n_q, n_db, dim, int(row0), float(thr), float(margin),
                    C.c_void_p(out_i.data_ptr()), C.c_void_p(out_j.data_ptr()), C.c_void_p(out_s.data_ptr()), cap,
                    C.c_void_p(counts.data_ptr()), C.c_void_p(ws.data_ptr()), ws.numel(), C.c_void_p(stream),
                )
                _native.check(rc, "vfp_join_threshold")
                n_out, n_cand = (int(v) for v in counts.tolist())
                if n_cand > cand_cap:  # screen overflow: the candidate count is now known
                    if n_cand + 1024 > _MAX_CANDIDATES and n_q > 1:
                        return None  # too many for one call: the caller splits the query block
                    cand_cap = n_cand + 1024
                    cap = max(cap, min(n_cand, 4 * cap))
                    continue
                if n_out > cap:
                    cap = n_out + 1024
                    continue
                return out_i[:n_out], out_j[:n_out], out_s[:n_out]

    def solve(lo: int, hi: int, cap: int):
        # self joins pass the SAME tensor for q and db when the block is the whole matrix (the library then converts it once)
        qb = q if (lo == 0 and hi == q.shape[0]) else q[lo:hi]
        out = run(qb, q_row0 + lo, cap)
        if out is not None:
            return [out]
        mid = (lo + hi) // 2
        return solve(lo, mid, cap) + solve(mid, hi, cap)

    parts = solve(0, q.shape[0], int(capacity) if capacity else max(4096, 8 * q.shape[0]))
    if len(parts) == 1:
        return parts[0]
    return tuple(torch.cat([p[c] for p in parts]) for c in range(3))


def threshold_join(db, thr: float, q=None, q_row0: int = 0) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """Host view of the join, sorted by (i, j) - the order np.where visits a row (fingerprint.py:499)."""
    i, j, s = threshold_join_device(db, thr, q, q_row0)
    i, j, s = i.cpu().numpy().astype(np.int64), j.cpu().numpy().astype(np.int64), s.cpu().numpy()
    order = np.lexsort((j, i))
    return i[order], j[order], s[order]


def duplicate_pairs(db, thr: float) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """The pairs the greedy grouping (fingerprint.py:495-511) can act on, sorted by (i, j): the self join restricted to rows
    with at least two hits. A row whose only hit is itself can neither seed a group (`len(similar) > 1`, :502) nor be marked
    by one, and at a million videos such rows are all but a few percent of the pair list - so they are dropped and the rest
    is ordered on the device (one bincount and one sort over the pair list) instead of on the host: 1 M embeddings, 1.08 M
    pairs: D2H + lexsort + grouping 300 ms -> a few ms next to the 175 ms join. `db` is (n, dim), 1 <= dim <= 512."""
    db, _ = _search_operands(db)
    n = db.shape[0]
    i, j, s = threshold_join_device(db, thr)
    i64 = i.to(torch.int64)
    hits = torch.bincount(i64, minlength=n)
    keep = hits[i64] >= 2
    i64, j64, s = i64[keep], j.to(torch.int64)[keep], s[keep]
    order = torch.argsort(i64 * n + j64)
    return i64[order].cpu().numpy(), j64[order].cpu().numpy(), s[order].cpu().numpy()


def topk_inner_product(q, db, k: int) -> Tuple[np.ndarray, np.ndarray]:
    """Exact flat-IP top-k: (scores (n_q,k) fp32 descending, indices (n_q,k) int64, ties by ascending index). `q` (n_q, dim)
    and `db` (n_db, dim) for any width dim of 1 to 512."""
    S, I = topk_inner_product_device(q, db, k)
    return S.cpu().numpy(), I.cpu().numpy()


def topk_inner_product_device(q, db, k: int) -> Tuple[torch.Tensor, torch.Tensor]:
    db, q = _search_operands(db, q)
    lib = _native.load()
    n_q, n_db, dim = q.shape[0], db.shape[0], db.shape[1]
    k = min(int(k), n_db)
    dev = db.device
    with torch.cuda.device(dev):
        ws = torch.empty(lib.vfp_topk_workspace_bytes_dim(n_q, n_db, k, dim), dtype=torch.uint8, device=dev)
        S = torch.empty((n_q, k), dtype=torch.float32, device=dev)
        I = torch.empty((n_q, k), dtype=torch.int64, device=dev)
        flags = torch.zeros(2, dtype=torch.int64, device=dev)
        rc = lib.vfp_topk_ip(
            C.c_void_p(q.data_ptr()), C.c_void_p(db.data_ptr()), n_q, n_db, dim, k, float(screen_margin(q, db)),
            C.c_void_p(S.data_ptr()), C.c_void_p(I.data_ptr()), C.c_void_p(flags.data_ptr()), C.c_void_p(ws.data_ptr()),
            ws.numel(), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream),
        )
        _native.check(rc, "vfp_topk_ip")
    return S, I


def preprocess_frames_device(frames, device=None) -> torch.Tensor:
    """Device restatement of ``_preprocess_frames`` (fingerprint.py:186-214) up to, not including, the ``/ 255`` and the
    HWC->CHW permute (both are fused into the stem kernel): decoded frames ``(T, H, W, 3)`` uint8 (a tensor, an array or a
    list of equally sized arrays) -> ``(T, 64, 64, 3)`` uint8 on the device, bit-exact with cv2.resize(INTER_AREA) +
    centre crop. Feed the result to ``model.fingerprint_packed(out, [T])``."""
    _native.require_cuda()
    lib = _native.load()
    if isinstance(frames, (list, tuple)):
        frames = np.stack(frames)
    if isinstance(frames, np.ndarray):
        frames = torch.from_numpy(np.ascontiguousarray(frames))
    if frames.dtype != torch.uint8 or frames.dim() != 4 or frames.shape[3] != 3:
        raise ValueError("frames must be uint8 (T, H, W, 3)")
    if not frames.is_cuda:
        frames = frames.cuda(device) if device is not None else frames.cuda()
    frames = frames.contiguous()
    t, h, w, _ = frames.shape
    dev = frames.device
    with torch.cuda.device(dev):
        out = torch.empty((t, 64, 64, 3), dtype=torch.uint8, device=dev)
        ws = torch.empty(lib.vfp_preprocess_workspace_bytes(h, w), dtype=torch.uint8, device=dev)
        st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        for f0 in range(0, t, 65535):
            n = min(65535, t - f0)
            _native.check(lib.vfp_preprocess_frames(C.c_void_p(frames[f0:].data_ptr()), n, h, w, C.c_void_p(out[f0:].data_ptr()),
                                                    C.c_void_p(ws.data_ptr()), ws.numel(), st), "vfp_preprocess_frames")
    return out


# ----------------------------------------------------------------------------------------------
# greedy grouping (host; sequential by definition - seeds are visited in ascending index order)
# ----------------------------------------------------------------------------------------------
def group_pairs_direct(n: int, pi: np.ndarray, pj: np.ndarray, ps: np.ndarray) -> List[List[Tuple[int, float]]]:
    """fingerprint.py:495-511 over a (row, col)-sorted pair list instead of a dense N x N matrix. Only rows
    with at least two hits can seed or mark anything, so only those are visited."""
    if len(pi) == 0:
        return []
    rows, starts, counts = np.unique(pi, return_index=True, return_counts=True)
    processed = np.zeros(n, dtype=bool)
    groups: List[List[Tuple[int, float]]] = []
    for r, st, ct in zip(rows.tolist(), starts.tolist(), counts.tolist()):
        if ct <= 1 or processed[r]:
            continue
        cols = pj[st : st + ct]
        fresh = ~processed[cols]
        members = cols[fresh]
        processed[members] = True
        if len(members) > 1:
            sims = ps[st : st + ct][fresh]
            groups.append([(int(m), float(s)) for m, s in zip(members, sims)])
    return groups


def group_pairs_topk(S: np.ndarray, I: np.ndarray, thr: float) -> List[List[Tuple[int, float]]]:
    """fingerprint.py:530-546: each unprocessed row claims its unprocessed top-k neighbours above thr."""
    n = S.shape[0]
    processed = np.zeros(max(n, int(I.max()) + 1 if I.size else n), dtype=bool)
    # the reference compares np.float32 scores with the Python float threshold (fingerprint.py:540), which NumPy 2
    # evaluates in float32: np.float32(0.95) >= 0.95 is True there. One mask, computed once, keeps exactly that rule.
    above = np.asarray(S, dtype=np.float32) >= np.float32(thr)
    hit_rows = np.nonzero(above.any(axis=1))[0]
    groups: List[List[Tuple[int, float]]] = []
    for r in hit_rows.tolist():
        if processed[r]:
            continue
        g = []
        for sim, idx, ok in zip(S[r].tolist(), I[r].tolist(), above[r].tolist()):
            if ok and not processed[idx]:
                processed[idx] = True
                g.append((int(idx), float(sim)))
        if len(g) > 1:
            groups.append(g)
    return groups


# ----------------------------------------------------------------------------------------------
# scanner
# ----------------------------------------------------------------------------------------------
class VideoFingerprintScanner:
    """Fingerprint extraction + duplicate search on pre-decoded frames."""

    def __init__(self, model_path: Optional[str] = None, device: str = "cuda", batch_size: int = 1, model=None, config: Optional[dict] = None):
        _native.require_cuda()  # the reference silently falls back to CPU (fingerprint.py:27); this build refuses
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _native.NativeError(f"device {device!r}: video_fingerprint_b200 runs on CUDA devices only (no CPU fallback)")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.batch_size = batch_size
        if model is not None:
            self.model, self.config = model, dict(config or {})
        else:
            self.model, self.config = self._load_model(model_path)
        self.model.eval()
        self.model_type = self.config.get("model_type", "attention")
        self.frame_size = self.config.get("frame_size", 64)
        self.max_frames = self.config.get("max_frames", 500)
        self.embedding_dim = self.config.get("embedding_dim", 256)

    def _load_model(self, model_path: str):
        """Checkpoint contract of fingerprint.py:51-72: keys `model_state_dict` and optional `config`."""
        checkpoint = torch.load(model_path, map_location="cpu")
        config = checkpoint.get("config", {})
        model = create_model(
            model_type=config.get("model_type", "attention"),
            spatial_dim=config.get("spatial_dim", 128),
            temporal_dim=config.get("temporal_dim", 256),
            embedding_dim=config.get("embedding_dim", 256),
            num_attention_blocks=config.get("num_attention_blocks", 4),
            frame_stride=config.get("frame_stride", 32),
        )
        model.load_state_dict(checkpoint["model_state_dict"])
        return model, config

    # -- per-video semantics (fingerprint.py:232-270) ---------------------------------------------
    def subsample(self, total_frames: int) -> List[int]:
        """Indices of the decoded frames the reference keeps (fingerprint.py:90-101)."""
        skip = max(1, total_frames // self.max_frames) if total_frames > self.max_frames else 1
        return list(range(0, total_frames, skip))[: self.max_frames]

    def _preprocess_frames(self, frames) -> torch.Tensor:
        """fingerprint.py:186-214 on the device: decoded (H, W, 3) uint8 frames -> the (T, 3, 64, 64) float clip in [0, 1] the
        reference returns (cv2 INTER_AREA + centre crop, bit-exact). ``extract_fingerprint_from_decoded`` skips the float
        round trip and hands the uint8 result straight to the stem kernel."""
        return preprocess_frames_device(frames).permute(0, 3, 1, 2).float() / 255.0

    def extract_fingerprint_from_decoded(self, frames) -> Optional[np.ndarray]:
        """Decoded frames of one video -> embedding: preprocessing and forward both on the device (fingerprint.py:232-270
        minus the PyAV decode). Fewer than 10 frames -> None like the reference (fingerprint.py:238-240)."""
        keep = self.subsample(len(frames))            # fingerprint.py:90-101: every skip-th frame, at most max_frames
        if len(keep) < 10:
            return None
        if len(keep) != len(frames):
            frames = frames[keep] if isinstance(frames, (np.ndarray, torch.Tensor)) else [frames[i] for i in keep]
        u8 = preprocess_frames_device(frames, self.device)
        emb = self.model.fingerprint_packed(u8, [u8.shape[0]])
        return emb[0].cpu().numpy()

    def extract_fingerprints_from_decoded(self, videos) -> List[Optional[np.ndarray]]:
        """Batched form of `extract_fingerprint_from_decoded`: decoded videos, each (T_v, H_v, W_v, 3) uint8 at its own
        resolution as an array, a tensor or a list of frames -> one embedding per video, or None where fewer than 10 frames
        are kept. Only the frames `subsample` keeps (a strided slice of the caller's frames) are uploaded and preprocessed on
        the device; the decoder-layout buffers of ALL videos then go through one `fingerprint_views` call. Row for row
        equal to `extract_fingerprint_from_decoded` on each video."""
        _native.require_cuda()
        views: List[torch.Tensor] = []
        rows: List[int] = []   # videos with a row in the result of fingerprint_views
        for v, frames in enumerate(videos):
            keep = self.subsample(len(frames))   # range(0, total, skip)[:max_frames]
            if len(keep) < 10:
                continue
            skip = keep[1] - keep[0]
            views.append(preprocess_frames_device(frames[: keep[-1] + 1 : skip], self.device))
            rows.append(v)
        result: List[Optional[np.ndarray]] = [None] * len(videos)
        if views:
            emb = self.model.fingerprint_views(views).cpu().numpy()
            for row, v in enumerate(rows):
                result[v] = emb[row]
        return result

    def window_starts_3d(self, total_frames: int) -> List[int]:
        """Start frames of the clip_length windows the 3-D scanner path fingerprints (fingerprint.py:293-303); one window
        starting at 0 (taking every frame) when the video is not longer than clip_length (fingerprint.py:280-291)."""
        clip_length = self.config.get("clip_length", 128)
        if total_frames <= clip_length:
            return [0]
        num_windows = min(5, max(3, total_frames // (clip_length * 2)))
        stride = (total_frames - clip_length) // (num_windows - 1) if num_windows > 1 else 0
        return [i * stride for i in range(num_windows)]

    def extract_fingerprint_3d_from_frames(self, frames: torch.Tensor) -> Optional[np.ndarray]:
        """3-D model path of the scanner (fingerprint.py:272-320) on preprocessed frames (T, 3, 64, 64): < 10 frames -> None;
        a video of at most clip_length frames is one clip; longer ones are 3..5 windows of clip_length frames whose embeddings
        are averaged and re-normalised. All windows go through ONE batched forward."""
        total = int(frames.shape[0])
        if total < 10:
            return None
        clip_length = self.config.get("clip_length", 128)
        if total <= clip_length:
            return self.model(frames.unsqueeze(0))[0].cpu().numpy()
        windows = torch.stack([frames[s : s + clip_length] for s in self.window_starts_3d(total)])
        emb = self.model(windows).cpu().numpy()
        final = np.mean(emb, axis=0)
        return final / np.linalg.norm(final)

    def extract_fingerprints_3d_from_frames(self, videos: Sequence[torch.Tensor]) -> List[Optional[np.ndarray]]:
        """Batched form of the reference's per-video 3-D scan loop (fingerprint.py:272-320, driven per video at :377-434):
        preprocessed (T_v, 3, 64, 64) videos of one dtype -> one embedding per video, with the rule of
        `extract_fingerprint_3d_from_frames` (< 10 frames -> None; at most clip_length frames -> one clip of the video's own
        length; longer -> the window_starts_3d windows, averaged and re-normalised). The clips of ALL videos go through one
        packed forward, so a corpus of short videos of many different lengths costs one launch sequence, not one per video."""
        clip_length = self.config.get("clip_length", 128)
        pieces: List[torch.Tensor] = []
        spans: List[Tuple[int, int, int]] = []   # (video, first row, rows) in the packed result
        for v, frames in enumerate(videos):
            total = int(frames.shape[0])
            if total < 10:
                continue
            starts = self.window_starts_3d(total)
            span = total if total <= clip_length else clip_length
            spans.append((v, len(pieces), len(starts)))
            pieces += [frames[s : s + span] for s in starts]
        result: List[Optional[np.ndarray]] = [None] * len(videos)
        if not pieces:
            return result
        emb = self.model.fingerprint_clips(pieces).cpu().numpy()
        self._combine_windows_3d(emb, spans, [int(v.shape[0]) for v in videos], result)
        return result

    def _combine_windows_3d(self, emb: np.ndarray, spans, totals: List[int], result: List[Optional[np.ndarray]]) -> None:
        """result[v] for every (video, first row, rows) span: the row itself for a video of at most clip_length frames, else
        the mean of its window rows, re-normalised (fingerprint.py:305-320)."""
        clip_length = self.config.get("clip_length", 128)
        for v, row, k in spans:
            if totals[v] <= clip_length:
                result[v] = emb[row]
            else:
                final = np.mean(np.ascontiguousarray(emb[row : row + k]), axis=0)
                result[v] = final / np.linalg.norm(final)

    def extract_fingerprints_3d_from_decoded(self, videos) -> List[Optional[np.ndarray]]:
        """Decoded videos -> one embedding (or None) per video with the rule of `extract_fingerprint_3d_from_frames`, with
        preprocessing and forward both on the device. Each video is (T_v, H_v, W_v, 3) uint8 at its own resolution, as an
        array, a tensor or a list of frames (what `preprocess_frames_device` accepts). Only frames inside some window are
        uploaded and resized (a 1 000-frame video at clip_length 128 needs at most 5 x 128), one decoder-layout buffer per run
        of overlapping windows; the windows of ALL videos are views into those buffers and go through one `fingerprint_views`
        call."""
        _native.require_cuda()
        clip_length = self.config.get("clip_length", 128)
        views: List[torch.Tensor] = []
        spans: List[Tuple[int, int, int]] = []   # (video, first row, rows) in the result of fingerprint_views
        totals = [len(frames) for frames in videos]
        for v, frames in enumerate(videos):
            total = totals[v]
            if total < 10:
                continue
            starts = self.window_starts_3d(total)
            span = min(total, clip_length)
            runs: List[List[int]] = []   # overlapping windows merged into runs [a, b) of frames
            for s in starts:
                if runs and s <= runs[-1][1]:
                    runs[-1][1] = s + span
                else:
                    runs.append([s, s + span])
            # a slice of an array or tensor is a view: each run is uploaded straight from the caller's frames, no host gather
            bufs = [(a, b, preprocess_frames_device(frames[a:b], self.device)) for a, b in runs]
            spans.append((v, len(views), len(starts)))
            views += [u8[s - a : s - a + span] for s in starts for a, b, u8 in bufs if a <= s < b]
        result: List[Optional[np.ndarray]] = [None] * len(totals)
        if not views:
            return result
        emb = self.model.fingerprint_views(views).cpu().numpy()
        self._combine_windows_3d(emb, spans, totals, result)
        return result

    def extract_fingerprint_3d_from_decoded(self, frames) -> Optional[np.ndarray]:
        """One decoded video (T, H, W, 3) uint8 -> its 3-D embedding, or None below 10 frames."""
        return self.extract_fingerprints_3d_from_decoded([frames])[0]

    def extract_fingerprint_from_frames(self, clip: torch.Tensor) -> Optional[np.ndarray]:
        """clip: (T,3,64,64) preprocessed frames (what _preprocess_frames returns). <10 frames -> None."""
        out = self.extract_fingerprints_from_frames([clip])
        return out[0]

    def extract_fingerprints_from_frames(self, clips: Sequence[torch.Tensor]) -> List[Optional[np.ndarray]]:
        """Batched form of the scanner loop: all clips with >= 10 frames go through one packed forward."""
        keep = [i for i, c in enumerate(clips) if c.shape[0] >= 10]
        for i, c in enumerate(clips):
            if c.shape[0] < 10:
                print(f"Video too short: clip {i} ({c.shape[0]} frames)")
        result: List[Optional[np.ndarray]] = [None] * len(clips)
        if keep:
            emb = self.model.fingerprint_clips([clips[i][: self.max_frames].to(self.device) for i in keep]).cpu().numpy()
            for row, i in enumerate(keep):
                result[i] = emb[row]
        return result

    # -- duplicate search (fingerprint.py:450-548) ------------------------------------------------
    def find_duplicates(self, fingerprints: Dict[str, dict], similarity_threshold: float = 0.95, use_faiss: bool = True) -> List[List[dict]]:
        if len(fingerprints) < 2:
            return []
        print(f"\nSearching for duplicates (threshold: {similarity_threshold})...")
        paths = list(fingerprints.keys())
        embeddings = np.array([fingerprints[p]["embedding"] for p in paths]).astype("float32")
        if use_faiss and len(embeddings) > 100:
            duplicate_groups = self._find_duplicates_faiss(embeddings, paths, fingerprints, similarity_threshold)
        else:
            duplicate_groups = self._find_duplicates_direct(embeddings, paths, fingerprints, similarity_threshold)
        for group in duplicate_groups:
            hashes = [item["file_hash"] for item in group]
            for item in group:
                item["exact_duplicate"] = hashes.count(item["file_hash"]) > 1
        return duplicate_groups

    @staticmethod
    def _materialise(groups, paths, fingerprints) -> List[List[dict]]:
        out = []
        for g in groups:
            items = []
            for idx, sim in g:
                item = fingerprints[paths[idx]].copy()
                item["similarity"] = sim
                items.append(item)
            out.append(items)
        return out

    def _find_duplicates_direct(self, embeddings, paths, fingerprints, threshold) -> List[List[dict]]:
        pi, pj, ps = duplicate_pairs(_as_device_f32(embeddings, getattr(self, "device", None)), threshold)
        return self._materialise(group_pairs_direct(len(embeddings), pi, pj, ps), paths, fingerprints)

    def _find_duplicates_faiss(self, embeddings, paths, fingerprints, threshold) -> List[List[dict]]:
        k = min(20, len(embeddings))
        E = _as_device_f32(embeddings, getattr(self, "device", None))
        S, I = topk_inner_product(E, E, k)
        return self._materialise(group_pairs_topk(S, I, threshold), paths, fingerprints)

    # -- JSON output (fingerprint.py:550-577; the reference crashes on np.float32 / ndarray members) -
    def save_results(self, fingerprints: Dict[str, dict], duplicate_groups: List[List[dict]], output_path: Path):
        def plain(v):
            if isinstance(v, np.ndarray):
                return v.tolist()
            if isinstance(v, np.generic):
                return v.item()
            return v

        results = {
            "metadata": {
                "scan_date": datetime.now().isoformat(),
                "total_videos": len(fingerprints),
                "duplicate_groups": len(duplicate_groups),
                "model_config": self.config,
                "model_type": self.model_type,
            },
            "fingerprints": {p: {k: plain(v) for k, v in d.items()} for p, d in fingerprints.items()},
            "duplicate_groups": [[{k: plain(v) for k, v in item.items()} for item in g] for g in duplicate_groups],
        }
        with open(output_path, "w", encoding="utf-8") as f:
            json.dump(results, f, indent=2, ensure_ascii=False)
        print(f"Results saved to {output_path}")
