"""Host-side mirror of the reference trainer's evaluation metrics (/root/reference/train.py):

* ``compute_discrimination_metrics(embeddings, video_ids, thresholds)``   train.py:285-358
* ``compute_retrieval_metrics(embeddings, video_ids, k_values)``          train.py:439-481 (``Trainer._compute_retrieval_metrics``)

Same arguments, same dictionary keys, same edge-case values (0 / 0.5 defaults, ``R@k`` skipped when k > n_videos - 1).
The reference builds the N x N similarity matrix on the host and walks it in Python; here ONE device pass
(``vfp_pair_stats``, csrc/metrics_kernels.cuh) visits every ordered pair in exact fp32 and returns the ranks of the
positives, the intra / inter moments, the threshold counts and the AUC rank sums, so the host work is O(N).
There is no CPU fallback: without a CUDA device these functions raise.

Tie handling (the reference's ``argpartition`` / unstable ``argsort`` order equal scores arbitrarily): ranks here use
(score descending, index ascending), the same canonical order as the top-k search.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Sequence, Tuple

import numpy as np
import torch

from . import _native

_MAX_THRESHOLDS = 8


def _positives(video_ids: np.ndarray) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """CSR list of the positives of every row: columns with the same video id, the row itself excluded, ascending."""
    n = len(video_ids)
    order = np.argsort(video_ids, kind="stable")
    sorted_ids = video_ids[order]
    starts = np.flatnonzero(np.r_[True, sorted_ids[1:] != sorted_ids[:-1]])
    sizes = np.diff(np.r_[starts, n])
    group_of = np.empty(n, np.int64)
    group_of[order] = np.repeat(np.arange(len(starts)), sizes)
    counts = sizes[group_of] - 1
    row_ptr = np.zeros(n + 1, np.int64)
    np.cumsum(counts, out=row_ptr[1:])
    pair_i = np.repeat(np.arange(n), counts)
    pos = np.empty(int(row_ptr[-1]), np.int64)
    for g, (s, k) in enumerate(zip(starts, sizes)):   # groups are small (a video's clips); rows of one group share members
        if k < 2:
            continue
        members = np.sort(order[s : s + k])
        for i in members:
            pos[row_ptr[i] : row_ptr[i + 1]] = members[members != i]
    return row_ptr, pair_i, pos


def _device_pass(embeddings, video_ids, thresholds: Sequence[float]):
    if isinstance(embeddings, torch.Tensor):
        E = embeddings.detach()
    else:
        E = torch.from_numpy(np.ascontiguousarray(embeddings, dtype=np.float32))
    if E.dim() != 2:
        raise ValueError(f"embeddings must be 2-D (n, dim), got shape {tuple(E.shape)}")
    ids_np = np.asarray(video_ids)
    if ids_np.ndim != 1 or len(ids_np) != E.shape[0]:
        raise ValueError(f"one video id per embedding: {E.shape[0]} embeddings, video_ids of shape {ids_np.shape}")
    if len(thresholds) > _MAX_THRESHOLDS:
        raise ValueError(f"at most {_MAX_THRESHOLDS} thresholds per pass")
    _native.require_cuda()
    lib = _native.load()
    E = E.float()
    if not E.is_cuda:
        E = E.cuda()
    # the pair kernels take rows of a multiple of 16 floats; zero columns add fmaf(0, 0, acc) = acc, so scores and ranks of
    # any width 1 .. 512 are those of the unpadded rows
    E = torch.nn.functional.pad(E, (0, -E.shape[1] % 16)).contiguous()
    _, ids_np = np.unique(ids_np, return_inverse=True)      # any hashable id -> dense int32
    ids_np = ids_np.astype(np.int32)
    n, dim = E.shape
    row_ptr, pair_i, pos = _positives(ids_np)
    m = int(row_ptr[-1])
    dev = E.device
    with torch.cuda.device(dev):
        st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        ids_d = torch.from_numpy(ids_np).to(dev)
        row_ptr_d = torch.from_numpy(row_ptr.astype(np.int32)).to(dev)
        pi_d = torch.from_numpy(pair_i.astype(np.int32)).to(dev)
        pos_d = torch.from_numpy(pos.astype(np.int32)).to(dev)
        score_d = torch.empty(max(m, 1), dtype=torch.float32, device=dev)
        _native.check(lib.vfp_pair_scores(C.c_void_p(E.data_ptr()), n, dim, C.c_void_p(pi_d.data_ptr()), C.c_void_p(pos_d.data_ptr()), m,
                                          C.c_void_p(score_d.data_ptr()), st), "vfp_pair_scores")
        sorted_d = torch.sort(score_d[:m]).values.contiguous() if m else score_d   # m values: bookkeeping, not the N^2 work
        greater = torch.zeros(max(m, 1), dtype=torch.int32, device=dev)
        tie = torch.zeros(max(m, 1), dtype=torch.int32, device=dev)
        sums = torch.zeros(4, dtype=torch.float64, device=dev)
        counts = torch.zeros(4 + 2 * _MAX_THRESHOLDS, dtype=torch.int64, device=dev)
        thr = (C.c_float * max(1, len(thresholds)))(*[float(t) for t in thresholds])
        _native.check(lib.vfp_pair_stats(
            C.c_void_p(E.data_ptr()), C.c_void_p(ids_d.data_ptr()), n, dim, C.c_void_p(row_ptr_d.data_ptr()), C.c_void_p(pos_d.data_ptr()),
            C.c_void_p(score_d.data_ptr()), C.c_void_p(sorted_d.data_ptr()), m, thr, len(thresholds), C.c_void_p(greater.data_ptr()),
            C.c_void_p(tie.data_ptr()), C.c_void_p(sums.data_ptr()), C.c_void_p(counts.data_ptr()), st), "vfp_pair_stats")
        out = dict(
            n=n, m=m, row_ptr=row_ptr, n_videos=int(ids_np.max()) + 1 if n else 0,
            rank=(greater[:m].cpu().numpy().astype(np.int64) + tie[:m].cpu().numpy().astype(np.int64) + 1),
            sums=sums.cpu().numpy(), counts=counts.cpu().numpy(),
        )
    return out


def compute_retrieval_metrics(embeddings, video_ids, k_values: Sequence[int] = (1, 5, 10)) -> Dict[str, float]:
    """R@k and mAP of every embedding against all others (train.py:439-481)."""
    r = _device_pass(embeddings, video_ids, [])
    n, row_ptr, rank = r["n"], r["row_ptr"], r["rank"]
    best = np.full(n, np.iinfo(np.int64).max)
    if r["m"]:
        np.minimum.at(best, np.repeat(np.arange(n), np.diff(row_ptr)), rank)
    metrics: Dict[str, float] = {}
    for k in k_values:
        if k > r["n_videos"] - 1:      # train.py:449-450
            continue
        metrics[f"R@{k}"] = float(np.mean(best <= k)) if n else 0.0
    # mAP (train.py:464-479). Reference quirk kept for drop-in parity: the row itself is masked to -inf, which sorts it LAST,
    # but it still carries its own video id - so it is one more "positive" at rank n, and a row without any true positive
    # has AP = 1/n instead of being skipped.
    aps = np.empty(n, np.float64)
    for i in range(n):
        rk = np.sort(rank[row_ptr[i] : row_ptr[i + 1]])
        rk = np.r_[rk, n]
        aps[i] = np.mean(np.arange(1, len(rk) + 1) / rk)
    metrics["mAP"] = float(np.mean(aps)) if n else 0.0
    return metrics


def compute_discrimination_metrics(embeddings, video_ids, thresholds: Sequence[float] = (0.7, 0.8, 0.85, 0.9)) -> Dict[str, float]:
    """Intra / inter similarity statistics, threshold precision / recall / F1 / FPR and AUC-ROC (train.py:285-358)."""
    thr32 = [float(np.float32(t)) for t in thresholds]    # the reference compares its fp32 scores with the fp32-rounded threshold
    r = _device_pass(embeddings, video_ids, thr32)
    s_intra, q_intra, s_inter, q_inter = (float(x) for x in r["sums"])
    c = r["counts"]
    n_intra, n_inter, sum_upper, sum_lower = (int(x) for x in c[:4])

    def mean_std(s, q, k):
        if k == 0:
            return 0.0, 0.0
        mu = s / k
        return mu, float(np.sqrt(max(q / k - mu * mu, 0.0)))

    mu_a, sd_a = mean_std(s_intra, q_intra, n_intra)
    mu_e, sd_e = mean_std(s_inter, q_inter, n_inter)
    both = n_intra > 0 and n_inter > 0
    metrics: Dict[str, float] = {
        "intra_sim_mean": mu_a, "intra_sim_std": sd_a, "inter_sim_mean": mu_e, "inter_sim_std": sd_e,
        "separation_gap": (mu_a - mu_e) if both else 0.0,
    }
    for t, threshold in enumerate(thresholds):
        if not both:
            continue
        tp, fp = int(c[4 + t]), int(c[4 + _MAX_THRESHOLDS + t])
        fn, tn = n_intra - tp, n_inter - fp
        precision = tp / (tp + fp) if (tp + fp) > 0 else 0.0
        recall = tp / (tp + fn) if (tp + fn) > 0 else 0.0
        f1 = 2 * precision * recall / (precision + recall) if (precision + recall) > 0 else 0.0
        metrics[f"precision@{threshold:.2f}"] = precision
        metrics[f"recall@{threshold:.2f}"] = recall
        metrics[f"f1@{threshold:.2f}"] = f1
        metrics[f"fpr@{threshold:.2f}"] = fp / (fp + tn) if (fp + tn) > 0 else 0.0
    if both:
        # P(intra > inter) + P(intra == inter) / 2 over all (intra, inter) pairs = sklearn's roc_auc_score
        wins = n_inter * n_intra - sum_upper          # sum over inter scores of #{intra > s}
        ties = sum_upper - sum_lower
        metrics["auc_roc"] = (wins + 0.5 * ties) / (n_intra * n_inter)
    else:
        metrics["auc_roc"] = 0.5
    return metrics
