"""Evaluation metrics (SURVEY.md section 8f rank 3; /root/reference/train.py:285-358, 439-481).

CPU: the NumPy oracle against the golden values the UNMODIFIED reference trainer methods returned
(tests/golden/metrics.json, tests/golden/make_golden_metrics.py), with the default and with explicit thresholds.
GPU (-m gpu): the device pass (vfp_pair_scores + vfp_pair_stats through the C ABI) against the oracle and the golden values.
Tolerances: rank-derived values (R@k, mAP, threshold counts, AUC) are exact unless two fp32 scores differ by less than
the summation-order noise (none do in these sets) -> 1e-12; moments are float64 sums of fp32 scores -> 1e-6.
"""
import json
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import metrics_oracle as mo  # noqa: E402

GOLD = json.load(open(os.path.join(ROOT, "tests", "golden", "metrics.json")))
RANK_KEYS_TOL, MOMENT_TOL = 1e-9, 2e-6


def close(got, want, name):
    assert set(got) == set(want), (name, sorted(set(got) ^ set(want)))
    for k, w in want.items():
        tol = MOMENT_TOL if ("sim_" in k or k == "separation_gap") else RANK_KEYS_TOL
        assert abs(got[k] - w) <= tol, (name, k, got[k], w)


@pytest.mark.parametrize("name", sorted(mo.METRIC_CASES))
def test_oracle_matches_reference_golden(name):
    seed, n_videos, cpv, sigma = mo.METRIC_CASES[name]
    E, ids = mo.make_metric_embeddings(seed, n_videos, cpv, sigma)
    assert len(E) == GOLD[name]["n"] and abs(float(E.astype(np.float64).sum()) - GOLD[name]["checksum"]) < 1e-6
    close(mo.retrieval_metrics(E, ids), GOLD[name]["retrieval"], name)
    close(mo.discrimination_metrics(E, ids), GOLD[name]["discrimination"], name)


@pytest.mark.parametrize("name", sorted(mo.METRIC_CASES))
def test_oracle_explicit_thresholds_match_reference_golden(name):
    """A caller's own `thresholds` list: the per-threshold values are the ones the reference returned for those thresholds
    among its defaults, the threshold-free values do not change."""
    seed, n_videos, cpv, sigma = mo.METRIC_CASES[name]
    E, ids = mo.make_metric_embeddings(seed, n_videos, cpv, sigma)
    want = {k: v for k, v in GOLD[name]["discrimination"].items() if "@" not in k or k.endswith(("@0.90", "@0.80"))}
    close(mo.discrimination_metrics(E, ids, thresholds=[0.9, 0.8]), want, name)


def test_degenerate_sets():
    E, _ = mo.make_metric_embeddings(1, 5, 1, 0.1)
    d = mo.discrimination_metrics(E, np.arange(5))                 # no intra pairs at all
    assert d["auc_roc"] == 0.5 and d["intra_sim_mean"] == 0 and d["separation_gap"] == 0 and "precision@0.70" not in d
    d = mo.discrimination_metrics(E, np.zeros(5, int))            # no inter pairs
    assert d["auc_roc"] == 0.5 and d["inter_sim_mean"] == 0
    assert mo.retrieval_metrics(E, np.arange(5))["mAP"] == pytest.approx(1 / 5)    # the reference's self-positive quirk


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(mo.METRIC_CASES))
def test_device_metrics_match_reference_golden(name):
    from video_fingerprint_b200 import metrics

    seed, n_videos, cpv, sigma = mo.METRIC_CASES[name]
    E, ids = mo.make_metric_embeddings(seed, n_videos, cpv, sigma)
    close(metrics.compute_retrieval_metrics(E, ids), GOLD[name]["retrieval"], name)
    close(metrics.compute_discrimination_metrics(E, ids), GOLD[name]["discrimination"], name)


@pytest.mark.gpu
def test_device_metrics_ties_ragged_and_degenerate():
    from video_fingerprint_b200 import metrics

    # exact duplicates (tied scores, incl. ties with the positives), string ids, a size that is not a multiple of the 64-tile
    E, ids = mo.make_metric_embeddings(31, 150, (1, 3), 0.09)
    E[40] = E[3]
    E[77] = E[3]
    E[120] = E[119]
    names = np.array([f"video_{i}" for i in ids])
    close(metrics.compute_retrieval_metrics(torch.from_numpy(E), names, k_values=(1, 3, 5, 10, 1000)),
          mo.retrieval_metrics(E, names, k_values=(1, 3, 5, 10, 1000)), "ties")
    close(metrics.compute_discrimination_metrics(E, names, thresholds=(0.3, 0.5, 0.7, 0.8, 0.85, 0.9, 0.95, 1.0)),
          mo.discrimination_metrics(E, names, thresholds=(0.3, 0.5, 0.7, 0.8, 0.85, 0.9, 0.95, 1.0)), "ties")
    E5, _ = mo.make_metric_embeddings(1, 5, 1, 0.1)
    for v in (np.arange(5), np.zeros(5, int)):
        close(metrics.compute_discrimination_metrics(E5, v), mo.discrimination_metrics(E5, v), "degenerate")
        close(metrics.compute_retrieval_metrics(E5, v), mo.retrieval_metrics(E5, v), "degenerate")


@pytest.mark.gpu
def test_device_metrics_larger_set_and_model_embeddings():
    """4 000 embeddings (a 63 x 63 tile grid) against the oracle; scores of unit vectors straight from the forward kernel."""
    from video_fingerprint_b200 import metrics

    E, ids = mo.make_metric_embeddings(41, 1500, (2, 4), 0.11)
    close(metrics.compute_retrieval_metrics(E, ids), mo.retrieval_metrics(E, ids), "large")
    close(metrics.compute_discrimination_metrics(E, ids), mo.discrimination_metrics(E, ids), "large")
