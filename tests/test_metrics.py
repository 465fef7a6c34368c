"""Evaluation metrics (SURVEY §8 f4): the reference's compute_metrics / classification_report inputs
(/root/reference/ViT-Training.py:112-118,139-146).  CPU: the count → score arithmetic against sklearn.  GPU: the
on-device counter kernel against sklearn on logits that include the threshold's edge cases."""
import numpy as np
import pytest
import torch

import chest_x_ray_vit_b200 as pkg


def _reference_predictions(logits: torch.Tensor) -> np.ndarray:
    probs = torch.nn.Sigmoid()(torch.Tensor(logits))           # exactly the reference's lines
    return (probs >= 0.5).int().cpu().numpy()


def _counts(y_true: np.ndarray, y_pred: np.ndarray) -> torch.Tensor:
    tp = (y_true == 1) & (y_pred == 1)
    fp = (y_true == 0) & (y_pred == 1)
    fn = (y_true == 1) & (y_pred == 0)
    tn = (y_true == 0) & (y_pred == 0)
    return torch.tensor(np.stack([tp.sum(0), fp.sum(0), fn.sum(0), tn.sum(0)], axis=1), dtype=torch.int64)


def _check_against_sklearn(scores, y_true, y_pred):
    skm = pytest.importorskip("sklearn.metrics")
    assert scores["f1_micro"] == pytest.approx(skm.f1_score(y_true=y_true, y_pred=y_pred, average="micro", zero_division=0), abs=1e-12)
    for avg in ("micro", "macro", "weighted"):
        p, r, f, _ = skm.precision_recall_fscore_support(y_true, y_pred, average=avg, zero_division=0)
        assert scores[f"f1_{avg}"] == pytest.approx(f, abs=1e-12)
        if avg != "weighted":
            assert scores[f"precision_{avg}"] == pytest.approx(p, abs=1e-12) and scores[f"recall_{avg}"] == pytest.approx(r, abs=1e-12)
    p, r, f, s = skm.precision_recall_fscore_support(y_true, y_pred, average=None, zero_division=0)
    assert np.allclose(scores["per_class"]["precision"], p) and np.allclose(scores["per_class"]["recall"], r)
    assert np.allclose(scores["per_class"]["f1"], f) and list(scores["per_class"]["support"]) == list(s)


def test_scores_from_counts_match_sklearn():
    g = torch.Generator().manual_seed(0)
    logits = torch.randn(257, 14, generator=g) * 2 - 1
    y = (torch.rand(257, 14, generator=g) < 0.1).float()
    y[:, 5] = 0                                        # a class with no positives: zero_division=0 paths
    logits[:, 7] = -5.0                                # a class never predicted
    y_true, y_pred = y.int().numpy(), _reference_predictions(logits)
    _check_against_sklearn(pkg.metrics.scores_from_counts(_counts(y_true, y_pred)), y_true, y_pred)


@pytest.mark.gpu
def test_device_counter_matches_sklearn_over_batches():
    g = torch.Generator().manual_seed(1)
    n, C = 1000, 14
    logits = torch.randn(n, C, generator=g) * 3
    logits[::17, 3] = 0.0                              # sigmoid(0) = 0.5 -> positive
    logits[1::17, 3] = -1e-9                           # rounds to exactly 0.5 in fp32 -> positive, as in the reference
    logits[2::17, 3] = -1e-3
    logits[3::17, 4] = float("inf")
    logits[4::17, 4] = float("-inf")
    y = (torch.rand(n, C, generator=g) < 0.15).float()
    ctr = pkg.metrics.MultilabelCounter(C)
    for lo in range(0, n, 64):                         # an evaluation loop of ragged batches
        ctr.update(logits[lo:lo + 64].cuda(), y[lo:lo + 64])
    scores = ctr.compute()
    y_true, y_pred = y.int().numpy(), _reference_predictions(logits)
    assert scores["counts"] == _counts(y_true, y_pred).tolist()
    _check_against_sklearn(scores, y_true, y_pred)
    ctr.reset()
    assert ctr.compute()["f1_micro"] == 0.0


@pytest.mark.gpu
def test_device_counter_at_the_label_limit():
    """C = 4096, the most labels the counter kernel accepts: its [C][4] shared-memory counters take 64 KB."""
    g = torch.Generator().manual_seed(2)
    B, C = 3, 4096
    logits = torch.randn(B, C, generator=g) * 2
    y = (torch.rand(B, C, generator=g) < 0.3).float()
    counts = torch.zeros((C, 4), dtype=torch.int64, device="cuda")
    pkg.ops.multilabel_counts(logits.cuda(), y.cuda(), counts)
    assert torch.equal(counts.cpu(), _counts(y.int().numpy(), _reference_predictions(logits)))
