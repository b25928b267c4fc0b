"""CPU half of the ranking metrics of the fused evaluation step: helpers.curves_from_hist and helpers.sample_curves
against sklearn. With the bin index as the score, the binned AUROC / AP and the ROC / PR points are sklearn's exactly;
against unquantised scores the AUROC lies within the tie bound that curves_from_hist reports."""
import math

import numpy as np
import pytest

sk = pytest.importorskip("sklearn.metrics")


def _hist(y, bins_of, k, t):
    """[K,2,T] histogram of per-class bin indices bins_of [n,K] with labels y [n]."""
    h = np.zeros((k, 2, t), dtype=np.int64)
    for c in range(k):
        np.add.at(h[c, 0], bins_of[y == c, c], 1)
        np.add.at(h[c, 1], bins_of[y != c, c], 1)
    return h


def _random_case(seed, k, t, n=4000):
    rng = np.random.default_rng(seed)
    y = rng.integers(0, k, n)
    b = rng.integers(0, t, (n, k))
    # some classes use a few bins only, so that most bins are empty
    for c in range(0, k, 2):
        b[:, c] = rng.choice(rng.choice(t, size=min(5, t), replace=False), n)
    b[y == 1, 1] = np.minimum(b[y == 1, 1] + t // 3, t - 1)   # class 1 better than chance
    return y, b


@pytest.mark.parametrize("k,t,seed", [(2, 16, 0), (5, 64, 1), (13, 256, 2), (16, 1024, 3), (3, 1000, 4)])
def test_curves_match_sklearn_on_bin_index(k, t, seed):
    from innovative3D.helpers import curves_from_hist
    y, b = _random_case(seed, k, t)
    cv = curves_from_hist(_hist(y, b, k, t))
    for c in range(k):
        yt, s = (y == c).astype(int), b[:, c]
        assert abs(cv["auroc"][c] - sk.roc_auc_score(yt, s)) <= 1e-12
        assert abs(cv["ap"][c] - sk.average_precision_score(yt, s)) <= 1e-12
        # ROC: sklearn's thresholds are the occurring scores (descending) after an initial +inf point, ours t_T..t_0
        fpr, tpr, th = sk.roc_curve(yt, s, drop_intermediate=False)
        occupied = np.unique(s)
        idx = np.concatenate([[t], occupied[::-1]])           # threshold index i of each sklearn point
        ours_thr = cv["roc_thresholds"][c]
        pos = t - idx                                          # position of t_i in the descending arrays
        np.testing.assert_array_equal(cv["fpr"][c][pos], fpr)
        np.testing.assert_array_equal(cv["tpr"][c][pos], tpr)
        np.testing.assert_array_equal(ours_thr[pos[1:]], th[1:] / t)
        # PR: sklearn's ascending occurring thresholds plus its final (recall 0, precision 1) point
        prec, rec, pth = sk.precision_recall_curve(yt, s)
        sel = np.searchsorted(cv["pr_thresholds"][c], pth / t)
        np.testing.assert_array_equal(cv["pr_thresholds"][c][sel], pth / t)
        np.testing.assert_allclose(cv["precision"][c][sel], prec[:-1], rtol=1e-15, atol=0)
        np.testing.assert_allclose(cv["recall"][c][sel], rec[:-1], rtol=1e-15, atol=0)
        # every PR point has TP + FP > 0, and the PR thresholds run from 0 to the highest occupied bin
        assert cv["pr_thresholds"][c][0] == 0 and cv["pr_thresholds"][c][-1] == occupied.max() / t


def test_nan_rules_and_macro_nanmean():
    from innovative3D.helpers import curves_from_hist
    k, t = 4, 16
    rng = np.random.default_rng(5)
    y = rng.choice([0, 2], 500)                               # class 1 and class 3: no positives
    b = rng.integers(0, t, (500, k))
    h = _hist(y, b, k, t)
    h[3] = 0
    h[3, 0, 4] = 7                                            # class 3: every counted voxel positive (N = 0)
    cv = curves_from_hist(h)
    assert math.isnan(cv["auroc"][1]) and math.isnan(cv["ap"][1]) and math.isnan(cv["auroc_tie_bound"][1])
    assert math.isnan(cv["auroc"][3]) and cv["ap"][3] == 1.0
    assert not math.isnan(cv["auroc"][0]) and not math.isnan(cv["auroc"][2])
    assert cv["macro_auroc"] == cv["auroc"][2]                # nanmean over classes 1..K-1
    assert abs(cv["macro_ap"] - np.mean([cv["ap"][2], cv["ap"][3]])) <= 1e-15
    # all-empty histogram: everything undefined
    empty = curves_from_hist(np.zeros((3, 2, t), np.int64))
    assert np.isnan(empty["auroc"]).all() and math.isnan(empty["macro_auroc"]) and math.isnan(empty["macro_ap"])


@pytest.mark.parametrize("t", [16, 256, 1000])
def test_tie_bound_covers_unquantised_auroc(t):
    from innovative3D.helpers import curves_from_hist
    rng = np.random.default_rng(t)
    k, n = 5, 20000
    y = rng.integers(0, k, n)
    logits = rng.normal(size=(n, k)) + 1.5 * np.eye(k)[y] * rng.random((n, 1))
    p = np.exp(logits - logits.max(1, keepdims=True))
    p /= p.sum(1, keepdims=True)
    b = np.minimum(np.floor(p * t).astype(np.int64), t - 1)
    cv = curves_from_hist(_hist(y, b, k, t))
    for c in range(k):
        exact = sk.roc_auc_score((y == c).astype(int), p[:, c])
        assert abs(cv["auroc"][c] - exact) <= cv["auroc_tie_bound"][c] + 1e-12, (c, cv["auroc"][c], exact)
    assert cv["auroc_tie_bound"].max() < (0.1 if t == 16 else 0.01)   # the bound shrinks with the resolution


def test_sample_curves_rows_equal_curves_from_hist():
    import torch
    from innovative3D.helpers import curves_from_hist, sample_curves
    k, t = 6, 32
    rows = np.stack([_hist(*_random_case(s, k, t, n=800), k, t) for s in range(4)])
    rows[2, 4] = 0                                            # a class absent from one case
    per = sample_curves(torch.from_numpy(rows))
    assert len(per) == 4
    for i, (auroc, ap, m_auroc, m_ap) in enumerate(per):
        cv = curves_from_hist(rows[i])
        np.testing.assert_array_equal(auroc, cv["auroc"])
        np.testing.assert_array_equal(ap, cv["ap"])
        assert (m_auroc == cv["macro_auroc"]) and (m_ap == cv["macro_ap"])
    assert math.isnan(per[2][0][4]) and math.isnan(per[2][1][4])


def test_bad_histogram_shapes_are_rejected():
    from innovative3D.helpers import curves_from_hist, sample_curves
    with pytest.raises(ValueError):
        curves_from_hist(np.zeros((3, 3, 16), np.int64))
    with pytest.raises(ValueError):
        sample_curves(np.zeros((3, 2, 16), np.int64))
