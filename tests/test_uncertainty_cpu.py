"""CPU half of the ensemble's uncertainty and calibration: helpers.calibration_from_hist against a direct numpy
computation on the voxels a histogram was made from, error detection against sklearn, exact re-binning, the NaN rules,
per-case rows, and the sample-group sizing with and without the entropy plane."""
import numpy as np
import pytest
import torch
from sklearn.metrics import average_precision_score, roc_auc_score

FIX = 2.0 ** -24


def _voxels(n, seed, acc_shift=0.0):
    """(confidence fp32, correct bool) of n synthetic voxels: confidences in [1/13, 1], accuracy near confidence."""
    rng = np.random.default_rng(seed)
    conf = (1 / 13 + (1 - 1 / 13) * rng.beta(5, 1.5, n)).astype(np.float32)
    conf[: n // 50] = 1.0                                          # the top edge goes to bin T - 1
    correct = rng.random(n) < np.clip(conf + acc_shift, 0, 1)
    return conf, correct


def _hist(conf, correct, t):
    """The kernel's [3,T] histogram: bin min(floor(conf * T), T - 1) in fp32, confidence rounded to 2^-24 per voxel."""
    b = np.minimum(np.floor(conf * np.float32(t)).astype(np.int64), t - 1)
    h = np.zeros((3, t), dtype=np.int64)
    np.add.at(h[0], b, 1)
    np.add.at(h[1], b, correct.astype(np.int64))
    np.add.at(h[2], b, np.rint(conf.astype(np.float64) / FIX).astype(np.int64))
    return h


@pytest.mark.parametrize("t,e", [(960, 15), (64, 8), (30, 10), (2, 2)])
def test_calibration_from_hist_against_voxels(t, e):
    from innovative3D.helpers import calibration_from_hist
    conf, correct = _voxels(20000, seed=t, acc_shift=-0.05)
    n = conf.size
    brier_v = np.random.default_rng(1).random(n)                   # any per-voxel Brier terms: the mean is checked
    c = calibration_from_hist(_hist(conf, correct, t), brier_v.sum(), ece_bins=e)
    cb = np.minimum(np.floor(conf.astype(np.float64) * e).astype(np.int64), e - 1)
    ece = mce = 0.0
    for b in range(e):
        m = cb == b
        if not m.any():
            assert c["reliability"]["count"][b] == 0 and np.isnan(c["reliability"]["accuracy"][b])
            continue
        acc, cf = correct[m].mean(), conf[m].astype(np.float64).mean()
        ece += m.sum() / n * abs(acc - cf)
        mce = max(mce, abs(acc - cf))
        assert c["reliability"]["count"][b] == m.sum()
        assert c["reliability"]["accuracy"][b] == pytest.approx(acc, abs=1e-12)
        assert c["reliability"]["confidence"][b] == pytest.approx(cf, abs=FIX)
    assert c["ece"] == pytest.approx(ece, abs=FIX)
    assert c["mce"] == pytest.approx(mce, abs=FIX)
    assert c["brier"] == pytest.approx(brier_v.mean(), rel=1e-12)
    assert c["counted"] == n and c["errors"] == int((~correct).sum()) and c["ece_bins"] == e
    # risk-coverage: keep the voxels of fine bins >= i, most confident first
    fb = np.minimum(np.floor(conf * np.float32(t)).astype(np.int64), t - 1)
    cov, risk = [], []
    for i in range(t - 1, -1, -1):
        kept = fb >= i
        if kept.any():
            cov.append(kept.sum() / n)
            risk.append((~correct[kept]).mean())
    np.testing.assert_allclose(c["coverage"], cov, rtol=1e-12)
    np.testing.assert_allclose(c["risk"], risk, rtol=1e-12)
    assert c["coverage"][-1] == 1.0
    aurc = risk[0] * cov[0] + np.trapezoid(risk, cov)
    assert c["aurc"] == pytest.approx(aurc, rel=1e-12)


@pytest.mark.parametrize("t", [960, 16, 2])
def test_error_detection_is_sklearn(t):
    from innovative3D.helpers import calibration_from_hist
    conf, correct = _voxels(5000, seed=7 + t)
    c = calibration_from_hist(_hist(conf, correct, t), ece_bins=t)
    fb = np.minimum(np.floor(conf * np.float32(t)).astype(np.int64), t - 1)
    score = (t - 1 - fb).astype(np.float64)                      # 1 - confidence, binned
    err = ~correct
    assert c["error_auroc"] == pytest.approx(roc_auc_score(err, score), abs=1e-12)
    assert c["error_ap"] == pytest.approx(average_precision_score(err, score), abs=1e-12)
    exact = roc_auc_score(err, 1.0 - conf.astype(np.float64))
    assert abs(c["error_auroc"] - exact) <= c["error_auroc_tie_bound"] + 1e-12


def test_rebinning_is_exact_and_needs_a_divisor():
    from innovative3D.helpers import calibration_from_hist
    conf, correct = _voxels(30000, seed=3)
    fine = calibration_from_hist(_hist(conf, correct, 960))
    coarse = calibration_from_hist(_hist(conf, correct, 15))        # the kernel binning straight into 15 bins
    assert fine["ece"] == pytest.approx(coarse["ece"], abs=1e-15)
    assert fine["mce"] == pytest.approx(coarse["mce"], abs=1e-15)
    np.testing.assert_array_equal(fine["reliability"]["count"], coarse["reliability"]["count"])
    with pytest.raises(ValueError, match="ece_bins"):
        calibration_from_hist(_hist(conf, correct, 1000))
    with pytest.raises(ValueError, match=r"\[3,T\]"):
        calibration_from_hist(np.zeros((2, 15), dtype=np.int64))


def test_nan_rules():
    from innovative3D.helpers import calibration_from_hist
    empty = calibration_from_hist(np.zeros((3, 30), dtype=np.int64), 0.0)
    for key in ("ece", "mce", "brier", "error_auroc", "error_ap", "aurc", "mean_entropy", "mean_mutual_info"):
        assert np.isnan(empty[key]), key
    assert empty["counted"] == 0 and empty["coverage"].size == 0
    conf = np.array([0.5, 0.9, 0.99], dtype=np.float32)
    no_err = calibration_from_hist(_hist(conf, np.ones(3, bool), 30), 0.1)
    assert np.isnan(no_err["error_auroc"]) and np.isnan(no_err["error_ap"]) and no_err["aurc"] == 0.0
    assert not np.isnan(no_err["ece"]) and no_err["brier"] == pytest.approx(0.1 / 3)
    all_err = calibration_from_hist(_hist(conf, np.zeros(3, bool), 30), ece_bins=15)
    assert np.isnan(all_err["error_auroc"]) and all_err["error_ap"] == 1.0 and all_err["aurc"] == 1.0
    assert np.isnan(all_err["brier"])                                 # no Brier sum given
    u = calibration_from_hist(_hist(conf, np.ones(3, bool), 30), unc=np.array([3 << 24, 1 << 23]), voxels=4)
    assert u["mean_entropy"] == 0.75 and u["mean_mutual_info"] == 0.125


def test_sample_calibration_rows():
    from innovative3D.helpers import calibration_from_hist, sample_calibration
    rows, briers = [], []
    for i in range(3):
        conf, correct = _voxels(2000, seed=40 + i, acc_shift=-0.1 * i)
        rows.append(_hist(conf, correct, 960))
        briers.append(10.0 * (i + 1))
    rows.append(np.zeros((3, 960), dtype=np.int64))
    briers.append(0.0)
    got = sample_calibration(torch.from_numpy(np.stack(rows)), torch.tensor(briers, dtype=torch.float64))
    assert len(got) == 4
    for row, br, (ece, brier, auroc) in zip(rows[:3], briers, got):
        c = calibration_from_hist(row, br)
        assert (ece, brier, auroc) == (c["ece"], c["brier"], c["error_auroc"])
    assert all(np.isnan(v) for v in got[3])
    with pytest.raises(ValueError, match=r"\[B,3,T\]"):
        sample_calibration(np.zeros((3, 960)))


def test_sample_group_sizing_with_entropy_plane(monkeypatch):
    """Without uncertainty the ensemble keeps its group size; the mutual information adds the fp32 entropy plane
    (4 B per position: 1/16 level-1 unit) per sample."""
    from spff_b200.engine import ENSEMBLE_UNITS, ENTROPY_UNITS, SpffEngine, ensemble_units
    free = 170 * 2 ** 30
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda device=None: (free, 183 * 2 ** 30))
    unit = 5 * 512 * 512 * 64
    assert ensemble_units(False) == ENSEMBLE_UNITS and ENTROPY_UNITS == 4 / 64
    assert ensemble_units(True) == ENSEMBLE_UNITS + 4 / 64
    assert SpffEngine.fit_group(256, 5, 512, 512, "cuda:0", train=False, extra=ensemble_units(False)) == 55
    got = SpffEngine.fit_group(256, 5, 512, 512, "cuda:0", train=False, extra=ensemble_units(True))
    assert got == int(0.45 * free / ((16.7 + ENSEMBLE_UNITS + 1 / 16) * unit)) == 54
    assert SpffEngine.fit_group(256, 5, 128, 128, "cuda:0", train=False, extra=ensemble_units(True)) == 256

def test_calibration_argument_validation():
    from innovative3D.models import _calib_buffers
    assert tuple(_calib_buffers(960, "cpu").shape) == (3, 960)
    assert _calib_buffers(None, "cpu") is None
    for bad in (1, 1025):
        with pytest.raises(ValueError, match="bin count"):
            _calib_buffers(bad, "cpu")
    with pytest.raises(ValueError, match=r"\[3,T\]"):
        _calib_buffers(torch.zeros(2, 16, dtype=torch.int64), "cpu")
    with pytest.raises(ValueError, match=r"\[3,T\]"):
        _calib_buffers(torch.zeros(3, 16, dtype=torch.int32), "cpu")
    c = torch.zeros(3, 16, dtype=torch.int64)
    assert _calib_buffers(c, "cpu") is c
