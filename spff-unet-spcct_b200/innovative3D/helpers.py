"""Loss and step metrics of the hot path, on the B200 kernels.

Same call surface as the reference's `innovative3D/helpers.py`:
  ce_plus_macro_dice_loss(logits, labels, num_classes, ignore_index=255, smooth=1e-6) -> Tensor   (:797-803)
  macro_dice_loss(logits, labels, num_classes, ignore_index=255, smooth=1e-6) -> float            (:782-795)
  per_class_metrics_3d / _2d(preds, labels, num_classes, smooth=1e-6, ignore_index=None) -> 9-tuple (:668-779)

The reference evaluates these with ~140 boolean-mask reductions and `.item()` host syncs per step
(SURVEY.md §2.3 K9/K10). Here ONE kernel pass (`spff_ce_confusion`) over logits + labels produces the
sufficient statistics — sum of nll, number of valid voxels, the [label][argmax] tally — and
everything else is derived from those 171 integers; the CE gradient is `spff_ce_grad`. A tally is
cached per (logits, labels) pair so that the loss and the metrics of one step share one pass.
There is no CPU path: CPU tensors raise.
"""
from __future__ import annotations

import math
import weakref
from typing import List, Optional

import numpy as np
import torch

from spff_b200 import ops
from spff_b200.engine import LossTally

_NO_IGNORE = -1   # label value that never occurs: "no ignore_index"


def _prep(logits: torch.Tensor, labels: torch.Tensor):
    if not logits.is_cuda:
        raise RuntimeError("innovative3D.helpers (B200 build) needs CUDA tensors; there is no CPU fallback")
    if logits.dim() == 4:      # 2-D models: [B,K,H,W] is a depth-1 volume
        logits = logits.unsqueeze(2)
        labels = labels.unsqueeze(1) if labels.dim() == 3 else labels
    if logits.dim() != 5:
        raise ValueError(f"logits must be [B,K,D,H,W] or [B,K,H,W], got {tuple(logits.shape)}")
    lg = logits.detach()
    if lg.dtype != torch.float32 or not lg.is_contiguous():
        lg = lg.float().contiguous()
    lb = labels.to(logits.device)
    if lb.dtype not in (torch.uint8, torch.int64):
        lb = lb.long()
    lb = lb.contiguous()
    n, k, d, h, w = lg.shape
    if tuple(lb.shape) != (n, d, h, w):
        raise ValueError(f"labels {tuple(lb.shape)} do not match logits {tuple(lg.shape)}")
    return lg, lb


class _TallyCache:
    """Tally of the most recent (logits, labels) pair, so that the loss and the metrics of one step
    share one kernel pass. A hit needs the SAME live tensor objects at the same version — data_ptr
    alone is not an identity (the caching allocator hands a freed block to the next tensor)."""
    logits_ref = None
    labels_ref = None
    versions = None
    ign = None
    tally: Optional[LossTally] = None


def _tally(logits: torch.Tensor, labels: torch.Tensor, ignore_index: Optional[int]) -> LossTally:
    ign = _NO_IGNORE if ignore_index is None else int(ignore_index)
    c = _TallyCache
    if (c.tally is not None and c.logits_ref is not None and c.logits_ref() is logits and c.labels_ref() is labels
            and c.versions == (logits._version, labels._version) and c.ign == ign):
        return c.tally
    lg, lb = _prep(logits, labels)
    t = LossTally(lg.shape[1], lg.device)
    ops.ce_confusion(lg, lb, ign, t.nll, t.count, t.confusion)
    c.logits_ref, c.labels_ref = weakref.ref(logits), weakref.ref(labels)
    c.versions, c.ign, c.tally = (logits._version, labels._version), ign, t
    return t


class _CrossEntropyFn(torch.autograd.Function):
    """F.cross_entropy(logits, labels, ignore_index) (mean over valid voxels), helpers.py:798-801."""

    @staticmethod
    def forward(ctx, logits, labels, ignore_index, t):
        ctx.save_for_backward(logits, labels, t.count)
        ctx.ignore_index = ignore_index
        return (t.nll[0] / t.count[0].double()).to(torch.float32)   # 0/0 = nan when nothing is valid, as torch

    @staticmethod
    def backward(ctx, g):
        logits, labels, count = ctx.saved_tensors
        lg, lb = _prep(logits, labels)
        dl = torch.empty_like(lg)
        ops.ce_grad(lg, lb, int(ctx.ignore_index), count, g.detach().reshape(1).float().contiguous(), dl)
        return dl.view_as(logits).to(logits.dtype), None, None, None


def masked_ce_loss(logits, labels, ignore_index=255):
    """Sum of the valid voxels' nll over max(#valid, 1): `_weighted_softmax_ce` of the Cicek wrapper with
    class_weights None and no voxel weights (models.py:779-798). Shares the tally pass with the metrics."""
    ign = _NO_IGNORE if ignore_index is None else int(ignore_index)
    t = _tally(logits, labels, ign)
    clamped = LossTally.__new__(LossTally)           # same statistics, denominator clamped like .clamp_min(1.0)
    clamped.k, clamped.nll, clamped.count, clamped.confusion = t.k, t.nll, t.count.clamp(min=1), t.confusion
    return _CrossEntropyFn.apply(logits, labels, ign, clamped)


def _dice_from_tally(t: LossTally, smooth: float) -> torch.Tensor:
    cm = t.confusion.double()
    tp = cm.diagonal()[1:]
    fp = cm.sum(0)[1:] - tp
    fn = cm.sum(1)[1:] - tp
    if tp.numel() == 0:
        return cm.new_ones(())
    return ((2 * tp + smooth) / (2 * tp + fp + fn + smooth)).mean()


def macro_dice_loss(logits, labels, num_classes, ignore_index=255, smooth=1e-6) -> float:
    """1 - hard macro Dice over classes 1..K-1 on argmax(logits); a Python float like the reference's
    (helpers.py:782-795), hence one host sync. ce_plus_macro_dice_loss does not call this."""
    return float(1.0 - _dice_from_tally(_tally(logits, labels, ignore_index), smooth))


def ce_plus_macro_dice_loss(logits, labels, num_classes, ignore_index=255, smooth=1e-6):
    """CE(ignore_index) + 0.5 * (1 - hard macro Dice) (helpers.py:797-803). The Dice term carries no
    gradient in the reference (argmax + .item()); here it stays on the device, so the call does not
    synchronise the host."""
    ign = _NO_IGNORE if ignore_index is None else int(ignore_index)
    t = _tally(logits, labels, ign)        # one pass; per_class_metrics_3d on the same tensors reuses it
    ce = _CrossEntropyFn.apply(logits, labels, ign, t)
    dice = _dice_from_tally(t, smooth)
    return ce + (0.5 * (1.0 - dice)).to(torch.float32)


def metrics_from_confusion(cm: np.ndarray, total_voxels: int, smooth: float = 1e-6):
    """The 9-tuple of per_class_metrics_3d (helpers.py:668-725) from the [label][argmax] tally over
    valid voxels. `total_voxels` counts every voxel, ignored ones included: the reference's true
    negatives are `(~pred_c & ~label_c).sum()` with both masks cleared on ignored voxels (:684-690),
    so ignored voxels are true negatives of every class."""
    k = cm.shape[0]
    row, col, diag = cm.sum(1), cm.sum(0), np.diagonal(cm)
    dice_l: List[float] = []
    sens_l: List[float] = []
    spec_l: List[float] = []
    for c in range(k):
        tp = int(diag[c]); fp = int(col[c] - diag[c]); fn = int(row[c] - diag[c])
        tn = int(total_voxels) - tp - fp - fn
        if (tp + fn) == 0 and fp == 0:          # absent in GT and never predicted (:693-696)
            dice = sens = float("nan")
        else:
            dice = (2 * tp + smooth) / (2 * tp + fp + fn + smooth)
            sens = (tp + smooth) / (tp + fn + smooth) if (tp + fn) > 0 else float("nan")
        spec = (tn + smooth) / (tn + fp + smooth) if (tn + fp) > 0 else float("nan")
        dice_l.append(dice); sens_l.append(sens); spec_l.append(spec)

    def _nanmean_fg(v):
        if k <= 1:
            return float("nan")
        vals = [x for x in v[1:] if not math.isnan(x)]
        return float(np.mean(vals)) if vals else float("nan")

    tp_s = int(diag[1:].sum()); fp_s = int((col[1:] - diag[1:]).sum()); fn_s = int((row[1:] - diag[1:]).sum())
    tn_s = int(cm[0, 0])
    den = 2 * tp_s + fp_s + fn_s
    micro_dice = (2 * tp_s + smooth) / (den + smooth) if den > 0 else float("nan")
    micro_sens = (tp_s + smooth) / (tp_s + fn_s + smooth) if (tp_s + fn_s) > 0 else float("nan")
    micro_spec = (tn_s + smooth) / (tn_s + fp_s + smooth) if (tn_s + fp_s) > 0 else float("nan")
    return (dice_l, sens_l, spec_l, _nanmean_fg(dice_l), _nanmean_fg(sens_l), _nanmean_fg(spec_l),
            micro_dice, micro_sens, micro_spec)


def per_class_metrics_3d(preds, labels, num_classes, smooth=1e-6, ignore_index=None):
    """(dice_list, sens_list, spec_list, macro_dice, macro_sens, macro_spec, micro_dice, micro_sens,
    micro_spec) as helpers.py:668-725 — one small device->host copy instead of 102 `.item()` calls."""
    t = _tally(preds, labels, ignore_index)
    cm = t.confusion.cpu().numpy()
    return metrics_from_confusion(cm, labels.numel(), smooth)


def sample_metrics(per_sample, voxels_per_sample: int, smooth: float = 1e-6) -> List[tuple]:
    """Per-case metrics: one per_class_metrics_3d 9-tuple per sample from the per-sample tallies of `eval_step`
    (`per_sample` = (nll [B], count [B], confusion [B,K,K]); only the confusion rows are read). `voxels_per_sample`
    counts every voxel of one sample as given, ignored ones included (metrics_from_confusion)."""
    cm = per_sample[2]
    cm = cm.cpu().numpy() if torch.is_tensor(cm) else np.asarray(cm)
    return [metrics_from_confusion(row, voxels_per_sample, smooth) for row in cm]


def _nanmean_fg(v) -> float:
    """per_class_metrics_3d's macro convention: the nanmean over classes 1..K-1 (NaN when none is defined)."""
    vals = [float(x) for x in list(v)[1:] if not math.isnan(float(x))]
    return float(np.mean(vals)) if vals else float("nan")


def _ranking(hist: np.ndarray):
    """(auroc [K], ap [K], auroc_tie_bound [K], tp [K,T+1], fp [K,T+1]) of one [K,2,T] histogram.
    tp[:, i] / fp[:, i] count the positives / negatives in bins >= i (threshold i / T); column T is 0."""
    h = np.asarray(hist, dtype=np.float64)
    pos, neg = h[:, 0], h[:, 1]
    k, bins = pos.shape
    zero = np.zeros((k, 1))
    tp = np.concatenate([np.cumsum(pos[:, ::-1], axis=1)[:, ::-1], zero], axis=1)
    fp = np.concatenate([np.cumsum(neg[:, ::-1], axis=1)[:, ::-1], zero], axis=1)
    P, N = tp[:, 0], fp[:, 0]
    with np.errstate(invalid="ignore", divide="ignore"):
        # trapezoids between the ROC points of thresholds i + 1 and i: width neg_i / N, mean height (tp_{i+1} + pos_i / 2) / P
        auroc = (neg * (tp[:, 1:] + 0.5 * pos)).sum(1) / (P * N)
        # sklearn's step AP: recall steps pos_i / P at precision tp_i / (tp_i + fp_i); empty steps add nothing
        prec = np.where(pos > 0, tp[:, :bins] / np.maximum(tp[:, :bins] + fp[:, :bins], 1), 0.0)
        ap = (pos * prec).sum(1) / P
        bound = 0.5 * (pos * neg).sum(1) / (P * N)
    undefined = (P == 0) | (N == 0)
    auroc[undefined] = np.nan
    bound[undefined] = np.nan
    ap[P == 0] = np.nan
    return auroc, ap, bound, tp, fp


def _as_numpy(t) -> np.ndarray:
    return t.detach().cpu().numpy() if torch.is_tensor(t) else np.asarray(t)


def curves_from_hist(hist) -> dict:
    """Per-class ROC and precision-recall curves from the softmax histogram of `eval_step(curves=T)` / `evaluate`
    (int64 [K,2,T]: hist[c,0,b] positives and hist[c,1,b] negatives of class c whose probability falls in bin b).

    Thresholds are t_i = i / T, i = 0..T; TP_i / FP_i count the positives / negatives in bins >= i. Per class c:
    ROC points (FP_i / N_c, TP_i / P_c) in order of falling threshold (`roc_thresholds` = t_T..t_0), PR points
    (recall TP_i / P_c, precision TP_i / (TP_i + FP_i)) for the i with TP_i + FP_i > 0 in order of rising threshold
    (`pr_thresholds`). `auroc` is the trapezoid area under the ROC points (NaN when P_c or N_c is 0), `ap` sklearn's
    step average precision sum_i (R_i - R_{i+1}) * Prec_i (NaN when P_c is 0): both equal sklearn's roc_auc_score /
    average_precision_score with the bin index as the score. Binning makes every positive-negative pair inside one
    bin a tie worth 1/2, so the unbinned AUROC differs by at most `auroc_tie_bound` = 1/2 sum_b pos_b * neg_b /
    (P_c * N_c). `macro_auroc` / `macro_ap` are the nanmeans over classes 1..K-1, as in per_class_metrics_3d."""
    h = _as_numpy(hist)
    if h.ndim != 3 or h.shape[1] != 2:
        raise ValueError(f"expected a [K,2,T] histogram, got {h.shape}")
    auroc, ap, bound, tp, fp = _ranking(h)
    k, bins = h.shape[0], h.shape[2]
    thr = np.arange(bins + 1, dtype=np.float64) / bins
    out = {k_: [] for k_ in ("fpr", "tpr", "roc_thresholds", "precision", "recall", "pr_thresholds")}
    for c in range(k):
        P, N = tp[c, 0], fp[c, 0]
        with np.errstate(invalid="ignore", divide="ignore"):
            out["fpr"].append(fp[c, ::-1] / N)
            out["tpr"].append(tp[c, ::-1] / P)
            out["roc_thresholds"].append(thr[::-1].copy())
            keep = (tp[c] + fp[c]) > 0
            out["precision"].append(tp[c][keep] / (tp[c][keep] + fp[c][keep]))
            out["recall"].append(tp[c][keep] / P)
            out["pr_thresholds"].append(thr[keep])
    out.update(auroc=auroc, ap=ap, auroc_tie_bound=bound, macro_auroc=_nanmean_fg(auroc), macro_ap=_nanmean_fg(ap))
    return out


def sample_curves(per_sample_hist) -> List[tuple]:
    """Per-case ranking metrics: one (auroc [K], ap [K], macro_auroc, macro_ap) per sample from the per-sample
    histograms of `eval_step(curves=T, per_sample=True)` ([B,K,2,T]), as curves_from_hist defines them. The ranking
    counterpart of `sample_metrics`."""
    h = _as_numpy(per_sample_hist)
    if h.ndim != 4 or h.shape[2] != 2:
        raise ValueError(f"expected a [B,K,2,T] histogram, got {h.shape}")
    out = []
    for row in h:
        auroc, ap, _, _, _ = _ranking(row)
        out.append((auroc, ap, _nanmean_fg(auroc), _nanmean_fg(ap)))
    return out


FIX24 = 2.0 ** -24   # unit of the fixed-point sums of the ensemble's confidence and uncertainty


def calibration_from_hist(calib, brier_sum=None, ece_bins: int = 15, unc=None, voxels=None) -> dict:
    """Calibration of the top-label confidence from the histogram of `SpctEnsemble.eval_step(calibration=T)` /
    `evaluate` (int64 [3,T]: per confidence bin b, i.e. conf in [b/T, (b+1)/T), the counted voxels n_b, the correct
    ones k_b (arg-max == label) and the summed confidence s_b in units of 2^-24; conf = max_c p̄_c).

    - `ece` / `mce`: expected / maximum calibration error over `ece_bins` equal-width bins, sum_B |k_B - s_B| / N and
      max_B |k_B / n_B - s_B / n_B| over non-empty B. The fine bins carry the confidence sum, so merging T / ece_bins
      of them is exact; T % ece_bins must be 0 (ValueError otherwise). calibration=960 gives the standard 15-bin ECE.
    - `reliability`: {"confidence", "accuracy", "count"} per coarse bin (NaN for empty bins).
    - `brier`: brier_sum / N, the mean over counted voxels of sum_c (p̄_c - [c == y])^2 (NaN without brier_sum).
    - `error_auroc` / `error_ap` / `error_auroc_tie_bound`: detecting errors (positives) by 1 - confidence, as
      curves_from_hist ranks (equal to sklearn's roc_auc_score / average_precision_score with the reversed bin index as
      the score; voxels of one bin are ties).
    - `coverage` / `risk` / `aurc`: keeping the voxels of bins >= i (most confident first) covers C_i / N of them at
      risk E_i / C_i (errors / kept), points in order of rising coverage for the non-empty prefixes; `aurc` is the
      trapezoid area under them from coverage 0, the first point's risk held down to 0.
    - `mean_entropy` / `mean_mutual_info`: the uncertainty sums `unc` (int64 [2], 2^-24 nats) over `voxels` positions
      (NaN without them).
    - `counted`, `errors`, `ece_bins`: N, its errors and the number of ECE bins.

    NaN rules: with no counted voxel every statistic above is NaN; with no error error_auroc is NaN (and error_ap, no
    positive); with no correct voxel error_auroc is NaN and error_ap is 1."""
    h = np.asarray(_as_numpy(calib), dtype=np.float64)
    if h.ndim != 2 or h.shape[0] != 3:
        raise ValueError(f"expected a [3,T] calibration histogram, got {h.shape}")
    bins = h.shape[1]
    if ece_bins < 1 or bins % ece_bins:
        raise ValueError(f"the {bins} confidence bins cannot be merged exactly into {ece_bins} (T % ece_bins != 0)")
    cnt, cor, csum = h[0], h[1], h[2] * FIX24
    n = cnt.sum()
    err = cnt - cor
    g = bins // ece_bins
    cn, kn, sn = (v.reshape(ece_bins, g).sum(1) for v in (cnt, cor, csum))
    with np.errstate(invalid="ignore", divide="ignore"):
        acc_b, conf_b = kn / cn, sn / cn
        gap = np.abs(kn - sn)
        ece = gap.sum() / n if n else float("nan")
        mce = float(np.max(np.abs(acc_b - conf_b)[cn > 0])) if n else float("nan")
        brier = float(brier_sum) / n if (brier_sum is not None and n) else float("nan")
    # error detection: score 1 - confidence, i.e. the bins in reverse order
    auroc, ap, bound, _, _ = _ranking(np.stack([err[::-1], cor[::-1]])[None])
    kept = np.cumsum(cnt[::-1])
    kept_err = np.cumsum(err[::-1])
    nz = kept > 0
    coverage = kept[nz] / n if n else np.zeros(0)
    risk = kept_err[nz] / kept[nz]
    if n:
        aurc = float(risk[0] * coverage[0] + np.sum(0.5 * (risk[1:] + risk[:-1]) * np.diff(coverage)))
    else:
        aurc = float("nan")
    mean_ent = mean_mi = float("nan")
    if unc is not None and voxels:
        u = np.asarray(_as_numpy(unc), dtype=np.float64) * FIX24
        mean_ent, mean_mi = float(u[0] / voxels), float(u[1] / voxels)
    return {"ece": float(ece), "mce": mce, "reliability": {"confidence": conf_b, "accuracy": acc_b, "count": cn},
            "brier": brier, "error_auroc": float(auroc[0]), "error_ap": float(ap[0]),
            "error_auroc_tie_bound": float(bound[0]), "coverage": coverage, "risk": risk, "aurc": aurc,
            "mean_entropy": mean_ent, "mean_mutual_info": mean_mi, "counted": int(n), "errors": int(err.sum()),
            "ece_bins": ece_bins}


def sample_calibration(per_sample_calib, per_sample_brier=None, ece_bins: int = 15) -> List[tuple]:
    """Per-case calibration: one (ece, brier, error_auroc) per sample from the per-sample histograms of
    `SpctEnsemble.eval_step(calibration=T, per_sample=True)` ([B,3,T]) and its per-sample Brier sums ([B]), as
    calibration_from_hist defines them. The calibration counterpart of `sample_curves`."""
    h = _as_numpy(per_sample_calib)
    if h.ndim != 3 or h.shape[1] != 3:
        raise ValueError(f"expected a [B,3,T] calibration histogram, got {h.shape}")
    b = _as_numpy(per_sample_brier) if per_sample_brier is not None else [None] * len(h)
    out = []
    for row, br in zip(h, b):
        c = calibration_from_hist(row, br, ece_bins)
        out.append((c["ece"], c["brier"], c["error_auroc"]))
    return out


def temperature_grid(t_max: float = 8.0, points: int = 33) -> np.ndarray:
    """The inverse temperatures β = 1/T of `SpctEnsemble.fit_temperature`'s grid, ascending, rounded to fp32 (the values
    the fit kernel evaluates): `points` (odd, 5..63) temperatures spaced geometrically over [1/t_max, t_max] (t_max > 1
    and finite), so that T = 1 is the middle point, exactly."""
    if isinstance(points, bool) or int(points) != points or not 5 <= points <= 63 or points % 2 == 0:
        raise ValueError(f"points must be an odd integer in [5, 63], got {points!r}")
    if not (math.isfinite(t_max) and t_max > 1.0):
        raise ValueError(f"t_max must be finite and > 1, got {t_max!r}")
    half = (int(points) - 1) // 2
    e = np.arange(-half, half + 1, dtype=np.float64) / half
    beta = np.power(float(t_max), e)
    beta[half] = 1.0
    return beta.astype(np.float32).astype(np.float64)


def temperature_from_sums(betas, sums, counted) -> dict:
    """The temperature that minimises the mean nll of the tempered pooled softmax, from the fit statistics of
    `ops.prob_temp_fit` on a grid of inverse temperatures: betas [G] ascending, sums [2,G] (sum over the counted voxels
    of the nll f(β_g) and of its derivative f'(β_g) = dnll/dβ), counted voxels.

    f is convex in β, so f' is non-decreasing: the minimum lies in the interval where the summed f' changes sign. There
    the estimate is the minimiser of the cubic Hermite interpolant of the nll from its values and derivatives at both
    ends (the secant root of f' if the cubic has no minimum inside); with no sign change on the grid it is the end point
    the slope points to and `at_bound` is True.

    Returns {"temperature": 1/β̂, "nll": the INTERPOLATED mean nll at β̂, "nll_at_1": the mean nll at β = 1 (None when
    1 is not a grid point), "grid": {"temperature": 1/betas, "nll": mean f, "dnll": mean f' (per unit β)},
    "counted", "at_bound"}. ValueError when no voxel was counted."""
    b = np.asarray(_as_numpy(betas), dtype=np.float64).reshape(-1)
    s = np.asarray(_as_numpy(sums), dtype=np.float64)
    n = int(np.asarray(_as_numpy(counted) if torch.is_tensor(counted) else counted).reshape(-1)[0])
    if s.shape != (2, b.size):
        raise ValueError(f"sums must be [2,{b.size}], got {s.shape}")
    if b.size < 2 or np.any(np.diff(b) <= 0) or b[0] <= 0 or not np.all(np.isfinite(b)):
        raise ValueError("betas must be at least two positive, finite, strictly ascending values")
    if n <= 0:
        raise ValueError("no counted voxel: every label is ignore_index or outside [0, K)")
    f, d = s[0] / n, s[1] / n
    at_bound = False
    if d[0] >= 0.0 or d[-1] <= 0.0:
        i = 0 if d[0] >= 0.0 else b.size - 1
        at_bound = d[i] != 0.0
        beta, nll = b[i], f[i]
    else:
        i = int(np.argmax(d >= 0.0)) - 1           # d[i] < 0 <= d[i + 1]
        a, h = b[i], b[i + 1] - b[i]
        c1 = h * d[i]
        c2 = 3.0 * (f[i + 1] - f[i]) - h * (2.0 * d[i] + d[i + 1])
        c3 = 2.0 * (f[i] - f[i + 1]) + h * (d[i] + d[i + 1])
        t = None
        if c3 != 0.0:                              # p'(t) = c1 + 2 c2 t + 3 c3 t^2: the root where p'' > 0
            disc = c2 * c2 - 3.0 * c1 * c3
            if disc >= 0.0:
                q = -(c2 + math.copysign(math.sqrt(disc), c2))
                for r in ((q / (3.0 * c3)) if q != 0.0 else None, (c1 / q) if q != 0.0 else None):
                    if r is not None and 0.0 <= r <= 1.0 and 2.0 * c2 + 6.0 * c3 * r > 0.0:
                        t = r
                        break
        elif c2 > 0.0:
            t = -c1 / (2.0 * c2)
        if t is None or not 0.0 <= t <= 1.0:      # the cubic degenerates: secant root of f'
            t = -d[i] / (d[i + 1] - d[i])
        beta = a + t * h
        nll = f[i] + t * (c1 + t * (c2 + t * c3))
    one = np.flatnonzero(b == 1.0)
    return {"temperature": float(1.0 / beta), "nll": float(nll), "nll_at_1": float(f[one[0]]) if one.size else None,
            "grid": {"temperature": 1.0 / b, "nll": f, "dnll": d}, "counted": n, "at_bound": bool(at_bound)}


def per_class_metrics_2d(preds, labels, num_classes, smooth=1e-6, ignore_index=None):
    """2-D twin (helpers.py:728-779): same counting rules on [B,K,H,W] logits."""
    return per_class_metrics_3d(preds, labels, num_classes, smooth, ignore_index)


LOSS_REGISTRY = {
    "ce_plus_macro_dice": lambda logits, labels, nc, ignore_index: ce_plus_macro_dice_loss(
        logits, labels, nc, ignore_index=ignore_index),
}


# Everything else of the reference's helpers.py (DICOM ingest, legacy augmentation, visualisers, unused losses:
# helpers.py:43-662, 811-943) is outside the hot path; those names resolve to the reference's module when a reference
# checkout is on sys.path, so `innovative3D/datasets.py:31-34` of the reference imports them from here unchanged.
from ._fallthrough import module_getattr as _module_getattr  # noqa: E402

__getattr__ = _module_getattr(__name__, "helpers", "only the loss / step-metric functions of the hot path are rebuilt here")
