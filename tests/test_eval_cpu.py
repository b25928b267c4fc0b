"""CPU half of the fused evaluation step: the per-case metrics (helpers.sample_metrics) and the voxel count that SP_UNet's
padded evaluation uses, against the oracle's per_class_metrics_3d."""
import math

import numpy as np
import torch


def _same(a, b):
    """9-tuples equal, NaN == NaN (absent classes), to fp64 rounding."""
    for x, y in zip(a, b):
        xs, ys = (list(x), list(y)) if isinstance(x, (list, tuple)) else ([x], [y])
        assert len(xs) == len(ys)
        for u, v in zip(xs, ys):
            assert (math.isnan(u) and math.isnan(v)) or abs(u - v) <= 1e-12 * max(1.0, abs(v)), (u, v)


def test_sample_metrics_match_per_class_metrics_3d_per_sample():
    from innovative3D.helpers import sample_metrics
    from oracle import spff_oracle as O
    k, f, h, w = 6, 5, 7, 9
    g = torch.Generator().manual_seed(3)
    logits = torch.randn(4, k, f, h, w, generator=g)
    labels = torch.randint(0, k, (4, f, h, w), generator=g)
    labels[1][labels[1] == 3] = 2                      # class 3 absent in sample 1's labels ...
    logits[1, 3] = -1e3                                # ... and never predicted there: NaN Dice / sensitivity
    labels[2][labels[2] == 4] = 5                      # class 4 absent in sample 2's labels but predicted: Dice 0
    labels[torch.rand(labels.shape, generator=g) < 0.15] = 255   # ignored voxels: true negatives of every class
    labels[3] = 255                                    # a sample with nothing valid
    cm = np.stack([O.confusion(logits[i].argmax(0), labels[i], k, 255) for i in range(4)])
    got = sample_metrics((None, None, torch.from_numpy(cm)), f * h * w)
    assert len(got) == 4
    for i in range(4):
        _same(got[i], O.per_class_metrics_3d(logits[i:i + 1], labels[i:i + 1], k, ignore_index=255))
    assert math.isnan(got[1][0][3]) and math.isnan(got[1][1][3])
    assert got[2][0][4] < 1e-6


def test_sp_unet_padded_evaluation_counts_the_unpadded_voxels():
    """SP_UNet evaluates on the padded grid with ignore_index outside the crop; its metrics equal those of the cropped
    logits only when the voxel count is the unpadded one (ignored voxels are true negatives)."""
    from innovative3D import models as M
    from innovative3D.helpers import metrics_from_confusion
    from oracle import spff_oracle as O
    k = 13
    g = torch.Generator().manual_seed(5)
    x = torch.randn(2, 1, 5, 24, 40, generator=g)
    y = torch.randint(0, k, (2, 5, 24, 40), generator=g)
    y[torch.rand(y.shape, generator=g) < 0.05] = 255
    lit = M.LitSPCT_SEspec(num_classes=k)
    x_pad, y_pad, orig = lit._padded_batch((x, y))
    assert tuple(x_pad.shape[2:]) == (16, 32, 48) and orig == (5, 24, 40)
    assert int((y_pad != 255).sum()) == int((y != 255).sum())
    logits_pad = torch.randn(2, k, *x_pad.shape[2:], generator=g)
    cm = O.confusion(logits_pad.argmax(1), y_pad, k, 255)
    voxels = M._eval_voxels((x, y))
    assert voxels == y.numel()
    _same(metrics_from_confusion(cm, voxels),
          O.per_class_metrics_3d(M._center_crop_to_3d(logits_pad, orig), y, k, ignore_index=255))
    padded = metrics_from_confusion(cm, y_pad.numel())
    assert padded[2] != O.per_class_metrics_3d(M._center_crop_to_3d(logits_pad, orig), y, k, ignore_index=255)[2]
