"""CPU: the C-ABI library loads and exports every symbol include/spff_b200.h declares; the plugin
surface (config.VARIANTS, module classes, parameter names, same-seed initialisation) matches the
reference fixtures; host-side metric logic matches the reference's outputs; no-GPU behaviour is loud."""
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def header_symbols():
    src = open(os.path.join(ROOT, "include", "spff_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(spff_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from spff_b200 import _lib
    syms = header_symbols()
    assert len(syms) >= 30
    for s in syms:
        assert hasattr(_lib.lib, s), f"{s} declared in include/spff_b200.h but not exported"
    assert sorted(_lib.exported_symbols()) == syms, "ctypes prototypes and header disagree"
    assert _lib.lib.spff_version() >= 100


def test_no_gpu_is_an_error_not_a_fallback():
    from spff_b200 import _lib
    if torch.cuda.is_available():
        pytest.skip("needs a machine without a GPU")
    assert _lib.lib.spff_device_check() == -2          # SPFF_ERR_UNSUPPORTED_ARCH
    assert b"CUDA" in _lib.lib.spff_last_error() or b"device" in _lib.lib.spff_last_error()
    from innovative3D import config as C
    lit = C.VARIANTS[0][1]()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        lit(torch.zeros(1, 1, 5, 16, 16))
    from innovative3D import helpers as H
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        H.ce_plus_macro_dice_loss(torch.zeros(1, 13, 5, 8, 8), torch.zeros(1, 5, 8, 8, dtype=torch.long), 13)


def test_variants_registry_surface():
    from innovative3D import config as C
    names = [v[0] for v in C.VARIANTS]
    assert names[:1] == ["SPFF-UNet"] and {"E_SP_UNet", "FG_SP_UNet", "SP_UNet", "PlainCore_UNet", "3DUNet"} <= set(names)
    assert (C.NUM_CLASSES, C.NUM_FRAMES, C.IGNORE_INDEX, C.BATCH_SIZE, C.BEST_LR, C.SEEDS) == (13, 5, 255, 1, 1e-4, [42, 123, 999])
    assert names[:6] == C.B200_VARIANT_NAMES     # the reference's other families (if a checkout is on the path) come after
    for name, builder, dm, ckpt in C.VARIANTS[:6]:
        lit = builder()
        assert hasattr(lit, "model") and lit.hparams.num_classes == 13 and callable(dm)
        opt = lit.configure_optimizers()
        if name == "3DUNet":     # SGD like the paper (config.py:287-290, models.py:844-846)
            assert isinstance(opt, torch.optim.SGD) and opt.defaults["momentum"] == 0.99 and opt.defaults["lr"] == 1e-2
            continue
        assert isinstance(opt["optimizer"], torch.optim.Adam) and opt["lr_scheduler"]["monitor"] == "val_macro_dice"


@pytest.mark.usefixtures("reference_threads")
def test_same_seed_same_init_and_keys_as_reference():
    """Constructing with the same seed draws bit-identical weights to the reference's constructors
    (checksums in tests/golden/init_seed42.npz come from the reference itself)."""
    from innovative3D import config as C
    z = np.load(os.path.join(GOLD, "init_seed42.npz"))
    ref = {}
    for key in z.files:
        variant, name = key.split("|")
        ref.setdefault(variant, {})[name] = z[key]
    builders = dict((v[0], v[1]) for v in C.VARIANTS)
    for variant, entries in ref.items():
        torch.manual_seed(42)
        sd = builders[variant]().state_dict()
        assert sorted(sd) == sorted(entries), variant
        for name, rec in entries.items():
            t = sd[name].double()
            assert tuple(t.shape) == tuple(int(v) for v in rec[:-2]), (variant, name)
            assert float(t.sum()) == rec[-2] and float(t.abs().sum()) == rec[-1], (variant, name)


def test_lazy_freq_mask_quirk():
    """FourierGate's mask appears at the first forward (models.py:1532-1535): absent from a fresh
    state_dict, present (under both aliases) afterwards, loadable from a checkpoint that has it."""
    from innovative3D import models as M
    g = M.FourierGate3D()
    assert list(g.state_dict()) == ["mag_scale"]
    assert g.ensure_mask(5, "cpu") and not g.ensure_mask(5, "cpu")
    assert sorted(g.state_dict()) == ["_mask", "freq_mask", "mag_scale"] and g.freq_mask.shape == (1, 1, 3, 1, 1)
    g2 = M.FourierGate3D()
    sd = {k: v * 2 for k, v in g.state_dict().items()}
    g2.load_state_dict(sd)
    assert float(g2.freq_mask.sum()) == 6.0
    with pytest.raises(RuntimeError):
        g(torch.zeros(1, 4, 5, 8, 8))        # sub-modules have no eager path


def test_metrics_from_confusion_matches_reference_fixture():
    from innovative3D import helpers as H
    from oracle import spff_oracle as O
    for path in sorted(p for p in os.listdir(GOLD) if p.startswith("case")):
        z = np.load(os.path.join(GOLD, path))
        variant, b, h, w, ign, seed = [str(v) for v in z["case"]]
        _, lab = O.phantom_batch(int(b), int(h), int(w), seed=int(seed), ignore_frac=float(ign))
        logits = torch.from_numpy(z["logits"])
        cm = O.confusion(logits.argmax(1), lab, 13, 255)
        m = H.metrics_from_confusion(cm, lab.numel())
        np.testing.assert_allclose(np.array(m[0]), z["dice_list"], rtol=1e-12, equal_nan=True)
        np.testing.assert_allclose(np.array(m[1]), z["sens_list"], rtol=1e-12, equal_nan=True)
        np.testing.assert_allclose(np.array(m[2]), z["spec_list"], rtol=1e-12, equal_nan=True)
        np.testing.assert_allclose(np.array(m[3:]), z["scalars"], rtol=1e-12, equal_nan=True)


def test_metrics_edge_cases():
    from innovative3D import helpers as H
    cm = np.zeros((13, 13), np.int64)
    m = H.metrics_from_confusion(cm, 0)                      # empty input: everything undefined
    assert all(np.isnan(v) for v in m[0]) and np.isnan(m[3]) and np.isnan(m[6])
    cm[0, 0] = 10                                            # background only
    m = H.metrics_from_confusion(cm, 10)
    assert m[0][0] == pytest.approx(1.0) and np.isnan(m[3]) and np.isnan(m[6]) and m[8] == pytest.approx(1.0)
    cm[3, 5] = 4                                             # class 3 present but always predicted as 5
    m = H.metrics_from_confusion(cm, 14)
    assert m[0][3] == pytest.approx(1e-6 / (4 + 1e-6)) and m[0][5] == pytest.approx(1e-6 / (4 + 1e-6))
    assert np.isnan(m[1][5]) and m[1][3] == pytest.approx(1e-6 / (4 + 1e-6))


def test_shard_range_partitions():
    from spff_b200 import dp
    for total in (0, 1, 7, 256, 1000):
        for world in (1, 2, 3, 8):
            parts = [dp.shard_range(total, r, world) for r in range(world)]
            assert parts[0][0] == 0 and parts[-1][1] == total
            assert all(a[1] == b[0] for a, b in zip(parts, parts[1:]))
            sizes = [hi - lo for lo, hi in parts]
            assert max(sizes) - min(sizes) <= 1


def test_plateau_lr_matches_torch_scheduler():
    """PlateauLR == torch ReduceLROnPlateau(mode='max', factor=0.5, patience=5) on the same metric series."""
    from spff_b200.sched import PlateauLR
    import random
    rnd = random.Random(0)
    series = [0.1, 0.2, 0.25] + [0.25 + rnd.uniform(-0.02, 0.00001) for _ in range(40)] + [0.6] + [0.5] * 20
    p = torch.nn.Parameter(torch.zeros(1))
    opt = torch.optim.Adam([p], lr=1e-4)
    sch = torch.optim.lr_scheduler.ReduceLROnPlateau(opt, mode="max", factor=0.5, patience=5)
    mine = PlateauLR(1e-4, mode="max", factor=0.5, patience=5)
    for v in series:
        sch.step(v)
        assert mine.step(v) == pytest.approx(opt.param_groups[0]["lr"], rel=1e-12, abs=0)
    assert mine.lr < 1e-4


def test_sample_group_sizing(monkeypatch):
    """SpffEngine.fit_group: the largest group <= the request whose buffers fit in 45 % of the free HBM
    (26.5 level-1 tensors per slice for a training step, 16.7 for inference)."""
    from spff_b200.engine import SpffEngine
    free = 170 * 2 ** 30
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda device=None: (free, 183 * 2 ** 30))
    # the bench slices (5 x 128 x 128): 139 MB per slice for training -> the requested 256 fits
    assert SpffEngine.fit_group(256, 5, 128, 128, "cuda:0", train=True) == 256
    # native 512 x 512 slices: 2.2 GB per slice for training, 1.4 GB for inference
    per_train = 26.5 * 5 * 512 * 512 * 64
    assert SpffEngine.fit_group(256, 5, 512, 512, "cuda:0", train=True) == int(0.45 * free / per_train) == 36
    assert SpffEngine.fit_group(256, 5, 512, 512, "cuda:0", train=False) == int(0.45 * free / (16.7 * 5 * 512 * 512 * 64)) == 58
    assert SpffEngine.fit_group(8, 5, 512, 512, "cuda:0", train=True) == 8
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda device=None: (2 ** 30, 183 * 2 ** 30))
    assert SpffEngine.fit_group(256, 5, 512, 512, "cuda:0", train=True) == 1      # never below one slice
    assert SpffEngine._groups(10, 4) == [(0, 4), (4, 8), (8, 10)]                  # ragged last group


def test_depth_matrix_matches_interpolate():
    """spff_b200.cicek.depth_matrix == F.interpolate(mode='trilinear', align_corners=False) along D (models.py:153-163)."""
    from spff_b200.cicek import depth_matrix
    for din, dout in ((5, 16), (16, 5), (3, 16), (16, 16), (7, 4)):
        eye = torch.eye(din).reshape(din, 1, din, 1, 1)
        ref = torch.nn.functional.interpolate(eye, size=(dout, 1, 1), mode="trilinear", align_corners=False)
        assert torch.allclose(depth_matrix(din, dout), ref.reshape(din, dout).t(), atol=1e-6), (din, dout)
