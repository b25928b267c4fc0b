"""GPU: the Lightning surface this package's callers drive. The fit loop of the Lightning stand-in
(`innovative3D._lightning`: `Trainer`, `ModelCheckpoint`, `EarlyStopping`, `CSVLogger`, checkpoint files, reload and
resume) trains SPFF-UNet on a synthetic DataModule the way the reference's `train.py` sets it up (train.py:1398-1583)
and reloads it the way `test.py:615-644` does. The step surface of the SPCT classes (`_shared_step`, `training_step`,
`validation_step`, `apply_unified_loss`: reference models.py:479-588, unified_loss.py:114-144) is checked against the
oracle. Lightning itself is the repo's stand-in when the real package is absent."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _synthetic_datamodule():
    from torch.utils.data import DataLoader, Dataset

    from oracle import spff_oracle as O

    class Phantoms(Dataset):
        """(img [1,F,H,W] fp32, lbl [F,H,W] int64) like DicomDataset3D.__getitem__ (datasets.py:227-238)."""

        def __init__(self, n, seed):
            x, lab = O.phantom_batch(n, 64, 64, seed=seed, ignore_frac=0.01)
            self.x, self.lab = x, lab

        def __len__(self):
            return len(self.x)

        def __getitem__(self, i):
            return self.x[i], self.lab[i]

    class SyntheticDataModule:
        """Constructor and loader methods of MultiDicomDataModule3D (datasets.py:280-340)."""

        def __init__(self, configs, batch_size=1, num_frames=5):
            self.configs, self.batch_size, self.num_frames = configs, batch_size, num_frames
            self.stages = []

        def setup(self, stage=None):
            self.stages.append(stage)
            self.train_set, self.val_set, self.test_set = Phantoms(6, 1), Phantoms(2, 2), Phantoms(2, 3)

        def train_dataloader(self):
            return DataLoader(self.train_set, batch_size=self.batch_size, shuffle=True)

        def val_dataloader(self):
            return DataLoader(self.val_set, batch_size=self.batch_size, shuffle=False)

        def test_dataloader(self):
            return DataLoader(self.test_set, batch_size=self.batch_size, shuffle=False)

    return SyntheticDataModule


def _fit(builder, folder, max_epochs, ckpt_path=None):
    """One `Trainer(...).fit` with the callbacks train.py:1430-1458 configures: last + best checkpoint on
    val_macro_dice, early stopping on it, a CSV logger. Returns the module, its logger and its best-checkpoint callback."""
    from innovative3D import _lightning as L
    dm = _synthetic_datamodule()([], batch_size=1, num_frames=5)
    dm.setup("fit")
    lit = builder()
    best = L.ModelCheckpoint(dirpath=folder, filename="best-{epoch:02d}-{val_macro_dice:.4f}", monitor="val_macro_dice",
                             mode="max", save_last=True, save_top_k=1)
    stop = L.EarlyStopping(monitor="val_macro_dice", mode="max", patience=10)
    logger = L.CSVLogger(save_dir=str(folder), name="logs")
    L.Trainer(max_epochs=max_epochs, accelerator="gpu", devices=1, logger=logger,
              callbacks=[best, stop]).fit(lit, datamodule=dm, ckpt_path=ckpt_path)
    return lit, logger, best


def test_trainer_fit_checkpoints_reload_and_resume(tmp_path):
    from innovative3D import _lightning as L
    from innovative3D import config as C
    variants = dict((v[0], v[1]) for v in C.VARIANTS)
    builder = variants["SPFF-UNet"]
    folder = tmp_path / "SPFF-UNet" / "seed42"
    L.seed_everything(42)
    lit, logger, best = _fit(builder, folder, max_epochs=2)
    assert (folder / "last.ckpt").is_file()
    best_files = sorted(folder.glob("best-*.ckpt"))
    assert len(best_files) == 1 and str(best_files[0]) == best.best_model_path, best_files
    # one train and one val row per epoch, val_macro_dice monitored
    train_rows = [r for r in logger.rows if "train_loss" in r]
    val_rows = [r for r in logger.rows if "val_macro_dice" in r]
    assert [r["epoch"] for r in train_rows] == [0, 1] and [r["epoch"] for r in val_rows] == [0, 1]
    assert all(np.isfinite(r["val_macro_dice"]) for r in val_rows) and all(np.isfinite(r["train_loss"]) for r in train_rows)
    assert float(train_rows[-1]["train_loss"]) < float(train_rows[0]["train_loss"])

    # ---- reload like test.py:615-644: prototype from the registry, PL restore, manual fallback ------------------
    ckpt_path = str(folder / "last.ckpt")
    proto = builder()
    ModelCls = proto.__class__
    dev = torch.device("cuda")
    # "PL restore attempt" (test.py:626-630). For this class it raises with real Lightning and the reference's own
    # module too: the saved hyper-parameter `is_3d` travels through **kw into UNet3D_SpectralCore.__init__
    # (models.py:1558-1564 -> :1547-1555 -> :654) - which is why test.py carries the manual fallback below
    with pytest.raises(TypeError):
        ModelCls.load_from_checkpoint(ckpt_path, map_location=dev)
    ck = torch.load(ckpt_path, map_location=dev, weights_only=False)
    assert {"state_dict", "optimizer_states", "epoch", "global_step", "hyper_parameters"} <= set(ck)
    assert ck["epoch"] == 1 and ck["global_step"] == 12
    proto.load_state_dict(ck["state_dict"], strict=False)
    manual = proto.to(dev).eval()
    x = _synthetic_datamodule()([], 1, 5)
    x.setup("test")
    xb, _ = next(iter(x.test_dataloader()))
    # a class without **kw restores through the PL path: SP_UNet (models.py:1585-1592)
    sp = variants["SP_UNet"]()
    sp_path = str(tmp_path / "sp_unet.ckpt")
    torch.save({"state_dict": sp.state_dict(), "hyper_parameters": dict(sp.hparams)}, sp_path)
    sp2 = type(sp).load_from_checkpoint(sp_path, map_location=dev)
    assert all(torch.equal(a.cpu(), b.cpu()) for a, b in zip(sp.state_dict().values(), sp2.state_dict().values()))
    with torch.no_grad():
        a, b = manual(xb.to(dev)), manual(xb.to(dev))
    assert a.shape == (1, 13, 5, 64, 64) and torch.equal(a, b)
    for k, v in ck["state_dict"].items():                       # the trained weights, not the seed's
        assert torch.equal(manual.state_dict()[k].cpu(), v.cpu()), k
    fresh = builder().to(dev).eval()
    with torch.no_grad():
        assert not torch.equal(fresh(xb.to(dev)), a)

    # ---- resume: a second fit from last.ckpt (train.py:504-509, 1509-1516) runs only the missing epoch ---------
    _, logger2, _ = _fit(builder, folder, max_epochs=3, ckpt_path=ckpt_path)
    epochs = sorted(int(r["epoch"]) for r in logger.rows + logger2.rows)
    assert epochs == [0, 0, 1, 1, 2, 2]
    ck2 = torch.load(folder / "last.ckpt", map_location="cpu", weights_only=False)
    assert ck2["epoch"] == 2 and ck2["global_step"] == 18


@pytest.mark.parametrize("variant", ["SPFF-UNet", "PlainCore_UNet", "SP_UNet"])
def test_lightning_step_surface_matches_the_oracle(variant):
    """training_step returns the differentiable ce_plus_macro_dice loss and logs the reference's metric names;
    validation_step returns {'val_loss': ...} and logs val_macro_dice (the monitored quantity)."""
    from innovative3D import config as C
    from oracle import spff_oracle as O
    lit = dict((v[0], v[1]) for v in C.VARIANTS)[variant]().cuda()
    x, lab = O.phantom_batch(2, 32, 32, seed=77, ignore_frac=0.02)
    batch = (x.cuda(), lab.cuda())
    loss = lit.training_step(batch, 0)
    assert loss.requires_grad and loss.dim() == 0
    with torch.no_grad():
        logits = lit(batch[0]).cpu()
    want = O.ce_plus_macro_dice_loss(logits, lab)
    assert abs(float(loss) - float(want)) < 1e-5
    mo = O.per_class_metrics_3d(logits, lab, 13, ignore_index=255)
    names = {"train_loss", "train_macro_dice", "train_micro_dice", "train_macro_sens", "train_macro_spec", "train_micro_sens",
             "train_micro_spec"} | {f"train_{m}_class_{i}" for m in ("dice", "sens", "spec") for i in range(13)}
    assert names <= set(lit.logged), sorted(names - set(lit.logged))
    assert abs(float(lit.logged["train_macro_dice"]) - mo[3]) < 1e-12
    np.testing.assert_allclose([float(lit.logged[f"train_dice_class_{i}"]) for i in range(13)], mo[0], rtol=1e-12, equal_nan=True)
    loss.backward()
    g = [p.grad for p in lit.parameters() if p.grad is not None]
    assert len(g) >= 40 and all(torch.isfinite(t).all() for t in g)
    # the same through a dict batch and list-wrapped tensors (models.py:480-481)
    loss2 = lit.training_step({"image": [batch[0]], "label": [batch[1]]}, 0)
    assert abs(float(loss2) - float(loss)) < 1e-6
    lit.eval()
    with torch.no_grad():
        out = lit.validation_step(batch, 0)
    assert set(out) == {"val_loss"} and abs(float(out["val_loss"]) - float(want)) < 1e-5
    assert abs(float(lit.logged["val_macro_dice"]) - mo[3]) < 1e-12
    with torch.no_grad():
        t = lit.test_step(batch, 0)
    assert abs(float(t) - float(want)) < 1e-5 and "test_macro_dice" in lit.logged


def test_apply_unified_loss_patches_every_lit_class():
    """unified_loss.apply_unified_loss (unified_loss.py:114-144): every Lightning class of innovative3D.models except
    BaseLitModel gets the unified train/val/test steps; they compute the same loss and log the macro/micro metrics."""
    from innovative3D import models as M
    from innovative3D import unified_loss as U
    from oracle import spff_oracle as O
    saved = {n: (c.training_step, c.validation_step, c.test_step) for n, c in vars(M).items()
             if isinstance(c, type) and issubclass(c, M.pl.LightningModule)}
    try:
        patched = U.apply_unified_loss()
        assert "BaseLitModel" not in patched
        assert {"LitSPCT_EFiLM_FourierGate", "LitSPCT_ControlUNet", "LitSPCT_SEspec", "LitCicek3DUNet_DepthAdapter_Published"} <= set(patched)
        lit = M.LitSPCT_EFiLM_FourierGate().cuda()
        assert lit.training_step.__func__ is U._training_step
        x, lab = O.phantom_batch(2, 32, 32, seed=78, ignore_frac=0.02)
        # labels as [B,1,F,H,W] exercise the canonicalisation (unified_loss.py:56-75, models.py:68-83)
        loss = lit.training_step((x.cuda(), lab.cuda().unsqueeze(1)), 0)
        with torch.no_grad():
            logits = lit(x.cuda()).cpu()
        assert abs(float(loss) - float(O.ce_plus_macro_dice_loss(logits, lab))) < 1e-5 and loss.requires_grad
        mo = O.per_class_metrics_3d(logits, lab, 13, ignore_index=255)
        assert abs(float(lit.logged["train_macro_dice"]) - mo[3]) < 1e-12
        assert abs(float(lit.logged["train_micro_dice"]) - mo[6]) < 1e-12
        with torch.no_grad():
            v = lit.validation_step({"image": x.cuda(), "label": lab.cuda()}, 0)
        assert abs(float(v) - float(loss)) < 1e-5 and "val_macro_dice" in lit.logged
    finally:
        for n, (a, b, c) in saved.items():
            cls = getattr(M, n)
            cls.training_step, cls.validation_step, cls.test_step = a, b, c
