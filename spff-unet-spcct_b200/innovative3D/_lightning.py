"""Minimal stand-in for the parts of pytorch_lightning the hot path's callers touch, used only when the real
package is not installed (it is a third-party dependency of the reference, `requirements.txt:70`, and absent from
this image). With Lightning present, `innovative3D.models` subclasses the real `pl.LightningModule` and nothing here
is used.

Two levels:
  * `LightningModule`, `LightningDataModule`, `seed_everything` — what `innovative3D.models` itself needs.
  * `Trainer`, `Callback`, `ModelCheckpoint`, `EarlyStopping`, `Logger`, `rank_zero_only` and `install()` — a
    single-device, epoch-based fit loop with Lightning's call order, metric aggregation (`self.log(..., on_epoch=True)`
    -> epoch means in `trainer.callback_metrics` -> logger / callbacks), `ReduceLROnPlateau` monitoring, checkpoint
    files with Lightning's key names (`state_dict`, `optimizer_states`, `hyper_parameters`, `epoch`, `global_step`) and
    resume. `install()` registers these under the `pytorch_lightning` module names so that the reference's unmodified
    `train.py` / `test.py` can drive this package on a machine without Lightning (tests/test_trainpy_gpu.py runs the
    fit loop, checkpoints, reload and resume).
    It is deliberately small: one optimizer, no distributed strategies, no sanity-check / test / predict loops.
"""
from __future__ import annotations

import inspect
import os
import random
import sys
import types
from pathlib import Path
from types import SimpleNamespace
from typing import Any, Dict, List, Optional

import torch
import torch.nn as nn

__version__ = "0.0-spff-standin"


class _HParams(dict):
    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError as e:
            raise AttributeError(k) from e

    def __setattr__(self, k, v):
        self[k] = v


class LightningModule(nn.Module):
    def __init__(self, *a, **kw):
        super().__init__()
        self._hparams = _HParams()
        self.logged: Dict[str, Any] = {}
        self.trainer: Optional["Trainer"] = None

    @property
    def hparams(self):
        return self._hparams

    def save_hyperparameters(self, *args, **kwargs):
        for a in args:
            if isinstance(a, dict):
                self._hparams.update(a)
        self._hparams.update(kwargs)

    def log(self, name, value, *a, **kw):
        self.logged[name] = value
        if self.trainer is not None:
            self.trainer._record(name, value)

    def log_dict(self, d, *a, **kw):
        for k, v in d.items():
            self.log(k, v, *a, **kw)

    @property
    def device(self):
        try:
            return next(self.parameters()).device
        except StopIteration:
            return torch.device("cpu")

    @property
    def current_epoch(self) -> int:
        return self.trainer.current_epoch if self.trainer is not None else 0

    @property
    def global_step(self) -> int:
        return self.trainer.global_step if self.trainer is not None else 0

    @classmethod
    def load_from_checkpoint(cls, checkpoint_path, map_location=None, strict: bool = True, **kwargs):
        """cls(**hyper_parameters) + load_state_dict, as Lightning restores a module (test.py:626-629)."""
        ckpt = torch.load(checkpoint_path, map_location=map_location, weights_only=False)
        hp = dict(ckpt.get("hyper_parameters", {}))
        hp.update(kwargs)
        params = inspect.signature(cls.__init__).parameters
        if not any(p.kind == inspect.Parameter.VAR_KEYWORD for p in params.values()):
            hp = {k: v for k, v in hp.items() if k in params}
        obj = cls(**hp)
        obj.load_state_dict(ckpt["state_dict"], strict=strict)
        if map_location is not None and not isinstance(map_location, dict):
            obj = obj.to(map_location)
        return obj


class LightningDataModule:
    def prepare_data(self):
        pass

    def setup(self, stage=None):
        pass


def seed_everything(seed: int, workers: bool = False):
    import numpy as np
    random.seed(seed)
    np.random.seed(seed)
    torch.manual_seed(seed)
    return seed


def rank_zero_only(fn):
    """Single process here (or one process per GPU under torchrun: only RANK 0 runs `fn`)."""
    def wrapped(*a, **kw):
        if int(os.environ.get("RANK", "0")) == 0:
            return fn(*a, **kw)
        return None
    wrapped.__name__ = getattr(fn, "__name__", "wrapped")
    return wrapped


class Callback:
    def setup(self, trainer, pl_module, stage=None): pass
    def on_fit_start(self, trainer, pl_module): pass
    def on_train_start(self, trainer, pl_module): pass
    def on_train_epoch_start(self, trainer, pl_module): pass
    def on_train_batch_end(self, trainer, pl_module, outputs, batch, batch_idx): pass
    def on_validation_epoch_start(self, trainer, pl_module): pass
    def on_validation_batch_end(self, trainer, pl_module, outputs, batch, batch_idx, dataloader_idx=0): pass
    def on_validation_epoch_end(self, trainer, pl_module): pass
    def on_validation_end(self, trainer, pl_module): pass
    def on_train_epoch_end(self, trainer, pl_module): pass
    def on_train_end(self, trainer, pl_module): pass
    def on_fit_end(self, trainer, pl_module): pass


def _scalar(v) -> float:
    if torch.is_tensor(v):
        return float(v.detach().float().mean().cpu())
    return float(v)


class ModelCheckpoint(Callback):
    """`save_last` -> <dirpath>/last.ckpt every epoch; `monitor` + `save_top_k=1` -> the best epoch under `filename`
    (train.py:1430-1448). Timing follows `save_on_train_epoch_end`."""

    def __init__(self, dirpath=None, filename=None, monitor=None, mode="min", save_last=False, save_top_k=1,
                 auto_insert_metric_name=True, save_on_train_epoch_end=None, every_n_epochs=1, **_ignored):
        self.dirpath = Path(dirpath) if dirpath is not None else None
        self.filename, self.monitor, self.mode = filename, monitor, mode
        self.save_last, self.save_top_k = bool(save_last), int(save_top_k)
        self.auto_insert_metric_name = auto_insert_metric_name
        self.save_on_train_epoch_end = save_on_train_epoch_end
        self.every_n_epochs = max(1, int(every_n_epochs or 1))
        self.best_model_path, self.best_model_score, self.last_model_path = "", None, ""

    def _format(self, trainer) -> str:
        vals = {"epoch": trainer.current_epoch, "step": trainer.global_step}
        vals.update({k: v for k, v in trainer.callback_metrics.items()})
        name = self.filename or "epoch={epoch}-step={step}"
        try:
            return name.format(**vals)
        except (KeyError, ValueError, IndexError):
            return f"epoch={trainer.current_epoch}-step={trainer.global_step}"

    def _save(self, trainer):
        if self.dirpath is None or (trainer.current_epoch + 1) % self.every_n_epochs:
            return
        self.dirpath.mkdir(parents=True, exist_ok=True)
        if self.save_last:
            self.last_model_path = str(self.dirpath / "last.ckpt")
            trainer.save_checkpoint(self.last_model_path)
        if self.monitor is not None and self.save_top_k != 0 and self.monitor in trainer.callback_metrics:
            score = trainer.callback_metrics[self.monitor]
            better = self.best_model_score is None or (score > self.best_model_score if self.mode == "max"
                                                       else score < self.best_model_score)
            if better and score == score:
                old = self.best_model_path
                self.best_model_score = score
                self.best_model_path = str(self.dirpath / (self._format(trainer) + ".ckpt"))
                trainer.save_checkpoint(self.best_model_path)
                if old and old != self.best_model_path and os.path.exists(old):
                    os.remove(old)

    def on_validation_end(self, trainer, pl_module):
        if self.save_on_train_epoch_end is False or (self.save_on_train_epoch_end is None and self.monitor is not None):
            self._save(trainer)

    def on_train_epoch_end(self, trainer, pl_module):
        if self.save_on_train_epoch_end or (self.save_on_train_epoch_end is None and self.monitor is None):
            self._save(trainer)


class EarlyStopping(Callback):
    def __init__(self, monitor=None, mode="min", patience=3, min_delta=0.0, check_on_train_epoch_end=None, verbose=False,
                 **_ignored):
        self.monitor, self.mode, self.patience = monitor, mode, int(patience)
        self.min_delta, self.verbose = abs(float(min_delta)), verbose
        self.best_score, self.wait_count = None, 0

    def on_validation_end(self, trainer, pl_module):
        if self.monitor not in trainer.callback_metrics:
            return
        score = trainer.callback_metrics[self.monitor]
        if self.best_score is None:
            improved = True
        elif self.mode == "max":
            improved = score > self.best_score + self.min_delta
        else:
            improved = score < self.best_score - self.min_delta
        if improved:
            self.best_score, self.wait_count = score, 0
        else:
            self.wait_count += 1
            if self.wait_count >= self.patience:
                trainer.should_stop = True


class LearningRateMonitor(Callback):
    def __init__(self, *a, **kw):
        pass


class Logger:
    def __init__(self, *a, **kw):
        pass

    @property
    def name(self):
        return "logger"

    @property
    def version(self):
        return ""

    def log_metrics(self, metrics: dict, step=None):
        pass

    def log_hyperparams(self, params):
        pass

    def save(self):
        pass

    def finalize(self, status):
        pass


class CSVLogger(Logger):
    def __init__(self, save_dir=".", name="logs", version=None, **_ignored):
        self.save_dir, self._name, self._version = save_dir, name, version
        self.rows: List[dict] = []

    @property
    def name(self):
        return self._name

    @property
    def log_dir(self):
        return os.path.join(self.save_dir, self._name)

    def log_metrics(self, metrics: dict, step=None):
        self.rows.append({**metrics, "step": step})


class Trainer:
    """Single-device fit loop in Lightning's order: per epoch — train batches (zero_grad, training_step, backward,
    optimizer step), validation batches under no_grad/eval, `on_validation_end` callbacks, plateau scheduler on its
    monitor, train-epoch-end logging + callbacks; stops at `max_epochs` or when a callback sets `should_stop`."""

    def __init__(self, max_epochs=1, accelerator="cpu", devices=1, logger=None, callbacks=None, limit_train_batches=None,
                 limit_val_batches=None, limit_test_batches=None, **_ignored):
        self.max_epochs = max_epochs
        self.fit_loop = SimpleNamespace(max_epochs=max_epochs)
        self.accelerator = accelerator
        self.logger = logger
        self.callbacks: List[Callback] = list(callbacks or [])
        self.limit_train_batches, self.limit_val_batches = limit_train_batches, limit_val_batches
        self.current_epoch, self.global_step = 0, 0
        self.should_stop = False
        self.is_global_zero = int(os.environ.get("RANK", "0")) == 0
        self.callback_metrics: Dict[str, float] = {}
        self.optimizers: List[torch.optim.Optimizer] = []
        self._sums: Dict[str, List[float]] = {}
        self._model: Optional[LightningModule] = None
        self._sched = None
        self.datamodule = None

    # -- logging -----------------------------------------------------------------------------------
    def _record(self, name, value):
        s = self._sums.setdefault(name, [0.0, 0])
        s[0] += _scalar(value)
        s[1] += 1

    def _flush(self, prefix_filter) -> Dict[str, float]:
        out = {}
        for k in [k for k in self._sums if prefix_filter(k)]:
            tot, n = self._sums.pop(k)
            out[k] = tot / max(1, n)
        self.callback_metrics.update(out)
        return out

    # -- checkpoints -------------------------------------------------------------------------------
    def save_checkpoint(self, path):
        m = self._model
        ckpt = {
            "epoch": self.current_epoch, "global_step": self.global_step,
            "pytorch-lightning_version": __version__,
            "state_dict": m.state_dict(),
            "optimizer_states": [o.state_dict() for o in self.optimizers],
            "lr_schedulers": [self._sched["scheduler"].state_dict()] if self._sched else [],
            "hyper_parameters": dict(getattr(m, "hparams", {})),
            "callbacks": {type(c).__name__: {k: v for k, v in vars(c).items() if isinstance(v, (int, float, str, type(None)))}
                          for c in self.callbacks},
        }
        if hasattr(m, "on_save_checkpoint"):
            m.on_save_checkpoint(ckpt)
        Path(path).parent.mkdir(parents=True, exist_ok=True)
        torch.save(ckpt, path)

    def _device(self):
        if self.accelerator in ("gpu", "cuda") and torch.cuda.is_available():
            return torch.device("cuda", torch.cuda.current_device())
        return torch.device("cpu")

    @staticmethod
    def _to(batch, device):
        if torch.is_tensor(batch):
            return batch.to(device, non_blocking=True)
        if isinstance(batch, dict):
            return {k: Trainer._to(v, device) for k, v in batch.items()}
        if isinstance(batch, (list, tuple)):
            return type(batch)(Trainer._to(v, device) for v in batch)
        return batch

    def _call(self, hook, *a):
        for c in self.callbacks:
            getattr(c, hook)(self, self._model, *a)

    # -- fit ---------------------------------------------------------------------------------------
    def fit(self, model, datamodule=None, ckpt_path=None, train_dataloaders=None, val_dataloaders=None):
        dev = self._device()
        self._model = model.to(dev)
        model.trainer = self
        self.datamodule = datamodule
        max_epochs = getattr(self.fit_loop, "max_epochs", None) or self.max_epochs
        cfg = model.configure_optimizers()
        sched = None
        if isinstance(cfg, dict):
            opt, sched = cfg["optimizer"], cfg.get("lr_scheduler")
        elif isinstance(cfg, (list, tuple)):
            opt = cfg[0][0] if isinstance(cfg[0], (list, tuple)) else cfg[0]
            if len(cfg) > 1 and cfg[1]:
                sched = cfg[1][0] if isinstance(cfg[1], (list, tuple)) else cfg[1]
        else:
            opt = cfg
        if sched is not None and not isinstance(sched, dict):
            sched = {"scheduler": sched}
        self.optimizers, self._sched = [opt], sched
        start = 0
        if ckpt_path:
            ck = torch.load(ckpt_path, map_location=dev, weights_only=False)
            model.load_state_dict(ck["state_dict"], strict=True)
            if hasattr(model, "on_load_checkpoint"):
                model.on_load_checkpoint(ck)
            if ck.get("optimizer_states"):
                try:
                    opt.load_state_dict(ck["optimizer_states"][0])
                except ValueError:      # parameter registered lazily after the optimizer was built (FourierGate masks)
                    pass
            if sched and ck.get("lr_schedulers"):
                sched["scheduler"].load_state_dict(ck["lr_schedulers"][0])
            start = int(ck.get("epoch", -1)) + 1
            self.global_step = int(ck.get("global_step", 0))
        for c in self.callbacks:
            c.setup(self, model, "fit")
        self._call("on_fit_start")
        self._call("on_train_start")
        for epoch in range(start, max_epochs):
            self.current_epoch = epoch
            model.train()
            self._call("on_train_epoch_start")
            dl = train_dataloaders if train_dataloaders is not None else datamodule.train_dataloader()
            for i, batch in enumerate(dl):
                if self.limit_train_batches is not None and i >= self.limit_train_batches:
                    break
                batch = self._to(batch, dev)
                opt.zero_grad(set_to_none=True)
                out = model.training_step(batch, i)
                loss = out["loss"] if isinstance(out, dict) else out
                loss.backward()
                opt.step()
                self.global_step += 1
                self._call("on_train_batch_end", out, batch, i)
            # validation (Lightning runs it inside the training epoch, before on_train_epoch_end)
            vdl = val_dataloaders if val_dataloaders is not None else (
                datamodule.val_dataloader() if datamodule is not None and hasattr(datamodule, "val_dataloader") else None)
            if vdl is not None:
                model.eval()
                self._call("on_validation_epoch_start")
                with torch.no_grad():
                    for i, batch in enumerate(vdl):
                        if self.limit_val_batches is not None and i >= self.limit_val_batches:
                            break
                        batch = self._to(batch, dev)
                        out = model.validation_step(batch, i)
                        self._call("on_validation_batch_end", out, batch, i)
                val = self._flush(lambda k: k.startswith("val"))
                self._call("on_validation_epoch_end")
                if self.logger is not None and val:
                    self.logger.log_metrics({**val, "epoch": epoch}, step=self.global_step)
                self._call("on_validation_end")
                model.train()
                if sched is not None:
                    s = sched["scheduler"]
                    if isinstance(s, torch.optim.lr_scheduler.ReduceLROnPlateau):
                        mon = sched.get("monitor")
                        if mon in self.callback_metrics:
                            s.step(self.callback_metrics[mon])
                    else:
                        s.step()
            tr = self._flush(lambda k: not k.startswith("val"))
            if self.logger is not None and tr:
                self.logger.log_metrics({**tr, "epoch": epoch}, step=self.global_step)
            self._call("on_train_epoch_end")
            if self.should_stop:
                break
        self._call("on_train_end")
        self._call("on_fit_end")
        if self.logger is not None:
            self.logger.finalize("success")


pl = SimpleNamespace(LightningModule=LightningModule, LightningDataModule=LightningDataModule,
                     seed_everything=seed_everything, Trainer=Trainer, Callback=Callback)


def install(force: bool = False) -> bool:
    """Register this stand-in as `pytorch_lightning` (+ the sub-modules `train.py:39,52-55` / `test.py` import) unless the
    real package is importable. Returns True when the stand-in is what `import pytorch_lightning` now yields."""
    if not force:
        try:
            import pytorch_lightning as real
            return getattr(real, "__spff_standin__", False)
        except ImportError:
            pass

    def mod(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    root = mod("pytorch_lightning", LightningModule=LightningModule, LightningDataModule=LightningDataModule,
               Trainer=Trainer, seed_everything=seed_everything, Callback=Callback, __version__=__version__,
               __spff_standin__=True)
    root.callbacks = mod("pytorch_lightning.callbacks", Callback=Callback, ModelCheckpoint=ModelCheckpoint,
                         EarlyStopping=EarlyStopping, LearningRateMonitor=LearningRateMonitor)
    root.loggers = mod("pytorch_lightning.loggers", Logger=Logger, CSVLogger=CSVLogger)
    root.loggers.logger = mod("pytorch_lightning.loggers.logger", Logger=Logger)
    root.utilities = mod("pytorch_lightning.utilities", rank_zero_only=rank_zero_only)
    return True
