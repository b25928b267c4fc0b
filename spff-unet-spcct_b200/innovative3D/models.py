"""SPCT-family network modules and Lightning wrappers — the reference's `innovative3D/models.py`
surface for the hot path, executed by the B200 engine.

Kept from the reference, name for name, so that `config.VARIANTS`, `train.py` and `test.py` work
unchanged: the constructor signatures, the `.model` attribute, the parameter names / shapes /
initialisation order (a checkpoint of either implementation loads into the other, and the same seed
gives bit-identical initial weights), `forward(x) -> logits [B,K,F,H,W]`, `compute_loss`,
`training_step / validation_step / test_step`, `configure_optimizers`, the logged metric names.

What differs is below `UNet3D_SpectralCore.forward`: the reference walks its sub-modules and
dispatches ~1500 ATen / cuDNN / cuFFT calls per step (SURVEY.md §2.3); here the sub-modules are
parameter containers and the whole graph — forward, and backward through one autograd node — is
scheduled by `spff_b200.engine.SpffEngine` onto libspff_b200.so. There is no eager fallback: on
anything but an sm_100 device `forward` raises.

In scope (SURVEY.md §8a, §8f-3): LitSPCT_EFiLM_FourierGate ("SPFF-UNet"), LitSPCT_EnergyFiLM, LitSPCT_FourierGate,
LitSPCT_SEspec ("SP_UNet", depth padded 5 -> 16), LitSPCT_ControlUNet ("PlainCore_UNet"). Options of the reference core that no in-scope variant turns on
(`use_spatial`, `use_skip_gate`, `ksd != 3`, non-instance norms, `use_moe`) raise NotImplementedError.
"""
from __future__ import annotations

import copy
import dataclasses
import math
import os
from typing import Dict, List, Optional

import torch
import torch.nn as nn

try:  # the real Lightning when it is installed (the reference pins 2.6.1, requirements.txt:70)
    import pytorch_lightning as pl
except ImportError:  # not in this image: a minimal stand-in with the same method names
    from ._lightning import pl

from spff_b200 import dp, ops
from spff_b200.engine import LossTally, NetConfig, SpffEngine, StagedBatch, run_ensemble
from spff_b200.sched import PlateauLR

from .config import BEST_LR, IGNORE_INDEX, NUM_CLASSES, NUM_FRAMES
from .helpers import (LOSS_REGISTRY, calibration_from_hist, ce_plus_macro_dice_loss, curves_from_hist,
                      metrics_from_confusion, per_class_metrics_2d, per_class_metrics_3d, temperature_from_sums,
                      temperature_grid)

LOG_PER_CLASS = os.getenv("LOG_PER_CLASS", "1") == "1"
# samples per group of the engine's schedule (activations of one group live at a time in fit_step)
SAMPLE_GROUP = int(os.getenv("SPFF_SAMPLE_GROUP", "256"))


def _pick_first_if_seq(x):
    return x[0] if isinstance(x, (list, tuple)) else x


def _canonicalize_targets_2d(lbls):
    """(B,F,H,W) -> max over frames; (H,W) -> (1,H,W); long (models.py:58-66)."""
    lbls = _pick_first_if_seq(lbls)
    if not torch.is_tensor(lbls):
        lbls = torch.as_tensor(lbls)
    if lbls.ndim == 4:
        lbls = lbls.max(dim=1).values
    elif lbls.ndim == 2:
        lbls = lbls.unsqueeze(0)
    return lbls.long()


def _canonicalize_targets_3d(lbls):
    """Normalise labels to (B,F,H,W) long (models.py:68-83)."""
    lbls = _pick_first_if_seq(lbls)
    if not torch.is_tensor(lbls):
        lbls = torch.as_tensor(lbls)
    if lbls.ndim == 5 and lbls.size(1) == 1:
        lbls = lbls[:, 0]
    if lbls.ndim == 5 and lbls.size(-1) == 1:
        lbls = lbls[..., 0]
    if lbls.ndim == 3:
        lbls = lbls.unsqueeze(0)
    assert lbls.ndim == 4, f"Need (B,F,H,W) labels, got {tuple(lbls.shape)}"
    return lbls.long()


# --------------------------------------------------------------------------------------------------
# parameter containers (same attribute names and construction order as the reference modules)
# --------------------------------------------------------------------------------------------------
class _EngineOwned(nn.Module):
    """Sub-modules hold parameters; their math runs inside the fused engine schedule."""

    def forward(self, *a, **kw):
        raise RuntimeError(f"{type(self).__name__} is executed by the B200 engine as part of "
                           "UNet3D_SpectralCore.forward; it has no stand-alone eager path")


def _norm3d(c: int, kind: str = "instance") -> nn.Module:
    if not (kind or "instance").lower().startswith("inst"):
        raise NotImplementedError("only norm='instance' is on the B200 hot path (models.py:168-173)")
    return nn.InstanceNorm3d(c, affine=True, eps=1e-5)


def _act(kind: str = "lrelu") -> nn.Module:
    if not (kind or "lrelu").lower().startswith("lrel"):
        raise NotImplementedError("only act='lrelu' is on the B200 hot path (models.py:175-181)")
    return nn.LeakyReLU(1e-2, inplace=True)


def _conv3x3xk(cin, cout, ksd=1, bias=False):
    if ksd != 3 or bias:
        raise NotImplementedError("the B200 conv kernels implement the (3,3,3), bias-free convolution the SPCT "
                                  "variants use (ksd=3, config.py:414)")
    return nn.Conv3d(cin, cout, kernel_size=(3, 3, 3), padding=(1, 1, 1), bias=False)


class _SEChannelLite(_EngineOwned):
    """Channel squeeze-excite, hidden max(4, c // r) (models.py:600-609)."""

    def __init__(self, c, r=16):
        super().__init__()
        h = max(4, c // r)
        self.pool = nn.AdaptiveAvgPool3d(1)
        self.fc = nn.Sequential(nn.Conv3d(c, h, 1, bias=True), nn.ReLU(inplace=True),
                                nn.Conv3d(h, c, 1, bias=True), nn.Sigmoid())


class _SpectralSE(_EngineOwned):
    """x * sigmoid(mean over (C,H,W)) per energy bin (models.py:611-614); parameter free."""


class _DoubleConvSpectral(_EngineOwned):
    """conv-IN-LReLU twice (models.py:620-625)."""

    def __init__(self, cin, cout, ksd=1, norm="instance", act="lrelu"):
        super().__init__()
        self.b1 = nn.Sequential(_conv3x3xk(cin, cout, ksd, bias=False), _norm3d(cout, norm), _act(act))
        self.b2 = nn.Sequential(_conv3x3xk(cout, cout, ksd, bias=False), _norm3d(cout, norm), _act(act))


class EnergyFiLM3D(_EngineOwned):
    """Per-energy-bin FiLM: (gamma, beta) from a 1x1 Conv1d MLP over a sinusoidal code of the bin
    index (models.py:1479-1512). Input independent -> evaluated once per step as a [C,F] table
    (spff_b200.tables.efilm_tables)."""

    def __init__(self, channels: int, hidden: int = 32, pe_dims: int = 16):
        super().__init__()
        self.channels = int(channels)
        self.pe_dims = int(pe_dims)
        self.mlp = nn.Sequential(nn.Conv1d(self.pe_dims, hidden, 1, bias=True), nn.ReLU(inplace=True),
                                 nn.Conv1d(hidden, 2 * self.channels, 1, bias=True))


class FourierGate3D(_EngineOwned):
    """Gate over the energy axis through a learnable rFFT magnitude mask (models.py:1515-1544).
    Like the reference, `freq_mask` ([1,1,F//2+1,1,1], ones) is registered lazily at the first
    forward (models.py:1532-1535) — so it is absent from a fresh module's state_dict and from an
    optimizer built before the first forward. `learn_phase=True` is not on the hot path."""

    def __init__(self, learn_phase: bool = False):
        super().__init__()
        if learn_phase:
            raise NotImplementedError("FourierGate3D(learn_phase=True) is not used by any in-scope variant")
        self.learn_phase = False
        self.mag_scale = nn.Parameter(torch.ones(1))
        self._mask = None

    def ensure_mask(self, frames: int, device) -> bool:
        """Register (or re-register when F changes) the lazy mask; True if a new parameter was made."""
        length = frames // 2 + 1
        if self._mask is not None and self._mask.shape[2] == length:
            return False
        self._mask = nn.Parameter(torch.ones(1, 1, length, 1, 1, device=device, dtype=torch.float32))
        self.register_parameter("freq_mask", self._mask)
        return True

    def _load_from_state_dict(self, state_dict, prefix, *args, **kwargs):
        # a checkpoint saved after the first forward carries freq_mask: make room for it
        key = prefix + "freq_mask"
        if key in state_dict and (self._mask is None or self._mask.shape != state_dict[key].shape):
            self._mask = nn.Parameter(torch.ones_like(state_dict[key], dtype=torch.float32,
                                                      device=self.mag_scale.device))
            self.register_parameter("freq_mask", self._mask)
        super()._load_from_state_dict(state_dict, prefix, *args, **kwargs)


class _DoubleConvSpectral_Novel(_EngineOwned):
    """conv-IN-LReLU twice + EnergyFiLM + FourierGate (models.py:1448-1478)."""

    def __init__(self, cin, cout, ksd=1, norm="instance", act="lrelu", use_efilm: bool = False,
                 use_fouriergate: bool = False, use_moe: bool = False, moe_K: int = 3):
        super().__init__()
        if use_moe:
            raise NotImplementedError("use_moe refers to SpectralMoE3D, which the reference does not define "
                                      "(models.py:1464)")
        self.pre = nn.Sequential(_conv3x3xk(cin, cout, ksd, bias=False), _norm3d(cout, norm), _act(act))
        self.body = nn.Sequential(_conv3x3xk(cout, cout, ksd, bias=False), _norm3d(cout, norm), _act(act))
        self.efilm = EnergyFiLM3D(cout) if use_efilm else nn.Identity()
        self.fgate = FourierGate3D() if use_fouriergate else nn.Identity()


class _CoreFn(torch.autograd.Function):
    """The whole network as one autograd node: forward keeps the engine's saved activations,
    backward returns the gradient of every parameter (none for the images)."""

    @staticmethod
    def forward(ctx, x, core, *params):
        logits, state = core.engine.forward_saved(x, group=core.sample_group)
        ctx.core, ctx.state = core, state
        return logits

    @staticmethod
    def backward(ctx, dlogits):
        core = ctx.core
        if ctx.state is None:
            raise RuntimeError("UNet3D_SpectralCore (B200 build): the activations of this forward were released by its "
                               "first backward; retain_graph / a second backward through the same forward is not supported")
        flat = torch.zeros(core._flat_numel, device=dlogits.device)
        G = core._views(flat)
        core.engine.backward_saved(ctx.state, dlogits, G)
        ctx.state = None
        return (None, None) + tuple(G[n] for n in core._names)


class UNet3D_SpectralCore(nn.Module):
    """Depth-preserving 4-level U-Net over [B,1,F,H,W] (models.py:647-701): pooling / upsampling in
    (H,W) only, 3x3x3 convs mixing the energy bins, optional Channel-SE + Spectral-SE after every
    encoder stage. Same constructor as the reference; H and W must be multiples of 8."""

    def __init__(self, in_channels=1, num_classes=2, base=32, ksd=3, use_se=False, use_specse=False,
                 use_spatial=False, use_skip_gate=False, norm="instance", act="lrelu"):
        super().__init__()
        if in_channels != 1:
            raise NotImplementedError("the SPCT family feeds energy bins on the depth axis: in_channels=1 (models.py:1551)")
        if int(base) != 32:
            raise NotImplementedError("the B200 kernels are built for base=32 (config.py:413)")
        if use_spatial or use_skip_gate:
            raise NotImplementedError("use_spatial / use_skip_gate are off in every in-scope variant (config.py:416-418)")
        if not 0 < num_classes <= 16:
            raise NotImplementedError("the head / loss kernels support up to 16 classes")
        f = int(base)
        P = (1, 2, 2)
        self.enc1 = _DoubleConvSpectral(in_channels, f, ksd, norm, act)
        self.pool1 = nn.MaxPool3d(P)
        self.enc2 = _DoubleConvSpectral(f, 2 * f, ksd, norm, act)
        self.pool2 = nn.MaxPool3d(P)
        self.enc3 = _DoubleConvSpectral(2 * f, 4 * f, ksd, norm, act)
        self.pool3 = nn.MaxPool3d(P)
        self.bott = _DoubleConvSpectral(4 * f, 8 * f, ksd, norm, act)
        self.up3 = nn.ConvTranspose3d(8 * f, 4 * f, kernel_size=P, stride=P)
        self.dec3 = _DoubleConvSpectral(8 * f, 4 * f, ksd, norm, act)
        self.up2 = nn.ConvTranspose3d(4 * f, 2 * f, kernel_size=P, stride=P)
        self.dec2 = _DoubleConvSpectral(4 * f, 2 * f, ksd, norm, act)
        self.up1 = nn.ConvTranspose3d(2 * f, f, kernel_size=P, stride=P)
        self.dec1 = _DoubleConvSpectral(2 * f, f, ksd, norm, act)
        self.out = nn.Conv3d(f, num_classes, 1)
        self.se = nn.ModuleList([_SEChannelLite(c) if use_se else nn.Identity() for c in (f, 2 * f, 4 * f, 8 * f)])
        self.sp = nn.ModuleList([_SpectralSE() if use_specse else nn.Identity() for _ in range(4)])
        self.sa = nn.ModuleList([nn.Identity() for _ in range(4)])
        self.g3 = self.g2 = self.g1 = None
        self._num_classes, self._base = int(num_classes), f
        self._use_se, self._use_specse = bool(use_se), bool(use_specse)
        self.sample_group = SAMPLE_GROUP
        self._engine: Optional[SpffEngine] = None
        self._flat: Optional[torch.Tensor] = None
        self._names: List[str] = []
        self._slots: Dict[str, tuple] = {}
        self._flat_numel = 0
        self._n_eager = 0     # elements of the flat buffer that existed before any lazy registration

    def __deepcopy__(self, memo):
        """`copy.deepcopy(core)` (train.py:1288 copies the core for its compute read-out; EMA / SWA helpers do the same):
        parameters are cloned, the engine, the flat buffer and its views are NOT shared — the copy rebuilds them at its
        first forward."""
        new = self.__class__.__new__(self.__class__)
        memo[id(self)] = new
        lazy = {"_engine": None, "_flat": None, "_param_objs": {}, "_param_data": {}, "_copy_stream": None,
                "_names": [], "_slots": {}, "_flat_numel": 0, "_n_eager": 0}
        for k, v in self.__dict__.items():
            new.__dict__[k] = copy.deepcopy(lazy[k]) if k in lazy else copy.deepcopy(v, memo)
        for m in new.modules():      # the two names of a lazy mask must stay ONE parameter in the copy
            if isinstance(m, FourierGate3D) and "freq_mask" in m._parameters:
                m._mask = m._parameters["freq_mask"]
        return new

    # -- structure -----------------------------------------------------------------------------
    def net_config(self) -> NetConfig:
        blk = self.enc1
        novel = isinstance(blk, _DoubleConvSpectral_Novel)
        return NetConfig(num_classes=self._num_classes, base=self._base,
                         conv_names=("pre", "body") if novel else ("b1", "b2"),
                         efilm=novel and isinstance(blk.efilm, EnergyFiLM3D),
                         fgate=novel and isinstance(blk.fgate, FourierGate3D),
                         specse=self._use_specse, chanse=self._use_se)

    @property
    def engine(self) -> SpffEngine:
        if self._engine is None:
            self._engine = SpffEngine(self.net_config(), lambda: self._param_data,
                                      lambda: tuple(p._version for p in self._param_objs.values()))
        return self._engine

    # -- flat parameter storage ------------------------------------------------------------------
    def _views(self, flat: torch.Tensor) -> Dict[str, torch.Tensor]:
        return {n: flat[o:o + k].view(shape) for n, (o, k, shape) in self._slots.items()}

    def materialize(self, frames: int = NUM_FRAMES):
        """Register the lazy FourierGate masks for `frames` bins and (re)build the flat fp32 parameter
        buffer: every parameter's `.data` becomes a view of it (names, shapes and values unchanged),
        so the gradient all-reduce and the fused Adam run over one contiguous range. The lazily
        registered masks sit at the tail of the buffer, after `self._n_eager` elements."""
        dev = self.out.weight.device
        if dev.type != "cuda":
            raise RuntimeError("UNet3D_SpectralCore (B200 build) must live on a CUDA sm_100 device: there is no CPU "
                               "fallback. Call .to('cuda') / .cuda() first.")
        for m in self.modules():
            if isinstance(m, FourierGate3D):
                m.ensure_mask(frames, dev)
        # named_parameters() de-duplicates the two aliases of a lazy mask and yields `fgate._mask`
        # (the attribute assignment registers first, as in the reference); the engine and the flat
        # buffer use the public name `fgate.freq_mask`
        named = [(n.replace("fgate._mask", "fgate.freq_mask"), p) for n, p in self.named_parameters()]
        ok = self._flat is not None and self._flat.device == dev and len(named) == len(self._names)
        if ok:
            base, end = self._flat.data_ptr(), self._flat.data_ptr() + 4 * self._flat_numel
            ok = all(base <= p.data_ptr() < end and p.dtype == torch.float32 for _, p in named)
        if ok:
            return
        eager = [(n, p) for n, p in named if not n.endswith("freq_mask")]
        lazy = [(n, p) for n, p in named if n.endswith("freq_mask")]
        slots, off = {}, 0
        for n, p in eager + lazy:
            k = p.numel()
            slots[n] = (off, k, tuple(p.shape))
            off += (k + 3) // 4 * 4          # 16-byte aligned slices
            if n == eager[-1][0]:
                self._n_eager = off
        flat = torch.zeros(off, dtype=torch.float32, device=dev)
        for n, p in eager + lazy:
            o, k, shape = slots[n]
            v = flat[o:o + k].view(shape)
            v.copy_(p.data)
            p.data = v
        self._flat, self._slots, self._flat_numel = flat, slots, off
        self._names = [n for n, _ in named]
        self._param_objs = dict(named)
        self._param_data = {n: p.data for n, p in named}
        if self._engine is not None:
            self._engine.invalidate_weights()

    def stage_ranges(self):
        """[lo, hi) of the flat buffer per backward stage, in the order their gradients complete: "decoder" (up3 .. out),
        "bott", "enc3", "enc2", "enc1" (each block with its EFiLM / FourierGate parameters), and "tail" (the SE modules
        and the lazily registered masks, final only when the whole backward is)."""
        out = {"decoder": self.decoder_range()}
        for b in ("enc1", "enc2", "enc3", "bott"):
            names = [n for n in self._slots if n.split(".")[0] == b and not n.endswith("freq_mask")]
            lo = min(self._slots[n][0] for n in names)
            hi = max(self._slots[n][0] + (self._slots[n][1] + 3) // 4 * 4 for n in names)
            inside = [n for n, (o, k, _) in self._slots.items() if lo <= o < hi]
            assert sorted(inside) == sorted(names), f"{b} parameters are not contiguous in the flat buffer"
            out[b] = (lo, hi)
        out["tail"] = (out["decoder"][1], self._flat_numel)
        covered = sorted(out.values())
        assert covered[0][0] == 0 and all(a[1] == b[0] for a, b in zip(covered, covered[1:])) and covered[-1][1] == self._flat_numel
        return out

    def decoder_range(self):
        """[lo, hi) of the flat buffer holding up3 .. out (transposed convs, decoder blocks, head): contiguous
        because parameters are laid out in registration order (enc1..bott, up3, dec3, up2, dec2, up1, dec1, out, se)."""
        names = [n for n in self._slots if n.split(".")[0] in ("up3", "dec3", "up2", "dec2", "up1", "dec1", "out")
                 and not n.endswith("freq_mask")]
        lo = min(self._slots[n][0] for n in names)
        hi = max(self._slots[n][0] + (self._slots[n][1] + 3) // 4 * 4 for n in names)
        inside = [n for n, (o, k, _) in self._slots.items() if lo <= o < hi]
        assert sorted(inside) == sorted(names), "decoder parameters are not contiguous in the flat buffer"
        return lo, hi

    # -- forward ---------------------------------------------------------------------------------
    def forward(self, x):
        x = _pick_first_if_seq(x)
        if x.ndim == 4:
            x = x.unsqueeze(1)
        self.materialize(x.shape[2])
        x = x.to(self.out.weight.device)
        params = [self._param_objs[n] for n in self._names]
        if torch.is_grad_enabled() and any(p.requires_grad for p in params):
            return _CoreFn.apply(x, self, *params)
        return self.engine.infer(x, group=self.sample_group)

    @torch.no_grad()
    def predict_labels(self, x) -> torch.Tensor:
        """uint8 label map [B,F,H,W] = argmax over classes, fused into the head kernel (the label
        maps `test.py:710-722` derives from softmax + argmax on the host)."""
        x = _pick_first_if_seq(x)
        self.materialize(x.shape[2])
        return self.engine.infer(x.to(self.out.weight.device), group=self.sample_group, argmax=True)


    @torch.no_grad()
    def predict_labels_streamed(self, x_host: torch.Tensor, out_host: Optional[torch.Tensor] = None) -> torch.Tensor:
        """`predict_labels` for a scan held in host memory (pinned for overlap): images stream in and label maps
        stream out group by group on a copy stream while the kernels run. Returns the host uint8 [B,F,H,W] tensor
        (complete on return)."""
        x_host = _pick_first_if_seq(x_host)
        if x_host.ndim == 4:
            x_host = x_host.unsqueeze(1)
        self.materialize(x_host.shape[2])
        dev = self.out.weight.device
        if out_host is None:
            out_host = torch.empty(x_host.shape[0], *x_host.shape[2:], dtype=torch.uint8).pin_memory()
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = torch.cuda.Stream(device=dev)
        self.engine.infer_streamed(x_host, out_host, dev, self._copy_stream, group=self.sample_group)
        self._copy_stream.synchronize()
        return out_host


def upgrade_spct_with_novel_blocks(m: nn.Module, use_efilm: bool = True, use_fouriergate: bool = True,
                                   use_moe: bool = False, moe_K: int = 3):
    """Replace every `_DoubleConvSpectral` child by the novel block, keeping channels
    (models.py:1416-1446). New blocks are constructed in `named_children` order like the
    reference, so a seeded construction draws the same initial weights."""
    for name, child in list(m.named_children()):
        if isinstance(child, _DoubleConvSpectral):
            conv1, conv2 = child.b1[0], child.b2[0]
            setattr(m, name, _DoubleConvSpectral_Novel(int(conv1.in_channels), int(conv2.out_channels),
                                                       ksd=int(conv1.kernel_size[0]), use_efilm=use_efilm,
                                                       use_fouriergate=use_fouriergate, use_moe=use_moe, moe_K=moe_K))
        else:
            upgrade_spct_with_novel_blocks(child, use_efilm, use_fouriergate, use_moe, moe_K)
    if isinstance(m, UNet3D_SpectralCore):
        m._engine = None
    return m


def build_spct_energyfilm_fourier(num_classes=NUM_CLASSES, base=32, ksd=3, use_se=True, use_specse=True,
                                  use_spatial=False, use_skip_gate=False, **kw):
    """models.py:1547-1555."""
    core = UNet3D_SpectralCore(in_channels=1, num_classes=num_classes, base=base, ksd=ksd, use_se=use_se,
                               use_specse=use_specse, use_spatial=use_spatial, use_skip_gate=use_skip_gate, **kw)
    return upgrade_spct_with_novel_blocks(core, use_efilm=True, use_fouriergate=True, use_moe=False)


# --------------------------------------------------------------------------------------------------
# Lightning wrappers
# --------------------------------------------------------------------------------------------------
class BaseLitModel(pl.LightningModule):
    """Step driver (models.py:466-594): forward, ce_plus_macro_dice_loss, per-step metrics, Adam +
    ReduceLROnPlateau on `val_macro_dice`. `fit_step` is the B200-native fused equivalent of
    Lightning's training_step + backward + optimizer step."""

    def __init__(self, num_classes=NUM_CLASSES, lr=BEST_LR, is_3d=True, **kwargs):
        super().__init__()
        self.is_3d = bool(is_3d)
        self.save_hyperparameters({"num_classes": num_classes, "lr": float(lr), "is_3d": bool(is_3d), **kwargs})
        self._fused = None
        self._copy_stream = None

    def __deepcopy__(self, memo):
        """The fused optimizer state, the copy stream and the trainer back-reference stay with the original."""
        new = self.__class__.__new__(self.__class__)
        memo[id(self)] = new
        drop = {"_fused": None, "_copy_stream": None, "trainer": None, "_trainer": None}
        for k, v in self.__dict__.items():
            new.__dict__[k] = drop[k] if k in drop else copy.deepcopy(v, memo)
        return new

    def _normalize_input(self, x):
        return _pick_first_if_seq(x)

    def forward(self, x):
        return self.model(self._normalize_input(x))

    def compute_loss(self, logits, labels):
        return ce_plus_macro_dice_loss(logits, labels, self.hparams.num_classes, ignore_index=IGNORE_INDEX)

    def _log_metrics(self, prefix, loss, metrics):
        (dice_list, sens_list, spec_list, macro_dice, macro_sens, macro_spec, micro_dice, micro_sens,
         micro_spec) = metrics
        kw = dict(on_step=False, on_epoch=True, sync_dist=True)
        self.log(f"{prefix}_loss", loss, prog_bar=(prefix == "train"), **kw)
        self.log(f"{prefix}_macro_dice", macro_dice, prog_bar=(prefix != "test"), **kw)
        for name, v in (("micro_dice", micro_dice), ("macro_sens", macro_sens), ("macro_spec", macro_spec),
                        ("micro_sens", micro_sens), ("micro_spec", micro_spec)):
            self.log(f"{prefix}_{name}", v, prog_bar=True, **kw)
        for i, (d, s, sp) in enumerate(zip(dice_list, sens_list, spec_list)):
            self.log(f"{prefix}_dice_class_{i}", d, prog_bar=False, **kw)
            self.log(f"{prefix}_sens_class_{i}", s, prog_bar=False, **kw)
            self.log(f"{prefix}_spec_class_{i}", sp, prog_bar=False, **kw)

    def _shared_step(self, batch, prefix):
        """models.py:479-586 without the test-only sklearn PR/ROC curves (CPU post-processing the
        reference's own test pass in train.py:676-878 repeats; outside the hot path)."""
        imgs, lbls = batch if isinstance(batch, (list, tuple)) else (batch["image"], batch["label"])
        imgs = _pick_first_if_seq(imgs)
        lbls = _pick_first_if_seq(lbls)
        if not self.is_3d:
            lbls = _canonicalize_targets_2d(lbls)
        logits = self(imgs)
        lbls = lbls.to(logits.device).long()
        loss = self.compute_loss(logits, lbls)
        fn = per_class_metrics_3d if self.is_3d else per_class_metrics_2d
        self._log_metrics(prefix, loss, fn(logits, lbls, self.hparams.num_classes, ignore_index=IGNORE_INDEX))
        return loss

    def training_step(self, batch, batch_idx, dataloader_idx=0):
        return self._shared_step(batch, "train")

    def validation_step(self, batch, batch_idx, dataloader_idx=0):
        return {"val_loss": self._shared_step(batch, "val")}

    def test_step(self, batch, batch_idx):
        return self._shared_step(batch, "test")

    def configure_optimizers(self):
        opt = torch.optim.Adam(self.parameters(), lr=self.hparams.lr)
        sch = torch.optim.lr_scheduler.ReduceLROnPlateau(opt, mode="max", factor=0.5, patience=5)
        return {"optimizer": opt, "lr_scheduler": {"scheduler": sch, "monitor": "val_macro_dice"}}

    # -- B200-native fused training step ---------------------------------------------------------
    def fit_step(self, batch, optimize: bool = True, sample_group: Optional[int] = None):
        """forward + ce_plus_macro_dice_loss + backward (+ data-parallel gradient all-reduce + Adam
        step) in the engine's sample-group schedule, without materialising the batch's activations
        or logits. Equivalent to `loss = training_step(batch); loss.backward(); optimizer.step()` with
        `torch.optim.Adam(lr=hparams.lr)`; like the reference (models.py:1532-1535 + :591-594) the
        lazily registered `freq_mask` parameters receive gradients but are not stepped.

        Under torch.distributed (one process per GPU) every rank passes its own shard of the batch;
        gradients are summed with ONE NCCL all-reduce over the flat buffer and scaled by 1/world in
        the Adam kernel — DistributedDataParallel's mean-of-rank-gradients.

        Returns {"loss": device scalar, "tally": LossTally}; nothing synchronises the host."""
        imgs, lbls = batch if isinstance(batch, (list, tuple)) else (batch["image"], batch["label"])
        imgs = _pick_first_if_seq(imgs)
        lbls = _pick_first_if_seq(lbls)
        core: UNet3D_SpectralCore = self.model
        if imgs.ndim == 4:
            imgs = imgs.unsqueeze(1)
        core.materialize(imgs.shape[2])
        dev = core._flat.device
        if lbls.dtype not in (torch.uint8, torch.int64):
            lbls = lbls.long()
        group = sample_group or core.sample_group
        staged = None
        if not imgs.is_cuda and not lbls.is_cuda:
            # host batch: stream it in group by group on a copy stream, overlapped with the kernels
            if self._copy_stream is None:
                self._copy_stream = torch.cuda.Stream(device=dev)
            staged = StagedBatch(imgs, lbls, dev, group, self._copy_stream)
            imgs, lbls = staged.x, staged.labels
        else:
            imgs = imgs.to(dev, non_blocking=True)
            lbls = lbls.to(dev, non_blocking=True)
        st = self._fused
        if st is None or st["flat"] is not core._flat:
            st = self._fused = dict(flat=core._flat, grad=torch.zeros_like(core._flat), m=torch.zeros_like(core._flat),
                                    v=torch.zeros_like(core._flat), step=0,
                                    tally=LossTally(self.hparams.num_classes, dev))
            st["G"] = core._views(st["grad"])
        st["grad"].zero_()
        st["tally"].zero()
        with torch.no_grad():
            # data parallel: ONE flat gradient buffer, reduced range by range as the last group's backward completes
            # them (decoder, bottleneck, enc3, enc2, enc1: async on the NCCL stream, overlapping the rest of the
            # backward); only the small tail (SE modules, lazy masks: ~50 KB) is reduced after the backward.
            pending = []
            hook = None
            if dp.world()[1] > 1:
                if "ranges" not in st:
                    st["ranges"] = core.stage_ranges()
                ranges = st["ranges"]
                def hook(stage):
                    g = st["grad"][ranges[stage][0]:ranges[stage][1]]
                    ops.scale_by_count(g, st["tally"].n_valid)          # sum-CE gradients -> this rank's mean CE
                    pending.append(dp.allreduce_async(g))
            core.engine.train_step(imgs, lbls, st["G"], st["tally"], group=group, ignore_index=IGNORE_INDEX,
                                   staged=staged, stage_done=hook)
            if pending:
                ev = dp.exposed_timer_start()
                lo, hi = ranges["tail"]
                ops.scale_by_count(st["grad"][lo:hi], st["tally"].n_valid)
                gscale = dp.allreduce_grads(st["grad"][lo:hi])
                for w in pending:
                    w.wait()
                dp.exposed_timer_stop(ev)
            else:
                ops.scale_by_count(st["grad"], st["tally"].n_valid)      # the engine back-propagates the CE sum
                gscale = dp.allreduce_grads(st["grad"])
            if optimize:
                st["step"] += 1
                n = core._n_eager
                ops.adam_step(core._flat[:n], st["grad"][:n], st["m"][:n], st["v"][:n], float(self.hparams.lr), 0.9, 0.999,
                              1e-8, st["step"], gscale)
                core.engine.invalidate_weights()   # written behind torch's back: re-pack the bf16 operands
            loss = st["tally"].loss()
        return {"loss": loss, "tally": st["tally"]}

    def fused_lr_step(self, val_macro_dice: float) -> float:
        """ReduceLROnPlateau(mode='max', factor=0.5, patience=5) on `val_macro_dice` for the fused Adam
        (the schedule `configure_optimizers` hands to Lightning, models.py:593-594). Returns the new lr."""
        if getattr(self, "_plateau", None) is None:
            self._plateau = PlateauLR(float(self.hparams.lr), mode="max", factor=0.5, patience=5)
        self.hparams["lr"] = self._plateau.step(val_macro_dice)
        return self.hparams["lr"]

    @torch.no_grad()
    def predict_labels_sharded(self, x) -> tuple:
        """Inference over a scan whose slices are independent units (SURVEY.md §8e): this rank runs the
        contiguous shard `dp.shard_range(len(x))` of the slices and returns ((lo, hi), uint8 labels
        [hi-lo,F,H,W]). No collective: the caller concatenates shards in rank order."""
        x = _pick_first_if_seq(x)
        lo, hi = dp.shard_range(x.shape[0])
        return (lo, hi), self.model.predict_labels(x[lo:hi])

    def fused_grads(self) -> Dict[str, torch.Tensor]:
        """Gradient views (by core parameter name) of the last fit_step."""
        return self._fused["G"]

    def fused_optimizer_state(self) -> Dict[str, object]:
        """State of the fused Adam (first / second moments over the flat parameter buffer, step count, current lr and
        the plateau scheduler) for checkpoint / resume — what `optimizer.state_dict()` holds on the Lightning path.
        Save it next to `state_dict()`."""
        st = self._fused
        if st is None:
            return {"step": 0}
        out = {"step": int(st["step"]), "exp_avg": st["m"].detach().cpu(), "exp_avg_sq": st["v"].detach().cpu(),
               "lr": float(self.hparams.lr)}
        pl_ = getattr(self, "_plateau", None)
        if pl_ is not None:
            out["plateau"] = dict(vars(pl_))
        return out

    def load_fused_optimizer_state(self, state: Dict[str, object]) -> None:
        """Inverse of `fused_optimizer_state` (call after `load_state_dict`, on the device the model trains on)."""
        core = self.model
        core.materialize(self._frames_of(core))
        if not state or int(state.get("step", 0)) == 0:
            self._fused = None
            return
        flat = core._flat
        if state["exp_avg"].numel() != flat.numel():
            raise ValueError(f"optimizer state holds {state['exp_avg'].numel()} elements, the model {flat.numel()}")
        self._fused = dict(flat=flat, grad=torch.zeros_like(flat), m=state["exp_avg"].to(flat), v=state["exp_avg_sq"].to(flat),
                           step=int(state["step"]), tally=LossTally(self.hparams.num_classes, flat.device))
        self._fused["G"] = core._views(self._fused["grad"])
        self.hparams["lr"] = float(state.get("lr", self.hparams.lr))
        if "plateau" in state:
            self._plateau = PlateauLR(float(self.hparams.lr), mode="max", factor=0.5, patience=5)
            vars(self._plateau).update(state["plateau"])

    @staticmethod
    def _frames_of(core) -> int:
        for m in core.modules():
            if isinstance(m, FourierGate3D) and m._mask is not None:
                return 2 * (m._mask.shape[2] - 1) + 1
        return NUM_FRAMES

    def step_metrics(self, tally: LossTally, total_voxels: int):
        """per_class_metrics_3d's 9-tuple from a fit_step tally (one device->host copy)."""
        return metrics_from_confusion(tally.confusion.cpu().numpy(), total_voxels)

    # -- B200-native fused evaluation step --------------------------------------------------------
    @torch.no_grad()
    def eval_step(self, batch, tally: Optional[LossTally] = None, per_sample: bool = False, return_labels: bool = False,
                  sample_group: Optional[int] = None, curves=None):
        """The loss statistics of `ce_plus_macro_dice_loss(model(x), y)` and `per_class_metrics_3d` without the logits:
        forward, head, CE and confusion tally in the engine's sample-group schedule. Takes the batch forms `fit_step`
        takes (tuple or dict; host or device; uint8 or int64 labels) and accumulates into `tally` (a fresh LossTally when
        None). Touches no parameter, gradient or optimizer state and does not synchronise the host.

        `curves`: None, a bin count T in [16, 1024], or an int64 [K,2,T] histogram to accumulate into (as `tally`): the
        head also bins every class's softmax probability of the counted voxels, positives and negatives apart, which is
        what `helpers.curves_from_hist` turns into ROC / PR curves, AUROC and AP.

        Returns {"loss": device scalar of the tally so far, "tally", "per_sample": (nll fp64 [B], count int64 [B],
        confusion int64 [B,K,K]) or None, "labels": uint8 arg-max map [B,F,H,W] or None, "hist": int64 [K,2,T] or None,
        "per_sample_hist": int64 [B,K,2,T] with curves and per_sample, else None}."""
        imgs, lbls = batch if isinstance(batch, (list, tuple)) else (batch["image"], batch["label"])
        imgs, lbls = _pick_first_if_seq(imgs), _pick_first_if_seq(lbls)
        core: UNet3D_SpectralCore = self.model
        if imgs.ndim == 4:
            imgs = imgs.unsqueeze(1)
        core.materialize(imgs.shape[2])
        dev = core._flat.device
        if lbls.dtype not in (torch.uint8, torch.int64):
            lbls = lbls.long()
        group = sample_group or core.sample_group
        staged = None
        if not imgs.is_cuda and not lbls.is_cuda:
            if self._copy_stream is None:
                self._copy_stream = torch.cuda.Stream(device=dev)
            staged = StagedBatch(imgs, lbls, dev, group, self._copy_stream)
            imgs, lbls = staged.x, staged.labels
        else:
            imgs = imgs.to(dev, non_blocking=True)
            lbls = lbls.to(dev, non_blocking=True)
        k = self.hparams.num_classes
        tally = LossTally(k, dev) if tally is None else tally
        bsz = imgs.shape[0]
        rows = (torch.zeros(bsz, dtype=torch.float64, device=dev), torch.zeros(bsz, dtype=torch.int64, device=dev),
                torch.zeros(bsz, k, k, dtype=torch.int64, device=dev)) if per_sample else None
        labels = torch.empty(bsz, *imgs.shape[2:], dtype=torch.uint8, device=dev) if return_labels else None
        hist, sample_hist = _curve_buffers(curves, k, bsz, per_sample, dev)
        core.engine.eval_step(imgs, lbls, tally, group=group, ignore_index=IGNORE_INDEX, per_sample=rows, labels_out=labels,
                              staged=staged, hist=hist, sample_hist=sample_hist)
        return {"loss": self._tally_loss(tally), "tally": tally, "per_sample": rows, "labels": labels, "hist": hist,
                "per_sample_hist": sample_hist}

    def _tally_loss(self, tally: LossTally) -> torch.Tensor:
        """ce_plus_macro_dice_loss from its statistics: CE over the valid voxels + 0.5 * (1 - hard macro Dice)."""
        return tally.loss()

    @torch.no_grad()
    def evaluate(self, batches, sample_group: Optional[int] = None, curves: Optional[int] = None):
        """`eval_step` over an iterable of batches into one tally: the validation / test loss and metrics of the whole
        set. Under torch.distributed every rank passes its own batches and gets the result of all of them. Returns
        {"loss": float, "metrics": per_class_metrics_3d's 9-tuple, "tally", "voxels"}; with `curves` = T bins also
        "hist" (int64 [K,2,T] on the device) and "curves" (`helpers.curves_from_hist`: per-class ROC / PR curves, AUROC,
        AP and their macro averages)."""
        return _evaluate(self.hparams.num_classes, next(self.parameters()).device, self._tally_loss, batches,
                         lambda b, t, h: self.eval_step(b, tally=t, sample_group=sample_group, curves=h), curves)


def _eval_voxels(batch) -> int:
    """Voxels of a batch as given, before any padding: ignored voxels count as true negatives in
    `metrics_from_confusion`, padding voxels must not."""
    lbls = batch[1] if isinstance(batch, (list, tuple)) else batch["label"]
    return int(_pick_first_if_seq(lbls).numel())


def _curve_buffers(curves, k: int, bsz: int, per_sample: bool, dev):
    """(hist [K,2,T], per-sample hist [B,K,2,T] or None) for `eval_step(curves=...)`; (None, None) without curves.
    `curves` is a bin count T (fresh zeros) or a [K,2,T] int64 histogram on `dev` to accumulate into."""
    if curves is None:
        return None, None
    if torch.is_tensor(curves):
        hist = curves
        if hist.dtype != torch.int64 or hist.dim() != 3 or tuple(hist.shape[:2]) != (k, 2) or not hist.is_contiguous() \
                or hist.device != torch.device(dev):
            raise ValueError(f"curves must be a contiguous int64 [{k},2,T] histogram on {dev}, got {hist.dtype} "
                             f"{tuple(hist.shape)} on {hist.device}")
    else:
        hist = torch.zeros(k, 2, int(curves), dtype=torch.int64, device=dev)
    bins = hist.shape[-1]
    if not 16 <= bins <= 1024:
        raise ValueError(f"curves: the bin count must be in [16, 1024], got {bins}")
    sample_hist = torch.zeros(bsz, k, 2, bins, dtype=torch.int64, device=dev) if per_sample else None
    return hist, sample_hist


def _calib_buffers(calibration, dev):
    """[3,T] int64 confidence histogram for `eval_step(calibration=...)`, or None: `calibration` is a bin count T (fresh
    zeros) or a contiguous int64 [3,T] histogram on `dev` to accumulate into, T in [2, 1024]."""
    if calibration is None:
        return None
    if torch.is_tensor(calibration):
        calib = calibration
        if calib.dtype != torch.int64 or calib.dim() != 2 or calib.shape[0] != 3 or not calib.is_contiguous() \
                or calib.device != torch.device(dev):
            raise ValueError(f"calibration must be a contiguous int64 [3,T] histogram on {dev}, got {calib.dtype} "
                             f"{tuple(calib.shape)} on {calib.device}")
    else:
        calib = torch.zeros(3, int(calibration), dtype=torch.int64, device=dev)
    if not 2 <= calib.shape[1] <= 1024:
        raise ValueError(f"calibration: the bin count must be in [2, 1024], got {calib.shape[1]}")
    return calib


def _evaluate(k: int, dev, loss_fn, batches, step, curves: Optional[int] = None, calibration: Optional[int] = None):
    """Shared driver of the `evaluate` methods: one tally (and, with `curves` = T, one [K,2,T] softmax histogram) over
    the batches, ONE all-reduce of the tally (plus the voxel count and the histogram) under data parallelism, ONE
    device->host copy at the end. k classes, `dev` the device of the tallies, loss_fn(tally) -> device scalar.
    `calibration` = T (ensembles only: step(batch, tally, hist, cal) takes a fourth argument, the dict of
    SpctEnsemble.eval_step's calibration outputs) adds a [3,T] confidence histogram, the Brier sum and the uncertainty
    sums to the all-reduce and the copy, and "calibration" (helpers.calibration_from_hist) to the result."""
    tally, voxels = None, 0
    hist = _curve_buffers(curves, k, 0, False, dev)[0]
    cal = None
    if calibration is not None:
        cal = {"calib": _calib_buffers(calibration, dev), "brier": torch.zeros(1, dtype=torch.float64, device=dev),
               "unc": torch.zeros(2, dtype=torch.int64, device=dev)}
    for batch in batches:
        tally = (step(batch, tally, hist) if cal is None else step(batch, tally, hist, cal))["tally"]
        voxels += _eval_voxels(batch)
    if tally is None:   # a rank without batches still joins the all-reduce
        tally = LossTally(k, dev)
    vox = torch.tensor([voxels], dtype=torch.int64, device=tally._buf.device)
    if dp.world()[1] > 1:
        dp.allreduce_tally(tally.nll, tally.count, tally.confusion)
        torch.distributed.all_reduce(vox)
        if hist is not None:
            dp.allreduce_hist(hist)
        if cal is not None:
            dp.allreduce_calibration(cal["calib"], cal["brier"], cal["unc"])
    loss = loss_fn(tally).double().reshape(1)
    # one copy: [nll (fp64 bits), count, confusion..., voxels, loss (fp64 bits), histogram..., calibration...]
    parts = [tally._buf, vox, loss.view(torch.int64)] + ([hist.view(-1)] if hist is not None else [])
    if cal is not None:
        parts += [cal["calib"].view(-1), cal["brier"].view(torch.int64), cal["unc"]]
    host = torch.cat(parts).cpu()
    cm = host[2:2 + k * k].view(k, k).numpy()
    voxels = int(host[2 + k * k])
    out = {"loss": float(host[3 + k * k:4 + k * k].view(torch.float64)[0]), "metrics": metrics_from_confusion(cm, voxels),
           "tally": tally, "voxels": voxels}
    if hist is not None:
        out["hist"] = hist
        out["curves"] = curves_from_hist(host[4 + k * k:4 + k * k + hist.numel()].view(hist.shape).numpy())
    if cal is not None:
        c0 = 4 + k * k + (hist.numel() if hist is not None else 0)
        ch = host[c0:c0 + cal["calib"].numel()].view(cal["calib"].shape)
        rest = host[c0 + ch.numel():]
        out["calib"] = cal["calib"]
        bins = ch.shape[1]
        out["calibration"] = calibration_from_hist(ch.numpy(), float(rest[:1].view(torch.float64)[0]),
                                                   ece_bins=15 if bins % 15 == 0 else bins, unc=rest[1:3].numpy(),
                                                   voxels=voxels)
    return out


def _next_mult(n: int, m: int = 16) -> int:
    return ((n + m - 1) // m) * m


def _pad_to_mult_3d(x: torch.Tensor, m: int = 16):
    """Replicate-pad [B,C,D,H,W] so that D/H/W are multiples of m (models.py:109-120); (x_pad, (D,H,W)) or (x, None)."""
    if x.ndim != 5:
        raise ValueError(f"expect [B,C,D,H,W], got {tuple(x.shape)}")
    _, _, D, H, W = x.shape
    pd, ph, pw = _next_mult(D, m) - D, _next_mult(H, m) - H, _next_mult(W, m) - W
    if not (pd or ph or pw):
        return x, None
    x = torch.nn.functional.pad(x, (pw // 2, pw - pw // 2, ph // 2, ph - ph // 2, pd // 2, pd - pd // 2), mode="replicate")
    return x, (D, H, W)


def _center_crop_to_3d(x: torch.Tensor, orig_dhw):
    """models.py:122-127."""
    if orig_dhw is None:
        return x
    D, H, W = orig_dhw
    sd, sh, sw = (x.shape[2] - D) // 2, (x.shape[3] - H) // 2, (x.shape[4] - W) // 2
    return x[:, :, sd:sd + D, sh:sh + H, sw:sw + W]


_pad_to_mult16_3d = _pad_to_mult16 = _pad_to_mult_3d
_center_crop_3d = _center_crop = _center_crop_to_3d


class _LitSPCT_Base(BaseLitModel):
    """Pads the input to multiples of `pad_multiple` in (D,H,W) — the 5 energy bins become 16 planes — runs
    the core and centre-crops the logits (models.py:703-712). The pad / crop are tiny tensor ops around the
    engine's autograd node; `fit_step` pads the labels with ignore_index instead of cropping the logits."""

    def __init__(self, num_classes=NUM_CLASSES, lr=BEST_LR, pad_multiple: int = 16):
        super().__init__(num_classes=num_classes, lr=lr, is_3d=True)
        self._pad_multiple = int(pad_multiple)

    def forward(self, x):
        x = _pick_first_if_seq(x)
        if x.ndim == 4:
            x = x.unsqueeze(1)
        x_pad, orig = _pad_to_mult16_3d(x.float(), self._pad_multiple)
        return _center_crop_3d(self.model(x_pad), orig)

    def _padded_batch(self, batch):
        """(x_pad, labels, orig): the images padded as `forward` pads them, the labels placed at the crop and
        ignore_index outside it (voxels outside the crop carry no loss and no tally), orig (D,H,W) or None."""
        imgs, lbls = batch if isinstance(batch, (list, tuple)) else (batch["image"], batch["label"])
        imgs, lbls = _pick_first_if_seq(imgs), _pick_first_if_seq(lbls)
        if imgs.ndim == 4:
            imgs = imgs.unsqueeze(1)
        x_pad, orig = _pad_to_mult16_3d(imgs.float(), self._pad_multiple)
        if orig is not None:
            D, H, W = orig
            full = torch.full((lbls.shape[0],) + tuple(x_pad.shape[2:]), IGNORE_INDEX, dtype=torch.int64, device=lbls.device)
            sd, sh, sw = (x_pad.shape[2] - D) // 2, (x_pad.shape[3] - H) // 2, (x_pad.shape[4] - W) // 2
            full[:, sd:sd + D, sh:sh + H, sw:sw + W] = lbls
            lbls = full
        return x_pad, lbls, orig

    def fit_step(self, batch, optimize: bool = True, sample_group: Optional[int] = None):
        x_pad, lbls, _ = self._padded_batch(batch)
        return super().fit_step((x_pad, lbls), optimize=optimize, sample_group=sample_group)

    def eval_step(self, batch, tally: Optional[LossTally] = None, per_sample: bool = False, return_labels: bool = False,
                  sample_group: Optional[int] = None, curves=None):
        """BaseLitModel.eval_step on the padded batch; the returned label map is cropped back to the input's size. The
        padding carries ignore_index, so the histograms count the input's voxels only."""
        x_pad, lbls, orig = self._padded_batch(batch)
        out = super().eval_step((x_pad, lbls), tally=tally, per_sample=per_sample, return_labels=return_labels,
                                sample_group=sample_group, curves=curves)
        if out["labels"] is not None and orig is not None:
            out["labels"] = _center_crop_to_3d(out["labels"].unsqueeze(1), orig)[:, 0].contiguous()
        return out


class LitSPCT_SEspec(_LitSPCT_Base):
    """"SP_UNet": plain double-conv blocks + Channel-SE + Spectral-SE at all encoder stages (models.py:1585-1592)."""

    def __init__(self, num_classes=NUM_CLASSES, lr=BEST_LR, base=32, pad_multiple=16):
        super().__init__(num_classes=num_classes, lr=lr, pad_multiple=pad_multiple)
        self.model = UNet3D_SpectralCore(in_channels=1, num_classes=num_classes, base=base, ksd=3, use_se=True,
                                         use_specse=True, use_spatial=False, use_skip_gate=False)


class LitSPCT_EFiLM_FourierGate(BaseLitModel):
    """"SPFF-UNet" (models.py:1558-1564, config.py:423-428)."""

    def __init__(self, num_classes=NUM_CLASSES, lr=BEST_LR, base=32, ksd=3, use_se=True, use_specse=True,
                 use_spatial=False, use_skip_gate=False, **kw):
        super().__init__(num_classes=num_classes, lr=lr, is_3d=True)
        self.model = build_spct_energyfilm_fourier(num_classes=num_classes, base=base, ksd=ksd, use_se=use_se,
                                                   use_specse=use_specse, use_spatial=use_spatial,
                                                   use_skip_gate=use_skip_gate, **kw)


class LitSPCT_EnergyFiLM(BaseLitModel):
    """"E_SP_UNet": EnergyFiLM only (models.py:1565-1573)."""

    def __init__(self, num_classes=NUM_CLASSES, lr=BEST_LR, base=32, ksd=3, use_se=True, use_specse=True,
                 use_spatial=False, use_skip_gate=False, **kw):
        super().__init__(num_classes=num_classes, lr=lr, is_3d=True, **kw)
        core = UNet3D_SpectralCore(in_channels=1, num_classes=num_classes, base=base, ksd=ksd, use_se=use_se,
                                   use_specse=use_specse, use_spatial=use_spatial, use_skip_gate=use_skip_gate)
        self.model = upgrade_spct_with_novel_blocks(core, use_efilm=True, use_fouriergate=False, use_moe=False)


class LitSPCT_FourierGate(BaseLitModel):
    """"FG_SP_UNet": FourierGate only (models.py:1575-1583)."""

    def __init__(self, num_classes=NUM_CLASSES, lr=BEST_LR, base=32, ksd=3, use_se=True, use_specse=True,
                 use_spatial=False, use_skip_gate=False, **kw):
        super().__init__(num_classes=num_classes, lr=lr, is_3d=True, **kw)
        core = UNet3D_SpectralCore(in_channels=1, num_classes=num_classes, base=base, ksd=ksd, use_se=use_se,
                                   use_specse=use_specse, use_spatial=use_spatial, use_skip_gate=use_skip_gate)
        self.model = upgrade_spct_with_novel_blocks(core, use_efilm=False, use_fouriergate=True, use_moe=False)


class LitSPCT_ControlUNet(BaseLitModel):
    """"PlainCore_UNet": the same core with plain double-conv blocks and no gates (models.py:1594-1607)."""

    def __init__(self, num_classes=NUM_CLASSES, lr=BEST_LR, base=32, ksd=3, use_se=False, use_specse=False,
                 use_spatial=False, use_skip_gate=False, **kw):
        super().__init__(num_classes=num_classes, lr=lr, is_3d=True, **kw)
        self.model = UNet3D_SpectralCore(in_channels=1, num_classes=num_classes, base=base, ksd=ksd, use_se=use_se,
                                         use_specse=use_specse, use_spatial=use_spatial, use_skip_gate=use_skip_gate)


# --------------------------------------------------------------------------------------------------
# "3DUNet" control: Cicek 3D U-Net behind a depth adapter (models.py:153-163, 718-846; config.py:283-311)
# --------------------------------------------------------------------------------------------------
def _resize_depth_like(x: torch.Tensor, target_depth: int):
    """[B,C,D,H,W] -> D resized to target_depth by the trilinear rule (models.py:153-157), as a plane-mixing
    matrix on the device (spff_depth_resample). Used by callers outside the fused path."""
    B, C, D, H, W = x.shape
    if D == target_depth:
        return x
    from spff_b200.cicek import depth_matrix
    if not x.is_cuda:
        raise RuntimeError("_resize_depth_like (B200 build) needs a CUDA tensor; there is no CPU fallback")
    xin = x.float().contiguous().view(B * C, D, H * W)
    if (H * W) % 4:
        raise ValueError("H*W must be a multiple of 4")
    out = torch.empty(B * C, target_depth, H * W, device=x.device)
    ops.depth_resample(xin, out, depth_matrix(D, target_depth).to(x.device))
    return out.view(B, C, target_depth, H, W)


_resize_logits_depth_like = _resize_depth_like


class _CicekFn(torch.autograd.Function):
    """Cicek3DUNet (+ depth adapter) as one autograd node."""

    @staticmethod
    def forward(ctx, x, net, target_depth, *params):
        if not net.training:
            # the backward kernels implement training-mode BatchNorm (batch statistics: mean / projection terms in dx);
            # eval-mode BatchNorm has a different input gradient, so gradients in eval() would be silently wrong
            raise NotImplementedError("Cicek3DUNet (B200 build): gradients through eval-mode BatchNorm (running statistics) "
                                      "are not implemented; call .train(), or run the forward under torch.no_grad()")
        logits, state = net.engine.forward_saved(x, target_depth, training=True)
        ctx.net, ctx.state = net, state
        return logits

    @staticmethod
    def backward(ctx, dlogits):
        net = ctx.net
        if ctx.state is None:
            raise RuntimeError("Cicek3DUNet (B200 build): the activations of this forward were released by its first "
                               "backward; retain_graph / a second backward through the same forward is not supported")
        flat = torch.zeros(net._flat_numel, device=dlogits.device)
        G = net._views(flat)
        net.engine.backward_saved(ctx.state, dlogits, G)
        ctx.state = None
        return (None, None, None) + tuple(G[n] for n in net._names)


class Cicek3DUNet(nn.Module):
    """Çiçek et al. 3-D U-Net (models.py:718-751): five levels of (3x3x3 conv, BatchNorm3d, ReLU) x 2,
    MaxPool3d(2), ConvTranspose3d(2, stride 2), cat([up, skip]), 1x1x1 head; base 32 -> 512 channels at the
    bottleneck. Same constructor, attribute names and construction order as the reference (so the same seed
    draws the same weights and checkpoints interchange); the sub-modules are parameter containers and the graph
    runs in `spff_b200.cicek.CicekEngine`. D, H, W must be multiples of 16."""

    def __init__(self, num_classes: int, base: int = 32, use_bn: bool = True):
        super().__init__()
        if not use_bn:
            raise NotImplementedError("the B200 path implements the BatchNorm configuration the variant uses "
                                      "(use_bn=True, config.py:299)")
        if int(base) != 32:
            raise NotImplementedError("the B200 kernels are built for base=32 (models.py:767)")
        if not 0 < num_classes <= 16:
            raise NotImplementedError("the head / loss kernels support up to 16 classes")

        def block(ci, co):
            return nn.Sequential(nn.Conv3d(ci, co, 3, padding=1, bias=False), nn.BatchNorm3d(co), nn.ReLU(inplace=True),
                                 nn.Conv3d(co, co, 3, padding=1, bias=False), nn.BatchNorm3d(co), nn.ReLU(inplace=True))

        self.enc1 = block(1, base); self.pool1 = nn.MaxPool3d(2)
        self.enc2 = block(base, base * 2); self.pool2 = nn.MaxPool3d(2)
        self.enc3 = block(base * 2, base * 4); self.pool3 = nn.MaxPool3d(2)
        self.enc4 = block(base * 4, base * 8); self.pool4 = nn.MaxPool3d(2)
        self.bott = block(base * 8, base * 16)
        self.up4 = nn.ConvTranspose3d(base * 16, base * 8, 2, stride=2)
        self.dec4 = block(base * 8 + base * 8, base * 8)
        self.up3 = nn.ConvTranspose3d(base * 8, base * 4, 2, stride=2)
        self.dec3 = block(base * 4 + base * 4, base * 4)
        self.up2 = nn.ConvTranspose3d(base * 4, base * 2, 2, stride=2)
        self.dec2 = block(base * 2 + base * 2, base * 2)
        self.up1 = nn.ConvTranspose3d(base * 2, base, 2, stride=2)
        self.dec1 = block(base + base, base)
        self.out = nn.Conv3d(base, num_classes, 1)
        self._num_classes, self._base = int(num_classes), int(base)
        self._engine = None
        self._flat: Optional[torch.Tensor] = None
        self._names: List[str] = []
        self._slots: Dict[str, tuple] = {}
        self._flat_numel = 0

    @property
    def engine(self):
        if self._engine is None:
            from spff_b200.cicek import CicekEngine
            self._engine = CicekEngine(self._num_classes, self._base, lambda: self._param_data, lambda: self._buffer_data,
                                       lambda: tuple(p._version for p in self._param_objs.values()))
        return self._engine

    def _views(self, flat: torch.Tensor) -> Dict[str, torch.Tensor]:
        return {n: flat[o:o + k].view(shape) for n, (o, k, shape) in self._slots.items()}

    def materialize(self):
        """(Re)build the flat fp32 parameter buffer: every parameter's `.data` becomes a view of it, so the gradient
        all-reduce and the fused SGD run over one contiguous range. BatchNorm buffers stay where they are."""
        from spff_b200.cicek import flat_names
        dev = self.out.weight.device
        if dev.type != "cuda":
            raise RuntimeError("Cicek3DUNet (B200 build) must live on a CUDA sm_100 device: there is no CPU fallback. "
                               "Call .to('cuda') / .cuda() first.")
        named = list(self.named_parameters())
        ok = self._flat is not None and self._flat.device == dev
        if ok:
            base, end = self._flat.data_ptr(), self._flat.data_ptr() + 4 * self._flat_numel
            ok = all(base <= p.data_ptr() < end and p.dtype == torch.float32 for _, p in named)
        if not ok:
            slots, total = flat_names(named)
            flat = torch.zeros(total, dtype=torch.float32, device=dev)
            for n, p in named:
                o, k, shape = slots[n]
                v = flat[o:o + k].view(shape)
                v.copy_(p.data)
                p.data = v
            self._flat, self._slots, self._flat_numel = flat, slots, total
            self._names = [n for n, _ in named]
            self._param_objs = dict(named)
            self._param_data = {n: p.data for n, p in named}
            if self._engine is not None:
                self._engine.invalidate_weights()
        self._buffer_data = dict(self.named_buffers())   # .to() / load_state_dict may have replaced them

    def _run(self, x, target_depth: Optional[int]):
        x = _pick_first_if_seq(x)
        if x.ndim == 4:
            x = x.unsqueeze(1)
        self.materialize()
        x = x.to(self.out.weight.device)
        params = [self._param_objs[n] for n in self._names]
        if torch.is_grad_enabled() and any(p.requires_grad for p in params):
            return _CicekFn.apply(x, self, target_depth, *params)
        return self.engine.infer(x, target_depth, training=self.training)

    def forward(self, x):
        """logits [B,K,D,H,W] of x [B,1,D,H,W] (D, H, W multiples of 16)."""
        return self._run(x, None)

    def forward_adapted(self, x, target_depth: int):
        """resize D -> target_depth, the network, resize back — fused (no 16-plane logits in memory)."""
        return self._run(x, int(target_depth))


class LitCicek3DUNet_DepthAdapter_Published(pl.LightningModule):
    """"3DUNet" (models.py:753-846 as configured by config.py:283-303): trilinear depth adapter 5 -> 16 -> 5 around
    Cicek3DUNet, plain CE over valid voxels, SGD(lr 1e-2, momentum 0.99). Same constructor as the reference; the
    options its configuration leaves off (class / voxel weights, the soft Dice term, use_bn=False) raise."""

    def __init__(self, num_classes: int, target_depth: int = 16, lr: float = 1e-2, momentum: float = 0.99,
                 nesterov: bool = False, weight_decay: float = 0.0, ignore_index: Optional[int] = 255,
                 class_weights: Optional[list] = None, voxel_weight_key: Optional[str] = None, ce_weight: float = 1.0,
                 dice_weight: float = 0.0, use_bn: bool = True, include_bg_in_dice: bool = False, *args, **kwargs):
        super().__init__()
        self.save_hyperparameters(dict(num_classes=num_classes, target_depth=target_depth, lr=lr, momentum=momentum,
                                       nesterov=nesterov, weight_decay=weight_decay, ignore_index=ignore_index,
                                       class_weights=class_weights, voxel_weight_key=voxel_weight_key, ce_weight=ce_weight,
                                       dice_weight=dice_weight, use_bn=use_bn, include_bg_in_dice=include_bg_in_dice))
        if class_weights is not None or voxel_weight_key is not None:
            raise NotImplementedError("class / voxel weighted CE is off in the 3DUNet variant (config.py:293-294)")
        if float(dice_weight) > 0.0:
            raise NotImplementedError("the soft Dice term is off in the 3DUNet variant (dice_weight=0, config.py:297)")
        self.backbone = Cicek3DUNet(num_classes=num_classes, base=32, use_bn=use_bn)
        self.target_depth = int(target_depth)
        self.class_weights = None
        self.voxel_weight_key = None
        self.ignore_index = ignore_index
        self.include_bg_in_dice = include_bg_in_dice
        self.ce_weight, self.dice_weight = float(ce_weight), float(dice_weight)
        self._fused = None

    @property
    def model(self):
        """`.model` is what the callers' profilers read (train.py:1416); for this wrapper it is the backbone."""
        return self.backbone

    def forward(self, x):
        return self.backbone.forward_adapted(x, self.target_depth)

    def _weighted_softmax_ce(self, logits, target, voxel_weights=None):
        from .helpers import masked_ce_loss
        if voxel_weights is not None:
            raise NotImplementedError("voxel weights are off in the 3DUNet variant")
        if target.ndim == 5 and target.shape[1] == 1:
            target = target[:, 0]
        return masked_ce_loss(logits, target, self.ignore_index)

    def _loss_and_log(self, logits, y, stage: str, voxel_w=None, log_metrics: bool = True):
        y = _canonicalize_targets_3d(y).to(logits.device)
        loss = self._weighted_softmax_ce(logits, y, voxel_w) * self.ce_weight
        self.log(f"{stage}_loss", loss, prog_bar=(stage == "train"), on_step=False, on_epoch=True, sync_dist=True)
        if log_metrics:
            macro_dice = per_class_metrics_3d(logits, y, self.hparams.num_classes, ignore_index=self.ignore_index)[3]
            self.log(f"{stage}_macro_dice", macro_dice, on_step=False, on_epoch=True, prog_bar=True, sync_dist=True)
        return loss

    def _unpack(self, batch):
        if isinstance(batch, (list, tuple)):
            x, y = batch
            return x, y, None
        return batch["image"], batch["label"], None

    def training_step(self, batch, _):
        x, y, vw = self._unpack(batch)
        return self._loss_and_log(self(x), y, "train", voxel_w=vw)

    def validation_step(self, batch, _):
        x, y, vw = self._unpack(batch)
        return self._loss_and_log(self(x), y, "val", voxel_w=vw, log_metrics=True)

    def test_step(self, batch, _):
        x, y, vw = self._unpack(batch)
        return self._loss_and_log(self(x), y, "test", voxel_w=vw)

    def configure_optimizers(self):
        return torch.optim.SGD(self.parameters(), lr=self.hparams.lr, momentum=self.hparams.momentum,
                               nesterov=bool(self.hparams.nesterov), weight_decay=self.hparams.weight_decay)

    # -- B200-native fused training step ---------------------------------------------------------
    def fit_step(self, batch, optimize: bool = True):
        """forward + CE + backward (+ data-parallel gradient all-reduce + SGD step) without materialising logits:
        `loss = training_step(batch); loss.backward(); optimizer.step()` of the reference with
        torch.optim.SGD(lr, momentum, nesterov, weight_decay). BatchNorm runs in training mode over the whole
        (per-rank) batch. Returns {"loss": device scalar, "tally": LossTally}; nothing synchronises the host."""
        x, y, _ = self._unpack(batch)
        x, y = _pick_first_if_seq(x), _pick_first_if_seq(y)
        net = self.backbone
        if x.ndim == 4:
            x = x.unsqueeze(1)
        net.materialize()
        dev = net._flat.device
        y = _canonicalize_targets_3d(y) if y.dtype not in (torch.uint8, torch.int64) or y.ndim != 4 else y
        x = x.to(dev, non_blocking=True)
        y = y.to(dev, non_blocking=True)
        st = self._fused
        if st is None or st["flat"] is not net._flat:
            st = self._fused = dict(flat=net._flat, grad=torch.zeros_like(net._flat), buf=torch.zeros_like(net._flat),
                                    step=0, tally=LossTally(self.hparams.num_classes, dev))
            st["G"] = net._views(st["grad"])
        st["grad"].zero_()
        st["tally"].zero()
        ign = -1 if self.ignore_index is None else int(self.ignore_index)
        with torch.no_grad():
            net.engine.train_step(x, y, st["G"], st["tally"], self.target_depth, ignore_index=ign)
            gscale = dp.allreduce_grads(st["grad"])
            if optimize:
                ops.sgd_step(net._flat, st["grad"], st["buf"], float(self.hparams.lr), float(self.hparams.momentum),
                             float(self.hparams.weight_decay), bool(self.hparams.nesterov), st["step"] == 0,
                             gscale * self.ce_weight)
                st["step"] += 1
                net.engine.invalidate_weights()
            t = st["tally"]
            loss = (self.ce_weight * t.nll[0] / t.count[0].clamp(min=1).double()).float()
        return {"loss": loss, "tally": t}

    def fused_grads(self) -> Dict[str, torch.Tensor]:
        return self._fused["G"]

    # -- B200-native fused evaluation step --------------------------------------------------------
    @torch.no_grad()
    def eval_step(self, batch, tally: Optional[LossTally] = None, per_sample: bool = False, return_labels: bool = False,
                  curves=None):
        """`_loss_and_log`'s loss and per_class_metrics_3d's statistics without the logits, BatchNorm in the module's
        mode (as `forward` under no_grad; BatchNorm couples the samples, so the batch runs whole). Batch forms,
        accumulation, `curves` and return value as BaseLitModel.eval_step; the loss is ce_weight * CE over
        max(#valid, 1)."""
        x, y, _ = self._unpack(batch)
        x, y = _pick_first_if_seq(x), _pick_first_if_seq(y)
        net = self.backbone
        if x.ndim == 4:
            x = x.unsqueeze(1)
        net.materialize()
        dev = net._flat.device
        y = _canonicalize_targets_3d(y) if y.dtype not in (torch.uint8, torch.int64) or y.ndim != 4 else y
        x = x.to(dev, non_blocking=True)
        y = y.to(dev, non_blocking=True)
        k = self.hparams.num_classes
        tally = LossTally(k, dev) if tally is None else tally
        bsz = x.shape[0]
        rows = (torch.zeros(bsz, dtype=torch.float64, device=dev), torch.zeros(bsz, dtype=torch.int64, device=dev),
                torch.zeros(bsz, k, k, dtype=torch.int64, device=dev)) if per_sample else None
        labels = torch.empty(bsz, *x.shape[2:], dtype=torch.uint8, device=dev) if return_labels else None
        ign = -1 if self.ignore_index is None else int(self.ignore_index)
        hist, sample_hist = _curve_buffers(curves, k, bsz, per_sample, dev)
        net.engine.eval_step(x, y, tally, self.target_depth, ignore_index=ign, training=net.training, per_sample=rows,
                             labels_out=labels, hist=hist, sample_hist=sample_hist)
        return {"loss": self._tally_loss(tally), "tally": tally, "per_sample": rows, "labels": labels, "hist": hist,
                "per_sample_hist": sample_hist}

    def _tally_loss(self, tally: LossTally) -> torch.Tensor:
        return (self.ce_weight * tally.nll[0] / tally.count[0].clamp(min=1).double()).float()

    @torch.no_grad()
    def evaluate(self, batches, curves: Optional[int] = None):
        """BaseLitModel.evaluate for this variant (loss: ce_weight * CE, no Dice term)."""
        return _evaluate(self.hparams.num_classes, next(self.parameters()).device, self._tally_loss, batches,
                         lambda b, t, h: self.eval_step(b, tally=t, curves=h), curves)

    def fused_optimizer_state(self) -> Dict[str, object]:
        """Momentum buffer + step count of the fused SGD, for checkpoint / resume (save next to `state_dict()`)."""
        st = self._fused
        if st is None:
            return {"step": 0}
        return {"step": int(st["step"]), "momentum_buffer": st["buf"].detach().cpu(), "lr": float(self.hparams.lr)}

    def load_fused_optimizer_state(self, state: Dict[str, object]) -> None:
        net = self.backbone
        net.materialize()
        if not state or int(state.get("step", 0)) == 0:
            self._fused = None
            return
        flat = net._flat
        if state["momentum_buffer"].numel() != flat.numel():
            raise ValueError(f"optimizer state holds {state['momentum_buffer'].numel()} elements, the model {flat.numel()}")
        self._fused = dict(flat=flat, grad=torch.zeros_like(flat), buf=state["momentum_buffer"].to(flat), step=int(state["step"]),
                           tally=LossTally(self.hparams.num_classes, flat.device))
        self._fused["G"] = net._views(self._fused["grad"])
        self.hparams["lr"] = float(state.get("lr", self.hparams.lr))

    @torch.no_grad()
    def predict_labels(self, x) -> torch.Tensor:
        """uint8 label map [B,D,H,W] (argmax fused into the head kernel); BatchNorm as the module's mode says."""
        x = _pick_first_if_seq(x)
        if x.ndim == 4:
            x = x.unsqueeze(1)
        net = self.backbone
        net.materialize()
        return net.engine.infer(x.to(net._flat.device), self.target_depth, training=net.training, argmax=True)


class SpctEnsemble:
    """Seed ensembles and mirror test-time augmentation of the depth-preserving SPCT family: the softmax averaged over
    members and input flips, on the device, with no logits in memory.

    `members`: Lightning wrappers whose `.model` is a UNet3D_SpectralCore (SPFF-UNet, E_SP_UNet, FG_SP_UNet,
    PlainCore_UNet) or such cores themselves, of one `net_config()` and one device; the ensemble holds references to
    them (no copies of weights) and touches no optimizer or fused-step state. `tta`: None (the input as given) or
    "flip" (identity, H, W and H+W mirrors; the depth axis holds the energy bins and is not a symmetry).

    Every pass runs the member on the (flipped) input and adds its softmax, mirrored back, into an fp32 accumulator of
    one sample group; p̄ = the mean over members x flips. `predict_labels` / `predict_proba` give its arg-max / p̄,
    `eval_step` / `evaluate` the loss, metrics and curves of BaseLitModel's on p̄: the loss is ce_plus_macro_dice_loss on
    the averaged probabilities (CE of p̄ + 0.5 * (1 - hard macro Dice of its arg-max)).

    `predict_uncertainty` gives per-voxel uncertainty maps (the predictive entropy H[p̄] and the mutual information
    between prediction and pass, H[p̄] - mean over passes of H[p]), and `eval_step` / `evaluate(calibration=T)` the
    calibration statistics of p̄ (helpers.calibration_from_hist). For one model, use SpctEnsemble([lit]): its MI is 0
    and its entropy and calibration are the single model's.

    `temperature` T (> 0, finite; settable as `ens.temperature`) recalibrates the pooled distribution:
    p̃_c = p̄_c^(1/T) / sum_c' p̄_c'^(1/T), which is softmax(z / T) for one member without TTA. p̃ replaces p̄ in
    `predict_proba`, `predict_uncertainty`'s entropy, and the loss, curves and calibration of `eval_step` / `evaluate`;
    the arg-max (labels, confusion, Dice) does not change, and the mutual information stays H[p̄] - mean H[p] of the
    untempered passes (a temperature on the pool does not model the members' disagreement), bit for bit.
    T = 1 is exactly the untempered computation. `fit_temperature` fits T on a validation set in one pass."""

    def __init__(self, members, tta: Optional[str] = None, temperature: float = 1.0):
        if tta not in (None, "flip"):
            raise ValueError(f"tta must be None or 'flip', got {tta!r}")
        members = list(members)
        if not members:
            raise ValueError("an ensemble needs at least one member")
        cores = []
        for i, m in enumerate(members):
            if isinstance(m, _LitSPCT_Base):
                raise NotImplementedError(f"member {i}: SP_UNet pads the depth to 16 planes and crops its logits back; the "
                                          "ensemble averages the softmax of depth-preserving cores only")
            if isinstance(m, (LitCicek3DUNet_DepthAdapter_Published, Cicek3DUNet)):
                raise NotImplementedError(f"member {i}: the 3DUNet's BatchNorm couples the samples of a batch, so its "
                                          "output cannot be computed sample group by sample group like the SPCT family's")
            core = m if isinstance(m, UNet3D_SpectralCore) else getattr(m, "model", None)
            if not isinstance(core, UNet3D_SpectralCore):
                raise TypeError(f"member {i}: expected a UNet3D_SpectralCore or a Lightning wrapper of one, got "
                                f"{type(m).__name__}")
            cores.append(core)
        cfg0, dev0 = cores[0].net_config(), cores[0].out.weight.device
        for i, core in enumerate(cores[1:], 1):
            cfg = core.net_config()
            for f in dataclasses.fields(cfg):
                if getattr(cfg, f.name) != getattr(cfg0, f.name):
                    raise ValueError(f"member {i}: net_config field {f.name!r} is {getattr(cfg, f.name)!r}, member 0 has "
                                     f"{getattr(cfg0, f.name)!r}")
            if core.out.weight.device != dev0:
                raise ValueError(f"member {i} lives on {core.out.weight.device}, member 0 on {dev0}")
        self.members, self.cores, self.tta = members, cores, tta
        self.num_classes = cfg0.num_classes
        self.flips = (0, 1, 2, 3) if tta == "flip" else (0,)
        self._copy_stream = None
        self.temperature = temperature

    @property
    def temperature(self) -> float:
        return self._temperature

    @temperature.setter
    def temperature(self, t: float):
        t = float(t)
        if not (math.isfinite(t) and t > 0.0):
            raise ValueError(f"temperature must be positive and finite, got {t}")
        self._temperature = t

    @property
    def device(self) -> torch.device:
        return self.cores[0].out.weight.device

    def _engines(self, frames: int):
        for core in self.cores:
            core.materialize(frames)
        return [core.engine for core in self.cores]

    def _images(self, x) -> torch.Tensor:
        x = _pick_first_if_seq(x)
        return x.unsqueeze(1) if x.ndim == 4 else x

    @torch.no_grad()
    def predict_labels(self, x, sample_group: Optional[int] = None) -> torch.Tensor:
        """uint8 label map [B,F,H,W]: the arg-max (first maximum) of the averaged softmax."""
        x = self._images(x)
        engines = self._engines(x.shape[2])
        b, _, d, h, w = x.shape
        out = torch.empty(b, d, h, w, dtype=torch.uint8, device=self.device)
        run_ensemble(engines, x.to(self.device), self.flips, sample_group or self.cores[0].sample_group, labels_out=out)
        return out

    @torch.no_grad()
    def predict_proba(self, x, sample_group: Optional[int] = None) -> torch.Tensor:
        """float16 [B,K,F,H,W]: the averaged softmax (the layout of softmax(model(x), 1))."""
        x = self._images(x)
        engines = self._engines(x.shape[2])
        b, _, d, h, w = x.shape
        out = torch.empty(b, self.num_classes, d, h, w, dtype=torch.float16, device=self.device)
        run_ensemble(engines, x.to(self.device), self.flips, sample_group or self.cores[0].sample_group, proba_out=out,
                     inv_temperature=1.0 / self.temperature)
        return out

    @torch.no_grad()
    def predict_uncertainty(self, x, sample_group: Optional[int] = None) -> Dict[str, torch.Tensor]:
        """One pass over members x flips: {"labels": uint8 [B,F,H,W] (predict_labels), "entropy": float16 [B,F,H,W]
        (H[p̄] = -sum_c p̄_c log p̄_c, nats; H[p̃] with a temperature), "mutual_info": float16 [B,F,H,W] (H[p̄] - mean over
        passes of H[p], clamped at 0: the members' / flips' disagreement; untempered whatever the temperature),
        "case_entropy", "case_mutual_info": float64 [B] (their means over the voxels of each case, from sums of the
        per-voxel values rounded to 2^-24)}."""
        x = self._images(x)
        engines = self._engines(x.shape[2])
        b, _, d, h, w = x.shape
        dev = self.device
        labels = torch.empty(b, d, h, w, dtype=torch.uint8, device=dev)
        ent = torch.empty(b, d, h, w, dtype=torch.float16, device=dev)
        mi = torch.empty_like(ent)
        sums = torch.zeros(2, dtype=torch.int64, device=dev)
        rows = torch.zeros(b, 2, dtype=torch.int64, device=dev)
        run_ensemble(engines, x.to(dev), self.flips, sample_group or self.cores[0].sample_group, labels_out=labels,
                     entropy_out=ent, mi_out=mi, unc=sums, sample_unc=rows, inv_temperature=1.0 / self.temperature)
        case = rows.double() * (2.0 ** -24) / (d * h * w)
        return {"labels": labels, "entropy": ent, "mutual_info": mi, "case_entropy": case[:, 0],
                "case_mutual_info": case[:, 1]}

    def _batch(self, batch, sample_group: Optional[int]):
        """(engines, images, labels, StagedBatch or None, group) of an evaluation batch: tuple or dict, host or device,
        uint8 or int64 labels; host batches are staged group by group on the copy stream."""
        imgs, lbls = batch if isinstance(batch, (list, tuple)) else (batch["image"], batch["label"])
        imgs, lbls = self._images(imgs), _pick_first_if_seq(lbls)
        engines = self._engines(imgs.shape[2])
        dev = self.device
        if lbls.dtype not in (torch.uint8, torch.int64):
            lbls = lbls.long()
        group = sample_group or self.cores[0].sample_group
        staged = None
        if not imgs.is_cuda and not lbls.is_cuda:
            if self._copy_stream is None:
                self._copy_stream = torch.cuda.Stream(device=dev)
            staged = StagedBatch(imgs, lbls, dev, group, self._copy_stream)
            imgs, lbls = staged.x, staged.labels
        else:
            imgs = imgs.to(dev, non_blocking=True)
            lbls = lbls.to(dev, non_blocking=True)
        return engines, imgs, lbls, staged, group

    @torch.no_grad()
    def eval_step(self, batch, tally: Optional[LossTally] = None, per_sample: bool = False, return_labels: bool = False,
                  sample_group: Optional[int] = None, curves=None, calibration=None):
        """BaseLitModel.eval_step for the ensemble: the tally, per-sample rows, arg-max map and histograms of the
        averaged softmax p̄ (same arguments, batch forms and return dict).

        `calibration`: a bin count T in [2, 1024] (fresh zeros) or a contiguous int64 [3,T] histogram on the device to
        accumulate into (as `curves`); adds "calib" ([3,T]: per confidence bin min(floor(conf * T), T - 1), conf = the
        largest p̄_c, the counted voxels, the correct ones and the summed confidence in units of 2^-24), "brier" (fp64
        [1], the summed Brier score) and "uncertainty" (int64 [2], the summed H[p̄] and mutual information in units of
        2^-24 nats); with per_sample=True also "per_sample_calib" [B,3,T], "per_sample_brier" [B] and
        "per_sample_uncertainty" (float64 [B,2], the mean H[p̄] and MI per case). helpers.calibration_from_hist /
        sample_calibration turn them into ECE, reliability diagrams and error detection. With a temperature, everything
        but the arg-max and the mutual information is computed on p̃ (see the class)."""
        engines, imgs, lbls, staged, group = self._batch(batch, sample_group)
        dev = self.device
        k = self.num_classes
        tally = LossTally(k, dev) if tally is None else tally
        bsz = imgs.shape[0]
        rows = (torch.zeros(bsz, dtype=torch.float64, device=dev), torch.zeros(bsz, dtype=torch.int64, device=dev),
                torch.zeros(bsz, k, k, dtype=torch.int64, device=dev)) if per_sample else None
        labels = torch.empty(bsz, *imgs.shape[2:], dtype=torch.uint8, device=dev) if return_labels else None
        hist, sample_hist = _curve_buffers(curves, k, bsz, per_sample, dev)
        cal = {}
        if calibration is not None:
            calib = _calib_buffers(calibration, dev)
            bins = calib.shape[1]
            cal = dict(calib=calib, brier=torch.zeros(1, dtype=torch.float64, device=dev),
                       unc=torch.zeros(2, dtype=torch.int64, device=dev))
            if per_sample:
                cal.update(sample_calib=torch.zeros(bsz, 3, bins, dtype=torch.int64, device=dev),
                           sample_brier=torch.zeros(bsz, dtype=torch.float64, device=dev),
                           sample_unc=torch.zeros(bsz, 2, dtype=torch.int64, device=dev))
        run_ensemble(engines, imgs, self.flips, group, labels=lbls, tally=tally, ignore_index=IGNORE_INDEX,
                     per_sample=rows, labels_out=labels, hist=hist, sample_hist=sample_hist, staged=staged,
                     unc=cal.get("unc"), sample_unc=cal.get("sample_unc"), calib=cal.get("calib"),
                     sample_calib=cal.get("sample_calib"), brier=cal.get("brier"), sample_brier=cal.get("sample_brier"),
                     inv_temperature=1.0 / self.temperature)
        out = {"loss": tally.loss(), "tally": tally, "per_sample": rows, "labels": labels, "hist": hist,
               "per_sample_hist": sample_hist}
        if calibration is not None:
            out.update(calib=cal["calib"], brier=cal["brier"], uncertainty=cal["unc"])
            if per_sample:
                vox = imgs.shape[2] * imgs.shape[3] * imgs.shape[4]
                out.update(per_sample_calib=cal["sample_calib"], per_sample_brier=cal["sample_brier"],
                           per_sample_uncertainty=cal["sample_unc"].double() * (2.0 ** -24) / vox)
        return out

    @torch.no_grad()
    def evaluate(self, batches, sample_group: Optional[int] = None, curves: Optional[int] = None,
                 calibration: Optional[int] = None):
        """BaseLitModel.evaluate for the ensemble: {"loss", "metrics", "tally", "voxels"} (+ "hist", "curves"). With
        `calibration` = T confidence bins also "calib" (int64 [3,T] on the device) and "calibration"
        (helpers.calibration_from_hist: ECE / MCE, reliability diagram, Brier score, error-detection AUROC / AP,
        risk-coverage and the mean entropy and mutual information). The ECE is over 15 bins when T is a multiple of 15
        and over the T bins otherwise ("ece_bins" says which): calibration=960 gives the standard 15-bin ECE exactly
        (960 = 15 * 64)."""
        k, dev = self.num_classes, self.device
        if calibration is None:
            return _evaluate(k, dev, lambda t: t.loss(), batches,
                             lambda b, t, h: self.eval_step(b, tally=t, sample_group=sample_group, curves=h), curves)

        def step(b, t, h, cal):
            out = self.eval_step(b, tally=t, sample_group=sample_group, curves=h, calibration=cal["calib"])
            cal["brier"] += out["brier"]
            cal["unc"] += out["uncertainty"]
            return out
        return _evaluate(k, dev, lambda t: t.loss(), batches, step, curves, calibration)

    @torch.no_grad()
    def fit_temperature(self, batches, t_max: float = 8.0, points: int = 33, sample_group: Optional[int] = None,
                        apply: bool = True) -> dict:
        """Temperature scaling fitted on a validation set in ONE pass over `batches` (the batch forms `evaluate` takes):
        the T that minimises the mean nll of the tempered pooled softmax p̃ over the counted voxels (label in [0, K),
        not the ignore index). Every group's accumulator is reduced on the device to the nll and its derivative at
        each of `points` (odd, 5..63) temperatures spaced geometrically over [1/t_max, t_max] (T = 1 among them);
        no probabilities are kept. Under torch.distributed every rank passes its own batches, the statistics are
        all-reduced once and every rank gets the same T. The host then takes the minimiser of the cubic Hermite
        interpolant in the bracketing interval (helpers.temperature_from_sums).

        Returns {"temperature", "nll" (the INTERPOLATED mean nll at that temperature), "nll_at_1" (mean nll at T = 1,
        untempered), "grid": {"temperature", "nll", "dnll" (d nll / d(1/T))} over the grid, "counted",
        "at_bound" (True when the slope has no sign change on the grid: the temperature is then the end point; widen
        t_max)}. With `apply` the ensemble's temperature is set to it. ValueError when no voxel is counted."""
        betas_h = temperature_grid(t_max, points)
        g, dev = betas_h.size, self.device
        betas = torch.tensor(betas_h, dtype=torch.float32, device=dev)
        sums = torch.zeros(2, g, dtype=torch.float64, device=dev)
        counted = torch.zeros(1, dtype=torch.int64, device=dev)
        for batch in batches:
            engines, imgs, lbls, staged, group = self._batch(batch, sample_group)
            run_ensemble(engines, imgs, self.flips, group, labels=lbls, ignore_index=IGNORE_INDEX, staged=staged,
                         temp_fit=(betas, sums, counted))
        dp.allreduce_temp_fit(sums, counted)
        host = torch.cat([sums.view(-1), counted.double()]).cpu()   # one copy; the count is exact in fp64 below 2^53
        out = temperature_from_sums(betas_h, host[:-1].view(2, g).numpy(), int(host[-1]))
        if apply:
            self.temperature = out["temperature"]
        return out


# Model families outside the hot path (UNETR / SwinUNETR wrappers, R2U-Net, ResUNet++, their helper blocks and losses:
# reference models.py:254-462, 858-1412) are not rebuilt: a name this module does not define resolves to the reference's
# own PyTorch implementation when a reference checkout is on sys.path, so the other `config.VARIANTS` entries keep working.
from ._fallthrough import module_getattr as _module_getattr  # noqa: E402

__getattr__ = _module_getattr(__name__, "models", "only the SPCT family and the 3DUNet control run on the B200 kernels")
