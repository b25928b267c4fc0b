"""Execution engine of the depth-preserving SPCT U-Net family on the B200 kernels.

This is the host-side schedule behind `innovative3D.models.UNet3D_SpectralCore.forward` of this tree:
it turns one forward (+ loss + backward) of the reference graph

    UNet3D_SpectralCore.forward                      reference innovative3D/models.py:693-701
      _DoubleConvSpectral(_Novel).forward            models.py:620-625, 1473-1478
      _post = SpectralSE -> ChannelSE                models.py:684-685
      MaxPool3d((1,2,2)) / ConvTranspose3d / cat     models.py:658-672, 687-691
      out = Conv3d(32, K, 1)                         models.py:674
    ce_plus_macro_dice_loss                          helpers.py:797-803

into launches of the C ABI (include/spff_b200.h). Everything here is enqueue-only: no host
synchronisation, no `.item()`. There is no PyTorch fallback for any of the compute.

Data layout in HBM. Activations are bf16, position-major [n, d, h, w, C] (channels innermost). The
three skip concatenations never happen as copies: a level owns ONE buffer `cat[l]` of 2*C_l
channels, the transposed conv writes channels [0, C_l) ("up first", models.py:691) and the encoder
block of that level writes its output into channels [C_l, 2*C_l) — the decoder conv reads the buffer
as a plain 2*C_l-channel tensor. Gradients mirror that (`dcat[l]`).

Samples are independent through the whole graph (InstanceNorm and every gate are per sample), so a
batch is processed in sample groups ("micro-batches") whose buffers are reused; weight gradients
accumulate (beta = 1) into one flat fp32 buffer, the CE normaliser N_valid is counted over the whole
batch first. This is exact, not an approximation (SURVEY.md §7.4-5).
"""
from __future__ import annotations

import os
from dataclasses import dataclass
from typing import Callable, Dict, List, Optional, Tuple

import torch

from . import ops
from ._lib import Shape

GATE_EFILM, GATE_FOURIER, GATE_SPECSE, GATE_CHANSE = 1, 2, 4, 8
BLOCKS = ("enc1", "enc2", "enc3", "bott", "dec3", "dec2", "dec1")
_LEVEL = {"enc1": 1, "enc2": 2, "enc3": 3, "bott": 4, "dec3": 3, "dec2": 2, "dec1": 1}
_STAGE = {"enc1": 0, "enc2": 1, "enc3": 2, "bott": 3}
SLOPE = 0.01      # nn.LeakyReLU(1e-2)            models.py:175-181
EPS = 1e-5        # nn.InstanceNorm3d(eps=1e-5)   models.py:170


@dataclass(frozen=True)
class NetConfig:
    """Static structure of one variant (what `config.VARIANTS` builders pass to the core)."""
    num_classes: int = 13
    base: int = 32
    conv_names: Tuple[str, str] = ("pre", "body")   # ("b1", "b2") for the plain _DoubleConvSpectral
    efilm: bool = True
    fgate: bool = True
    specse: bool = True
    chanse: bool = True

    def block_flags(self, block: str) -> int:
        f = (GATE_EFILM if self.efilm else 0) | (GATE_FOURIER if self.fgate else 0)
        if block in _STAGE:  # `_post` runs on encoder / bottleneck outputs only (models.py:694-697)
            f |= (GATE_SPECSE if self.specse else 0) | (GATE_CHANSE if self.chanse else 0)
        return f

    def channels(self, block: str) -> Tuple[int, int]:
        f = self.base
        return {"enc1": (1, f), "enc2": (f, 2 * f), "enc3": (2 * f, 4 * f), "bott": (4 * f, 8 * f),
                "dec3": (8 * f, 4 * f), "dec2": (4 * f, 2 * f), "dec1": (2 * f, f)}[block]


class _Pool:
    """Bump allocator over one zero-able device buffer (statistics and reduction targets that the
    kernels accumulate into: one memset per pass instead of one per tensor)."""

    def __init__(self, dtype, device):
        self.dtype, self.device = dtype, device
        self.items: List[Tuple[Tuple[int, ...], int]] = []
        self.total = 0
        self.buf: Optional[torch.Tensor] = None

    def reserve(self, *shape) -> int:
        n = 1
        for s in shape:
            n *= s
        n = (n + 3) // 4 * 4   # keep 16-byte alignment for fp32 / 32 for fp64
        self.items.append((tuple(shape), self.total))
        self.total += n
        return len(self.items) - 1

    def commit(self):
        self.buf = torch.zeros(max(self.total, 4), dtype=self.dtype, device=self.device)

    def get(self, idx: int) -> torch.Tensor:
        shape, off = self.items[idx]
        n = 1
        for s in shape:
            n *= s
        return self.buf[off:off + n].view(shape)

    def zero(self):
        self.buf.zero_()


class _GroupBuffers:
    """Every activation, statistic and scratch gradient of one sample group of fixed shape."""

    def __init__(self, cfg: NetConfig, n: int, d: int, h: int, w: int, device, train: bool):
        if h % 8 or w % 8:
            raise ValueError(f"H, W must be multiples of 8 for the SPCT family (got {h} x {w}); the reference's "
                             "trilinear fallback for odd sizes (models.py:689-690) is not on this path")
        self.n, self.d, self.h, self.w, self.train = n, d, h, w, train
        f = cfg.base
        if os.getenv("SPFF_POISON", "0") == "1":   # test hook: every activation starts as NaN
            bf = lambda hh, ww, c: torch.full((n, d, hh, ww, c), float("nan"), dtype=torch.bfloat16, device=device)
        else:
            bf = lambda hh, ww, c: torch.empty(n, d, hh, ww, c, dtype=torch.bfloat16, device=device)
        self.C = {l: f * 2 ** (l - 1) for l in (1, 2, 3, 4)}
        self.HW = {l: (h >> (l - 1), w >> (l - 1)) for l in (1, 2, 3, 4)}
        self.cat = {l: bf(*self.HW[l], 2 * self.C[l]) for l in (1, 2, 3)}
        self.pool = {l: bf(*self.HW[l + 1], self.C[l]) for l in (1, 2, 3)}    # pooled output of level l
        # training: which corner of each pooling window held the maximum (one byte per pooled element), so that the
        # backward need not read the full-resolution activation again
        self.pool_argmax = {l: torch.empty(n, d, *self.HW[l + 1], self.C[l], dtype=torch.uint8, device=device)
                            for l in (1, 2, 3)} if train else {l: None for l in (1, 2, 3)}
        self.x1, self.a1, self.x2, self.out = {}, {}, {}, {}
        self.partial: Dict[str, torch.Tensor] = {}
        self.slots: Dict[str, int] = {}
        self.f32 = _Pool(torch.float32, device)
        self.idx: Dict[str, int] = {}
        for b in BLOCKS:
            l = _LEVEL[b]
            c = self.C[l]
            hh, ww = self.HW[l]
            self.x1[b] = bf(hh, ww, c)
            self.a1[b] = bf(hh, ww, c)
            self.x2[b] = bf(hh, ww, c)
            self.out[b] = self.cat[l][..., c:] if b.startswith("enc") else bf(hh, ww, c)
            self.idx[f"{b}.S"] = self.f32.reserve(n, d, c)
            # per-item partial statistics written by the conv epilogue (no zeroing needed)
            self.slots[b] = ops.conv3d_k3_stat_slots(Shape(n, d, hh, ww))
            for j in (1, 2):
                if not (b == "enc1" and j == 1):
                    self.partial[f"{b}.{j}"] = torch.empty(n, self.slots[b], 2, c, device=device)
        self.stem_slots = ops.conv3d_stem_stat_slots(Shape(n, d, h, w))
        self.partial["enc1.1"] = torch.empty(n, self.stem_slots, 2, f, device=device)
        self.f32.commit()
        self.coef = {f"{b}.{j}": torch.empty(n, self.C[_LEVEL[b]], 4, device=device) for b in BLOCKS for j in (1, 2)}
        self.P = {b: torch.empty(n, d, self.C[_LEVEL[b]], device=device) for b in BLOCKS}
        self.Q = {b: torch.empty(n, d, self.C[_LEVEL[b]], device=device) for b in BLOCKS}
        self._logits_shape = (n, cfg.num_classes, d, h, w)
        self._logits = None
        self._device = device
        self.x_in: Optional[torch.Tensor] = None   # fp32 [n,1,d,h,w] network input of this group
        if train:
            self.dcat = {l: bf(*self.HW[l], 2 * self.C[l]) for l in (1, 2, 3)}
            self.gout = {l: bf(*self.HW[l], self.C[l]) for l in (1, 2, 3, 4)}
            self.t1 = {l: bf(*self.HW[l], self.C[l]) for l in (1, 2, 3, 4)}
            self.t2 = {l: bf(*self.HW[l], self.C[l]) for l in (1, 2, 3, 4)}
            self.dpool = {l: bf(*self.HW[l + 1], self.C[l]) for l in (1, 2, 3)}
            self.b32 = _Pool(torch.float32, device)
            for b in BLOCKS:
                c = self.C[_LEVEL[b]]
                for j in (1, 2):
                    self.idx[f"{b}.R{j}"] = self.b32.reserve(n, d, c, 6)
            # column statistics of a decoder block's input gradient (dgrad epilogue): their first C_l columns sum to the
            # bias gradient of the transposed conv of that level
            self.dpartial = {l: torch.empty(n, self.slots[dec], 2, 2 * self.C[l], device=device)
                             for l, dec in ((3, "dec3"), (2, "dec2"), (1, "dec1"))}
            self.b32.commit()
            self.bcoef = {f"{b}.{j}": torch.empty(n, self.C[_LEVEL[b]], 4, device=device) for b in BLOCKS for j in (1, 2)}
            self.dSa = {b: torch.empty(n, d, self.C[_LEVEL[b]], device=device) for b in BLOCKS}
            self.Pout = {b: torch.empty(n, d, self.C[_LEVEL[b]], device=device) for b in BLOCKS}

    @property
    def logits(self) -> torch.Tensor:
        """fp32 [n,K,d,h,w] scratch, allocated on first use (the fused training step never needs it)."""
        if self._logits is None:
            self._logits = torch.empty(self._logits_shape, device=self._device)
        return self._logits

    def shape(self, level: int) -> Shape:
        hh, ww = self.HW[level]
        return Shape(self.n, self.d, hh, ww)


class GateTables:
    """Per-step parameter-only tensors of the gates plus their gradient accumulators.

    EnergyFiLM's (g1, bt) [C,F] come from an MLP over a constant sinusoidal code of the bin index (reference
    models.py:1494-1512) and FourierGate's mask acts as a circular convolution with kernel kfg [F] = irfft(freq_mask *
    mag_scale) (models.py:1537-1542): both depend on parameters only. One kernel per block builds them
    (spff_gate_tables_fwd), the gate kernels accumulate the table gradients (dg1, dbt, dkfg) over the sample groups, and
    `finish()` folds those into the parameter gradients with one kernel per block (spff_gate_tables_bwd)."""

    def __init__(self, cfg: NetConfig, params: Dict[str, torch.Tensor], frames: int, need_grad: bool):
        self.cfg, self.params, self.frames = cfg, params, frames
        self.g1: Dict[str, Optional[torch.Tensor]] = {}
        self.bt: Dict[str, Optional[torch.Tensor]] = {}
        self.kfg: Dict[str, Optional[torch.Tensor]] = {}
        self.se: Dict[str, Optional[tuple]] = {}
        self.dg1: Dict[str, Optional[torch.Tensor]] = {}
        self.dbt: Dict[str, Optional[torch.Tensor]] = {}
        self.dkfg: Dict[str, Optional[torch.Tensor]] = {}
        self._done: set = set()
        dev = next(iter(params.values())).device
        # one allocation for the tables, one zero-filled allocation for their gradient accumulators
        sizes = {b: cfg.channels(b)[1] * frames for b in BLOCKS}
        per = {b: (2 * sizes[b] if cfg.efilm else 0) + (frames if cfg.fgate else 0) for b in BLOCKS}
        total = sum((v + 3) // 4 * 4 for v in per.values())
        tab = torch.empty(max(total, 4), device=dev)
        acc = torch.zeros(max(total, 4), device=dev) if need_grad else None
        off = 0
        for b in BLOCKS:
            c = cfg.channels(b)[1]
            self.g1[b] = self.bt[b] = self.kfg[b] = self.se[b] = None
            self.dg1[b] = self.dbt[b] = self.dkfg[b] = None
            o = off

            def take(n, shape):
                nonlocal o
                t = tab[o:o + n].view(shape)
                a = acc[o:o + n].view(shape) if acc is not None else None
                o += n
                return t, a
            if cfg.efilm:
                self.g1[b], self.dg1[b] = take(sizes[b], (c, frames))
                self.bt[b], self.dbt[b] = take(sizes[b], (c, frames))
            if cfg.fgate:
                self.kfg[b], self.dkfg[b] = take(frames, (frames,))
            off += (per[b] + 3) // 4 * 4
            if cfg.efilm or cfg.fgate:
                ops.gate_tables_fwd(*self._table_params(b), c, frames, self.g1[b], self.bt[b], self.kfg[b])
            if cfg.chanse and b in _STAGE:
                i = _STAGE[b]
                w1 = params[f"se.{i}.fc.0.weight"]
                w2 = params[f"se.{i}.fc.2.weight"]
                self.se[b] = (w1.reshape(w1.shape[0], w1.shape[1]), params[f"se.{i}.fc.0.bias"],
                              w2.reshape(w2.shape[0], w2.shape[1]), params[f"se.{i}.fc.2.bias"])

    def _table_params(self, b: str):
        p, cfg = self.params, self.cfg
        e = [p[f"{b}.efilm.mlp.0.weight"], p[f"{b}.efilm.mlp.0.bias"], p[f"{b}.efilm.mlp.2.weight"],
             p[f"{b}.efilm.mlp.2.bias"]] if cfg.efilm else [None] * 4
        f = [p[f"{b}.fgate.freq_mask"], p[f"{b}.fgate.mag_scale"]] if cfg.fgate else [None] * 2
        return e + f

    @staticmethod
    def _d(t):
        return t

    def finish(self, G: Dict[str, torch.Tensor], blocks: Optional[Tuple[str, ...]] = None):
        """G[name] += gradient of the EFiLM MLP / FourierGate parameters of `blocks` (default: every block
        not finished yet) from the accumulated table gradients (dg1, dbt, dkfg)."""
        cfg = self.cfg
        if not (cfg.efilm or cfg.fgate):
            return
        for b in (blocks or BLOCKS):
            if b in self._done:
                continue
            self._done.add(b)
            ge = [G[f"{b}.efilm.mlp.0.weight"], G[f"{b}.efilm.mlp.0.bias"], G[f"{b}.efilm.mlp.2.weight"],
                  G[f"{b}.efilm.mlp.2.bias"]] if cfg.efilm else [None] * 4
            gf = [G[f"{b}.fgate.freq_mask"], G[f"{b}.fgate.mag_scale"]] if cfg.fgate else [None] * 2
            ops.gate_tables_bwd(*self._table_params(b), cfg.channels(b)[1], self.frames, self.dg1[b], self.dbt[b], self.dkfg[b],
                                *ge, *gf)


class SpffEngine:
    """Forward / backward schedule of one SPCT-family network over the C ABI.

    `params` maps the core module's parameter names (no `model.` prefix: `enc1.pre.0.weight`, …,
    the key surface of SURVEY.md §8b) to CUDA fp32 tensors. The engine never owns parameters; the
    packed bf16 GEMM operands it derives from them are refreshed by `refresh_weights()`.
    """

    def __init__(self, cfg: NetConfig, params: Callable[[], Dict[str, torch.Tensor]],
                 versions: Optional[Callable[[], tuple]] = None):
        self.cfg = cfg
        self._params = params
        self._versions = versions    # changes whenever a parameter was written through torch
        self._packed: Dict[str, Tuple[torch.Tensor, Optional[torch.Tensor]]] = {}
        self._packed_key = None
        self._bufs: Dict[tuple, _GroupBuffers] = {}
        self._fit: Dict[tuple, int] = {}
        self._ones: Dict[str, torch.Tensor] = {}

    # ------------------------------------------------------------------------------------------
    def params(self) -> Dict[str, torch.Tensor]:
        return self._params()

    def refresh_weights(self, force: bool = False):
        """Re-pack conv / transposed-conv weights into the bf16 operand layouts when any changed."""
        p = self.params()
        names = [f"{b}.{cn}.0.weight" for b in BLOCKS for cn in self.cfg.conv_names] + ["up3.weight", "up2.weight", "up1.weight"]
        key = (tuple(p[n].data_ptr() for n in names), self._versions() if self._versions else None)
        if self._versions is None:
            force = True
        if not force and key == self._packed_key:
            return
        for b in BLOCKS:
            for j, cn in enumerate(self.cfg.conv_names):
                if b == "enc1" and j == 0:
                    continue   # the Cin = 1 stem reads the fp32 weight directly
                self._packed[f"{b}.{j + 1}"] = ops.pack_conv3_weight(p[f"{b}.{cn}.0.weight"])
        for up in ("up3", "up2", "up1"):
            self._packed[up] = ops.pack_convt_weight(p[f"{up}.weight"])
        self._packed_key = key

    def invalidate_weights(self):
        self._packed_key = None

    def _one(self, device) -> torch.Tensor:
        t = self._ones.get(str(device))
        if t is None:
            t = self._ones[str(device)] = torch.ones(1, dtype=torch.int64, device=device)
        return t

    def buffers(self, n, d, h, w, device, train: bool, fresh: bool = False) -> _GroupBuffers:
        if fresh:
            return _GroupBuffers(self.cfg, n, d, h, w, device, train)
        key = (n, d, h, w, str(device), train)
        b = self._bufs.get(key)
        if b is None:
            b = self._bufs[key] = _GroupBuffers(self.cfg, n, d, h, w, device, train)
        return b

    def release_buffers(self):
        self._bufs.clear()

    # ------------------------------------------------------------------------------------------
    # forward of one sample group
    # ------------------------------------------------------------------------------------------
    def _block_fwd(self, B: _GroupBuffers, T: GateTables, b: str, xin: Optional[torch.Tensor], pool_to):
        cfg, p = self.cfg, self.params()
        l = _LEVEL[b]
        cin, c = cfg.channels(b)
        cn1, cn2 = cfg.conv_names
        shp = B.shape(l)
        count = B.d * shp.h * shp.w
        # conv1 -> IN statistics -> a1 = lrelu(IN(x1))
        # (the tensor-core convs produce the InstanceNorm statistics in their epilogue; the stem needs a pass)
        if b == "enc1":   # the Cin = 1 stem takes its statistics in its own epilogue, like the tensor-core convs
            ops.conv3d_stem_fwd_stats(B.x_in, p[f"{b}.{cn1}.0.weight"], B.x1[b], c, B.partial[f"{b}.1"])
            ops.in_coeffs_from_partials(B.partial[f"{b}.1"], B.stem_slots, p[f"{b}.{cn1}.1.weight"], p[f"{b}.{cn1}.1.bias"],
                                        EPS, B.n, c, count, B.coef[f"{b}.1"])
        else:
            ops.conv3d_k3_fwd_stats(xin, cin, self._packed[f"{b}.1"][0], B.x1[b], c, B.partial[f"{b}.1"])
            ops.in_coeffs_from_partials(B.partial[f"{b}.1"], B.slots[b], p[f"{b}.{cn1}.1.weight"], p[f"{b}.{cn1}.1.bias"],
                                        EPS, B.n, c, count, B.coef[f"{b}.1"])
        ops.norm_act_apply(B.x1[b], B.coef[f"{b}.1"], B.a1[b], c, SLOPE)
        # conv2 -> IN statistics -> (S -> P,Q) -> out = lrelu(IN(x2))*P + Q (+ pooled copy)
        ops.conv3d_k3_fwd_stats(B.a1[b], c, self._packed[f"{b}.2"][0], B.x2[b], c, B.partial[f"{b}.2"])
        ops.in_coeffs_from_partials(B.partial[f"{b}.2"], B.slots[b], p[f"{b}.{cn2}.1.weight"], p[f"{b}.{cn2}.1.bias"],
                                    EPS, B.n, c, count, B.coef[f"{b}.2"])
        flags = cfg.block_flags(b)
        P = Q = None
        if flags:
            S = B.f32.get(B.idx[f"{b}.S"])
            ops.norm_act_reduce(B.x2[b], B.coef[f"{b}.2"], S, c, SLOPE, fixed_order=True)
            P, Q = B.P[b], B.Q[b]
            ops.gate_micro_fwd(S, T._d(T.g1[b]), T._d(T.bt[b]), T._d(T.kfg[b]), T.se[b], flags, c, shp, P, Q)
        ops.norm_act_affine_apply(B.x2[b], B.coef[f"{b}.2"], P, Q, B.out[b], pool_to, c, SLOPE,
                                  pool_argmax=B.pool_argmax[l] if pool_to is not None else None)

    def forward_group(self, B: _GroupBuffers, T: GateTables, x: torch.Tensor, head: str = "logits",
                      logits_out: Optional[torch.Tensor] = None, labels_out: Optional[torch.Tensor] = None):
        """x: fp32 [n,1,d,h,w] contiguous. head = "logits" (fp32 [n,K,d,h,w] into logits_out, default
        B.logits), "argmax" (uint8 label map [n,d,h,w] into labels_out) or "none"."""
        p = self.params()
        B.x_in = x
        B.f32.zero()
        self._block_fwd(B, T, "enc1", None, B.pool[1])
        self._block_fwd(B, T, "enc2", B.pool[1], B.pool[2])
        self._block_fwd(B, T, "enc3", B.pool[2], B.pool[3])
        self._block_fwd(B, T, "bott", B.pool[3], None)
        prev = B.out["bott"]
        for l, up, dec in ((3, "up3", "dec3"), (2, "up2", "dec2"), (1, "up1", "dec1")):
            cu = B.C[l]
            ops.convt_k122_fwd(prev, 2 * cu, self._packed[up][0], p[f"{up}.bias"], B.cat[l][..., :cu], cu)
            self._block_fwd(B, T, dec, B.cat[l], None)
            prev = B.out[dec]
        if head == "logits":
            ops.head_fwd(prev, p["out.weight"], p["out.bias"], B.logits if logits_out is None else logits_out)
        elif head == "argmax":
            ops.head_argmax(prev, p["out.weight"], p["out.bias"], labels_out)

    # ------------------------------------------------------------------------------------------
    # backward of one sample group
    # ------------------------------------------------------------------------------------------
    def _block_bwd(self, B: _GroupBuffers, T: GateTables, G: Dict[str, torch.Tensor], b: str, dout: torch.Tensor,
                   xin: Optional[torch.Tensor], dxin: Optional[torch.Tensor]):
        cfg, p = self.cfg, self.params()
        l = _LEVEL[b]
        cin, c = cfg.channels(b)
        cn1, cn2 = cfg.conv_names
        shp = B.shape(l)
        flags = cfg.block_flags(b)
        t1, t2 = B.t1[l], B.t2[l]
        # tail + IN2 + lrelu backward
        R2 = B.b32.get(B.idx[f"{b}.R2"])
        S = B.f32.get(B.idx[f"{b}.S"]) if flags else None
        ops.norm_act_bwd_reduce(dout, B.x2[b], B.coef[f"{b}.2"], R2, c, SLOPE, plain=(flags == 0), fixed_order=True, S=S)
        dse = None
        if flags & GATE_CHANSE:
            i = _STAGE[b]
            dse = (G[f"se.{i}.fc.0.weight"].view(-1, c), G[f"se.{i}.fc.0.bias"], G[f"se.{i}.fc.2.weight"].view(c, -1),
                   G[f"se.{i}.fc.2.bias"])
        ops.gate_micro_bwd(R2, S, B.coef[f"{b}.2"], p[f"{b}.{cn2}.1.weight"], T._d(T.g1[b]), T._d(T.bt[b]), T._d(T.kfg[b]),
                           T.se[b], flags, c, shp, B.bcoef[f"{b}.2"], B.dSa[b] if flags else None,
                           B.Pout[b] if flags else None, G[f"{b}.{cn2}.1.weight"], G[f"{b}.{cn2}.1.bias"],
                           T.dg1[b], T.dbt[b], T.dkfg[b], dse)
        ops.norm_act_bwd_apply(dout, B.x2[b], B.coef[f"{b}.2"], B.bcoef[f"{b}.2"], B.Pout[b] if flags else None,
                               B.dSa[b] if flags else None, t1, c, SLOPE)
        # conv2 backward
        ops.conv3d_k3_wgrad(B.a1[b], c, t1, c, G[f"{b}.{cn2}.0.weight"], 1.0)
        ops.conv3d_k3_dgrad(t1, c, self._packed[f"{b}.2"][1], t2, c)
        # IN1 + lrelu backward
        R1 = B.b32.get(B.idx[f"{b}.R1"])
        ops.norm_act_bwd_reduce(t2, B.x1[b], B.coef[f"{b}.1"], R1, c, SLOPE, plain=True, fixed_order=True)
        ops.gate_micro_bwd(R1, None, B.coef[f"{b}.1"], p[f"{b}.{cn1}.1.weight"], None, None, None, None, 0, c, shp,
                           B.bcoef[f"{b}.1"], None, None, G[f"{b}.{cn1}.1.weight"], G[f"{b}.{cn1}.1.bias"], None, None,
                           None, None)
        ops.norm_act_bwd_apply(t2, B.x1[b], B.coef[f"{b}.1"], B.bcoef[f"{b}.1"], None, None, t1, c, SLOPE)
        # conv1 backward
        if b == "enc1":
            ops.conv3d_stem_wgrad(B.x_in, t1, c, G[f"{b}.{cn1}.0.weight"], 1.0)
        else:
            ops.conv3d_k3_wgrad(xin, cin, t1, c, G[f"{b}.{cn1}.0.weight"], 1.0)
            if b.startswith("dec"):
                ops.conv3d_k3_dgrad_stats(t1, c, self._packed[f"{b}.1"][1], dxin, cin, B.dpartial[l])
            else:
                ops.conv3d_k3_dgrad(t1, c, self._packed[f"{b}.1"][1], dxin, cin)

    def backward_group(self, B: _GroupBuffers, T: GateTables, G: Dict[str, torch.Tensor],
                       dlogits: Optional[torch.Tensor], stage_done: Optional[Callable[[str], None]] = None):
        """Accumulates (+=) every parameter gradient of this group into the fp32 tensors of `G`
        (shaped like the parameters). dlogits: fp32 [n,K,d,h,w], or None when the fused head/loss
        kernel already left the head's input gradient in B.gout[1] (and its dW/db in G).
        `stage_done(stage)` is called as soon as every gradient of a stage has been enqueued: "decoder" (head, decoder
        blocks, transposed convs), then "bott", "enc3", "enc2", "enc1" (each with its SE / gate parameters)."""
        p = self.params()
        B.b32.zero()
        if dlogits is not None:
            ops.head_bwd(dlogits, B.out["dec1"], p["out.weight"], B.gout[1], G["out.weight"].view(-1, self.cfg.base),
                         G["out.bias"], 1.0)
        for l, up, dec, below in ((1, "up1", "dec1", "dec2"), (2, "up2", "dec2", "dec3"), (3, "up3", "dec3", "bott")):
            cu = B.C[l]
            self._block_bwd(B, T, G, dec, B.gout[l], B.cat[l], B.dcat[l])
            dy = B.dcat[l][..., :cu]
            xb = B.out[below]
            ops.convt_k122_wgrad(xb, 2 * cu, dy, cu, G[f"{up}.weight"], 1.0)
            ops.convt_k122_dgrad(dy, cu, self._packed[up][1], B.gout[l + 1], 2 * cu)
        if stage_done is not None:   # head / decoder / transposed-conv gradients of this group are complete
            self._up_bias_grads(B, G)
            stage_done("decoder")
        self._block_bwd(B, T, G, "bott", B.gout[4], B.pool[3], B.dpool[3])
        if stage_done is not None:
            stage_done("bott")
        for l, enc in ((3, "enc3"), (2, "enc2"), (1, "enc1")):
            c = B.C[l]
            dskip = B.dcat[l][..., c:]
            ops.maxpool_bwd_add_argmax(B.dpool[l], B.pool_argmax[l], dskip, c, True)
            if l > 1:
                self._block_bwd(B, T, G, enc, dskip, B.pool[l - 1], B.dpool[l - 1])
            else:
                self._block_bwd(B, T, G, enc, dskip, None, None)
            if stage_done is not None:
                stage_done(enc)
        if stage_done is None:
            self._up_bias_grads(B, G)

    @staticmethod
    def _up_bias_grads(B: _GroupBuffers, G: Dict[str, torch.Tensor]):
        """ConvTranspose3d bias gradient = column sums of dy = the `up` half of the decoder input gradient, summed by the
        dgrad epilogue per work item (fp32) and folded here in double (spff_partial_colsum)."""
        for l, up in ((3, "up3"), (2, "up2"), (1, "up1")):
            dp = B.dpartial[l]                      # [n, slots, 2, 2*C_l]: row (n, slot) holds {sums, sums of squares}
            ops.partial_colsum(dp, dp.shape[0] * dp.shape[1], 2 * dp.shape[3], B.C[l], G[f"{up}.bias"])

    # ------------------------------------------------------------------------------------------
    # batch-level drivers
    # ------------------------------------------------------------------------------------------
    @staticmethod
    def _check_input(x: torch.Tensor) -> torch.Tensor:
        if x.dim() != 5 or x.shape[1] != 1:
            raise ValueError(f"expected images [B,1,F,H,W] (energy bins on the depth axis), got {tuple(x.shape)}")
        if not x.is_cuda:
            raise RuntimeError("spff_b200 runs on a B200 (sm_100) device only; the input is on the CPU and there is "
                               "no CPU fallback")
        return x.float().contiguous()

    @staticmethod
    def fit_group(group: int, d: int, h: int, w: int, device, train: bool, extra: float = 0.0) -> int:
        """Largest sample group <= `group` whose buffers fit in ~45 % of the free HBM. One sample holds, in units of
        one level-1 32-channel bf16 tensor (d*h*w*64 bytes): x1/a1/x2/out per block, the concat and pooled buffers
        (16.7 units forward) plus the gradient scratch (26.5 units for a training step). `extra`: further units per
        sample that a caller keeps beside the buffers (ENSEMBLE_UNITS for run_ensemble)."""
        per = ((26.5 if train else 16.7) + extra) * d * h * w * 64
        try:
            free, _ = torch.cuda.mem_get_info(device)
        except Exception:
            return max(1, group)
        return max(1, min(group, int(0.45 * free / per)))

    def _fitted(self, group: int, d: int, h: int, w: int, device, train: bool, extra: float = 0.0) -> int:
        """fit_group, decided once per (shape, mode, requested group, extra) — before that shape's buffers exist, when
        the free-memory reading still describes what is available to them."""
        key = (group, d, h, w, str(device), train) + ((extra,) if extra else ())
        if key not in self._fit:
            if not any(k[1:4] == (d, h, w) for k in self._bufs):
                self._bufs.clear()          # buffers of another slice size would otherwise count as unavailable
            self._fit[key] = self.fit_group(group, d, h, w, device, train, extra)
        return self._fit[key]

    @staticmethod
    def _groups(batch: int, group: int):
        group = max(1, min(group, batch))
        return [(i, min(batch, i + group)) for i in range(0, batch, group)]

    def infer(self, x: torch.Tensor, group: int = 32, argmax: bool = False) -> torch.Tensor:
        """Forward only. Returns fp32 logits [B,K,F,H,W], or the uint8 label map [B,F,H,W] (argmax=True,
        first maximum wins as torch.argmax)."""
        x = self._check_input(x)
        bsz, _, d, h, w = x.shape
        self.refresh_weights()
        T = GateTables(self.cfg, self.params(), d, need_grad=False)
        if argmax:
            out = torch.empty(bsz, d, h, w, dtype=torch.uint8, device=x.device)
        else:
            out = torch.empty(bsz, self.cfg.num_classes, d, h, w, device=x.device)
        group = self._fitted(min(group, bsz), d, h, w, x.device, train=False)
        for lo, hi in self._groups(bsz, group):
            B = self.buffers(hi - lo, d, h, w, x.device, train=False)
            if argmax:
                self.forward_group(B, T, x[lo:hi], head="argmax", labels_out=out[lo:hi])
            else:
                self.forward_group(B, T, x[lo:hi], head="logits", logits_out=out[lo:hi])
        return out

    def infer_streamed(self, x_host: torch.Tensor, out_host: torch.Tensor, device, copy_stream: torch.cuda.Stream,
                       group: int = 32) -> None:
        """Label maps of a scan that lives in (pinned) HOST memory, written to a (pinned) host uint8 tensor [B,F,H,W]:
        group g+1 is copied in and the labels of group g-1 are copied out on `copy_stream` while group g computes, so
        neither transfer is exposed. The last device->host copy is complete when `copy_stream` is synchronised."""
        if x_host.dim() != 5 or x_host.shape[1] != 1 or x_host.is_cuda or out_host.is_cuda:
            raise ValueError("infer_streamed takes host tensors: images [B,1,F,H,W] and a uint8 output [B,F,H,W]")
        bsz, _, d, h, w = x_host.shape
        if tuple(out_host.shape) != (bsz, d, h, w) or out_host.dtype != torch.uint8:
            raise ValueError(f"out_host must be uint8 {(bsz, d, h, w)}")
        self.refresh_weights()
        T = GateTables(self.cfg, self.params(), d, need_grad=False)
        group = self._fitted(min(group, bsz), d, h, w, device, train=False)
        groups = self._groups(bsz, group)
        main = torch.cuda.current_stream(device)
        src = x_host if x_host.dtype == torch.float32 else x_host.float()
        xin = [torch.empty(group, 1, d, h, w, device=device) for _ in range(2)]         # double-buffered input
        lab = [torch.empty(group, d, h, w, dtype=torch.uint8, device=device) for _ in range(2)]
        loaded, computed, stored = {}, {}, {}
        copy_stream.wait_stream(main)

        def load(i):
            lo, hi = groups[i]
            with torch.cuda.stream(copy_stream):
                if i >= 2:
                    copy_stream.wait_event(computed[i - 2])      # the buffer's previous group has been consumed
                xin[i % 2][:hi - lo].copy_(src[lo:hi], non_blocking=True)
                loaded[i] = copy_stream.record_event()

        load(0)
        for i, (lo, hi) in enumerate(groups):
            if i + 1 < len(groups):
                load(i + 1)
            main.wait_event(loaded[i])
            if i >= 2:
                main.wait_event(stored[i - 2])                    # its label buffer has been copied out
            B = self.buffers(hi - lo, d, h, w, device, train=False)
            self.forward_group(B, T, xin[i % 2][:hi - lo], head="argmax", labels_out=lab[i % 2][:hi - lo])
            computed[i] = main.record_event()
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(computed[i])
                out_host[lo:hi].copy_(lab[i % 2][:hi - lo], non_blocking=True)
                stored[i] = copy_stream.record_event()
        for t in xin + lab:
            t.record_stream(copy_stream)

    def forward_saved(self, x: torch.Tensor, group: int = 32):
        """Forward that keeps every group's activations for a later `backward_saved` (the autograd
        path behind `model(x)`; memory grows with the batch, unlike `train_step`)."""
        x = self._check_input(x)
        bsz, _, d, h, w = x.shape
        self.refresh_weights()
        T = GateTables(self.cfg, self.params(), d, need_grad=True)
        logits = torch.empty(bsz, self.cfg.num_classes, d, h, w, device=x.device)
        saved = []
        for lo, hi in self._groups(bsz, group):
            B = self.buffers(hi - lo, d, h, w, x.device, train=True, fresh=True)
            self.forward_group(B, T, x[lo:hi], head="logits", logits_out=logits[lo:hi])
            saved.append((lo, hi, B))
        return logits, (T, saved)

    def backward_saved(self, state, dlogits: torch.Tensor, G: Dict[str, torch.Tensor]):
        T, saved = state
        dlogits = dlogits.float().contiguous()
        for lo, hi, B in saved:
            self.backward_group(B, T, G, dlogits[lo:hi])
        T.finish(G)

    def train_step(self, x: torch.Tensor, labels: torch.Tensor, G: Dict[str, torch.Tensor], tally: "LossTally",
                   group: int = 32, ignore_index: int = 255, staged: Optional["StagedBatch"] = None,
                   stage_done: Optional[Callable[[str], None]] = None):
        """Fused forward + CE/confusion + backward over the batch in sample groups. Accumulates into G the parameter
        gradients of the SUM over valid voxels of the CE terms, and leaves the number of valid voxels in `tally.n_valid`:
        the caller divides the finished gradients by it (ops.scale_by_count) to obtain the gradients of the batch-mean CE
        (helpers.py:798-801; the Dice term of the loss has no gradient, helpers.py:782-795). Back-propagating the sum
        keeps a group's backward independent of the other groups' labels. Loss statistics go into `tally`.
        `staged`: the batch is still arriving from pinned host memory on a copy stream (StagedBatch);
        each group waits only for its own images and labels.
        `stage_done(stage)`: called inside the LAST group's backward as soon as every gradient of a stage is final —
        "decoder" (head, decoder blocks, transposed convs), "bott", "enc3", "enc2", "enc1" — so that a data-parallel
        caller can start that range's all-reduce while the rest of the backward still runs."""
        x = self._check_input(x)
        bsz, _, d, h, w = x.shape
        if labels.shape != (bsz, d, h, w):
            raise ValueError(f"labels must be [B,F,H,W] = {(bsz, d, h, w)}, got {tuple(labels.shape)}")
        labels = labels.contiguous()
        self.refresh_weights()
        group = self._fitted(min(group, bsz), d, h, w, x.device, train=True)
        T = GateTables(self.cfg, self.params(), d, need_grad=True)
        p = self.params()
        one = self._one(x.device)      # normaliser of the per-voxel CE gradient inside the step: 1 (sum reduction)
        for lo, hi in self._groups(bsz, group):
            if staged is not None:
                staged.wait_images(hi)
            B = self.buffers(hi - lo, d, h, w, x.device, train=True)
            self.forward_group(B, T, x[lo:hi], head="none")
            if staged is not None:
                staged.wait_labels(hi)
            last = hi == bsz
            if last:                   # every label is on the device: the CE normaliser of the whole batch
                ops.count_valid(labels, ignore_index, tally.n_valid)
            # head + CE + confusion + their backward in one pass; the logits never reach memory
            ops.head_loss_fused(B.out["dec1"], p["out.weight"], p["out.bias"], labels[lo:hi], ignore_index, one, None,
                                tally.nll, tally.count, tally.confusion, B.gout[1],
                                G["out.weight"].view(-1, self.cfg.base), G["out.bias"], 1.0)
            hook = None
            if last and stage_done is not None:
                def hook(stage):
                    T.finish(G, ("dec3", "dec2", "dec1") if stage == "decoder" else (stage,))
                    stage_done(stage)
            self.backward_group(B, T, G, None, stage_done=hook)
        T.finish(G)

    def eval_step(self, x: torch.Tensor, labels: torch.Tensor, tally: "LossTally", group: int = 32,
                  ignore_index: int = 255, per_sample: Optional[Tuple[torch.Tensor, torch.Tensor, torch.Tensor]] = None,
                  labels_out: Optional[torch.Tensor] = None, staged: Optional["StagedBatch"] = None,
                  hist: Optional[torch.Tensor] = None, sample_hist: Optional[torch.Tensor] = None):
        """Forward + head + CE/confusion over the batch in sample groups, with no gradient: the loss statistics of
        `ce_plus_macro_dice_loss` / `per_class_metrics_3d` on `infer(x)` accumulate (+=) into `tally`, and the fp32 logits
        never reach memory. per_sample = (nll fp64 [B], count int64 [B], confusion int64 [B,K,K]) receives the same
        tally per sample (+=); labels_out (uint8 [B,F,H,W]) the arg-max the tally counts. `staged`: as in train_step.
        hist (int64 [K,2,T]) / sample_hist (int64 [B,K,2,T], with per_sample) receive (+=) the softmax histograms of
        ops.head_eval."""
        x = self._check_input(x)
        bsz, _, d, h, w = x.shape
        if labels.shape != (bsz, d, h, w):
            raise ValueError(f"labels must be [B,F,H,W] = {(bsz, d, h, w)}, got {tuple(labels.shape)}")
        labels = labels.contiguous()
        self.refresh_weights()
        group = self._fitted(min(group, bsz), d, h, w, x.device, train=False)
        T = GateTables(self.cfg, self.params(), d, need_grad=False)
        p = self.params()
        for lo, hi in self._groups(bsz, group):
            if staged is not None:
                staged.wait_images(hi)
            B = self.buffers(hi - lo, d, h, w, x.device, train=False)
            self.forward_group(B, T, x[lo:hi], head="none")
            if staged is not None:
                staged.wait_labels(hi)
            rows = tuple(t[lo:hi] for t in per_sample) if per_sample is not None else (None, None, None)
            ops.head_eval(B.out["dec1"], p["out.weight"], p["out.bias"], labels[lo:hi], ignore_index, tally.nll,
                          tally.count, tally.confusion, *rows, labels_out[lo:hi] if labels_out is not None else None,
                          hist=hist, sample_hist=sample_hist[lo:hi] if sample_hist is not None else None)


# per sample, in fit_group's units, of run_ensemble beside the inference buffers: the fp32 probability accumulator
# (16 classes x 4 B = 64 B per position, one unit) and the fp32 flipped input (4 B per position)
ENSEMBLE_UNITS = 1.0 + 1.0 / 16
# and, when the mutual information is wanted, the fp32 expected-entropy plane (4 B per position)
ENTROPY_UNITS = 1.0 / 16


def ensemble_units(entropy: bool) -> float:
    """fit_group's `extra` for run_ensemble: ENSEMBLE_UNITS, plus ENTROPY_UNITS when the entropy plane is allocated."""
    return ENSEMBLE_UNITS + (ENTROPY_UNITS if entropy else 0.0)


def flip_tables(n: int, h: int, w: int, flip: int, device="cpu"):
    """(amap int32 [n,h], bmap int32 [n,w]) that make spff_grid_aug's gather x[., ., amap[u], bmap[v]] torch.flip over H
    (flip & 1) and / or W (flip & 2)."""
    a = torch.arange(h, dtype=torch.int32)
    b = torch.arange(w, dtype=torch.int32)
    if flip & 1:
        a = a.flip(0)
    if flip & 2:
        b = b.flip(0)
    return a.to(device).expand(n, h).contiguous(), b.to(device).expand(n, w).contiguous()


class _FlipGather:
    """spff_grid_aug as a pure gather (not transposed, scale 1, shift 0, no noise or stamp): torch.flip of an fp32
    [n,1,d,h,w] group over H / W, for up to `n` samples."""

    def __init__(self, n: int, h: int, w: int, device):
        self.maps = {f: flip_tables(n, h, w, f, device) for f in (1, 2, 3)}
        self.zi = torch.zeros(n, dtype=torch.int32, device=device)
        self.one = torch.ones(n, device=device)
        self.zf = torch.zeros(n, device=device)
        self.seed = torch.zeros(n, dtype=torch.int64, device=device)

    def __call__(self, x: torch.Tensor, out: torch.Tensor, flip: int):
        n, _, d, h, w = x.shape
        a, b = self.maps[flip]
        ops.grid_aug(x.view(n, d, h, w), None, out.view(n, d, h, w), None, a[:n], b[:n], self.zi[:n], self.one[:n],
                     self.zf[:n], self.zf[:n], self.seed[:n], self.zi[:n], 0, 0)


def run_ensemble(engines: List[SpffEngine], x: torch.Tensor, flips: Tuple[int, ...], group: int = 32,
                 labels: Optional[torch.Tensor] = None, tally: Optional["LossTally"] = None, ignore_index: int = 255,
                 per_sample: Optional[Tuple[torch.Tensor, torch.Tensor, torch.Tensor]] = None,
                 labels_out: Optional[torch.Tensor] = None, proba_out: Optional[torch.Tensor] = None,
                 hist: Optional[torch.Tensor] = None, sample_hist: Optional[torch.Tensor] = None,
                 staged: Optional["StagedBatch"] = None, entropy_out: Optional[torch.Tensor] = None,
                 mi_out: Optional[torch.Tensor] = None, unc: Optional[torch.Tensor] = None,
                 sample_unc: Optional[torch.Tensor] = None, calib: Optional[torch.Tensor] = None,
                 sample_calib: Optional[torch.Tensor] = None, brier: Optional[torch.Tensor] = None,
                 sample_brier: Optional[torch.Tensor] = None, inv_temperature: float = 1.0,
                 temp_fit: Optional[Tuple[torch.Tensor, torch.Tensor, torch.Tensor]] = None):
    """Averaged softmax of several networks of one NetConfig over input flips (1 = H, 2 = W, 0 = none), sample group by
    sample group, with no logits in memory. Every member runs on the FIRST engine's inference buffers; for each group
    and member (outer) and flip (inner): flip the input (spff_grid_aug), forward, and add the head's softmax, mirrored
    back, into an fp32 [group,d,h,w,16] accumulator (ops.head_prob_accum). One ops.prob_finalize per group then writes
    p̄ = mean over the passes: labels_out (uint8 [B,F,H,W], arg-max), proba_out (fp16 [B,K,F,H,W]) and, with labels,
    the tally, per-sample rows and histograms of SpffEngine.eval_step computed on p̄. `staged`: as in train_step.

    Uncertainty and calibration (ops.Uncertainty): entropy_out / mi_out fp16 [B,F,H,W] maps of H[p̄] and of the mutual
    information H[p̄] - mean over passes of H[p]; unc int64 [2] / sample_unc int64 [B,2] (+=) their sums in units of
    2^-24 nats; with labels calib int64 [3,T] / sample_calib [B,3,T] and brier fp64 [1] / sample_brier fp64 [B] (+=).
    The fp32 [group,d,h,w] expected-entropy plane rides the member x flip loop only when mi_out, unc or sample_unc is
    given (the mutual information needs it); it is counted in the group size only then.

    Temperature scaling: `inv_temperature` β = 1/T tempers p̄ in the finishing pass (ops.prob_finalize; β == 1.0 is the
    untempered call). `temp_fit` = (betas fp32 [G], sums fp64 [2,G], counted int64 [1]), with labels, replaces the
    finishing pass by ops.prob_temp_fit on each group's accumulator (+= the tempered nll and its derivative at each
    β_g, and the counted voxels); no other output may be given then, and nothing is added to the group size."""
    first = engines[0]
    x = first._check_input(x)
    bsz, _, d, h, w = x.shape
    if temp_fit is not None and (labels is None or tally is not None or per_sample is not None or labels_out is not None
                                 or proba_out is not None or hist is not None or entropy_out is not None
                                 or mi_out is not None or unc is not None or calib is not None):
        raise ValueError("temp_fit needs labels and takes no other output")
    if labels is not None:
        if labels.shape != (bsz, d, h, w):
            raise ValueError(f"labels must be [B,F,H,W] = {(bsz, d, h, w)}, got {tuple(labels.shape)}")
        labels = labels.contiguous()
    tables = []
    for e in engines:   # once per call, not per group
        e.refresh_weights()
        tables.append(GateTables(e.cfg, e.params(), d, need_grad=False))
    want_mi = mi_out is not None or unc is not None or sample_unc is not None
    want_unc = want_mi or entropy_out is not None or calib is not None
    group = first._fitted(min(group, bsz), d, h, w, x.device, train=False, extra=ensemble_units(want_mi))
    acc = torch.empty(group, d, h, w, 16, device=x.device)
    ent = torch.empty(group, d, h, w, device=x.device) if want_mi else None
    flipped = any(flips)
    xf = torch.empty(group, 1, d, h, w, device=x.device) if flipped else None
    gather = _FlipGather(group, h, w, x.device) if flipped else None
    scale = 1.0 / (len(engines) * len(flips))
    tl = (tally.nll, tally.count, tally.confusion) if tally is not None else None

    def rows(t, lo, hi):
        return t[lo:hi] if t is not None else None
    for lo, hi in first._groups(bsz, group):
        n = hi - lo
        if staged is not None:
            staged.wait_images(hi)
        B = first.buffers(n, d, h, w, x.device, train=False)
        a = acc[:n]
        beta = 0
        for e, T in zip(engines, tables):
            p = e.params()
            for f in flips:
                xin = x[lo:hi]
                if f:
                    gather(xin, xf[:n], f)
                    xin = xf[:n]
                e.forward_group(B, T, xin, head="none")
                ops.head_prob_accum(B.out["dec1"], p["out.weight"], p["out.bias"], a, flip=f, beta=beta,
                                    ent=ent[:n] if ent is not None else None)
                beta = 1
        if staged is not None:
            staged.wait_labels(hi)
        if temp_fit is not None:
            ops.prob_temp_fit(a, first.cfg.num_classes, scale, rows(labels, lo, hi), temp_fit[0], temp_fit[1],
                              ignore_index=ignore_index, counted=temp_fit[2])
            continue
        u = ops.Uncertainty(ent=ent[:n] if ent is not None else None, entropy_out=rows(entropy_out, lo, hi),
                            mi_out=rows(mi_out, lo, hi), unc=unc, sample_unc=rows(sample_unc, lo, hi), calib=calib,
                            sample_calib=rows(sample_calib, lo, hi), brier=brier,
                            sample_brier=rows(sample_brier, lo, hi)) if want_unc else None
        ops.prob_finalize(a, first.cfg.num_classes, scale, labels=rows(labels, lo, hi), ignore_index=ignore_index,
                          tally=tl, per_sample=tuple(t[lo:hi] for t in per_sample) if per_sample is not None else None,
                          labels_out=rows(labels_out, lo, hi), hist=hist, sample_hist=rows(sample_hist, lo, hi),
                          proba_out=rows(proba_out, lo, hi), unc=u, inv_temperature=inv_temperature)


class StagedBatch:
    """Host -> device staging of one batch on a dedicated copy stream, group by group: the images of a group, then its
    labels. The compute stream waits per group (images before the forward, labels before the fused head / loss), so the
    transfer of group g+1 overlaps the kernels of group g and nothing waits for the whole batch. Host tensors should be
    pinned (a pageable source still works, synchronously)."""

    def __init__(self, imgs: torch.Tensor, labels: torch.Tensor, device, group: int, stream: torch.cuda.Stream):
        bsz = imgs.shape[0]
        self.x = torch.empty(imgs.shape, dtype=torch.float32, device=device)
        self.labels = torch.empty(labels.shape, dtype=labels.dtype, device=device)
        self.h2d_bytes = imgs.numel() * 4 + labels.numel() * labels.element_size()
        self._events = []       # (upper sample index, images there, labels there)
        stream.wait_stream(torch.cuda.current_stream(device))
        src = imgs if imgs.dtype == torch.float32 else imgs.float()
        with torch.cuda.stream(stream):
            for lo in range(0, bsz, max(1, group)):
                hi = min(bsz, lo + group)
                self.x[lo:hi].copy_(src[lo:hi], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(stream)
                self.labels[lo:hi].copy_(labels[lo:hi], non_blocking=True)
                evl = torch.cuda.Event()
                evl.record(stream)
                self._events.append((hi, ev, evl))
        self.x.record_stream(stream)
        self.labels.record_stream(stream)

    def _wait(self, upto: int, which: int):
        for rec in self._events:
            if rec[0] >= upto:
                torch.cuda.current_stream().wait_event(rec[which])
                return

    def wait_images(self, upto: int):
        self._wait(upto, 1)

    def wait_labels(self, upto: int):
        self._wait(upto, 2)


class LossTally:
    """Device-side sufficient statistics of ce_plus_macro_dice_loss and per_class_metrics_3d
    (helpers.py:668-725, 782-803): sum of nll, number of valid voxels, [label][argmax] tally — one 8-byte-element
    buffer (one memset per step), plus the CE normaliser of the batch and the loss scalar."""

    def __init__(self, num_classes: int, device):
        self.k = num_classes
        self._buf = torch.zeros(2 + num_classes * num_classes, dtype=torch.int64, device=device)
        self.nll = self._buf[0:1].view(torch.float64)
        self.count = self._buf[1:2]
        self.confusion = self._buf[2:].view(num_classes, num_classes)
        self.n_valid = torch.zeros(1, dtype=torch.int64, device=device)
        self._loss = torch.zeros(1, device=device)

    def zero(self):
        self._buf.zero_()

    def loss(self, smooth: float = 1e-6) -> torch.Tensor:
        """CE + 0.5 * (1 - hard macro Dice over classes 1..K-1) as a device scalar (no host sync, one kernel)."""
        out = torch.empty(1, device=self._buf.device)
        ops.loss_from_tally(self.nll, self.count, self.confusion, self.k, smooth, out)
        return out[0]
