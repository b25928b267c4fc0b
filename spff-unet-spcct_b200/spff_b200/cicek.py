"""Execution engine of the "3DUNet" control (Cicek 3D U-Net behind a depth adapter) on the B200 kernels.

Host-side schedule behind `innovative3D.models.Cicek3DUNet.forward` and
`LitCicek3DUNet_DepthAdapter_Published` of this tree. Reference graph:

    LitCicek3DUNet_DepthAdapter_Published.forward     reference innovative3D/models.py:773-777
      _resize_depth_like (trilinear, D 5 -> 16)        models.py:153-157
      Cicek3DUNet.forward                              models.py:741-751
        block = (Conv3d 3x3x3 no bias, BatchNorm3d, ReLU) x 2     models.py:722-726
        MaxPool3d(2) x 4, ConvTranspose3d(2, stride 2) x 4, cat([up, skip])
        out = Conv3d(32, K, 1)
      _resize_logits_depth_like (D 16 -> 5)            models.py:159-163
    _weighted_softmax_ce (plain CE over valid voxels)  models.py:779-798
    torch.optim.SGD(lr 1e-2, momentum 0.99)            models.py:844-846

The 3x3x3 convolutions (tcgen05 implicit GEMM), the normalise + ReLU passes (slope 0), the head and the
fused head + CE kernel are the SPFF-UNet kernels; only the (2,2,2) pool / transposed conv, the BatchNorm
coefficient kernels, the depth resample and SGD are specific to this variant (csrc/cicek.cu, csrc/convt.cu).

Differences from the SPCT engine (engine.py) that the math forces:
  * BatchNorm couples the samples of a batch, so the batch cannot run in independent sample groups: every layer
    runs over the whole (per-rank) batch and all activations of the step are resident. Per-rank statistics under
    data parallelism (no SyncBN), as the reference's commented-out DDP configuration would do (SURVEY.md §8e).
  * The two depth resizes are linear maps over the planes. The head (1x1x1 conv + bias) commutes with the
    output resize (its rows sum to 1), so the engine resamples the 32-channel decoder output 16 -> 5 planes and
    runs the head / fused loss kernel at the original depth: the 13-channel logits at 16 planes never exist.
Everything is enqueue-only; there is no PyTorch fallback for any of the compute.
"""
from __future__ import annotations

from typing import Callable, Dict, List, Optional, Tuple

import torch

from . import ops
from ._lib import Shape
from .engine import LossTally

ENC = ("enc1", "enc2", "enc3", "enc4", "bott")
DEC = ("dec4", "dec3", "dec2", "dec1")
BLOCKS = ENC + DEC
_LEVEL = {"enc1": 1, "enc2": 2, "enc3": 3, "enc4": 4, "bott": 5, "dec4": 4, "dec3": 3, "dec2": 2, "dec1": 1}
_UPS = ((4, "up4", "dec4", "bott"), (3, "up3", "dec3", "dec4"), (2, "up2", "dec2", "dec3"), (1, "up1", "dec1", "dec2"))
BN_EPS, BN_MOMENTUM = 1e-5, 0.1    # nn.BatchNorm3d defaults (models.py:721)
SLOPE = 0.0                        # nn.ReLU


def depth_matrix(din: int, dout: int) -> torch.Tensor:
    """[dout, din] fp32 matrix of F.interpolate(mode='trilinear', align_corners=False) along D when H and W are
    unchanged (models.py:153-163): source index (o + 0.5) * din / dout - 0.5 clamped at 0, two taps."""
    m = torch.zeros(dout, din, dtype=torch.float32)
    scale = din / dout
    for o in range(dout):
        src = max(0.0, (o + 0.5) * scale - 0.5)
        i0 = min(int(src), din - 1)
        i1 = i0 + (1 if i0 < din - 1 else 0)
        lam = src - i0
        m[o, i0] += 1.0 - lam
        m[o, i1] += lam
    return m


class _Buffers:
    """Every activation, statistic and scratch gradient of one batch of fixed shape."""

    def __init__(self, base: int, k: int, n: int, d0: int, d: int, h: int, w: int, device, train: bool):
        if d % 16 or h % 16 or w % 16:
            raise ValueError(f"3DUNet pools 4 times in (D,H,W): the adapted depth, H and W must be multiples of 16 "
                             f"(got {d} x {h} x {w})")
        self.n, self.d0, self.d, self.h, self.w, self.train = n, d0, d, h, w, train
        bf = lambda dd, hh, ww, c: torch.empty(n, dd, hh, ww, c, dtype=torch.bfloat16, device=device)
        self.C = {l: base * 2 ** (l - 1) for l in range(1, 6)}
        self.DHW = {l: (d >> (l - 1), h >> (l - 1), w >> (l - 1)) for l in range(1, 6)}
        self.x_in = torch.empty(n, 1, d, h, w, device=device) if d0 != d else None
        self.cat = {l: bf(*self.DHW[l], 2 * self.C[l]) for l in range(1, 5)}
        self.pool = {l: bf(*self.DHW[l + 1], self.C[l]) for l in range(1, 5)}
        self.x1, self.a1, self.x2, self.out = {}, {}, {}, {}
        self.partial: Dict[str, torch.Tensor] = {}
        self.slots: Dict[str, int] = {}
        self.coef: Dict[str, torch.Tensor] = {}
        for b in BLOCKS:
            l = _LEVEL[b]
            c = self.C[l]
            dhw = self.DHW[l]
            self.x1[b], self.a1[b], self.x2[b] = bf(*dhw, c), bf(*dhw, c), bf(*dhw, c)
            self.out[b] = self.cat[l][..., c:] if b.startswith("enc") else bf(*dhw, c)
            self.slots[b] = ops.conv3d_k3_stat_slots(Shape(n, *dhw))
            for j in (1, 2):
                if not (b == "enc1" and j == 1):
                    self.partial[f"{b}.{j}"] = torch.empty(n, self.slots[b], 2, c, device=device)
                self.coef[f"{b}.{j}"] = torch.empty(n, c, 4, device=device)
        self.stem_slots = ops.conv3d_stem_stat_slots(Shape(n, d, h, w))
        self.partial["enc1.1"] = torch.empty(n, self.stem_slots, 2, self.C[1], device=device)
        # decoder output resampled to the caller's depth: the head's input
        self.hx = bf(d0, h, w, base) if d0 != d else None
        self._logits_shape = (n, k, d0, h, w)
        self._device = device
        if train:
            self.dcat = {l: bf(*self.DHW[l], 2 * self.C[l]) for l in range(1, 5)}
            self.gout = {l: bf(*self.DHW[l], self.C[l]) for l in range(1, 6)}
            self.t1 = {l: bf(*self.DHW[l], self.C[l]) for l in range(1, 6)}
            self.t2 = {l: bf(*self.DHW[l], self.C[l]) for l in range(1, 6)}
            self.dpool = {l: bf(*self.DHW[l + 1], self.C[l]) for l in range(1, 5)}
            self.gh = bf(d0, h, w, base) if d0 != d else None
            self.R = {f"{b}.{j}": torch.zeros(n, self.DHW[_LEVEL[b]][0], self.C[_LEVEL[b]], 6, device=device)
                      for b in BLOCKS for j in (1, 2)}
            self.bcoef = {f"{b}.{j}": torch.empty(n, self.C[_LEVEL[b]], 4, device=device) for b in BLOCKS for j in (1, 2)}
            self.dpartial = {l: torch.empty(n, self.slots[dec], 2, 2 * self.C[l], device=device) for l, _, dec, _ in _UPS}

    def shape(self, level: int) -> Shape:
        return Shape(self.n, *self.DHW[level])


class CicekEngine:
    """Forward / backward schedule of Cicek3DUNet over the C ABI.

    `params()` maps the backbone's parameter names (`enc1.0.weight`, `enc1.1.weight`, `up4.bias`, `out.weight`, ...)
    to CUDA fp32 tensors, `buffers()` its BatchNorm buffers (`enc1.1.running_mean`, ...), both owned by the module.
    """

    def __init__(self, num_classes: int, base: int, params: Callable[[], Dict[str, torch.Tensor]],
                 buffers: Callable[[], Dict[str, torch.Tensor]], versions: Optional[Callable[[], tuple]] = None):
        self.k, self.base = int(num_classes), int(base)
        self._params, self._buffers, self._versions = params, buffers, versions
        self._packed: Dict[str, tuple] = {}
        self._packed_key = None
        self._bufs: Dict[tuple, _Buffers] = {}
        self._mats: Dict[tuple, torch.Tensor] = {}

    # ------------------------------------------------------------------------------------------
    def channels(self, block: str) -> Tuple[int, int]:
        f = self.base
        return {"enc1": (1, f), "enc2": (f, 2 * f), "enc3": (2 * f, 4 * f), "enc4": (4 * f, 8 * f),
                "bott": (8 * f, 16 * f), "dec4": (16 * f, 8 * f), "dec3": (8 * f, 4 * f), "dec2": (4 * f, 2 * f),
                "dec1": (2 * f, f)}[block]

    def refresh_weights(self, force: bool = False):
        p = self._params()
        names = [f"{b}.{i}.weight" for b in BLOCKS for i in (0, 3)] + [f"{up}.weight" for _, up, _, _ in _UPS]
        key = (tuple(p[n].data_ptr() for n in names), self._versions() if self._versions else None)
        if self._versions is None:
            force = True
        if not force and key == self._packed_key:
            return
        for b in BLOCKS:
            for j, i in ((1, 0), (2, 3)):
                if not (b == "enc1" and j == 1):   # the Cin = 1 stem reads the fp32 weight directly
                    self._packed[f"{b}.{j}"] = ops.pack_conv3_weight(p[f"{b}.{i}.weight"])
        for _, up, _, _ in _UPS:
            self._packed[up] = ops.pack_convt_weight_k222(p[f"{up}.weight"])
        self._packed_key = key

    def invalidate_weights(self):
        self._packed_key = None

    def matrix(self, din: int, dout: int, device, transpose: bool = False) -> torch.Tensor:
        key = (din, dout, str(device), transpose)
        m = self._mats.get(key)
        if m is None:
            m = depth_matrix(din, dout)
            m = self._mats[key] = (m.t().contiguous() if transpose else m).to(device)
        return m

    def buffers(self, n, d0, d, h, w, device, train: bool, fresh: bool = False) -> _Buffers:
        if fresh:
            return _Buffers(self.base, self.k, n, d0, d, h, w, device, train)
        key = (n, d0, d, h, w, str(device), train)
        b = self._bufs.get(key)
        if b is None:
            self._bufs.clear()     # one resident shape at a time: a batch of activations is tens of GB
            b = self._bufs[key] = _Buffers(self.base, self.k, n, d0, d, h, w, device, train)
        return b

    def release_buffers(self):
        self._bufs.clear()

    # ------------------------------------------------------------------------------------------
    def _bn(self, B: _Buffers, b: str, j: int, training: bool):
        p, bufs = self._params(), self._buffers()
        l = _LEVEL[b]
        c = B.C[l]
        dd, hh, ww = B.DHW[l]
        i = 1 if j == 1 else 4
        rm, rv = bufs[f"{b}.{i}.running_mean"], bufs[f"{b}.{i}.running_var"]
        if training:
            ops.bn_coeffs(p[f"{b}.{i}.weight"], p[f"{b}.{i}.bias"], BN_EPS, B.n, c, dd * hh * ww, B.coef[f"{b}.{j}"],
                          partial=B.partial[f"{b}.{j}"], slots=B.stem_slots if (b == "enc1" and j == 1) else B.slots[b],
                          momentum=BN_MOMENTUM, running_mean=rm, running_var=rv)
            bufs[f"{b}.{i}.num_batches_tracked"].add_(1)
        else:
            ops.bn_coeffs(p[f"{b}.{i}.weight"], p[f"{b}.{i}.bias"], BN_EPS, B.n, c, dd * hh * ww, B.coef[f"{b}.{j}"],
                          running_mean=rm, running_var=rv, eval_mode=True)

    def _block_fwd(self, B: _Buffers, b: str, xin: Optional[torch.Tensor], x_img: Optional[torch.Tensor], training: bool):
        p = self._params()
        l = _LEVEL[b]
        cin, c = self.channels(b)
        if b == "enc1":
            if training:
                ops.conv3d_stem_fwd_stats(x_img, p[f"{b}.0.weight"], B.x1[b], c, B.partial[f"{b}.1"])
            else:
                ops.conv3d_stem_fwd(x_img, p[f"{b}.0.weight"], B.x1[b], c)
            self._bn(B, b, 1, training)
        else:
            if training:
                ops.conv3d_k3_fwd_stats(xin, cin, self._packed[f"{b}.1"][0], B.x1[b], c, B.partial[f"{b}.1"])
            else:
                ops.conv3d_k3_fwd(xin, cin, self._packed[f"{b}.1"][0], B.x1[b], c)
            self._bn(B, b, 1, training)
        ops.norm_act_apply(B.x1[b], B.coef[f"{b}.1"], B.a1[b], c, SLOPE)
        if training:
            ops.conv3d_k3_fwd_stats(B.a1[b], c, self._packed[f"{b}.2"][0], B.x2[b], c, B.partial[f"{b}.2"])
        else:
            ops.conv3d_k3_fwd(B.a1[b], c, self._packed[f"{b}.2"][0], B.x2[b], c)
        self._bn(B, b, 2, training)
        ops.norm_act_affine_apply(B.x2[b], B.coef[f"{b}.2"], None, None, B.out[b], None, c, SLOPE)
        if b.startswith("enc"):
            ops.maxpool222_fwd(B.out[b], B.pool[l], c)

    def forward(self, B: _Buffers, x: torch.Tensor, training: bool) -> torch.Tensor:
        """x: fp32 [n,1,d0,h,w] contiguous. Returns the head's input: bf16 [n,d0,h,w,32] (the decoder output
        resampled to the caller's depth)."""
        p = self._params()
        if B.x_in is not None:
            ops.depth_resample(x.view(B.n, B.d0, -1), B.x_in.view(B.n, B.d, -1), self.matrix(B.d0, B.d, x.device))
            x_img = B.x_in
        else:
            x_img = x
        self._block_fwd(B, "enc1", None, x_img, training)
        for l, b in ((2, "enc2"), (3, "enc3"), (4, "enc4"), (5, "bott")):
            self._block_fwd(B, b, B.pool[l - 1], None, training)
        prev = B.out["bott"]
        for l, up, dec, _ in _UPS:
            cu = B.C[l]
            ops.convt_k222_fwd(prev, 2 * cu, self._packed[up][0], p[f"{up}.bias"], B.cat[l][..., :cu], cu)
            self._block_fwd(B, dec, B.cat[l], None, training)
            prev = B.out[dec]
        if B.hx is None:
            return prev
        ops.depth_resample(prev, B.hx, self.matrix(B.d, B.d0, x.device))
        return B.hx

    # ------------------------------------------------------------------------------------------
    def _block_bwd(self, B: _Buffers, G: Dict[str, torch.Tensor], b: str, dout: torch.Tensor, xin, dxin, x_img):
        p = self._params()
        l = _LEVEL[b]
        cin, c = self.channels(b)
        shp = B.shape(l)
        t1, t2 = B.t1[l], B.t2[l]
        # BN2 + ReLU backward
        ops.norm_act_bwd_reduce(dout, B.x2[b], B.coef[f"{b}.2"], B.R[f"{b}.2"], c, SLOPE, plain=True, fixed_order=True)
        ops.bn_bwd_coeffs(B.R[f"{b}.2"], B.coef[f"{b}.2"], p[f"{b}.4.weight"], c, shp, B.bcoef[f"{b}.2"],
                          G[f"{b}.4.weight"], G[f"{b}.4.bias"])
        ops.norm_act_bwd_apply(dout, B.x2[b], B.coef[f"{b}.2"], B.bcoef[f"{b}.2"], None, None, t1, c, SLOPE)
        ops.conv3d_k3_wgrad(B.a1[b], c, t1, c, G[f"{b}.3.weight"], 1.0)
        ops.conv3d_k3_dgrad(t1, c, self._packed[f"{b}.2"][1], t2, c)
        # BN1 + ReLU backward
        ops.norm_act_bwd_reduce(t2, B.x1[b], B.coef[f"{b}.1"], B.R[f"{b}.1"], c, SLOPE, plain=True, fixed_order=True)
        ops.bn_bwd_coeffs(B.R[f"{b}.1"], B.coef[f"{b}.1"], p[f"{b}.1.weight"], c, shp, B.bcoef[f"{b}.1"],
                          G[f"{b}.1.weight"], G[f"{b}.1.bias"])
        ops.norm_act_bwd_apply(t2, B.x1[b], B.coef[f"{b}.1"], B.bcoef[f"{b}.1"], None, None, t1, c, SLOPE)
        if b == "enc1":
            ops.conv3d_stem_wgrad(x_img, t1, c, G[f"{b}.0.weight"], 1.0)
        else:
            ops.conv3d_k3_wgrad(xin, cin, t1, c, G[f"{b}.0.weight"], 1.0)
            if b.startswith("dec"):   # + column sums of the input gradient: the transposed conv's bias gradient
                ops.conv3d_k3_dgrad_stats(t1, c, self._packed[f"{b}.1"][1], dxin, cin, B.dpartial[l])
            else:
                ops.conv3d_k3_dgrad(t1, c, self._packed[f"{b}.1"][1], dxin, cin)

    def backward(self, B: _Buffers, G: Dict[str, torch.Tensor], x: torch.Tensor, ghead: torch.Tensor):
        """ghead: gradient w.r.t. the head's input (bf16 [n,d0,h,w,32]). Accumulates (+=) every parameter
        gradient except the head's into the fp32 tensors of `G`."""
        if B.hx is not None:
            ops.depth_resample(ghead, B.gout[1], self.matrix(B.d, B.d0, x.device, transpose=True))
        elif ghead.data_ptr() != B.gout[1].data_ptr():
            B.gout[1].copy_(ghead)
        for l, up, dec, below in _UPS[::-1]:
            cu = B.C[l]
            self._block_bwd(B, G, dec, B.gout[l], B.cat[l], B.dcat[l], None)
            dy = B.dcat[l][..., :cu]
            ops.convt_k222_wgrad(B.out[below], 2 * cu, dy, cu, G[f"{up}.weight"], 1.0)
            ops.convt_k222_dgrad(dy, cu, self._packed[up][1], B.gout[l + 1], 2 * cu)
        self._block_bwd(B, G, "bott", B.gout[5], B.pool[4], B.dpool[4], None)
        x_img = B.x_in if B.x_in is not None else x
        for l, enc in ((4, "enc4"), (3, "enc3"), (2, "enc2"), (1, "enc1")):
            c = B.C[l]
            dskip = B.dcat[l][..., c:]
            ops.maxpool222_bwd_add(B.dpool[l], B.out[enc], dskip, c, True)
            if l > 1:
                self._block_bwd(B, G, enc, dskip, B.pool[l - 1], B.dpool[l - 1], None)
            else:
                self._block_bwd(B, G, enc, dskip, None, None, x_img)
        for l, up, _, _ in _UPS:   # ConvTranspose3d bias gradient = column sums of dy (dgrad epilogue partials)
            G[f"{up}.bias"].add_(B.dpartial[l][:, :, 0, :B.C[l]].double().sum((0, 1)).float())

    # ------------------------------------------------------------------------------------------
    def _check_input(self, x: torch.Tensor) -> torch.Tensor:
        if x.dim() != 5 or x.shape[1] != 1:
            raise ValueError(f"expected images [B,1,D,H,W], got {tuple(x.shape)}")
        if not x.is_cuda:
            raise RuntimeError("spff_b200 runs on a B200 (sm_100) device only; the input is on the CPU and there is "
                               "no CPU fallback")
        return x.float().contiguous()

    def infer(self, x: torch.Tensor, target_depth: Optional[int], training: bool = False, argmax: bool = False):
        """Forward only: fp32 logits [B,K,D0,H,W] or (argmax) the uint8 label map [B,D0,H,W]. `training` selects
        batch statistics (and updates the running buffers) as module.train() does for nn.BatchNorm3d."""
        x = self._check_input(x)
        n, _, d0, h, w = x.shape
        self.refresh_weights()
        B = self.buffers(n, d0, target_depth or d0, h, w, x.device, train=False)
        hx = self.forward(B, x, training)
        p = self._params()
        if argmax:
            out = torch.empty(n, d0, h, w, dtype=torch.uint8, device=x.device)
            ops.head_argmax(hx, p["out.weight"], p["out.bias"], out)
        else:
            out = torch.empty(n, self.k, d0, h, w, device=x.device)
            ops.head_fwd(hx, p["out.weight"], p["out.bias"], out)
        return out

    def forward_saved(self, x: torch.Tensor, target_depth: Optional[int], training: bool = True):
        x = self._check_input(x)
        n, _, d0, h, w = x.shape
        self.refresh_weights()
        B = self.buffers(n, d0, target_depth or d0, h, w, x.device, train=True, fresh=True)
        hx = self.forward(B, x, training)
        p = self._params()
        logits = torch.empty(n, self.k, d0, h, w, device=x.device)
        ops.head_fwd(hx, p["out.weight"], p["out.bias"], logits)
        return logits, (B, x, hx)

    def backward_saved(self, state, dlogits: torch.Tensor, G: Dict[str, torch.Tensor]):
        B, x, hx = state
        p = self._params()
        gh = B.gh if B.gh is not None else B.gout[1]
        ops.head_bwd(dlogits.float().contiguous(), hx, p["out.weight"], gh, G["out.weight"].view(-1, self.base),
                     G["out.bias"], 1.0)
        self.backward(B, G, x, gh)

    def train_step(self, x: torch.Tensor, labels: torch.Tensor, G: Dict[str, torch.Tensor], tally: LossTally,
                   target_depth: Optional[int], ignore_index: int = 255):
        """Fused forward + CE/confusion + backward over the whole batch (training-mode BatchNorm). Accumulates the
        gradient of the mean CE over valid voxels into G and the loss statistics into `tally`."""
        x = self._check_input(x)
        n, _, d0, h, w = x.shape
        if labels.shape != (n, d0, h, w):
            raise ValueError(f"labels must be [B,D,H,W] = {(n, d0, h, w)}, got {tuple(labels.shape)}")
        labels = labels.contiguous()
        self.refresh_weights()
        B = self.buffers(n, d0, target_depth or d0, h, w, x.device, train=True)
        hx = self.forward(B, x, True)
        p = self._params()
        n_valid = (labels != ignore_index).sum().clamp(min=1).reshape(1)    # .clamp_min(1.0), models.py:797
        gh = B.gh if B.gh is not None else B.gout[1]
        ops.head_loss_fused(hx, p["out.weight"], p["out.bias"], labels, ignore_index, n_valid, None, tally.nll,
                            tally.count, tally.confusion, gh, G["out.weight"].view(-1, self.base), G["out.bias"], 1.0)
        self.backward(B, G, x, gh)

    def eval_step(self, x: torch.Tensor, labels: torch.Tensor, tally: LossTally, target_depth: Optional[int],
                  ignore_index: int = 255, training: bool = False,
                  per_sample: Optional[Tuple[torch.Tensor, torch.Tensor, torch.Tensor]] = None,
                  labels_out: Optional[torch.Tensor] = None, hist: Optional[torch.Tensor] = None,
                  sample_hist: Optional[torch.Tensor] = None):
        """Forward + head + CE/confusion over the whole batch, with no gradient and no logits in memory: the tally of
        `infer(x, target_depth, training)` accumulates (+=) into `tally` (BatchNorm as `training` selects, like infer).
        per_sample / labels_out / hist / sample_hist as in SpffEngine.eval_step (at the original depth)."""
        x = self._check_input(x)
        n, _, d0, h, w = x.shape
        if labels.shape != (n, d0, h, w):
            raise ValueError(f"labels must be [B,D,H,W] = {(n, d0, h, w)}, got {tuple(labels.shape)}")
        labels = labels.contiguous()
        self.refresh_weights()
        B = self.buffers(n, d0, target_depth or d0, h, w, x.device, train=False)
        hx = self.forward(B, x, training)
        p = self._params()
        rows = per_sample if per_sample is not None else (None, None, None)
        ops.head_eval(hx, p["out.weight"], p["out.bias"], labels, ignore_index, tally.nll, tally.count, tally.confusion,
                      *rows, labels_out, hist=hist, sample_hist=sample_hist)


def flat_names(named_params: List[Tuple[str, torch.Tensor]]):
    """16-byte aligned slots of a flat fp32 buffer holding the given parameters in order: name -> (offset, numel, shape)."""
    slots, off = {}, 0
    for n, p in named_params:
        k = p.numel()
        slots[n] = (off, k, tuple(p.shape))
        off += (k + 3) // 4 * 4
    return slots, off
