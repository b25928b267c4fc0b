"""Tensor-level wrappers over the C ABI (include/spff_b200.h).

Activations are bf16 "position-major" views [N, D, H, W, C] whose last dimension is contiguous and
whose position pitch `ld` (= stride of W, in elements) may exceed C — a channel slice of a wider
buffer is passed as the sliced view itself. These functions only validate, extract pointers and
enqueue on the current CUDA stream.
"""
from __future__ import annotations

import ctypes
import dataclasses
import math
from typing import Optional

import torch

from . import _lib
from ._lib import Shape, UncOut, call, ptr, stream_ptr


def _view(t: torch.Tensor, c: int):
    """(shape, ld) of a position-major bf16 view holding >= c channels."""
    if t.dtype != torch.bfloat16 or t.dim() != 5 or not t.is_cuda:
        raise ValueError(f"expected a CUDA bf16 [N,D,H,W,C] view, got {t.dtype} {tuple(t.shape)} on {t.device}")
    n, d, h, w, cc = t.shape
    if cc < c:
        raise ValueError(f"view has {cc} channels, need {c}")
    ld = t.stride(3)
    if t.stride(4) != 1 or t.stride(2) != w * ld or t.stride(1) != h * w * ld or t.stride(0) != d * h * w * ld:
        raise ValueError(f"view is not position-major with a uniform pitch: strides {t.stride()}")
    return Shape(n, d, h, w), ld


def conv3_flops(s: Shape, cin: int, cout: int) -> float:
    """Algorithmic FLOPs of one 3x3x3 convolution pass (fwd, dgrad or wgrad): 2 * 27 * cin * cout per position."""
    return 2.0 * 27 * cin * cout * s.n * s.d * s.h * s.w


def conv3_kc(k_channels: int) -> int:
    return 64 if k_channels % 64 == 0 else 32


def pack_conv3_weight(w: torch.Tensor, fwd: bool = True, dgrad: bool = True):
    """nn.Conv3d weight [Cout,Cin,3,3,3] fp32 -> (w_fwd, w_dgrad) bf16 GEMM operands."""
    cout, cin = w.shape[0], w.shape[1]
    w = w.detach().contiguous().float()
    elems = int(_lib.lib.spff_conv3_packed_elems(cin, cout))
    wf = torch.empty(elems, dtype=torch.bfloat16, device=w.device) if fwd else None
    wd = torch.empty(elems, dtype=torch.bfloat16, device=w.device) if dgrad else None
    call("spff_pack_conv3_weight", ptr(w), ptr(wf), ptr(wd), cout, cin, stream_ptr())
    return wf, wd


def conv3d_k3_fwd(x, cin, w_fwd, y, cout):
    s, ldx = _view(x, cin)
    s2, ldy = _view(y, cout)
    assert (s.n, s.d, s.h, s.w) == (s2.n, s2.d, s2.h, s2.w)
    _lib.NOTE = conv3_flops(s, cin, cout)
    call("spff_conv3d_k3_fwd", ptr(x), ldx, cin, ptr(w_fwd), ptr(y), ldy, cout, s, stream_ptr())


def conv3d_k3_stat_slots(shape: Shape) -> int:
    return int(_lib.lib.spff_conv3d_k3_stat_slots(shape))


def conv3d_k3_fwd_stats(x, cin, w_fwd, y, cout, partial):
    """Forward conv + per-item InstanceNorm partial statistics of y (fp32 [n, slots, 2, cout])."""
    s, ldx = _view(x, cin)
    s2, ldy = _view(y, cout)
    assert (s.n, s.d, s.h, s.w) == (s2.n, s2.d, s2.h, s2.w)
    assert partial.dtype == torch.float32 and partial.is_contiguous()
    assert partial.numel() >= s.n * conv3d_k3_stat_slots(s) * 2 * cout
    _lib.NOTE = conv3_flops(s, cin, cout)
    call("spff_conv3d_k3_fwd_stats", ptr(x), ldx, cin, ptr(w_fwd), ptr(y), ldy, cout, s, ptr(partial), stream_ptr())


def in_coeffs_from_partials(partial, slots, gamma, beta, eps, n, c, count, coef):
    call("spff_in_coeffs_from_partials", ptr(partial), int(slots), ptr(gamma), ptr(beta), float(eps), n, c, int(count),
         ptr(coef), stream_ptr())


def conv3d_k3_dgrad(dy, cout, w_dgrad, dx, cin):
    s, lddy = _view(dy, cout)
    s2, lddx = _view(dx, cin)
    assert (s.n, s.d, s.h, s.w) == (s2.n, s2.d, s2.h, s2.w)
    _lib.NOTE = conv3_flops(s, cin, cout)
    call("spff_conv3d_k3_dgrad", ptr(dy), lddy, cout, ptr(w_dgrad), ptr(dx), lddx, cin, s, stream_ptr())


def conv3d_k3_dgrad_stats(dy, cout, w_dgrad, dx, cin, partial):
    """dgrad + per-item {sum, sum sq} partials of dx (fp32 [n, slots, 2, cin])."""
    s, lddy = _view(dy, cout)
    s2, lddx = _view(dx, cin)
    assert (s.n, s.d, s.h, s.w) == (s2.n, s2.d, s2.h, s2.w)
    assert partial.dtype == torch.float32 and partial.is_contiguous()
    assert partial.numel() >= s.n * conv3d_k3_stat_slots(s) * 2 * cin
    _lib.NOTE = conv3_flops(s, cin, cout)
    call("spff_conv3d_k3_dgrad_stats", ptr(dy), lddy, cout, ptr(w_dgrad), ptr(dx), lddx, cin, s, ptr(partial), stream_ptr())


_WS = {}


def workspace(nbytes: int, device) -> torch.Tensor:
    """Grow-only scratch buffer per device (the library itself allocates nothing)."""
    key = str(device)
    buf = _WS.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device)
        _WS[key] = buf
    return buf


def conv3d_k3_wgrad_workspace(cin, cout, x) -> torch.Tensor:
    s, _ = _view(x, cin)
    return workspace(int(_lib.lib.spff_conv3d_k3_wgrad_workspace(cin, cout, s)), x.device)


def conv3d_k3_wgrad(x, cin, dy, cout, dw, beta: float = 0.0, ws: torch.Tensor | None = None):
    """dw [Cout,Cin,3,3,3] fp32 = beta*dw + grad_weight."""
    s, ldx = _view(x, cin)
    s2, lddy = _view(dy, cout)
    assert (s.n, s.d, s.h, s.w) == (s2.n, s2.d, s2.h, s2.w)
    assert dw.dtype == torch.float32 and dw.is_contiguous() and tuple(dw.shape) == (cout, cin, 3, 3, 3)
    if ws is None:
        ws = conv3d_k3_wgrad_workspace(cin, cout, x)
    _lib.NOTE = conv3_flops(s, cin, cout)
    call("spff_conv3d_k3_wgrad", ptr(x), ldx, cin, ptr(dy), lddy, cout, s, ptr(dw), float(beta), ptr(ws),
         ws.numel(), stream_ptr())


# ------------------------------------------------------------------------------------------------
# stem / transposed conv
# ------------------------------------------------------------------------------------------------
def _shape5(x5):
    n, _, d, h, w = x5.shape
    return Shape(n, d, h, w)


def conv3d_stem_fwd(x, w, y, cout):
    """x fp32 [N,1,D,H,W] contiguous, w fp32 [cout,1,3,3,3] -> y bf16 view."""
    assert x.dtype == torch.float32 and x.is_contiguous() and x.shape[1] == 1
    s, ldy = _view(y, cout)
    call("spff_conv3d_stem_fwd", ptr(x), ptr(w), ptr(y), ldy, cout, s, stream_ptr())


def conv3d_stem_stat_slots(shape: Shape) -> int:
    return int(_lib.lib.spff_conv3d_stem_stat_slots(shape))


def conv3d_stem_fwd_stats(x, w, y, cout, partial):
    """Stem forward + {sum, sum sq} partials of y (fp32 [n, slots, 2, cout], slots = conv3d_stem_stat_slots)."""
    assert x.dtype == torch.float32 and x.is_contiguous() and x.shape[1] == 1
    s, ldy = _view(y, cout)
    assert partial.dtype == torch.float32 and partial.is_contiguous()
    assert partial.numel() >= s.n * conv3d_stem_stat_slots(s) * 2 * cout
    call("spff_conv3d_stem_fwd_stats", ptr(x), ptr(w), ptr(y), ldy, cout, s, ptr(partial), stream_ptr())


def conv3d_stem_wgrad(x, dy, cout, dw, beta=0.0):
    s, lddy = _view(dy, cout)
    ws = workspace(int(_lib.lib.spff_conv3d_stem_wgrad_workspace(cout)), x.device)
    call("spff_conv3d_stem_wgrad", ptr(x), ptr(dy), lddy, cout, s, ptr(dw), float(beta), ptr(ws), ws.numel(),
         stream_ptr())


def pack_convt_weight(w):
    """nn.ConvTranspose3d weight [Cin,Cout,1,2,2] fp32 -> (w_fwd, w_dgrad) bf16."""
    cin, cout = w.shape[0], w.shape[1]
    w = w.detach().contiguous().float()
    wf = torch.empty(4 * cin * cout, dtype=torch.bfloat16, device=w.device)
    wd = torch.empty(4 * cin * cout, dtype=torch.bfloat16, device=w.device)
    call("spff_pack_convt_weight", ptr(w), ptr(wf), ptr(wd), cin, cout, stream_ptr())
    return wf, wd


def convt_k122_fwd(x, cin, w_fwd, bias, y, cout):
    s, ldx = _view(x, cin)
    s2, ldy = _view(y, cout)
    assert (s2.h, s2.w) == (2 * s.h, 2 * s.w)
    call("spff_convt_k122_fwd", ptr(x), ldx, cin, ptr(w_fwd), ptr(bias), ptr(y), ldy, cout, s, stream_ptr())


def convt_k122_dgrad(dy, cout, w_dgrad, dx, cin):
    s, lddx = _view(dx, cin)
    s2, lddy = _view(dy, cout)
    assert (s2.h, s2.w) == (2 * s.h, 2 * s.w)
    call("spff_convt_k122_dgrad", ptr(dy), lddy, cout, ptr(w_dgrad), ptr(dx), lddx, cin, s, stream_ptr())


def convt_k122_wgrad(x, cin, dy, cout, dw, beta=0.0):
    s, ldx = _view(x, cin)
    _, lddy = _view(dy, cout)
    ws = workspace(int(_lib.lib.spff_convt_k122_wgrad_workspace(cin, cout, s)), x.device)
    call("spff_convt_k122_wgrad", ptr(x), ldx, cin, ptr(dy), lddy, cout, s, ptr(dw), float(beta), ptr(ws), ws.numel(),
         stream_ptr())


# ------------------------------------------------------------------------------------------------
# norm / act / SPFF tail
# ------------------------------------------------------------------------------------------------
def in_stats(x, c, stats):
    """stats fp64 [N,C,2] += {sum, sum sq}."""
    s, ldx = _view(x, c)
    call("spff_in_stats", ptr(x), ldx, c, s, ptr(stats), stream_ptr())


def in_coeffs(stats, gamma, beta, eps, n, c, count, coef, batch_stats=False):
    call("spff_in_coeffs", ptr(stats), ptr(gamma), ptr(beta), float(eps), n, c, int(count), int(batch_stats), ptr(coef),
         stream_ptr())


def norm_act_apply(x, coef, y, c, slope):
    s, ldx = _view(x, c)
    _, ldy = _view(y, c)
    call("spff_norm_act_apply", ptr(x), ldx, ptr(coef), ptr(y), ldy, c, s, float(slope), stream_ptr())


def norm_act_reduce(x, coef, S, c, slope, fixed_order=False):
    """fixed_order=True: S is overwritten by a bit-reproducible two-stage reduction (no zeroing needed);
    otherwise the blocks accumulate into S with atomics (zero S first)."""
    s, ldx = _view(x, c)
    ws, nbytes = None, 0
    if fixed_order:
        nbytes = int(_lib.lib.spff_norm_act_reduce_workspace(c, s))
        ws = workspace(nbytes, x.device) if nbytes else None
    call("spff_norm_act_reduce", ptr(x), ldx, ptr(coef), ptr(S), c, s, float(slope), ptr(ws), ws.numel() if ws is not None else 0,
         stream_ptr())


def norm_act_affine_apply(x, coef, P, Q, y, ypool, c, slope, pool_argmax=None):
    """pool_argmax: optional uint8 [n,d,h/2,w/2,c] (contiguous) receiving the corner 0..3 of every pooling window's first
    maximum, for maxpool_bwd_add_argmax."""
    s, ldx = _view(x, c)
    _, ldy = _view(y, c)
    ldp = _view(ypool, c)[1] if ypool is not None else 0
    if pool_argmax is not None:
        assert ypool is not None and pool_argmax.dtype == torch.uint8 and pool_argmax.is_contiguous()
        assert tuple(pool_argmax.shape) == (s.n, s.d, s.h // 2, s.w // 2, c)
    call("spff_norm_act_affine_apply", ptr(x), ldx, ptr(coef), ptr(P), ptr(Q), ptr(y), ldy, ptr(ypool), ldp, ptr(pool_argmax), c, s,
         float(slope), stream_ptr())


def gate_tables_fwd(w0, b0, w2, b2, mask, scale, c, frames, g1, bt, kfg):
    """g1 / bt [c, frames] from the EFiLM MLP, kfg [frames] from the FourierGate mask (None skips a gate)."""
    call("spff_gate_tables_fwd", ptr(w0), ptr(b0), ptr(w2), ptr(b2), ptr(mask), ptr(scale), c, frames, ptr(g1), ptr(bt), ptr(kfg),
         stream_ptr())


def gate_tables_bwd(w0, b0, w2, b2, mask, scale, c, frames, dg1, dbt, dkfg, dw0, db0, dw2, db2, dmask, dscale):
    """+= the parameter gradients from the accumulated table gradients."""
    call("spff_gate_tables_bwd", ptr(w0), ptr(b0), ptr(w2), ptr(b2), ptr(mask), ptr(scale), c, frames, ptr(dg1), ptr(dbt),
         ptr(dkfg), ptr(dw0), ptr(db0), ptr(dw2), ptr(db2), ptr(dmask), ptr(dscale), stream_ptr())


def gate_micro_fwd(S, g1, bt, kfg, se, flags, c, shape, P, Q):
    w1, b1, w2, b2 = se if se is not None else (None, None, None, None)
    hid = w1.shape[0] if w1 is not None else 0
    call("spff_gate_micro_fwd", ptr(S), ptr(g1), ptr(bt), ptr(kfg), ptr(w1), ptr(b1), ptr(w2), ptr(b2), hid, flags, c,
         shape, ptr(P), ptr(Q), stream_ptr())


def norm_act_bwd_reduce(dout, x, coef, R, c, slope, plain=False, fixed_order=False, S=None):
    """plain=True: only the two sums the gate-free InstanceNorm + LeakyReLU backward needs.
    S: the forward statistic of the same tensor (norm_act_reduce); with fixed_order it enables the lean first stage."""
    s, lddo = _view(dout, c)
    _, ldx = _view(x, c)
    ws, nbytes = None, 0
    if fixed_order:
        nbytes = int(_lib.lib.spff_norm_act_bwd_reduce_workspace(c, s, int(plain)))
        ws = workspace(nbytes, x.device) if nbytes else None
    call("spff_norm_act_bwd_reduce", ptr(dout), lddo, ptr(x), ldx, ptr(coef), ptr(R), ptr(S), c, s, float(slope), int(plain),
         ptr(ws), ws.numel() if ws is not None else 0, stream_ptr())


def gate_micro_bwd(R, S, coef, gamma, g1, bt, kfg, se, flags, c, shape, bcoef, dSa, Pout, dgamma, dbeta, dg1, dbt, dkfg,
                   dse):
    w1, b1, w2, b2 = se if se is not None else (None, None, None, None)
    dw1, db1, dw2, db2 = dse if dse is not None else (None, None, None, None)
    hid = w1.shape[0] if w1 is not None else 0
    call("spff_gate_micro_bwd", ptr(R), ptr(S), ptr(coef), ptr(gamma), ptr(g1), ptr(bt), ptr(kfg), ptr(w1), ptr(b1),
         ptr(w2), ptr(b2), hid, flags, c, shape, ptr(bcoef), ptr(dSa), ptr(Pout), ptr(dgamma), ptr(dbeta), ptr(dg1),
         ptr(dbt), ptr(dkfg), ptr(dw1), ptr(db1), ptr(dw2), ptr(db2), stream_ptr())


def norm_act_bwd_apply(dout, x, coef, bcoef, P, dSa, dx, c, slope):
    s, lddo = _view(dout, c)
    _, ldx = _view(x, c)
    _, lddx = _view(dx, c)
    call("spff_norm_act_bwd_apply", ptr(dout), lddo, ptr(x), ldx, ptr(coef), ptr(bcoef), ptr(P), ptr(dSa), ptr(dx), lddx,
         c, s, float(slope), stream_ptr())


def maxpool_bwd_add(dpool, y, dskip, c, accumulate):
    s, ldy = _view(y, c)
    _, ldp = _view(dpool, c)
    _, ldd = _view(dskip, c)
    call("spff_maxpool_bwd_add", ptr(dpool), ldp, ptr(y), ldy, ptr(dskip), ldd, c, s, int(accumulate), stream_ptr())


def maxpool_bwd_add_argmax(dpool, pool_argmax, dskip, c, accumulate):
    """dskip[window corner pool_argmax] += dpool, without reading the full-resolution activation."""
    s, ldd = _view(dskip, c)
    _, ldp = _view(dpool, c)
    assert pool_argmax.dtype == torch.uint8 and pool_argmax.is_contiguous()
    call("spff_maxpool_bwd_add_argmax", ptr(dpool), ldp, ptr(pool_argmax), ptr(dskip), ldd, c, s, int(accumulate), stream_ptr())


# ------------------------------------------------------------------------------------------------
# head / loss / optimizer
# ------------------------------------------------------------------------------------------------
def head_fwd(x, w, b, logits):
    """x bf16 view (32 ch), w fp32 [K,32] (any trailing 1-dims), logits fp32 [N,K,D,H,W] contiguous."""
    k = w.shape[0]
    s, ldx = _view(x, 32)
    assert logits.dtype == torch.float32 and logits.is_contiguous()
    call("spff_head_fwd", ptr(x), ldx, 32, ptr(w), ptr(b), ptr(logits), k, s, stream_ptr())


def head_argmax(x, w, b, labels):
    k = w.shape[0]
    s, ldx = _view(x, 32)
    assert labels.dtype == torch.uint8 and labels.is_contiguous()
    call("spff_head_argmax", ptr(x), ldx, 32, ptr(w), ptr(b), ptr(labels), k, s, stream_ptr())


def head_bwd(dlogits, x, w, dx, dw, db, beta=0.0):
    k = w.shape[0]
    s, ldx = _view(x, 32)
    lddx = _view(dx, 32)[1] if dx is not None else 0
    ws = workspace(int(_lib.lib.spff_head_bwd_workspace(k)), x.device)
    call("spff_head_bwd", ptr(dlogits), ptr(x), ldx, 32, ptr(w), ptr(dx), lddx, ptr(dw), ptr(db), float(beta), k, s,
         ptr(ws), ws.numel(), stream_ptr())


def _label_bytes(labels):
    if labels.dtype == torch.uint8:
        return 1
    if labels.dtype == torch.int64:
        return 8
    raise ValueError("labels must be uint8 or int64")


def ce_confusion(logits, labels, ignore_index, acc, counts, confusion):
    n, k, d, h, w = logits.shape
    assert logits.is_contiguous() and labels.is_contiguous()
    call("spff_ce_confusion", ptr(logits), ptr(labels), _label_bytes(labels), int(ignore_index), k, Shape(n, d, h, w),
         ptr(acc), ptr(counts), ptr(confusion), stream_ptr())


def ce_grad(logits, labels, ignore_index, n_valid, gscale, dlogits):
    n, k, d, h, w = logits.shape
    call("spff_ce_grad", ptr(logits), ptr(labels), _label_bytes(labels), int(ignore_index), k, Shape(n, d, h, w),
         ptr(n_valid), ptr(gscale), ptr(dlogits), stream_ptr())


def head_loss_fused(x, w, b, labels, ignore_index, n_valid, gscale, acc, counts, confusion, dx, dw, db, beta=0.0):
    """Fused training head (no logits in memory): loss statistics += , dx / dw / db of the batch-mean CE."""
    k = w.shape[0]
    s, ldx = _view(x, 32)
    lddx = _view(dx, 32)[1] if dx is not None else 0
    assert labels.is_contiguous() and labels.numel() == s.n * s.d * s.h * s.w
    ws = workspace(int(_lib.lib.spff_head_loss_workspace(k)), x.device)
    call("spff_head_loss_fused", ptr(x), ldx, 32, ptr(w), ptr(b), ptr(labels), _label_bytes(labels), int(ignore_index), k, s,
         ptr(n_valid), ptr(gscale), ptr(acc), ptr(counts), ptr(confusion), ptr(dx), lddx, ptr(dw), ptr(db), float(beta),
         ptr(ws), ws.numel(), stream_ptr())


def head_eval(x, w, b, labels, ignore_index, acc, counts, confusion, sample_acc=None, sample_counts=None,
              sample_confusion=None, labels_out=None, hist=None, sample_hist=None):
    """Fused evaluation head (no logits in memory): the loss statistics of head_fwd + ce_confusion += into acc /
    counts / confusion; optionally per sample (fp64 [n], int64 [n], int64 [n,K,K], +=) and the uint8 arg-max map
    [n,d,h,w] the tally counts. `hist` (int64 [K,2,T], +=) adds the per-class histogram of the softmax probability
    over T = hist.shape[-1] bins, positives in [c,0] and negatives in [c,1] (spff_head_eval_hist); `sample_hist`
    (int64 [n,K,2,T]) is the same per sample and goes with the per-sample tallies."""
    if hist is not None:
        k, bins = w.shape[0], hist.shape[-1]
        assert hist.dtype == torch.int64 and hist.is_contiguous() and tuple(hist.shape) == (k, 2, bins)
        if sample_hist is not None:
            n = x.shape[0]
            assert sample_hist.dtype == torch.int64 and sample_hist.is_contiguous()
            assert tuple(sample_hist.shape) == (n, k, 2, bins)
    else:
        assert sample_hist is None, "sample_hist needs hist"
    k = w.shape[0]
    s, ldx = _view(x, 32)
    assert labels.is_contiguous() and labels.numel() == s.n * s.d * s.h * s.w
    per = (sample_acc, sample_counts, sample_confusion)
    if any(t is not None for t in per):
        assert sample_acc.dtype == torch.float64 and sample_acc.numel() == s.n
        assert sample_counts.dtype == torch.int64 and sample_counts.numel() == s.n
        assert sample_confusion.dtype == torch.int64 and sample_confusion.is_contiguous()
        assert sample_confusion.numel() == s.n * k * k
    if labels_out is not None:
        assert labels_out.dtype == torch.uint8 and labels_out.is_contiguous() and labels_out.numel() == s.n * s.d * s.h * s.w
    if hist is None:
        call("spff_head_eval", ptr(x), ldx, 32, ptr(w), ptr(b), ptr(labels), _label_bytes(labels), int(ignore_index), k, s,
             ptr(acc), ptr(counts), ptr(confusion), *(ptr(t) for t in per), ptr(labels_out), stream_ptr())
    else:
        call("spff_head_eval_hist", ptr(x), ldx, 32, ptr(w), ptr(b), ptr(labels), _label_bytes(labels), int(ignore_index),
             k, s, ptr(acc), ptr(counts), ptr(confusion), *(ptr(t) for t in per), ptr(labels_out), int(hist.shape[-1]),
             ptr(hist), ptr(sample_hist), stream_ptr())


def head_prob_accum(x, w, b, acc, flip: int = 0, beta: int = 0, ent=None):
    """Head + softmax added into the probability accumulator acc (fp32 [n,d,h,w,16], contiguous, 16-byte aligned):
    acc[n,d,h',w',c] = beta * acc + p_c, with h' / w' mirrored back when bit 1 / 2 of `flip` is set (the inverse of an
    input flip). Classes >= K are written as 0 when beta = 0 and left alone when beta = 1 (spff_head_prob_accum).
    With `ent` (fp32 [n,d,h,w], contiguous) also ent[n,d,h',w'] = beta * ent + H(p), the entropy of this pass's
    softmax in nats (spff_head_prob_accum_ent)."""
    s, ldx = _view(x, 32)
    assert acc.dtype == torch.float32 and acc.is_contiguous() and acc.numel() == s.n * s.d * s.h * s.w * 16
    if ent is None:
        call("spff_head_prob_accum", ptr(x), ldx, 32, ptr(w), ptr(b), w.shape[0], s, int(flip), int(beta), ptr(acc),
             stream_ptr())
        return
    assert ent.dtype == torch.float32 and ent.is_contiguous() and ent.numel() == s.n * s.d * s.h * s.w
    call("spff_head_prob_accum_ent", ptr(x), ldx, 32, ptr(w), ptr(b), w.shape[0], s, int(flip), int(beta), ptr(acc),
         ptr(ent), stream_ptr())


@dataclasses.dataclass
class Uncertainty:
    """Outputs of prob_finalize(unc=...) (spff_unc_out); every field is optional. Per position of an accumulator of n
    samples: `ent` the expected-entropy plane of head_prob_accum(ent=...) (fp32 [n,d,h,w], the sum over the passes),
    `entropy_out` / `mi_out` fp16 [n,d,h,w] maps of H[p̄] and of the mutual information max(H[p̄] - scale * ent, 0)
    (needs ent); `unc` int64 [2] (+=) and `sample_unc` int64 [n,2] (+=) their sums in units of 2^-24 nats. With labels:
    `calib` int64 [3,T] (+=: per confidence bin the counted voxels, the correct ones and the summed confidence in
    units of 2^-24), `sample_calib` [n,3,T] (exactly when the per-sample tallies are given), `brier` fp64 [1] and
    `sample_brier` fp64 [n] (exactly with calib / sample_calib) the summed Brier score."""
    ent: Optional[torch.Tensor] = None
    entropy_out: Optional[torch.Tensor] = None
    mi_out: Optional[torch.Tensor] = None
    unc: Optional[torch.Tensor] = None
    sample_unc: Optional[torch.Tensor] = None
    calib: Optional[torch.Tensor] = None
    sample_calib: Optional[torch.Tensor] = None
    brier: Optional[torch.Tensor] = None
    sample_brier: Optional[torch.Tensor] = None


def _unc_struct(u: Uncertainty, n: int, vox: int) -> UncOut:
    def check(t, dtype, numel, name):
        if t is not None:
            assert t.dtype == dtype and t.is_contiguous() and t.numel() == numel, \
                f"{name}: expected contiguous {dtype} with {numel} elements, got {t.dtype} {tuple(t.shape)}"
    check(u.ent, torch.float32, vox, "ent")
    check(u.entropy_out, torch.float16, vox, "entropy_out")
    check(u.mi_out, torch.float16, vox, "mi_out")
    check(u.unc, torch.int64, 2, "unc")
    check(u.sample_unc, torch.int64, 2 * n, "sample_unc")
    bins = 0
    if u.calib is not None:
        bins = u.calib.shape[-1]
        check(u.calib, torch.int64, 3 * bins, "calib")
        check(u.sample_calib, torch.int64, n * 3 * bins, "sample_calib")
    check(u.brier, torch.float64, 1, "brier")
    check(u.sample_brier, torch.float64, n, "sample_brier")
    return UncOut(ptr(u.ent), ptr(u.entropy_out), ptr(u.mi_out), ptr(u.unc), ptr(u.sample_unc), int(bins), ptr(u.calib),
                  ptr(u.sample_calib), ptr(u.brier), ptr(u.sample_brier))


def prob_finalize(acc, k: int, scale: float, labels=None, ignore_index: int = 255, tally=None, per_sample=None,
                  labels_out=None, hist=None, sample_hist=None, proba_out=None, unc: Optional[Uncertainty] = None,
                  inv_temperature: float = 1.0):
    """One pass over a spff_head_prob_accum accumulator acc (fp32 [n,d,h,w,16]): p̄ = scale * acc. Optional outputs:
    labels_out (uint8 [n,d,h,w], the first arg-max of acc over classes < k), proba_out (fp16 [n,k,d,h,w], p̄), and with
    labels (uint8 / int64 [n,d,h,w]) the tally (nll fp64 [1], count int64 [1], confusion int64 [k,k], +=) of
    head_eval on p̄, per_sample rows (fp64 [n], int64 [n], int64 [n,k,k]), hist (int64 [k,2,T]) and sample_hist
    (int64 [n,k,2,T]) of p̄ (spff_prob_finalize). With `unc` (an Uncertainty) also its maps, sums and calibration
    histogram (spff_prob_finalize_unc); every other output is the same, bit for bit.

    `inv_temperature` β = 1/T != 1.0 tempers the pooled distribution, p̃_c ∝ p̄_c^β, and p̃ replaces p̄ in every output
    but the arg-max and the mutual information (spff_prob_finalize_tempered). β == 1.0 makes exactly the untempered
    call."""
    assert acc.dtype == torch.float32 and acc.dim() == 5 and acc.shape[-1] == 16 and acc.is_contiguous()
    n, d, h, w, _ = acc.shape
    vox = n * d * h * w
    s = Shape(n, d, h, w)
    lb = 0
    if labels is not None:
        assert labels.is_contiguous() and labels.numel() == vox
        lb = _label_bytes(labels)
    nll, cnt, conf = tally if tally is not None else (None, None, None)
    per = per_sample if per_sample is not None else (None, None, None)
    if per_sample is not None:
        assert per[0].dtype == torch.float64 and per[0].numel() == n
        assert per[1].dtype == torch.int64 and per[1].numel() == n
        assert per[2].dtype == torch.int64 and per[2].is_contiguous() and per[2].numel() == n * k * k
    if conf is not None:
        assert conf.dtype == torch.int64 and conf.is_contiguous() and conf.numel() == k * k
    bins = 0
    if hist is not None:
        bins = hist.shape[-1]
        assert hist.dtype == torch.int64 and hist.is_contiguous() and tuple(hist.shape) == (k, 2, bins)
        if sample_hist is not None:
            assert sample_hist.dtype == torch.int64 and sample_hist.is_contiguous()
            assert tuple(sample_hist.shape) == (n, k, 2, bins)
    if labels_out is not None:
        assert labels_out.dtype == torch.uint8 and labels_out.is_contiguous() and labels_out.numel() == vox
    if proba_out is not None:
        assert proba_out.dtype == torch.float16 and proba_out.is_contiguous() and tuple(proba_out.shape) == (n, k, d, h, w)
    beta = float(inv_temperature)
    if beta != 1.0:
        if not (math.isfinite(beta) and beta > 0.0):
            raise ValueError(f"inv_temperature must be positive and finite, got {inv_temperature}")
        u = _unc_struct(unc, n, vox) if unc is not None else None
        call("spff_prob_finalize_tempered", ptr(acc), int(k), s, float(scale), ptr(labels), lb, int(ignore_index),
             ptr(nll), ptr(cnt), ptr(conf), *(ptr(t) for t in per), ptr(labels_out), int(bins), ptr(hist),
             ptr(sample_hist), ptr(proba_out), ctypes.byref(u) if u is not None else None, beta, stream_ptr())
        return
    if unc is None:
        call("spff_prob_finalize", ptr(acc), int(k), s, float(scale), ptr(labels), lb, int(ignore_index), ptr(nll),
             ptr(cnt), ptr(conf), *(ptr(t) for t in per), ptr(labels_out), int(bins), ptr(hist), ptr(sample_hist),
             ptr(proba_out), stream_ptr())
        return
    u = _unc_struct(unc, n, vox)
    call("spff_prob_finalize_unc", ptr(acc), int(k), s, float(scale), ptr(labels), lb, int(ignore_index), ptr(nll),
         ptr(cnt), ptr(conf), *(ptr(t) for t in per), ptr(labels_out), int(bins), ptr(hist), ptr(sample_hist),
         ptr(proba_out), ctypes.byref(u), stream_ptr())


def prob_temp_fit(acc, k: int, scale: float, labels, betas, sums, ignore_index: int = 255, *, counted):
    """Temperature-fit statistics on a spff_head_prob_accum accumulator acc (fp32 [n,d,h,w,16], p̄ = scale * acc): for
    every voxel whose label (uint8 / int64 [n,d,h,w]) is in [0,k) and not ignore_index, and every β_g of `betas` (fp32
    [G] on the device, G in [1, 64], each positive and finite: the caller's duty, the values are not read back), sums
    (fp64 [2,G], +=) receives the tempered nll f(β_g) = log sum_c p̄_c^β - β log p̄_y in [0] and its derivative
    f'(β_g) = sum_c p̃_c log p̄_c - log p̄_y in [1]; counted (int64 [1], +=) the voxels (spff_prob_temp_fit).
    Bit-reproducible: per-block fp64 partials added in a fixed order."""
    assert acc.dtype == torch.float32 and acc.dim() == 5 and acc.shape[-1] == 16 and acc.is_contiguous()
    n, d, h, w, _ = acc.shape
    s = Shape(n, d, h, w)
    assert labels.is_contiguous() and labels.numel() == n * d * h * w
    g = betas.numel()
    assert betas.dtype == torch.float32 and betas.is_contiguous()
    assert sums.dtype == torch.float64 and sums.is_contiguous() and tuple(sums.shape) == (2, g)
    assert counted.dtype == torch.int64 and counted.numel() == 1
    ws = workspace(int(_lib.lib.spff_prob_temp_fit_workspace(int(k), s, g)), acc.device)
    call("spff_prob_temp_fit", ptr(acc), int(k), s, float(scale), ptr(labels), _label_bytes(labels), int(ignore_index),
         ptr(betas), g, ptr(sums), ptr(counted), ptr(ws), ws.numel(), stream_ptr())


def scale_by_count(g, count, factor: float = 1.0):
    """g (fp32, contiguous) *= factor / count[0]  (0 when the count is 0)."""
    assert g.dtype == torch.float32 and g.is_contiguous() and count.dtype == torch.int64
    call("spff_scale_by_count", ptr(g), g.numel(), ptr(count), float(factor), stream_ptr())


def count_valid(labels, ignore_index, out):
    """out (int64 [1]) = number of labels != ignore_index."""
    call("spff_count_valid", ptr(labels), _label_bytes(labels), labels.numel(), int(ignore_index), ptr(out), stream_ptr())


def loss_from_tally(nll, count, confusion, k, smooth, out):
    call("spff_loss_from_tally", ptr(nll), ptr(count), ptr(confusion), int(k), float(smooth), ptr(out), stream_ptr())


def partial_colsum(m, rows, row_stride, cols, out):
    """out[:cols] += column sums of the [rows, row_stride] fp32 matrix m (first `cols` columns)."""
    ws = workspace(int(_lib.lib.spff_partial_colsum_workspace(int(cols))), m.device)
    call("spff_partial_colsum", ptr(m), int(rows), int(row_stride), int(cols), ptr(out), ptr(ws), ws.numel(), stream_ptr())


def adam_step(p, g, m, v, lr, beta1, beta2, eps, step, grad_scale=1.0):
    call("spff_adam_step", ptr(p), ptr(g), ptr(m), ptr(v), p.numel(), float(lr), float(beta1), float(beta2), float(eps),
         int(step), float(grad_scale), stream_ptr())


# ------------------------------------------------------------------------------------------------
# "3DUNet" control (Cicek3DUNet): (2,2,2) transposed conv / pool, BatchNorm, depth resampling, SGD
# ------------------------------------------------------------------------------------------------
def pack_convt_weight_k222(w):
    """nn.ConvTranspose3d weight [Cin,Cout,2,2,2] fp32 -> (w_fwd, w_dgrad) bf16."""
    cin, cout = w.shape[0], w.shape[1]
    w = w.detach().contiguous().float()
    wf = torch.empty(8 * cin * cout, dtype=torch.bfloat16, device=w.device)
    wd = torch.empty(8 * cin * cout, dtype=torch.bfloat16, device=w.device)
    call("spff_pack_convt_weight_k222", ptr(w), ptr(wf), ptr(wd), cin, cout, stream_ptr())
    return wf, wd


def convt_k222_fwd(x, cin, w_fwd, bias, y, cout):
    s, ldx = _view(x, cin)
    s2, ldy = _view(y, cout)
    assert (s2.d, s2.h, s2.w) == (2 * s.d, 2 * s.h, 2 * s.w)
    call("spff_convt_k222_fwd", ptr(x), ldx, cin, ptr(w_fwd), ptr(bias), ptr(y), ldy, cout, s, stream_ptr())


def convt_k222_dgrad(dy, cout, w_dgrad, dx, cin):
    s, lddx = _view(dx, cin)
    s2, lddy = _view(dy, cout)
    assert (s2.d, s2.h, s2.w) == (2 * s.d, 2 * s.h, 2 * s.w)
    call("spff_convt_k222_dgrad", ptr(dy), lddy, cout, ptr(w_dgrad), ptr(dx), lddx, cin, s, stream_ptr())


def convt_k222_wgrad(x, cin, dy, cout, dw, beta=0.0):
    s, ldx = _view(x, cin)
    _, lddy = _view(dy, cout)
    assert dw.dtype == torch.float32 and dw.is_contiguous() and tuple(dw.shape) == (cin, cout, 2, 2, 2)
    ws = workspace(int(_lib.lib.spff_convt_k222_wgrad_workspace(cin, cout, s)), x.device)
    call("spff_convt_k222_wgrad", ptr(x), ldx, cin, ptr(dy), lddy, cout, s, ptr(dw), float(beta), ptr(ws), ws.numel(),
         stream_ptr())


def depth_resample(x, y, matrix):
    """y[n, do, ...] = sum_di matrix[do, di] * x[n, di, ...] for contiguous x [n, din, *inner], y [n, dout, *inner]
    (bf16 or fp32); matrix: CUDA fp32 [dout, din]."""
    assert x.is_contiguous() and y.is_contiguous() and x.dtype == y.dtype and x.dtype in (torch.bfloat16, torch.float32)
    n, din = x.shape[0], x.shape[1]
    dout = y.shape[1]
    inner = x[0, 0].numel()
    assert y.shape[0] == n and y[0, 0].numel() == inner and tuple(matrix.shape) == (dout, din)
    assert matrix.dtype == torch.float32 and matrix.is_contiguous() and matrix.is_cuda
    call("spff_depth_resample", ptr(x), ptr(y), x.element_size(), n, din, dout, inner, ptr(matrix), stream_ptr())


def bn_coeffs(gamma, beta, eps, n, c, count, coef, partial=None, slots=0, stats=None, momentum=0.1, running_mean=None,
              running_var=None, eval_mode=False):
    ws = workspace(int(_lib.lib.spff_bn_coeffs_workspace(c)), coef.device)
    call("spff_bn_coeffs", ptr(partial), int(slots), ptr(stats), ptr(gamma), ptr(beta), float(eps), n, c, int(count),
         float(momentum), ptr(running_mean), ptr(running_var), int(eval_mode), ptr(coef), ptr(ws), ws.numel(), stream_ptr())


def bn_bwd_coeffs(R, coef, gamma, c, shape, bcoef, dgamma, dbeta):
    call("spff_bn_bwd_coeffs", ptr(R), ptr(coef), ptr(gamma), c, shape, ptr(bcoef), ptr(dgamma), ptr(dbeta), stream_ptr())


def maxpool222_fwd(y, ypool, c):
    s, ldy = _view(y, c)
    s2, ldp = _view(ypool, c)
    assert (s2.d, s2.h, s2.w) == (s.d // 2, s.h // 2, s.w // 2)
    call("spff_maxpool222_fwd", ptr(y), ldy, ptr(ypool), ldp, c, s, stream_ptr())


def maxpool222_bwd_add(dpool, y, dskip, c, accumulate):
    s, ldy = _view(y, c)
    _, ldp = _view(dpool, c)
    _, ldd = _view(dskip, c)
    call("spff_maxpool222_bwd_add", ptr(dpool), ldp, ptr(y), ldy, ptr(dskip), ldd, c, s, int(accumulate), stream_ptr())


def sgd_step(p, g, buf, lr, momentum, weight_decay, nesterov, first_step, grad_scale=1.0):
    call("spff_sgd_step", ptr(p), ptr(g), ptr(buf), p.numel(), float(lr), float(momentum), float(weight_decay),
         int(bool(nesterov)), int(bool(first_step)), float(grad_scale), stream_ptr())


# ------------------------------------------------------------------------------------------------
# data path (SURVEY.md §8f-4)
# ------------------------------------------------------------------------------------------------
def roi_labels(rois, frames, height, width, device) -> torch.Tensor:
    """int64 [frames, height, width] label map of elliptical rois [(x0, y0, w0, h0, label), ...] (last one wins)."""
    import ctypes
    flat = [int(v) for r in rois for v in r]
    arr = (ctypes.c_int * max(1, len(flat)))(*flat)
    out = torch.empty(frames, height, width, dtype=torch.int64, device=device)
    with torch.cuda.device(out.device):
        call("spff_roi_labels", arr, len(rois), frames, height, width, ptr(out), stream_ptr())
    return out


def grid_aug(x, y, xo, yo, amap, bmap, transposed, scale, shift, noise_cap, seed, stamp, any_noise, any_stamp):
    """x fp32 [n,F,H,W] -> xo; y uint8/int64 [n,F,H,W] or None -> yo; the per-sample tables are CUDA tensors."""
    n, f, h, w = x.shape
    assert x.dtype == torch.float32 and x.is_contiguous() and xo.is_contiguous() and xo.shape == x.shape
    lb = 0
    if y is not None:
        assert y.is_contiguous() and yo.is_contiguous() and tuple(y.shape) == (n, f, h, w) and y.dtype == yo.dtype
        lb = _label_bytes(y)
    assert amap.dtype == torch.int32 and bmap.dtype == torch.int32 and tuple(amap.shape) == (n, h) and tuple(bmap.shape) == (n, w)
    ws = workspace(int(_lib.lib.spff_grid_aug_workspace(n)), x.device)
    call("spff_grid_aug", ptr(x), ptr(y), lb, ptr(xo), ptr(yo), n, f, h, w, ptr(amap), ptr(bmap), ptr(transposed), ptr(scale),
         ptr(shift), ptr(noise_cap), ptr(seed), ptr(stamp), int(any_noise), int(any_stamp), ptr(ws), ws.numel(), stream_ptr())
