"""ctypes binding of libspff_b200.so (C ABI: include/spff_b200.h).

The library is the product: there is no Python/PyTorch fallback behind these calls. Loading fails
loudly when the shared object is missing, and every compute entry point returns
SPFF_ERR_UNSUPPORTED_ARCH (raised here as RuntimeError) on anything that is not an sm_100 GPU.
"""
from __future__ import annotations

import ctypes
import os
import threading
from ctypes import POINTER, Structure, c_char_p, c_double, c_float, c_int, c_longlong, c_size_t, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libspff_b200.so")


class Shape(Structure):
    """spff_shape: samples, energy bins (depth), height, width."""

    _fields_ = [("n", c_int), ("d", c_int), ("h", c_int), ("w", c_int)]


class UncOut(Structure):
    """spff_unc_out: the uncertainty / calibration outputs of spff_prob_finalize_unc (device pointers, NULL = not
    wanted)."""

    _fields_ = [("ent", c_void_p), ("entropy_out", c_void_p), ("mi_out", c_void_p), ("unc", c_void_p),
                ("sample_unc", c_void_p), ("cal_bins", c_int), ("calib", c_void_p), ("sample_calib", c_void_p),
                ("brier", c_void_p), ("sample_brier", c_void_p)]


def _load() -> ctypes.CDLL:
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C spff-unet-spcct_b200/csrc`). spff_b200 has no fallback path."
        )
    return ctypes.CDLL(LIB_PATH)


lib = _load()
lib.spff_last_error.restype = c_char_p
lib.spff_version.restype = c_int

_P = c_void_p
_LL = c_longlong

# name -> argtypes, exactly the prototypes of include/spff_b200.h (restype int unless noted)
_PROTOTYPES = {
    "spff_device_check": [],
    "spff_debug_set": [c_int, _LL],
    "spff_conv3_packed_elems": [c_int, c_int],
    "spff_pack_conv3_weight": [_P, _P, _P, c_int, c_int, _P],
    "spff_conv3d_k3_fwd": [_P, _LL, c_int, _P, _P, _LL, c_int, Shape, _P],
    "spff_conv3d_k3_stat_slots": [Shape],
    "spff_conv3d_k3_fwd_stats": [_P, _LL, c_int, _P, _P, _LL, c_int, Shape, _P, _P],
    "spff_conv3d_k3_dgrad": [_P, _LL, c_int, _P, _P, _LL, c_int, Shape, _P],
    "spff_conv3d_k3_dgrad_stats": [_P, _LL, c_int, _P, _P, _LL, c_int, Shape, _P, _P],
    "spff_conv3d_k3_wgrad_workspace": [c_int, c_int, Shape],
    "spff_conv3d_k3_wgrad": [_P, _LL, c_int, _P, _LL, c_int, Shape, _P, c_float, _P, c_size_t, _P],
    "spff_conv3d_stem_fwd": [_P, _P, _P, _LL, c_int, Shape, _P],
    "spff_conv3d_stem_stat_slots": [Shape],
    "spff_conv3d_stem_fwd_stats": [_P, _P, _P, _LL, c_int, Shape, _P, _P],
    "spff_conv3d_stem_wgrad_workspace": [c_int],
    "spff_conv3d_stem_wgrad": [_P, _P, _LL, c_int, Shape, _P, c_float, _P, c_size_t, _P],
    "spff_pack_convt_weight": [_P, _P, _P, c_int, c_int, _P],
    "spff_convt_k122_fwd": [_P, _LL, c_int, _P, _P, _P, _LL, c_int, Shape, _P],
    "spff_convt_k122_dgrad": [_P, _LL, c_int, _P, _P, _LL, c_int, Shape, _P],
    "spff_convt_k122_wgrad_workspace": [c_int, c_int, Shape],
    "spff_convt_k122_wgrad": [_P, _LL, c_int, _P, _LL, c_int, Shape, _P, c_float, _P, c_size_t, _P],
    "spff_in_stats": [_P, _LL, c_int, Shape, _P, _P],
    "spff_in_coeffs": [_P, _P, _P, c_float, c_int, c_int, _LL, c_int, _P, _P],
    "spff_in_coeffs_from_partials": [_P, c_int, _P, _P, c_float, c_int, c_int, _LL, _P, _P],
    "spff_norm_act_apply": [_P, _LL, _P, _P, _LL, c_int, Shape, c_float, _P],
    "spff_norm_act_reduce_workspace": [c_int, Shape],
    "spff_norm_act_reduce": [_P, _LL, _P, _P, c_int, Shape, c_float, _P, c_size_t, _P],
    "spff_norm_act_affine_apply": [_P, _LL, _P, _P, _P, _P, _LL, _P, _LL, _P, c_int, Shape, c_float, _P],
    "spff_gate_tables_fwd": [_P] * 6 + [c_int, c_int] + [_P] * 3 + [_P],
    "spff_gate_tables_bwd": [_P] * 6 + [c_int, c_int] + [_P] * 9 + [_P],
    "spff_gate_micro_fwd": [_P] * 8 + [c_int, c_int, c_int, Shape, _P, _P, _P],
    "spff_norm_act_bwd_reduce_workspace": [c_int, Shape, c_int],
    "spff_norm_act_bwd_reduce": [_P, _LL, _P, _LL, _P, _P, _P, c_int, Shape, c_float, c_int, _P, c_size_t, _P],
    "spff_gate_micro_bwd": [_P] * 11 + [c_int, c_int, c_int, Shape] + [_P] * 12 + [_P],
    "spff_norm_act_bwd_apply": [_P, _LL, _P, _LL, _P, _P, _P, _P, _P, _LL, c_int, Shape, c_float, _P],
    "spff_maxpool_bwd_add": [_P, _LL, _P, _LL, _P, _LL, c_int, Shape, c_int, _P],
    "spff_maxpool_bwd_add_argmax": [_P, _LL, _P, _P, _LL, c_int, Shape, c_int, _P],
    "spff_head_fwd": [_P, _LL, c_int, _P, _P, _P, c_int, Shape, _P],
    "spff_head_argmax": [_P, _LL, c_int, _P, _P, _P, c_int, Shape, _P],
    "spff_head_bwd_workspace": [c_int],
    "spff_head_bwd": [_P, _P, _LL, c_int, _P, _P, _LL, _P, _P, c_float, c_int, Shape, _P, c_size_t, _P],
    "spff_ce_confusion": [_P, _P, c_int, c_int, c_int, Shape, _P, _P, _P, _P],
    "spff_ce_grad": [_P, _P, c_int, c_int, c_int, Shape, _P, _P, _P, _P],
    "spff_head_loss_workspace": [c_int],
    "spff_head_loss_fused": [_P, _LL, c_int, _P, _P, _P, c_int, c_int, c_int, Shape, _P, _P, _P, _P, _P, _P, _LL, _P, _P,
                             c_float, _P, c_size_t, _P],
    "spff_head_eval": [_P, _LL, c_int, _P, _P, _P, c_int, c_int, c_int, Shape, _P, _P, _P, _P, _P, _P, _P, _P],
    "spff_head_eval_hist": [_P, _LL, c_int, _P, _P, _P, c_int, c_int, c_int, Shape, _P, _P, _P, _P, _P, _P, _P, c_int, _P,
                            _P, _P],
    "spff_head_prob_accum": [_P, _LL, c_int, _P, _P, c_int, Shape, c_int, c_int, _P, _P],
    "spff_prob_finalize": [_P, c_int, Shape, c_float, _P, c_int, c_int, _P, _P, _P, _P, _P, _P, _P, c_int, _P, _P, _P, _P],
    "spff_head_prob_accum_ent": [_P, _LL, c_int, _P, _P, c_int, Shape, c_int, c_int, _P, _P, _P],
    "spff_prob_finalize_unc": [_P, c_int, Shape, c_float, _P, c_int, c_int, _P, _P, _P, _P, _P, _P, _P, c_int, _P, _P, _P,
                               POINTER(UncOut), _P],
    "spff_prob_finalize_tempered": [_P, c_int, Shape, c_float, _P, c_int, c_int, _P, _P, _P, _P, _P, _P, _P, c_int, _P, _P,
                                    _P, POINTER(UncOut), c_float, _P],
    "spff_prob_temp_fit_workspace": [c_int, Shape, c_int],
    "spff_prob_temp_fit": [_P, c_int, Shape, c_float, _P, c_int, c_int, _P, c_int, _P, _P, _P, c_size_t, _P],
    "spff_count_valid": [_P, c_int, _LL, c_int, _P, _P],
    "spff_scale_by_count": [_P, _LL, _P, c_float, _P],
    "spff_loss_from_tally": [_P, _P, _P, c_int, c_double, _P, _P],
    "spff_partial_colsum_workspace": [c_int],
    "spff_partial_colsum": [_P, _LL, _LL, c_int, _P, _P, c_size_t, _P],
    "spff_adam_step": [_P, _P, _P, _P, _LL, c_float, c_float, c_float, c_float, c_int, c_float, _P],
    "spff_pack_convt_weight_k222": [_P, _P, _P, c_int, c_int, _P],
    "spff_convt_k222_fwd": [_P, _LL, c_int, _P, _P, _P, _LL, c_int, Shape, _P],
    "spff_convt_k222_dgrad": [_P, _LL, c_int, _P, _P, _LL, c_int, Shape, _P],
    "spff_convt_k222_wgrad_workspace": [c_int, c_int, Shape],
    "spff_convt_k222_wgrad": [_P, _LL, c_int, _P, _LL, c_int, Shape, _P, c_float, _P, c_size_t, _P],
    "spff_depth_resample": [_P, _P, c_int, c_int, c_int, c_int, _LL, _P, _P],
    "spff_bn_coeffs_workspace": [c_int],
    "spff_bn_coeffs": [_P, c_int, _P, _P, _P, c_float, c_int, c_int, _LL, c_float, _P, _P, c_int, _P, _P, c_size_t, _P],
    "spff_bn_bwd_coeffs": [_P, _P, _P, c_int, Shape, _P, _P, _P, _P],
    "spff_maxpool222_fwd": [_P, _LL, _P, _LL, c_int, Shape, _P],
    "spff_maxpool222_bwd_add": [_P, _LL, _P, _LL, _P, _LL, c_int, Shape, c_int, _P],
    "spff_sgd_step": [_P, _P, _P, _LL, c_float, c_float, c_float, c_int, c_int, c_float, _P],
    "spff_roi_labels": [_P, c_int, c_int, c_int, c_int, _P, _P],
    "spff_grid_aug_workspace": [c_int],
    "spff_grid_aug": [_P, _P, c_int, _P, _P, c_int, c_int, c_int, c_int, _P, _P, _P, _P, _P, _P, _P, _P, c_int, c_int, _P,
                      c_size_t, _P],
}

_SIZE_T_FUNCS = {"spff_conv3d_k3_wgrad_workspace", "spff_conv3d_stem_wgrad_workspace",
                 "spff_convt_k122_wgrad_workspace", "spff_head_bwd_workspace", "spff_head_loss_workspace",
                 "spff_norm_act_reduce_workspace", "spff_norm_act_bwd_reduce_workspace",
                 "spff_convt_k222_wgrad_workspace", "spff_bn_coeffs_workspace", "spff_grid_aug_workspace",
                 "spff_partial_colsum_workspace", "spff_prob_temp_fit_workspace"}


def _declare():
    for name, argtypes in _PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = c_size_t if name in _SIZE_T_FUNCS else (c_longlong if name == "spff_conv3_packed_elems" else c_int)


_declare()


def exported_symbols():
    """Names this binding expects the shared object to export (checked by the CPU tests)."""
    return ["spff_version", "spff_last_error"] + list(_PROTOTYPES)


def check(code: int, what: str = "") -> None:
    if code != 0:
        msg = lib.spff_last_error()
        raise RuntimeError(f"libspff_b200 {what} failed ({code}): {msg.decode() if msg else ''}")


# C-ABI compute calls made by this process (each enqueues one or two kernels); bench.py reports the
# number issued inside its timed region as `gpu_launches`.
CALLS = 0


class Profile:
    """Optional per-call device timing (CUDA events on the launching stream around each C-ABI call
    whose name passes `select`). `note` carries the algorithmic work of the next call (FLOPs or
    bytes), set by the ops wrappers. Used by bench.py for the roofline line; off by default."""

    def __init__(self, select=None):
        self.select = select
        self.records = []   # (name, work, start_event, end_event)

    def summary(self):
        """name -> (launches, total ms, total work); synchronises."""
        import torch

        torch.cuda.synchronize()
        out = {}
        for name, work, e0, e1 in self.records:
            n, ms, w = out.get(name, (0, 0.0, 0.0))
            out[name] = (n + 1, ms + e0.elapsed_time(e1), w + (work or 0.0))
        return out


PROFILE = None   # set to a Profile() to time calls
NOTE = None      # algorithmic work of the next call


# Device of the tensor arguments of the call being assembled (per thread): `ptr()` records it, `stream_ptr()` hands out THAT device's
# current stream, `call()` makes it the current CUDA device around the C call (kernel launches and TMA descriptors are
# issued against the current device) and forgets it. Tensors of two devices in one call are an error.
_TLS = threading.local()     # forward runs on the main thread, backward on autograd's worker thread


def _enter_device():
    """(device index or None, previous device index or None) for the call being issued."""
    dev = getattr(_TLS, "dev", None)
    _TLS.dev = None
    if dev is None:
        return None
    import torch

    cur = torch.cuda.current_device()
    if cur == dev:
        return None
    torch.cuda.set_device(dev)
    return cur


def call(name: str, *args) -> None:
    global CALLS, NOTE
    CALLS += 1
    prev = _enter_device()
    try:
        _call(name, *args)
    finally:
        if prev is not None:
            import torch

            torch.cuda.set_device(prev)


def _call(name: str, *args) -> None:
    global NOTE
    prof = PROFILE
    if prof is not None and (prof.select is None or prof.select(name)):
        import torch

        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        rc = getattr(lib, name)(*args)
        e1.record()
        prof.records.append((name, NOTE, e0, e1))
        NOTE = None
        check(rc, name)
        return
    NOTE = None
    check(getattr(lib, name)(*args), name)


def ptr(t) -> c_void_p:
    """Device pointer of a torch tensor (or None). Records the tensor's device for the call being assembled."""
    if t is None:
        return c_void_p(0)
    d = t.device
    if d.type == "cuda":
        seen = getattr(_TLS, "dev", None)
        if seen is None:
            _TLS.dev = d.index
        elif seen != d.index:
            _TLS.dev = None
            raise RuntimeError(f"libspff_b200: tensors of one call live on different devices (cuda:{seen} and cuda:{d.index})")
    return c_void_p(t.data_ptr())


def stream_ptr() -> c_void_p:
    """Current stream of the device the call's tensors live on (not of whatever device happens to be current)."""
    import torch

    return c_void_p(torch.cuda.current_stream(getattr(_TLS, "dev", None)).cuda_stream)
