"""GPU: temperature scaling of ensembles and mirror test-time augmentation. The fit kernel (spff_prob_temp_fit) and the
tempered finishing pass (spff_prob_finalize_tempered) on given accumulators against fp64 torch; every argument error;
then SpctEnsemble on the weights the reference trained: T = 1 is the untempered path bit for bit, the fitted temperature
against scipy's minimiser of the fp64 nll of the unfused pooled softmax, the softmax(z / T) identity, host batches,
native 512 x 512 slices, memory and two ranks.

Tolerances. The fit sums are fp64 sums of per-voxel terms evaluated in fp32 with accurate logf / expf / log1pf; their
error is measured against the sum of the terms' magnitudes (the derivative sums cancel near the minimum). The tempered
p̃ is formed in fp32 from log p̄ (relative error about 1e-5 for the smallest probabilities at β = 8); fp16 outputs are
compared to half an fp16 ulp plus that. Histogram and calibration counts are exact outside voxels within DELTA = 3e-5 of
a bin edge."""
import math
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu

DELTA = 3e-5
FIX = 2.0 ** -24
FLT_MIN = float(np.finfo(np.float32).tiny)
NEG_LOG_FLT_MIN = float(-np.log(np.float32(FLT_MIN)))   # the fp32 constant the kernels add
FLIPS = {0: [], 1: [3], 2: [4], 3: [3, 4]}      # flip code -> dims of a [B,C,F,H,W] tensor


def entropy(p, dim=1):
    return -(p * torch.where(p > 0, p.log(), torch.zeros_like(p))).sum(dim)


def fp16_tol(ref, extra):
    return ref.abs() * 2.0 ** -11 + 2.0 ** -25 + extra


def tally_bufs(k, dev="cuda"):
    return (torch.zeros(1, dtype=torch.float64, device=dev), torch.zeros(1, dtype=torch.int64, device=dev),
            torch.zeros(k, k, dtype=torch.int64, device=dev))


def sample_bufs(n, k, dev="cuda"):
    return (torch.zeros(n, dtype=torch.float64, device=dev), torch.zeros(n, dtype=torch.int64, device=dev),
            torch.zeros(n, k, k, dtype=torch.int64, device=dev))


def tempered(pbar, beta):
    """fp64 p̃ = p̄^β / sum p̄^β over dim 1 (p̄ = 0 stays 0; an all-zero row stays 0)."""
    pb = pbar.double()
    lg = torch.where(pb > 0, pb.log(), torch.full_like(pb, -math.inf))
    m = lg.amax(1, keepdim=True)
    e = torch.where(pb > 0, torch.exp(beta * (lg - torch.where(torch.isfinite(m), m, torch.zeros_like(m)))),
                    torch.zeros_like(pb))
    s = e.sum(1, keepdim=True)
    return torch.where(s > 0, e / s.clamp(min=1e-300), torch.zeros_like(e))


def fit_terms(pbar, lab, k, beta, ignore_index=255):
    """Per counted voxel (fp64): f(β) = log sum_{p̄_c > 0} p̄_c^β - β log p̄_y and f'(β) = sum_c p̃_c log p̄_c -
    log p̄_y; -log FLT_MIN and 0 when p̄_y = 0. pbar [B,K,...], lab [B,...]."""
    counted = (lab != ignore_index) & (lab >= 0) & (lab < k)
    pb = pbar.double().movedim(1, -1)[counted]                 # [n,K]
    y = lab[counted].long()
    pos = pb > 0
    lg = torch.where(pos, pb.log(), torch.zeros_like(pb))
    py = pb.gather(1, y[:, None])[:, 0]
    ly = lg.gather(1, y[:, None])[:, 0]
    z = torch.where(pos, beta * lg, torch.full_like(pb, -math.inf))
    lse = torch.logsumexp(z, 1)
    pt = torch.where(pos, torch.exp(z - lse[:, None]), torch.zeros_like(pb))
    zero = py == 0
    f = torch.where(zero, torch.full_like(py, NEG_LOG_FLT_MIN), lse - beta * ly)
    d = torch.where(zero, torch.zeros_like(py), (pt * lg).sum(1) - ly)
    return f, d


def make_acc(n, d, h, w, k, seed, dtype):
    """An accumulator of 3 passes on a coarse grid (ties, zeros, a few all-zero rows) or a fine one, classes >= k set
    to 100 (must be ignored), and labels with ignored voxels, labels >= k and, for int64, negative labels."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    acc = torch.full((n, d, h, w, 16), 100.0, device="cuda")
    raw = torch.randint(0, 7, (n, d, h, w, k), device="cuda", generator=g).float() * 0.125
    fine = torch.rand(n, d, h, w, k, device="cuda", generator=g) ** 4 * 3
    acc[..., :k] = torch.where(torch.rand(n, d, h, w, 1, device="cuda", generator=g) < 0.5, raw, fine)
    lab = torch.randint(0, k, (n, d, h, w), device="cuda", generator=g)
    lab[torch.rand(n, d, h, w, device="cuda", generator=g) < 0.1] = 255          # ignored
    lab[torch.rand(n, d, h, w, device="cuda", generator=g) < 0.03] = 200         # not a class
    if dtype == torch.int64:
        lab[torch.rand(n, d, h, w, device="cuda", generator=g) < 0.02] = -3      # negative: not a class
    return acc, lab.to(dtype)


SHAPES = [(1, 5, 7, 9), (3, 5, 17, 31)]          # neither fills the blocks of the launch


# --------------------------------------------------------------------------------------------------------------------
# kernels
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.uint8, torch.int64])
@pytest.mark.parametrize("k", [2, 5, 13, 16])
@pytest.mark.parametrize("shape", SHAPES)
def test_prob_temp_fit(dtype, k, shape):
    """Each of the 2G sums within 1e-6 of the sum of the terms' magnitudes (plus 1e-9 per voxel) of the fp64 torch
    computation on the kernel's fp32 p̄; the count exact; two calls bit-identical; += accumulates."""
    from innovative3D.helpers import temperature_grid
    from spff_b200 import ops
    n, d, h, w = shape
    acc, lab = make_acc(n, d, h, w, k, seed=k * 31 + h, dtype=dtype)
    scale = 1.0 / 3.0
    pbar = (acc[..., :k] * scale).permute(0, 4, 1, 2, 3).contiguous()     # fp32, the kernel's p̄
    for g_ in (1, 33, 64):
        b_h = temperature_grid(8.0, 33) if g_ == 33 else np.geomspace(0.125, 8.0, g_).astype(np.float32).astype(float)
        betas = torch.tensor(b_h, dtype=torch.float32, device="cuda")
        sums = torch.zeros(2, g_, dtype=torch.float64, device="cuda")
        cnt = torch.zeros(1, dtype=torch.int64, device="cuda")
        ops.prob_temp_fit(acc, k, scale, lab, betas, sums, counted=cnt)
        sums2 = torch.zeros_like(sums)
        cnt2 = torch.zeros_like(cnt)
        ops.prob_temp_fit(acc, k, scale, lab, betas, sums2, counted=cnt2)
        assert torch.equal(sums, sums2) and torch.equal(cnt, cnt2)         # bit-reproducible
        ll = lab.long()
        counted = int(((ll != 255) & (ll >= 0) & (ll < k)).sum())
        assert int(cnt) == counted
        worst = 0.0
        for i, b in enumerate(b_h):
            f, dv = fit_terms(pbar, ll, k, float(b))
            for r, ref in ((0, f), (1, dv)):
                tol = 1e-6 * float(ref.abs().sum()) + 1e-9 * counted
                err = abs(float(sums[r, i]) - float(ref.sum()))
                worst = max(worst, err / tol)
                assert err <= tol, (g_, i, r, float(sums[r, i]), float(ref.sum()))
        print(f"k={k} {tuple(shape)} G={g_}: worst error / tolerance {worst:.3f}")
        ops.prob_temp_fit(acc, k, scale, lab, betas, sums2, counted=cnt2)  # +=
        assert torch.equal(sums2, sums * 2) and int(cnt2) == 2 * counted


@pytest.mark.parametrize("dtype", [torch.uint8, torch.int64])
@pytest.mark.parametrize("k,t,tc,beta", [(13, 256, 960, 0.37), (5, 16, 15, 2.5), (16, 1024, 1024, 8.0), (2, 0, 64, 0.125)])
@pytest.mark.parametrize("shape", SHAPES)
def test_prob_finalize_tempered(dtype, k, t, tc, beta, shape):
    """Against fp64 torch p̃: proba_out within fp16 rounding, nll within 1e-5, H[p̃] map, histogram and calibration
    counts exact outside the DELTA band, Brier; labels_out and the confusion bit-identical to spff_prob_finalize; the
    mutual information bit-identical to the untempered call."""
    from spff_b200 import ops
    n, d, h, w = shape
    acc, lab = make_acc(n, d, h, w, k, seed=k * 13 + t + h, dtype=dtype)
    scale = 1.0 / 3.0
    pbar = (acc[..., :k] * scale).permute(0, 4, 1, 2, 3).contiguous()
    pt = tempered(pbar, float(np.float32(beta)))                          # [n,k,d,h,w] fp64
    hb = entropy(pbar.double())
    g = torch.Generator(device="cuda").manual_seed(5)
    ent = (3 * hb * (0.5 + 0.5 * torch.rand(n, d, h, w, device="cuda", generator=g, dtype=torch.float64))).float()
    ll = lab.long()
    counted = (ll != 255) & (ll >= 0) & (ll < k)
    arg = acc[..., :k].argmax(-1)

    def run(inv_t):
        tl, per = tally_bufs(k), sample_bufs(n, k)
        out = torch.full((n, d, h, w), 77, dtype=torch.uint8, device="cuda")
        proba = torch.empty(n, k, d, h, w, dtype=torch.float16, device="cuda")
        hist = torch.zeros(k, 2, t, dtype=torch.int64, device="cuda") if t else None
        s_hist = torch.zeros(n, k, 2, t, dtype=torch.int64, device="cuda") if t else None
        z = lambda *s, dt=torch.int64: torch.zeros(*s, dtype=dt, device="cuda")   # noqa: E731
        u = ops.Uncertainty(ent=ent, entropy_out=torch.empty(n, d, h, w, dtype=torch.float16, device="cuda"),
                            mi_out=torch.empty(n, d, h, w, dtype=torch.float16, device="cuda"), unc=z(2),
                            sample_unc=z(n, 2), calib=z(3, tc), brier=z(1, dt=torch.float64), sample_calib=z(n, 3, tc),
                            sample_brier=z(n, dt=torch.float64))
        ops.prob_finalize(acc, k, scale, labels=lab, tally=tl, per_sample=per, labels_out=out, hist=hist,
                          sample_hist=s_hist, proba_out=proba, unc=u, inv_temperature=inv_t)
        return tl, per, out, proba, hist, s_hist, u

    base = run(1.0)
    got = run(beta)
    # the arg-max and the mutual information: bit for bit
    assert torch.equal(got[2], base[2]) and torch.equal(got[0][2], base[0][2]) and torch.equal(got[0][1], base[0][1])
    assert torch.equal(got[1][2], base[1][2])
    assert torch.equal(got[6].mi_out, base[6].mi_out)
    assert torch.equal(got[6].unc[1], base[6].unc[1]) and torch.equal(got[6].sample_unc[:, 1], base[6].sample_unc[:, 1])
    # without the uncertainty outputs the tally is the same
    tl2 = tally_bufs(k)
    ops.prob_finalize(acc, k, scale, labels=lab, tally=tl2, inv_temperature=beta)
    assert torch.equal(tl2[2], got[0][2]) and torch.equal(tl2[1], got[0][1])
    # proba within fp16 rounding of the fp64 p̃
    perr = (got[3].double() - pt).abs()
    assert (perr <= fp16_tol(pt, 1e-5 * pt + 1e-8)).all(), perr.max().item()
    # nll
    py = pt.gather(1, ll.clamp(0, k - 1)[:, None])[:, 0]
    nll_ref = float((-py.clamp(min=FLT_MIN).log())[counted].sum())
    assert abs(float(got[0][0]) - nll_ref) <= 1e-5 * nll_ref, (float(got[0][0]), nll_ref)
    # entropy map of p̃ and its sum
    u = got[6]
    ht = entropy(pt)
    e_err = (u.entropy_out.double() - ht).abs()
    assert (e_err <= fp16_tol(ht, 2e-6)).all(), e_err.max().item()
    vox = n * d * h * w
    assert abs(int(u.unc[0]) * FIX - float(ht.sum())) <= vox * FIX + float(ht.sum()) * 1e-5
    # histogram and calibration: exact outside the DELTA band of a bin edge
    lab_c = ll.clamp(0, k - 1)
    if t:
        v = pt.movedim(1, -1)[counted]                                   # [m,k]
        yy = lab_c[counted]
        ref = torch.zeros(k, 2, t, dtype=torch.int64, device="cuda")
        bins = (v * t).floor().long().clamp(max=t - 1)
        for c in range(k):
            pos = yy == c
            ref[c, 0] = torch.bincount(bins[pos, c], minlength=t)
            ref[c, 1] = torch.bincount(bins[~pos, c], minlength=t)
        frac = v * t - (v * t).round()
        near = int((frac.abs() < DELTA * t).sum())
        diff = int((got[4] - ref).abs().sum())
        assert diff <= 2 * near, (diff, near)
        assert torch.equal(got[5].sum(0), got[4])
    conf = pt.gather(1, arg[:, None])[:, 0][counted]
    cb = (conf * tc).floor().long().clamp(max=tc - 1)
    near = int(((conf * tc - (conf * tc).round()).abs() < DELTA * tc).sum())
    cal = u.calib
    assert int((cal[0] - torch.bincount(cb, minlength=tc)).abs().sum()) <= 2 * near
    correct = (arg == ll)[counted]
    assert int((cal[1] - torch.bincount(cb[correct], minlength=tc)).abs().sum()) <= 2 * near
    assert abs(float(cal[2].sum()) * FIX - float(conf.sum())) <= 1e-5 * float(conf.sum()) + conf.numel() * FIX
    assert torch.equal(u.sample_calib.sum(0), cal)
    onehot = torch.nn.functional.one_hot(lab_c, k).movedim(-1, 1).double()
    br = float(((pt - onehot) ** 2).sum(1)[counted].sum())
    assert abs(float(u.brier) - br) <= 1e-5 * br
    print(f"k={k} beta={beta}: max |proba - ref| {perr.max().item():.2e}, nll {float(got[0][0]):.6f} "
          f"(ref {nll_ref:.6f}), near-edge voxels {near}")


def test_temperature_kernels_reject_bad_arguments():
    import ctypes

    from spff_b200 import _lib
    from spff_b200._lib import Shape, UncOut, ptr, stream_ptr
    k = 13
    acc = torch.zeros(5 * 8 * 8 * 16 + 4, device="cuda")
    a, bad_acc = acc[:-4], acc[1:-3]
    lab = torch.zeros(1, 5, 8, 8, dtype=torch.uint8, device="cuda")
    tl = tally_bufs(k)
    s1 = Shape(1, 5, 8, 8)
    betas = torch.ones(64, device="cuda")
    sums = torch.zeros(2, 64, dtype=torch.float64, device="cuda")
    cnt = torch.zeros(1, dtype=torch.int64, device="cuda")
    ws_bytes = int(_lib.lib.spff_prob_temp_fit_workspace(k, s1, 33))
    assert ws_bytes > 0
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    assert int(_lib.lib.spff_prob_temp_fit_workspace(k, s1, 0)) == 0
    assert int(_lib.lib.spff_prob_temp_fit_workspace(k, s1, 65)) == 0
    assert int(_lib.lib.spff_prob_temp_fit_workspace(17, s1, 33)) == 0

    def fit(kk=k, s=s1, g=33, acc_=a, labels=lab, lb=1, b=betas, sm=sums, c=cnt, w=ws, nbytes=None, scale=1.0):
        return _lib.lib.spff_prob_temp_fit(ptr(acc_), kk, s, scale, ptr(labels), lb, 255, ptr(b), g, ptr(sm), ptr(c),
                                           ptr(w), ws_bytes if nbytes is None else nbytes, stream_ptr())

    def fin(inv_t, kk=k, s=s1, u=None):
        return _lib.lib.spff_prob_finalize_tempered(ptr(a), kk, s, 1.0, ptr(lab), 1, 255, *(ptr(v) for v in tl), None,
                                                    None, None, None, 0, None, None, None,
                                                    ctypes.byref(u) if u is not None else None, inv_t, stream_ptr())

    bad, small = -1, -4          # SPFF_ERR_BAD_ARGUMENT, SPFF_ERR_WORKSPACE
    for kk in (1, 17):
        assert fit(kk=kk) == bad and "classes" in _lib.lib.spff_last_error().decode()
        assert fin(1.5, kk=kk) == bad
    for g in (0, 65):
        assert fit(g=g) == bad and "grid points" in _lib.lib.spff_last_error().decode()
    for v in (0.0, -1.0, float("inf"), float("nan")):
        assert fin(v) == bad and "inv_temperature" in _lib.lib.spff_last_error().decode()
    for name, kw in (("acc_", None), ("labels", None), ("b", None), ("sm", None), ("c", None), ("w", None)):
        assert fit(**{name: kw}) == bad and "null pointer" in _lib.lib.spff_last_error().decode()
    assert fit(acc_=bad_acc) == bad and "16-byte aligned" in _lib.lib.spff_last_error().decode()
    assert fit(s=Shape(65536, 1, 1, 1)) == bad and fin(1.5, s=Shape(65536, 1, 1, 1)) == bad
    assert fit(s=Shape(1, 0, 8, 8)) == bad
    assert fit(lb=4) == bad and "uint8 or int64" in _lib.lib.spff_last_error().decode()
    assert fit(scale=0.0) == bad
    assert fit(nbytes=ws_bytes - 1) == small and "workspace" in _lib.lib.spff_last_error().decode()
    # the uncertainty struct's rules still apply
    u = UncOut(None, None, ptr(torch.zeros(1, 5, 8, 8, dtype=torch.float16, device="cuda")), None, None, 0, None, None,
               None, None)
    assert fin(1.5, u=u) == bad and "mi_out needs ent" in _lib.lib.spff_last_error().decode()
    assert fit() == 0 and fin(1.5) == 0
    torch.cuda.synchronize()
    assert int(cnt) == 5 * 8 * 8 and int(tl[1]) == 5 * 8 * 8
    from spff_b200 import ops
    with pytest.raises(ValueError, match="inv_temperature"):
        ops.prob_finalize(a.view(1, 5, 8, 8, 16), k, 1.0, inv_temperature=0.0)


# --------------------------------------------------------------------------------------------------------------------
# model, on the weights the reference trained
# --------------------------------------------------------------------------------------------------------------------
def _load_trained():
    from test_parity_trained import FIX as FIXTURE
    from test_parity_trained import init_state, trained_weights
    z = np.load(FIXTURE)
    lit = init_state()
    w = trained_weights(z, lit)
    lit = lit.cuda()
    lit.model.materialize(5)
    alias = {k.replace("freq_mask", "_mask"): v for k, v in w.items() if k.endswith("freq_mask")}
    lit.load_state_dict({**w, **alias}, strict=True)
    return lit


@pytest.fixture(scope="module")
def members():
    """The trained weights, plus two copies moved by a few fit_steps under other seeds (the three seeds of a variant)."""
    import copy

    from oracle import spff_oracle as O
    lit = _load_trained()
    out = [lit]
    for seed in (123, 999):
        m = copy.deepcopy(lit)
        x, lab = O.phantom_batch(8, 64, 64, seed=seed, ignore_frac=0.01)
        for _ in range(3):
            m.fit_step((x.cuda(), lab.cuda()))
        out.append(m)
    return out


def _batch(b=16, hw=128, seed=42, ignore=0.05):
    from oracle import spff_oracle as O
    x, lab = O.phantom_batch(b, hw, hw, seed=seed, ignore_frac=0.01)
    lab = lab.clone()
    g = torch.Generator().manual_seed(seed)
    lab[torch.rand(lab.shape, generator=g) < ignore] = 255
    return x.cuda(), lab.cuda()


def _with_group(members, g):
    for m in members:
        m.model.sample_group = g


@torch.no_grad()
def ref_pbar(cores, x, flips):
    """fp64 p̄ [B,K,F,H,W] of per-member, per-flip softmax(core(flip(x))) flipped back."""
    acc = None
    for core in cores:
        for f in flips:
            p = torch.flip(torch.softmax(core(torch.flip(x, FLIPS[f])).double(), 1), FLIPS[f])
            acc = p if acc is None else acc + p
            del p
    return acc / (len(cores) * len(flips))


def scipy_fit(pbar, lab, k, t_max=8.0):
    """(T, mean nll at T, mean nll at T = 1) minimising the fp64 mean nll of p̃ over β in [1/t_max, t_max]."""
    from scipy.optimize import minimize_scalar
    mean = lambda b: float(fit_terms(pbar, lab, k, b)[0].mean())   # noqa: E731
    r = minimize_scalar(mean, bounds=(1.0 / t_max, t_max), method="bounded", options={"xatol": 1e-9})
    return 1.0 / r.x, r.fun, mean(1.0)


def test_temperature_one_is_the_untempered_path(members):
    """temperature=1.0 (and a temperature set back to 1.0) gives every output of the untempered path bit for bit; the
    fp64 nll and Brier sums, which both paths add with fp64 atomics, to their order (1e-12)."""
    from innovative3D import models
    from spff_b200.engine import run_ensemble
    xg, lg = _batch(b=8, seed=5)
    plain = models.SpctEnsemble(members, tta="flip")
    ens = models.SpctEnsemble(members, tta="flip", temperature=1.0)
    ens.temperature = 2.0
    ens.temperature = 1.0

    def outputs(e):
        ev = e.eval_step((xg, lg), per_sample=True, return_labels=True, sample_group=4, curves=64, calibration=960)
        u = e.predict_uncertainty(xg, sample_group=4)
        exact = [ev["labels"], ev["tally"].count, ev["tally"].confusion, *ev["per_sample"][1:], ev["hist"],
                 ev["per_sample_hist"], ev["calib"], ev["uncertainty"], ev["per_sample_calib"],
                 e.predict_proba(xg, sample_group=4), *u.values()]
        return exact, [ev["tally"].nll, ev["per_sample"][0], ev["brier"], ev["per_sample_brier"]]

    (a, fa), (b, fb) = outputs(plain), outputs(ens)
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    for x, y in zip(fa, fb):
        assert torch.allclose(x, y, rtol=1e-12, atol=0)
    # and the engine without the argument (the call the ensemble made before temperatures existed)
    engines = plain._engines(5)
    proba = torch.empty_like(a[10])
    run_ensemble(engines, xg, plain.flips, 4, proba_out=proba)
    assert torch.equal(proba, a[10])


def test_fit_three_members_flip_against_scipy(members):
    """3 members x flip: the fitted T within 1e-3 of scipy's minimiser of the fp64 nll of the unfused pooled softmax,
    nll_at_1 equal to the reference nll at T = 1 to 1e-5; the fitted temperature lowers the validation nll of
    evaluate; predict_labels does not change."""
    from innovative3D import models
    k = 13
    xg, lg = _batch(seed=7)
    ens = models.SpctEnsemble(members, tta="flip")
    _with_group(members, 16)
    pbar = ref_pbar([m.model for m in members], xg, (0, 1, 2, 3))
    _with_group(members, 256)
    t_ref, nll_ref, nll1_ref = scipy_fit(pbar, lg, k)
    del pbar
    labels_before = ens.predict_labels(xg, sample_group=16)
    ev1 = ens.evaluate([(xg, lg)], sample_group=16, calibration=960)
    res = ens.fit_temperature([(xg, lg)], sample_group=16)
    print(f"3 x flip: T {res['temperature']:.6f} (scipy {t_ref:.6f}), nll {res['nll']:.6f} (ref {nll_ref:.6f}), "
          f"nll at 1 {res['nll_at_1']:.6f} (ref {nll1_ref:.6f}), at_bound {res['at_bound']}")
    assert not res["at_bound"]
    assert abs(res["temperature"] / t_ref - 1) <= 1e-3
    assert abs(res["nll_at_1"] - nll1_ref) <= 1e-5 * max(1.0, nll1_ref)
    assert res["nll"] <= res["nll_at_1"] and ens.temperature == res["temperature"]
    assert res["counted"] == int(((lg != 255) & (lg < k)).sum())
    assert res["grid"]["temperature"].size == 33 and res["grid"]["temperature"][16] == 1.0
    ev2 = ens.evaluate([(xg, lg)], sample_group=16, calibration=960)
    nll1 = float(ev1["tally"].nll) / int(ev1["tally"].count)
    nll2 = float(ev2["tally"].nll) / int(ev2["tally"].count)
    print(f"3 x flip: validation CE {nll1:.6f} -> {nll2:.6f}, ECE {ev1['calibration']['ece']:.5f} -> "
          f"{ev2['calibration']['ece']:.5f}")
    assert nll2 <= nll1 + 1e-7
    assert torch.equal(ev1["tally"].confusion, ev2["tally"].confusion)
    assert torch.equal(ens.predict_labels(xg, sample_group=16), labels_before)
    # apply=False leaves the temperature alone
    ens.temperature = 1.0
    again = ens.fit_temperature([(xg, lg)], sample_group=16, apply=False)
    assert ens.temperature == 1.0 and again["temperature"] == res["temperature"]


def test_scaled_head_scales_the_temperature(members):
    """One member without TTA: multiplying the head's weight and bias by s = 3 multiplies the fitted T by 3, to 1e-3
    (p̃ = softmax(z / T) end to end); predict_proba at a temperature is softmax(model(x) / T) within fp16 rounding."""
    import copy

    from innovative3D import models
    xg, lg = _batch(seed=11)
    lit = members[0]
    t1 = models.SpctEnsemble([lit]).fit_temperature([(xg, lg)], t_max=16.0, points=63, sample_group=16)
    m3 = copy.deepcopy(lit)
    with torch.no_grad():
        m3.model.out.weight.mul_(3.0)
        m3.model.out.bias.mul_(3.0)
    t3 = models.SpctEnsemble([m3]).fit_temperature([(xg, lg)], t_max=16.0, points=63, sample_group=16)
    print(f"one member: T {t1['temperature']:.6f}, with the head x 3: {t3['temperature']:.6f} "
          f"(ratio {t3['temperature'] / t1['temperature']:.6f})")
    assert not t1["at_bound"] and not t3["at_bound"]
    assert abs(t3["temperature"] / t1["temperature"] / 3.0 - 1) <= 1e-3
    for temp in (t1["temperature"], 0.5, 2.7):
        ens = models.SpctEnsemble([lit], temperature=temp)
        proba = ens.predict_proba(xg, sample_group=16)
        with torch.no_grad():
            ref = torch.softmax(lit(xg).double() / temp, 1)
        err = (proba.double() - ref).abs().max().item()
        print(f"T {temp:.4f}: max |proba - softmax(z / T)| {err:.2e}")
        assert err <= 5e-4


def test_fit_host_batches_and_dict_batches(members):
    """Host batches (pinned, uint8 labels) and dict batches give the device batches' temperature bit for bit."""
    from innovative3D import models
    xg, lg = _batch(b=12, seed=3)
    ens = models.SpctEnsemble(members[:2], tta="flip")
    a = ens.fit_temperature([(xg[:5], lg[:5]), (xg[5:], lg[5:])], sample_group=4, apply=False)
    b = ens.fit_temperature([(xg[:5].cpu().pin_memory(), lg[:5].cpu().to(torch.uint8).pin_memory()),
                             {"image": xg[5:].cpu(), "label": lg[5:].cpu()}], sample_group=4, apply=False)
    assert a["temperature"] == b["temperature"] and a["counted"] == b["counted"]
    np.testing.assert_array_equal(a["grid"]["nll"], b["grid"]["nll"])
    np.testing.assert_array_equal(a["grid"]["dnll"], b["grid"]["dnll"])
    with pytest.raises(ValueError, match="no counted voxel"):
        ens.fit_temperature([(xg[:1], torch.full_like(lg[:1], 255))], sample_group=4)


def test_fit_native_slices_two_members_flip(members):
    from innovative3D import models
    k = 13
    xg, lg = _batch(b=4, hw=512, seed=21)
    ens = models.SpctEnsemble(members[:2], tta="flip")
    _with_group(members[:2], 4)
    pbar = ref_pbar([m.model for m in members[:2]], xg, (0, 1, 2, 3))
    _with_group(members[:2], 256)
    t_ref, _, nll1_ref = scipy_fit(pbar, lg, k)
    del pbar
    res = ens.fit_temperature([(xg, lg)], sample_group=4)
    print(f"512 x 512: T {res['temperature']:.6f} (scipy {t_ref:.6f}), nll at 1 {res['nll_at_1']:.6f} "
          f"(ref {nll1_ref:.6f})")
    assert abs(res["temperature"] / t_ref - 1) <= 1e-3
    assert abs(res["nll_at_1"] - nll1_ref) <= 1e-5 * max(1.0, nll1_ref)


def test_fit_memory():
    """fit_temperature's peak above the resident set is no more than evaluate(calibration=960)'s plus 4 MB."""
    from innovative3D import config as C
    from innovative3D import models
    torch.manual_seed(42)
    lits = [dict((v[0], v[1]) for v in C.VARIANTS)["SPFF-UNet"]().cuda() for _ in range(3)]
    g = torch.Generator(device="cuda").manual_seed(9)
    b = 64
    x = torch.randn(b, 1, 5, 128, 128, device="cuda", generator=g)
    lab = torch.randint(0, 13, (b, 5, 128, 128), device="cuda", generator=g)
    ens = models.SpctEnsemble(lits, tta="flip")

    def peak(fn):
        fn()
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        fn()
        torch.cuda.synchronize()
        return torch.cuda.max_memory_allocated() - base

    ev = peak(lambda: ens.evaluate([(x, lab)], sample_group=16, calibration=960))
    fit = peak(lambda: ens.fit_temperature([(x, lab)], sample_group=16, apply=False))
    print(f"peak above the resident set: evaluate(calibration=960) {ev / 2**20:.1f} MB, fit_temperature "
          f"{fit / 2**20:.1f} MB")
    assert fit <= ev + 4 * 2**20


# --------------------------------------------------------------------------------------------------------------------
# data parallel (2 ranks over NCCL; skipped on a single-GPU box)
# --------------------------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _dp_setup():
    from innovative3D import config as C
    from innovative3D import models
    from oracle import spff_oracle as O
    lits = []
    for seed in (42, 123):
        torch.manual_seed(seed)
        lits.append(dict((v[0], v[1]) for v in C.VARIANTS)["SPFF-UNet"]().cuda())
    x, lab = O.phantom_batch(6, 32, 32, seed=79, ignore_frac=0.02)
    return models.SpctEnsemble(lits, tta="flip"), x, lab


def _worker(rank, world, port, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    ens, x, lab = _dp_setup()
    lo = rank * 3
    res = ens.fit_temperature([(x[lo:lo + 3].cuda(), lab[lo:lo + 3].cuda())], apply=False)
    out[rank] = dict(t=res["temperature"], counted=res["counted"], nll=res["grid"]["nll"].tolist())
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_fit_equals_single_process():
    world = 2
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    ens, x, lab = _dp_setup()
    res = ens.fit_temperature([(x[lo:lo + 3].cuda(), lab[lo:lo + 3].cuda()) for lo in (0, 3)], apply=False)
    for r in range(world):
        assert out[r]["t"] == res["temperature"] and out[r]["counted"] == res["counted"]
        assert out[r]["nll"] == res["grid"]["nll"].tolist()
