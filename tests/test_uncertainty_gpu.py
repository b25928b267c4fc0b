"""GPU: uncertainty maps and calibration of ensembles and mirror test-time augmentation. The two kernels
(spff_head_prob_accum_ent, spff_prob_finalize_unc) against torch and against the entry points they extend; every
argument error; three members x four flips on the weights the reference trained against the per-member
model(torch.flip(x)) -> fp64 softmax -> flip back reference, with the entropy and the mutual information formed in fp64;
the invariants with the existing paths; determinism, host batches, native 512 x 512 slices, memory, isolation from the
training state and two ranks.

Tolerances. The kernels' logits are about 1e-5 from the fp32 logits of model(x) (tensor-core head, W split into bf16
hi + lo) and the per-pass entropy uses __expf / __logf, so a pass's H(p) is within about 5e-5 nats of the fp64 entropy
of softmax(F.conv3d(...)). The fp16 maps are within half an fp16 ulp of the kernel's fp32 value. Calibration counts are
exact on given accumulators (the confidence and its bin are fp32 products torch reproduces); on the model they are
exact outside voxels within DELTA = 3e-5 of a bin edge or whose two largest probabilities are within NEAR_TIE = 1e-4
(the rules of test_ensemble_gpu)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DELTA = 3e-5
NEAR_TIE = 1e-4
FIX = 2.0 ** -24
FLIPS = {0: [], 1: [3], 2: [4], 3: [3, 4]}      # flip code -> dims of a [B,C,F,H,W] tensor


def pm(x, ld):  # NCDHW fp32 -> position-major bf16 channel slice of a wider buffer
    n, c, d, h, w = x.shape
    buf = torch.zeros(n, d, h, w, ld, dtype=torch.bfloat16, device=x.device)
    buf[..., :c] = x.permute(0, 2, 3, 4, 1).to(torch.bfloat16)
    return buf[..., :c]


def entropy(p, dim=1):
    """-sum p log p over `dim` (0 log 0 = 0), in the dtype of p."""
    return -(p * torch.where(p > 0, p.log(), torch.zeros_like(p))).sum(dim)


def fp16_tol(ref, extra):
    """Half an fp16 ulp of |ref| (normal range) plus `extra`."""
    return ref.abs() * 2.0 ** -11 + 2.0 ** -25 + extra


def tally_bufs(k, dev="cuda"):
    return (torch.zeros(1, dtype=torch.float64, device=dev), torch.zeros(1, dtype=torch.int64, device=dev),
            torch.zeros(k, k, dtype=torch.int64, device=dev))


def sample_bufs(n, k, dev="cuda"):
    return (torch.zeros(n, dtype=torch.float64, device=dev), torch.zeros(n, dtype=torch.int64, device=dev),
            torch.zeros(n, k, k, dtype=torch.int64, device=dev))


def unc_bufs(n, d, h, w, t, ent=None, per_sample=True, labels=True):
    from spff_b200 import ops
    z = lambda *s, dt=torch.int64: torch.zeros(*s, dtype=dt, device="cuda")   # noqa: E731
    u = ops.Uncertainty(ent=ent, entropy_out=torch.full((n, d, h, w), 9.0, dtype=torch.float16, device="cuda"),
                        mi_out=torch.full((n, d, h, w), 9.0, dtype=torch.float16, device="cuda") if ent is not None
                        else None, unc=z(2), sample_unc=z(n, 2) if per_sample else None)
    if labels:
        u.calib = z(3, t)
        u.brier = z(1, dt=torch.float64)
        if per_sample:
            u.sample_calib = z(n, 3, t)
            u.sample_brier = z(n, dt=torch.float64)
    return u


def ref_calib(conf, arg, lab, k, t, ignore_index=255):
    """[3,T] histogram of the confidences conf (fp32 [B,...]) of the counted voxels, by the kernel's rules."""
    counted = (lab != ignore_index) & (lab >= 0) & (lab < k)
    c = conf[counted]
    b = (c * np.float32(t)).floor().long().clamp(max=t - 1)
    h = torch.zeros(3, t, dtype=torch.int64, device=conf.device)
    h[0] = torch.bincount(b, minlength=t)
    h[1] = torch.bincount(b[arg[counted] == lab[counted]], minlength=t)
    h[2].index_add_(0, b, (c.double() / FIX).round().long())
    return h


def ref_brier(pbar, lab, k, ignore_index=255):
    counted = (lab != ignore_index) & (lab >= 0) & (lab < k)
    onehot = F.one_hot(lab.clamp(0, k - 1), k).movedim(-1, 1).double()
    return ((pbar.double() - onehot) ** 2).sum(1)[counted].sum()


# --------------------------------------------------------------------------------------------------------------------
# kernels
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [2, 5, 13, 16])
@pytest.mark.parametrize("n,d,h,w", [(1, 5, 7, 9), (3, 5, 17, 31), (2, 5, 16, 16)])
def test_head_prob_accum_ent(k, n, d, h, w):
    """acc bit-identical to spff_head_prob_accum; ent = sum over passes of H(p) within 5e-5 nats per pass of the fp64
    entropy of softmax(F.conv3d(...)), at the mirrored position; nothing past the plane is written."""
    from spff_b200 import ops
    torch.backends.cudnn.allow_tf32 = False
    torch.manual_seed(11 + k + h)
    xb = pm(torch.randn(n, 32, d, h, w, device="cuda") * 1.5, ld=64)
    wt = torch.randn(k, 32, 1, 1, 1, device="cuda") * 0.5
    b = torch.randn(k, device="cuda") * 0.1
    p = torch.softmax(F.conv3d(xb.permute(0, 4, 1, 2, 3).float(), wt, b).double(), 1)   # [n,k,d,h,w]
    hp = entropy(p)                                                                     # [n,d,h,w]
    vox = n * d * h * w
    acc_a = torch.empty(n, d, h, w, 16, device="cuda")
    acc_b = torch.empty_like(acc_a)
    store = torch.full((vox + 64,), 7.0, device="cuda")          # 64 guard floats past the plane
    ent = store[:vox].view(n, d, h, w)
    ref = torch.zeros(n, d, h, w, dtype=torch.float64, device="cuda")
    worst = 0.0
    for i, f in enumerate((0, 1, 2, 3, 3, 0)):
        beta = 0 if i == 0 else 1
        ops.head_prob_accum(xb, wt, b, acc_a, flip=f, beta=beta)
        ops.head_prob_accum(xb, wt, b, acc_b, flip=f, beta=beta, ent=ent)
        ref += torch.flip(hp, [d_ - 1 for d_ in FLIPS[f]])
        assert torch.equal(acc_a, acc_b)
        err = (ent.double() - ref).abs().max().item()
        worst = max(worst, err / (i + 1))
        assert err <= 5e-5 * (i + 1), (f, i, err)
    print(f"k={k}: max |ent - ref| per pass {worst:.2e}")
    assert torch.equal(store[vox:], torch.full((64,), 7.0, device="cuda"))
    ent.fill_(float("nan"))                                       # beta = 0 replaces whatever was there
    ops.head_prob_accum(xb, wt, b, acc_b, flip=1, beta=0, ent=ent)
    assert (ent.double() - torch.flip(hp, [2])).abs().max().item() <= 5e-5


@pytest.mark.parametrize("dtype", [torch.uint8, torch.int64])
@pytest.mark.parametrize("k,t,tc", [(13, 256, 960), (5, 16, 2), (16, 1024, 1024), (2, 0, 15)])
def test_prob_finalize_unc(dtype, k, t, tc):
    from spff_b200 import ops
    n, d, h, w = 3, 5, 17, 31
    g = torch.Generator(device="cuda").manual_seed(k * 7 + t + tc)
    # sums of 3 passes on a coarse grid (ties, zeros) plus a fine component (confidences spread over the bins)
    acc = torch.full((n, d, h, w, 16), 100.0, device="cuda")                # classes >= k must be ignored
    raw = torch.randint(0, 7, (n, d, h, w, k), device="cuda", generator=g).float() * 0.125
    fine = torch.rand(n, d, h, w, k, device="cuda", generator=g) ** 4 * 3
    acc[..., :k] = torch.where(torch.rand(n, d, h, w, 1, device="cuda", generator=g) < 0.5, raw, fine)
    scale = 1.0 / 3.0
    lab = torch.randint(0, k, (n, d, h, w), device="cuda", generator=g)
    lab[torch.rand(n, d, h, w, device="cuda", generator=g) < 0.1] = 255          # ignored
    lab[torch.rand(n, d, h, w, device="cuda", generator=g) < 0.03] = 200         # not a class: counted only
    lab = lab.to(dtype)
    pbar = (acc[..., :k] * scale).permute(0, 4, 1, 2, 3).contiguous()            # fp32, the kernel's p̄
    hb = entropy(pbar.double())
    ent = (3 * hb * (0.5 + 0.5 * torch.rand(n, d, h, w, device="cuda", generator=g, dtype=torch.float64))).float()
    mi = (hb - ent.double() * np.float32(scale)).clamp(min=0)
    arg = acc[..., :k].argmax(-1)
    conf = pbar.amax(1)
    vox = n * d * h * w

    def outputs(unc):
        tl, per = tally_bufs(k), sample_bufs(n, k)
        out = torch.full((n, d, h, w), 77, dtype=torch.uint8, device="cuda")
        proba = torch.empty(n, k, d, h, w, dtype=torch.float16, device="cuda")
        hist = torch.zeros(k, 2, t, dtype=torch.int64, device="cuda") if t else None
        s_hist = torch.zeros(n, k, 2, t, dtype=torch.int64, device="cuda") if t else None
        ops.prob_finalize(acc, k, scale, labels=lab, tally=tl, per_sample=per, labels_out=out, hist=hist,
                          sample_hist=s_hist, proba_out=proba, unc=unc)
        return tl, per, out, proba, hist, s_hist

    base = outputs(None)
    u = unc_bufs(n, d, h, w, tc, ent=ent)
    got = outputs(u)
    for a, b in zip(base, got):                       # everything spff_prob_finalize gives, bit for bit
        for x, y in zip(a if isinstance(a, tuple) else (a,), b if isinstance(b, tuple) else (b,)):
            if x is not None and x.dtype != torch.float64:
                assert torch.equal(x, y)
    assert torch.allclose(base[0][0], got[0][0], rtol=1e-12, atol=0)      # fp64 atomics: order only
    # maps
    e_err = (u.entropy_out.double() - hb).abs()
    assert (e_err <= fp16_tol(hb, 1e-6)).all(), e_err.max().item()
    m_err = (u.mi_out.double() - mi).abs()
    assert (m_err <= fp16_tol(mi, 2e-6)).all(), m_err.max().item()
    # sums: within the per-voxel rounding (2^-24 per voxel) plus the fp32 evaluation of H (2^-22 relative) of the fp64
    # values; these accumulators are not normalised, so H reaches 3.7 nats at K = 16
    assert abs(int(u.unc[0]) * FIX - float(hb.sum())) <= vox * FIX + float(hb.sum()) * 2.0 ** -22
    assert abs(int(u.unc[1]) * FIX - float(mi.sum())) <= vox * FIX + float(hb.sum()) * 2.0 ** -22
    # calibration: exact counts and confidence sums, Brier to fp32 rounding
    labl = lab.long()
    assert torch.equal(u.calib, ref_calib(conf, arg, labl, k, tc))
    br = ref_brier(pbar, labl, k)
    assert abs(float(u.brier) - float(br)) <= 1e-5 * float(br)
    for i in range(n):
        assert torch.equal(u.sample_calib[i], ref_calib(conf[i:i + 1], arg[i:i + 1], labl[i:i + 1], k, tc))
        assert abs(int(u.sample_unc[i, 0]) * FIX - float(hb[i].sum())) <= vox / n * FIX + float(hb[i].sum()) * 2.0 ** -22
    # per-sample rows sum exactly to the totals
    assert torch.equal(u.sample_unc.sum(0), u.unc) and torch.equal(u.sample_calib.sum(0), u.calib)
    assert torch.allclose(u.sample_brier.sum(), u.brier[0], rtol=1e-12, atol=0)
    # without labels: the maps and sums only, the same values
    v = unc_bufs(n, d, h, w, tc, ent=ent, labels=False)
    out2 = torch.empty(n, d, h, w, dtype=torch.uint8, device="cuda")
    ops.prob_finalize(acc, k, scale, labels_out=out2, unc=v)
    assert torch.equal(out2, got[2])
    assert torch.equal(v.entropy_out, u.entropy_out) and torch.equal(v.mi_out, u.mi_out)
    assert torch.equal(v.unc, u.unc) and torch.equal(v.sample_unc, u.sample_unc)
    # without ent: the entropy map, no MI
    w_ = unc_bufs(n, d, h, w, tc, labels=False)
    ops.prob_finalize(acc, k, scale, unc=w_)
    assert torch.equal(w_.entropy_out, u.entropy_out) and int(w_.unc[0]) == int(u.unc[0]) and int(w_.unc[1]) == 0


def test_unc_kernels_reject_bad_arguments():
    from spff_b200._lib import Shape, UncOut, call, ptr, stream_ptr
    import ctypes
    k = 13
    x = torch.zeros(1, 5, 8, 8, 32, dtype=torch.bfloat16, device="cuda")
    wt, b = torch.zeros(k, 32, device="cuda"), torch.zeros(k, device="cuda")
    acc = torch.zeros(5 * 8 * 8 * 16, device="cuda")
    store = torch.zeros(5 * 8 * 8 + 1, device="cuda")
    ent, bad_ent = store[:-1], store.view(torch.uint8)[1:1 + 5 * 8 * 8 * 4]
    lab = torch.zeros(1, 5, 8, 8, dtype=torch.uint8, device="cuda")
    tl, per = tally_bufs(k), sample_bufs(1, k)
    s1 = Shape(1, 5, 8, 8)
    z = lambda *s, dt=torch.int64: torch.zeros(*s, dtype=dt, device="cuda")   # noqa: E731

    def accum(e=ent):
        call("spff_head_prob_accum_ent", ptr(x), 32, 32, ptr(wt), ptr(b), k, s1, 0, 0, ptr(acc), ptr(e), stream_ptr())

    def fin(u, labels=True, p=(None, None, None)):
        call("spff_prob_finalize_unc", ptr(acc), k, s1, 1.0, ptr(lab) if labels else None, 1, 255,
             *(ptr(v) if labels else None for v in tl), *(ptr(v) for v in p), None, 0, None, None, None,
             ctypes.byref(u) if u is not None else None, stream_ptr())

    def U(**kw):
        f = dict(ent=None, entropy_out=None, mi_out=None, unc=None, sample_unc=None, cal_bins=0, calib=None,
                 sample_calib=None, brier=None, sample_brier=None)
        f.update(kw)
        return UncOut(*(ptr(v) if torch.is_tensor(v) else v for v in f.values()))

    calib, brier = z(3, 16), z(1, dt=torch.float64)
    with pytest.raises(RuntimeError, match="null pointer"):
        accum(e=None)
    with pytest.raises(RuntimeError, match="4-byte aligned"):
        accum(e=bad_ent)
    with pytest.raises(RuntimeError, match="null output struct"):
        fin(None)
    for tc in (1, 1025):
        with pytest.raises(RuntimeError, match="cal_bins"):
            fin(U(cal_bins=tc, calib=z(3, 2048), brier=brier))
    with pytest.raises(RuntimeError, match="calib needs labels"):
        fin(U(cal_bins=16, calib=calib, brier=brier), labels=False)
    with pytest.raises(RuntimeError, match="sample_calib needs"):
        fin(U(cal_bins=16, calib=calib, brier=brier, sample_calib=z(1, 3, 16), sample_brier=z(1, dt=torch.float64)))
    with pytest.raises(RuntimeError, match="sample_calib is given exactly"):
        fin(U(cal_bins=16, calib=calib, brier=brier), p=per)
    with pytest.raises(RuntimeError, match="brier is given exactly"):
        fin(U(cal_bins=16, calib=calib))
    with pytest.raises(RuntimeError, match="brier is given exactly"):
        fin(U(brier=brier))
    with pytest.raises(RuntimeError, match="sample_brier is given exactly"):
        fin(U(cal_bins=16, calib=calib, brier=brier, sample_calib=z(1, 3, 16)), p=per)
    with pytest.raises(RuntimeError, match="mi_out needs ent"):
        fin(U(mi_out=z(1, 5, 8, 8, dt=torch.float16)))
    with pytest.raises(RuntimeError, match="sample_unc needs unc"):
        fin(U(sample_unc=z(1, 2)))
    with pytest.raises(RuntimeError, match="4-byte aligned"):
        fin(U(ent=bad_ent))
    accum()
    sb = z(1, dt=torch.float64)
    fin(U(ent=ent, unc=z(2), cal_bins=16, calib=calib, brier=brier, sample_calib=z(1, 3, 16), sample_brier=sb), p=per)
    torch.cuda.synchronize()
    assert int(calib[0].sum()) == 5 * 8 * 8


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


@torch.no_grad()
def ref_uncertainty(cores, x, flips):
    """fp64 (p̄ [B,K,F,H,W], H[p̄], MI) of per-member, per-flip softmax(core(flip(x))) flipped back."""
    acc, hsum = None, None
    for core in cores:
        for f in flips:
            p = torch.flip(torch.softmax(core(torch.flip(x, FLIPS[f])).double(), 1), FLIPS[f])
            acc = p if acc is None else acc + p
            hp = entropy(p)
            hsum = hp if hsum is None else hsum + hp
            del p, hp
    passes = len(cores) * len(flips)
    pbar = acc / passes
    hb = entropy(pbar)
    return pbar, hb, hb - hsum / passes


def _with_group(members, g):
    for m in members:
        m.model.sample_group = g


def test_three_members_flip_against_torch(members):
    from innovative3D import models
    from sklearn.metrics import roc_auc_score
    k, t = 13, 960
    xg, lg = _batch(seed=7)
    ens = models.SpctEnsemble(members, tta="flip")
    _with_group(members, 16)
    pbar, hb, mi = ref_uncertainty([m.model for m in members], xg, (0, 1, 2, 3))
    _with_group(members, 256)
    out = ens.predict_uncertainty(xg, sample_group=16)
    assert out["entropy"].dtype == torch.float16 and tuple(out["entropy"].shape) == (16, 5, 128, 128)
    e_err = (out["entropy"].double() - hb).abs()
    m_err = (out["mutual_info"].double() - mi).abs()
    print(f"3 x flip: max |H - ref| {e_err.max().item():.2e}, max |MI - ref| {m_err.max().item():.2e}, "
          f"mean MI {mi.mean().item():.3e}")
    assert (e_err <= fp16_tol(hb, 5e-4)).all()
    assert (m_err <= fp16_tol(mi, 5e-4)).all()
    ce = (out["case_entropy"] - hb.mean(dim=(1, 2, 3))).abs().max().item()
    cm = (out["case_mutual_info"] - mi.clamp(min=0).mean(dim=(1, 2, 3))).abs().max().item()
    print(f"3 x flip: per-case mean entropy / MI error {ce:.2e} / {cm:.2e}")
    assert ce <= 1e-4 and cm <= 1e-4
    assert torch.equal(out["labels"], ens.predict_labels(xg, sample_group=16))
    # evaluate(calibration=960): ECE and error AUROC against the reference's confidences
    ev = ens.evaluate([(xg, lg)], sample_group=16, calibration=t)
    c = ev["calibration"]
    assert c["ece_bins"] == 15
    counted = (lg != 255) & (lg < k)
    conf = pbar.amax(1)[counted].cpu().numpy()
    err = (pbar.argmax(1) != lg)[counted].cpu().numpy()
    cb = np.minimum(np.floor(conf * 15).astype(np.int64), 14)
    ece = sum(abs((~err[cb == b]).sum() - conf[cb == b].sum()) for b in range(15)) / conf.size
    fb = np.minimum(np.floor(conf * t).astype(np.int64), t - 1)
    auroc = roc_auc_score(err, t - 1 - fb)
    top = pbar.topk(2, dim=1).values
    near = int(((top[:, 0] - top[:, 1]) < NEAR_TIE)[counted].sum())
    print(f"3 x flip: ECE {c['ece']:.5f} (ref {ece:.5f}), error AUROC {c['error_auroc']:.6f} (ref {auroc:.6f}), "
          f"Brier {c['brier']:.5f}, near ties {near}")
    assert abs(c["ece"] - ece) <= 1e-3
    assert abs(c["error_auroc"] - auroc) <= 1e-3
    assert c["counted"] == int(counted.sum())
    onehot = F.one_hot(lg.clamp(0, k - 1).long(), k).movedim(-1, 1).double()
    brier = float(((pbar - onehot) ** 2).sum(1)[counted].mean())
    assert abs(c["brier"] - brier) <= 1e-4
    assert abs(c["mean_entropy"] - float(hb.mean())) <= 1e-4
    assert abs(c["mean_mutual_info"] - float(mi.clamp(min=0).mean())) <= 1e-4


def test_invariants_with_the_existing_paths(members):
    """predict_uncertainty's labels are predict_labels'; calibration changes no loss, metric or curve; one member
    without TTA has no mutual information."""
    from innovative3D import models
    xg, lg = _batch(seed=5)
    ens = models.SpctEnsemble(members, tta="flip")
    a = ens.evaluate([(xg, lg)], sample_group=16, curves=256)
    b = ens.evaluate([(xg, lg)], sample_group=16, curves=256, calibration=960)
    assert torch.equal(a["tally"].confusion, b["tally"].confusion) and torch.equal(a["tally"].count, b["tally"].count)
    assert torch.equal(a["hist"], b["hist"])
    assert abs(a["loss"] - b["loss"]) <= 1e-12 * abs(a["loss"])
    for x, y in zip(a["metrics"], b["metrics"]):
        np.testing.assert_array_equal(np.asarray(x), np.asarray(y))
    np.testing.assert_array_equal(a["curves"]["auroc"], b["curves"]["auroc"])
    single = models.SpctEnsemble([members[0]])
    out = single.predict_uncertainty(xg, sample_group=16)
    print(f"one member: max MI {out['mutual_info'].float().max().item():.2e}")
    assert out["mutual_info"].float().min().item() >= 0 and out["mutual_info"].float().max().item() <= 1e-5
    assert torch.equal(out["labels"], single.predict_labels(xg, sample_group=16))


def test_determinism_and_host_batches(members):
    from innovative3D import models
    xg, lg = _batch(b=12, seed=3)
    ens = models.SpctEnsemble(members[:2], tta="flip")

    def run(x, lab):
        out = ens.eval_step((x, lab), sample_group=4, per_sample=True, calibration=64)
        return out["calib"], out["per_sample_calib"], out["uncertainty"], out["per_sample_uncertainty"]

    first = run(xg, lg)
    pu = ens.predict_uncertainty(xg, sample_group=4)
    for a, b in zip(first, run(xg, lg)):
        assert torch.equal(a, b)
    for a, b in zip(first, run(xg.cpu().pin_memory(), lg.cpu().to(torch.uint8).pin_memory())):
        assert torch.equal(a, b)
    again = ens.predict_uncertainty(xg.cpu(), sample_group=4)
    for key in pu:
        assert torch.equal(pu[key], again[key]), key
    # the uncertainty sums of eval_step are those of predict_uncertainty
    assert torch.equal(first[3], torch.stack([pu["case_entropy"], pu["case_mutual_info"]], 1))


def test_native_slices_two_members_flip(members):
    from innovative3D import models
    xg, _ = _batch(b=8, hw=512, seed=21)
    ens = models.SpctEnsemble(members[:2], tta="flip")
    _with_group(members[:2], 8)
    _, hb, mi = ref_uncertainty([m.model for m in members[:2]], xg, (0, 1, 2, 3))
    _with_group(members[:2], 256)
    out = ens.predict_uncertainty(xg, sample_group=8)
    e_err = (out["entropy"].double() - hb).abs()
    m_err = (out["mutual_info"].double() - mi).abs()
    print(f"512 x 512: max |H - ref| {e_err.max().item():.2e}, max |MI - ref| {m_err.max().item():.2e}")
    assert (e_err <= fp16_tol(hb, 5e-4)).all()
    assert (m_err <= fp16_tol(mi, 5e-4)).all()


def test_uncertainty_memory():
    from innovative3D import config as C
    from innovative3D import models
    torch.manual_seed(42)
    lits = [dict((v[0], v[1]) for v in C.VARIANTS)["SPFF-UNet"]().cuda() for _ in range(3)]
    g = torch.Generator(device="cuda").manual_seed(9)
    b = 64
    x = torch.randn(b, 1, 5, 128, 128, device="cuda", generator=g)
    ens = models.SpctEnsemble(lits, tta="flip")

    def peak(fn):
        fn()
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        fn()
        torch.cuda.synchronize()
        return torch.cuda.max_memory_allocated() - base

    labels = peak(lambda: ens.predict_labels(x, sample_group=16))
    unc = peak(lambda: ens.predict_uncertainty(x, sample_group=16))
    plane = 16 * 5 * 128 * 128 * 4
    outputs = 2 * b * 5 * 128 * 128 * 2 + 2 * 2**20
    print(f"peak above the resident set: predict_labels {labels / 2**20:.1f} MB, predict_uncertainty "
          f"{unc / 2**20:.1f} MB; entropy plane {plane / 2**20:.1f} MB + maps {outputs / 2**20:.1f} MB")
    assert unc - labels <= plane + outputs


def test_uncertainty_leaves_training_state_untouched():
    import copy

    from innovative3D import config as C
    from innovative3D import models
    from oracle import spff_oracle as O
    torch.manual_seed(42)
    a = dict((v[0], v[1]) for v in C.VARIANTS)["SPFF-UNet"]().cuda()
    x, lab = O.phantom_batch(4, 32, 32, seed=13, ignore_frac=0.02)
    a.fit_step((x.cuda(), lab.cuda()))
    snap = lambda m: ([p.detach().clone() for p in m.parameters()], m.fused_optimizer_state())   # noqa: E731
    before = snap(a)
    ens = models.SpctEnsemble([a, copy.deepcopy(a).model], tta="flip")
    ens.evaluate([(x.cuda(), lab.cuda()), (x, lab)], calibration=64)
    ens.eval_step((x, lab), per_sample=True, calibration=32)
    ens.predict_uncertainty(x.cuda())
    torch.cuda.synchronize()
    after = snap(a)
    assert all(torch.equal(p, q) for p, q in zip(after[0], before[0]))
    assert after[1]["step"] == before[1]["step"]
    assert torch.equal(after[1]["exp_avg"], before[1]["exp_avg"])
    assert torch.equal(after[1]["exp_avg_sq"], before[1]["exp_avg_sq"])
    assert all(p.grad is None for p in a.parameters())


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
    ev = ens.evaluate([(x[lo:lo + 1].cuda(), lab[lo:lo + 1].cuda()), (x[lo + 1:lo + 3], lab[lo + 1:lo + 3])],
                      calibration=64)
    out[rank] = dict(calib=ev["calib"].cpu(), cal={k: v for k, v in ev["calibration"].items() if np.isscalar(v)},
                     loss=ev["loss"])
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_calibration_equals_single_process():
    world = 2
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    ens, x, lab = _dp_setup()
    batches = [(x[lo:lo + 1].cuda(), lab[lo:lo + 1].cuda()) if i == 0 else (x[lo + 1:lo + 3], lab[lo + 1:lo + 3])
               for lo in (0, 3) for i in (0, 1)]
    ev = ens.evaluate(batches, calibration=64)
    for r in range(world):
        assert torch.equal(out[r]["calib"], ev["calib"].cpu())
        for key in ("ece", "mce", "error_auroc", "mean_entropy", "mean_mutual_info", "counted"):
            assert out[r]["cal"][key] == ev["calibration"][key], key
        assert abs(out[r]["cal"]["brier"] - ev["calibration"]["brier"]) <= 1e-12
        assert abs(out[r]["loss"] - ev["loss"]) <= 1e-12 * abs(ev["loss"])
