"""GPU: ensembles and mirror test-time augmentation (SpctEnsemble). The two kernels (spff_head_prob_accum,
spff_prob_finalize) against torch; the flip gather against torch.flip; one member without TTA against the single-model
fused path on the weights the reference trained; three members x four flips against the per-member
model(torch.flip(x)) -> fp64 softmax -> flip back -> mean reference; determinism, host batches, memory, isolation from
the training state, native 512 x 512 slices and two ranks.

Tolerances. The kernels' logits come from the tensor-core head (W split into bf16 hi + lo), about 1e-5 from the fp32
logits of model(x) (the CUDA-core head), so a probability is within about 3e-5 of the reference's. Arg-max maps are
compared exactly outside voxels whose two largest reference probabilities are within NEAR_TIE = 1e-4; histograms outside
pairs within DELTA = 3e-5 of a bin edge (as in test_curves_gpu)."""
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
FLT_MIN = float(np.finfo(np.float32).tiny)
FLIPS = {0: [], 1: [3], 2: [4], 3: [3, 4]}      # flip code -> dims of a [B,C,F,H,W] tensor


def pm(x, ld):  # NCDHW fp32 -> position-major bf16 channel slice of a wider buffer
    n, c, d, h, w = x.shape
    buf = torch.zeros(n, d, h, w, ld, dtype=torch.bfloat16, device=x.device)
    buf[..., :c] = x.permute(0, 2, 3, 4, 1).to(torch.bfloat16)
    return buf[..., :c]


def tally_bufs(k, dev="cuda"):
    return (torch.zeros(1, dtype=torch.float64, device=dev), torch.zeros(1, dtype=torch.int64, device=dev),
            torch.zeros(k, k, dtype=torch.int64, device=dev))


def sample_bufs(n, k, dev="cuda"):
    return (torch.zeros(n, dtype=torch.float64, device=dev), torch.zeros(n, dtype=torch.int64, device=dev),
            torch.zeros(n, k, k, dtype=torch.int64, device=dev))


def ref_tally(pbar, lab, k, ignore_index=255):
    """(nll fp64, count, confusion [k,k], arg-max) of p̄ (any float dtype, [B,K,...]) by the rules of spff_prob_finalize."""
    valid = lab != ignore_index
    inr = valid & (lab >= 0) & (lab < k)
    arg = pbar.argmax(1)
    py = pbar.gather(1, lab.clamp(0, k - 1).unsqueeze(1))[:, 0]
    nll = -(py[inr].double().clamp(min=FLT_MIN).log()).sum()
    conf = torch.bincount(lab[inr] * k + arg[inr], minlength=k * k).view(k, k)
    return nll, int(valid.sum()), conf, arg


def ref_hist(pbar, lab, k, t, ignore_index=255, delta=DELTA):
    """(hist int64 [K,2,T], pairs within `delta` of a bin edge per class [K]) of p̄ [B,K,...]."""
    counted = (lab != ignore_index) & (lab >= 0) & (lab < k)
    hist = torch.zeros(k, 2, t, dtype=torch.int64, device=pbar.device)
    near = torch.zeros(k, dtype=torch.int64)
    lb = lab[counted]
    for c in range(k):
        pc = pbar[:, c][counted]
        b = (pc * t).floor().clamp(max=t - 1).long()
        hist[c, 0] = torch.bincount(b[lb == c], minlength=t)
        hist[c, 1] = torch.bincount(b[lb != c], minlength=t)
        near[c] = int(((pc.double() * t - (pc.double() * t).round()).abs() < delta * t).sum())
    return hist, near


def near_ties(p):
    """Voxels [B,...] whose two largest probabilities of p [B,K,...] are within NEAR_TIE."""
    top = p.topk(2, dim=1).values
    return (top[:, 0] - top[:, 1]) < NEAR_TIE


def tally_loss(nll, count, conf, k):
    from spff_b200.engine import LossTally
    t = LossTally(k, "cuda")
    t.nll.fill_(float(nll))
    t.count.fill_(int(count))
    t.confusion.copy_(conf)
    return float(t.loss())


@torch.no_grad()
def ref_ensemble(cores, x, flips):
    """Mean over members and flips of flip(softmax(core(flip(x))), fp64) [B,K,F,H,W]."""
    acc = None
    for core in cores:
        for f in flips:
            p = torch.softmax(core(torch.flip(x, FLIPS[f])).double(), 1)
            p = torch.flip(p, FLIPS[f])
            acc = p if acc is None else acc + p
    return acc / (len(cores) * len(flips))


# --------------------------------------------------------------------------------------------------------------------
# kernels
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [2, 5, 13, 16])
@pytest.mark.parametrize("n,d,h,w", [(1, 5, 7, 9), (3, 5, 17, 31), (2, 5, 16, 16)])
def test_head_prob_accum(k, n, d, h, w):
    from spff_b200 import ops
    torch.backends.cudnn.allow_tf32 = False
    torch.manual_seed(5 + k + h)
    xb = pm(torch.randn(n, 32, d, h, w, device="cuda"), ld=64)
    wt = torch.randn(k, 32, 1, 1, 1, device="cuda") * 0.5
    b = torch.randn(k, device="cuda") * 0.1
    p = torch.softmax(F.conv3d(xb.permute(0, 4, 1, 2, 3).float(), wt, b).double(), 1)   # [n,k,d,h,w]
    total = n * d * h * w * 16
    store = torch.full((total + 64,), 7.0, device="cuda")       # 64 guard floats past the accumulator
    acc = store[:total].view(n, d, h, w, 16)
    ref = torch.zeros(n, d, h, w, 16, dtype=torch.float64, device="cuda")
    for i, f in enumerate((0, 1, 2, 3, 3, 0)):
        beta = 0 if i == 0 else 1
        ops.head_prob_accum(xb, wt, b, acc, flip=f, beta=beta)
        ref[..., :k] += torch.flip(p, FLIPS[f]).permute(0, 2, 3, 4, 1)
        if i == 0:
            assert torch.equal(acc[..., k:], torch.zeros_like(acc[..., k:]))      # beta = 0 writes the padding
            acc[..., k:] = 5.0                                                     # ... beta = 1 never touches it
        err = (acc[..., :k].double() - ref[..., :k]).abs().max().item()
        assert err <= 3e-5, (f, i, err)
    assert torch.equal(acc[..., k:], torch.full_like(acc[..., k:], 5.0))
    assert torch.equal(store[total:], torch.full((64,), 7.0, device="cuda"))
    # beta = 0 replaces whatever was there (no memset needed): NaN garbage included
    acc.fill_(float("nan"))
    ops.head_prob_accum(xb, wt, b, acc, flip=2, beta=0)
    assert not torch.isnan(acc).any()
    assert (acc[..., :k].double() - torch.flip(p, [4]).permute(0, 2, 3, 4, 1)).abs().max().item() <= 3e-5


@pytest.mark.parametrize("dtype", [torch.uint8, torch.int64])
@pytest.mark.parametrize("k,t", [(13, 256), (5, 16), (16, 1024), (2, 64)])
def test_prob_finalize(dtype, k, t):
    from spff_b200 import ops
    n, d, h, w = 3, 5, 17, 31
    g = torch.Generator(device="cuda").manual_seed(k * 7 + t)
    # sums of 3 passes on a coarse grid: many exact ties (the first maximum wins), zeros (the FLT_MIN clamp)
    acc = torch.full((n, d, h, w, 16), 100.0, device="cuda")           # classes >= k must be ignored
    acc[..., :k] = torch.randint(0, 7, (n, d, h, w, k), device="cuda", generator=g).float() * 0.125
    scale = 1.0 / 3.0
    lab = torch.randint(0, k, (n, d, h, w), device="cuda", generator=g)
    lab[torch.rand(n, d, h, w, device="cuda", generator=g) < 0.1] = 255          # ignored
    lab[torch.rand(n, d, h, w, device="cuda", generator=g) < 0.03] = 200         # not a class: counted only
    lab = lab.to(dtype)
    pbar = (acc[..., :k] * scale).permute(0, 4, 1, 2, 3).contiguous()            # fp32, the kernel's p̄
    nll_r, cnt_r, conf_r, arg_r = ref_tally(acc[..., :k].permute(0, 4, 1, 2, 3), lab.long(), k)
    # the arg-max is taken on acc, and the p̄ of the nll is the fp32 product
    nll_r = -(pbar.gather(1, lab.long().clamp(0, k - 1).unsqueeze(1))[:, 0][(lab.long() < k)].double()
              .clamp(min=FLT_MIN).log()).sum()
    hist_r, _ = ref_hist(pbar, lab.long(), k, t, delta=0)

    tl = tally_bufs(k)
    per = sample_bufs(n, k)
    out = torch.full((n, d, h, w), 77, dtype=torch.uint8, device="cuda")
    proba = torch.empty(n, k, d, h, w, dtype=torch.float16, device="cuda")
    hist = torch.zeros(k, 2, t, dtype=torch.int64, device="cuda")
    s_hist = torch.zeros(n, k, 2, t, dtype=torch.int64, device="cuda")
    ops.prob_finalize(acc, k, scale, labels=lab, tally=tl, per_sample=per, labels_out=out, hist=hist,
                      sample_hist=s_hist, proba_out=proba)
    assert torch.equal(out, arg_r.to(torch.uint8))
    assert torch.equal(proba, pbar.half())
    assert int(tl[1]) == cnt_r and torch.equal(tl[2], conf_r)
    assert abs(float(tl[0]) - float(nll_r)) <= 1e-5 * abs(float(nll_r))
    assert torch.equal(hist, hist_r)
    for i in range(n):
        nl, c, cf, _ = ref_tally(acc[i:i + 1, ..., :k].permute(0, 4, 1, 2, 3), lab[i:i + 1].long(), k)
        assert int(per[1][i]) == c and torch.equal(per[2][i], cf)
        hi, _ = ref_hist(pbar[i:i + 1], lab[i:i + 1].long(), k, t, delta=0)
        assert torch.equal(s_hist[i], hi)
    assert torch.allclose(per[0].sum(), tl[0], rtol=1e-12, atol=0)
    # without labels: the arg-max and the probabilities only; with labels but no extras: the same tally
    out2 = torch.empty_like(out)
    proba2 = torch.empty_like(proba)
    ops.prob_finalize(acc, k, scale, labels_out=out2, proba_out=proba2)
    assert torch.equal(out2, out) and torch.equal(proba2, proba)
    tl2 = tally_bufs(k)
    ops.prob_finalize(acc, k, scale, labels=lab, tally=tl2)
    assert torch.equal(tl2[1], tl[1]) and torch.equal(tl2[2], tl[2])


def test_prob_kernels_reject_bad_arguments():
    from spff_b200._lib import Shape, call, ptr, stream_ptr
    k = 13
    x = torch.zeros(1, 5, 8, 8, 32, dtype=torch.bfloat16, device="cuda")
    wt, b = torch.zeros(k, 32, device="cuda"), torch.zeros(k, device="cuda")
    store = torch.zeros(5 * 8 * 8 * 16 + 4, device="cuda")
    acc, bad = store[:-4], store[1:-3]          # 16-byte aligned / 4 bytes off
    lab = torch.zeros(1, 5, 8, 8, dtype=torch.uint8, device="cuda")
    tl = tally_bufs(k)
    per = sample_bufs(1, k)
    hist = torch.zeros(k, 2, 64, dtype=torch.int64, device="cuda")
    s1 = Shape(1, 5, 8, 8)

    def accum(kk=k, flip=0, a=acc, s=s1, beta=0):
        call("spff_head_prob_accum", ptr(x), 32, 32, ptr(wt), ptr(b), kk, s, flip, beta, ptr(a), stream_ptr())

    def fin(kk=k, a=acc, s=s1, bins=64, h=hist, p=(None, None, None), sh=None):
        call("spff_prob_finalize", ptr(a), kk, s, 1.0, ptr(lab), 1, 255, *(ptr(v) for v in tl), *(ptr(v) for v in p),
             None, bins, ptr(h), ptr(sh), None, stream_ptr())

    for kk in (1, 17):
        with pytest.raises(RuntimeError, match="classes"):
            accum(kk=kk)
        with pytest.raises(RuntimeError, match="classes"):
            fin(kk=kk)
    with pytest.raises(RuntimeError, match="flip"):
        accum(flip=4)
    with pytest.raises(RuntimeError, match="flip"):
        accum(flip=-1)
    with pytest.raises(RuntimeError, match="beta"):
        accum(beta=2)
    with pytest.raises(RuntimeError, match="aligned"):
        accum(a=bad)
    with pytest.raises(RuntimeError, match="aligned"):
        fin(a=bad)
    for bins in (8, 2048):
        with pytest.raises(RuntimeError, match="bins"):
            fin(bins=bins)
    with pytest.raises(RuntimeError, match="per-sample histogram"):
        fin(sh=torch.zeros(1, k, 2, 64, dtype=torch.int64, device="cuda"))
    with pytest.raises(RuntimeError, match="per-sample histogram"):
        fin(p=per)
    big = Shape(65536, 1, 1, 1)
    with pytest.raises(RuntimeError, match="65535"):
        accum(s=big)
    with pytest.raises(RuntimeError, match="65535"):
        fin(s=big)
    accum()
    fin(p=per, sh=torch.zeros(1, k, 2, 64, dtype=torch.int64, device="cuda"))
    torch.cuda.synchronize()
    assert int(tl[1]) == 5 * 8 * 8


@pytest.mark.parametrize("flip", [1, 2, 3])
def test_flip_gather_is_torch_flip(flip):
    from spff_b200.engine import _FlipGather
    x = torch.randn(6, 1, 5, 24, 40, device="cuda", generator=torch.Generator(device="cuda").manual_seed(flip))
    out = torch.full_like(x, float("nan"))
    _FlipGather(8, 24, 40, x.device)(x, out, flip)
    assert torch.equal(out, torch.flip(x, FLIPS[flip]))


# --------------------------------------------------------------------------------------------------------------------
# model, on the weights the reference trained
# --------------------------------------------------------------------------------------------------------------------
def _load_trained():
    from test_parity_trained import FIX, init_state, trained_weights
    z = np.load(FIX)
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


def _batch(b=16, hw=128, seed=42):
    from oracle import spff_oracle as O
    x, lab = O.phantom_batch(b, hw, hw, seed=seed, ignore_frac=0.01)
    return x.cuda(), lab.cuda()


def test_single_member_without_tta_is_the_single_model(members):
    from innovative3D import models
    lit = members[0]
    k = lit.hparams.num_classes
    xg, lg = _batch()
    ens = models.SpctEnsemble([lit])
    a = ens.eval_step((xg, lg), return_labels=True, sample_group=16)
    b = lit.eval_step((xg, lg), return_labels=True, sample_group=16)
    with torch.no_grad():
        p = torch.softmax(lit(xg).double(), 1)
    near = near_ties(p)
    diff = a["labels"] != b["labels"]
    print(f"identity: {int(diff.sum())} labels differ, {int(near.sum())} near-tie voxels")
    assert not (diff & ~near).any()
    assert int((a["tally"].confusion - b["tally"].confusion).abs().sum()) <= 2 * int(diff.sum())
    assert torch.equal(a["tally"].count, b["tally"].count)
    la, lb = float(a["loss"]), float(b["loss"])
    assert abs(la - lb) <= 1e-5 * abs(lb), (la, lb)
    pa = ens.predict_labels(xg, sample_group=16)
    lit.model.sample_group, sg = 16, lit.model.sample_group
    try:
        pb = lit.model.predict_labels(xg)
    finally:
        lit.model.sample_group = sg
    assert torch.equal(pa, a["labels"])
    assert not ((pa != pb) & ~near).any()


def test_three_members_flip_tta_against_torch(members):
    from innovative3D import models
    k, t = 13, 256
    xg, lg = _batch(seed=7)
    ens = models.SpctEnsemble(members, tta="flip")
    for m in members:
        m.model.sample_group = 16
    pref = ref_ensemble([m.model for m in members], xg, (0, 1, 2, 3))
    for m in members:
        m.model.sample_group = 256
    proba = ens.predict_proba(xg, sample_group=16)
    assert proba.dtype == torch.float16 and tuple(proba.shape) == (16, k, 5, 128, 128)
    err = (proba.double() - pref).abs().max().item()
    print(f"3 x flip: max |proba - ref| {err:.2e}")
    assert err <= 5e-4
    near = near_ties(pref)
    labels = ens.predict_labels(xg, sample_group=16)
    assert not ((labels.long() != pref.argmax(1)) & ~near).any()
    ev = ens.evaluate([(xg, lg)], sample_group=16, curves=t)
    nll_r, cnt_r, conf_r, _ = ref_tally(pref, lg, k)
    conf_d = int((ev["tally"].confusion - conf_r).abs().sum())
    print(f"3 x flip: confusion L1 difference {conf_d}, near-tie voxels {int(near.sum())}")
    assert conf_d <= 2 * int(near.sum()) and int(ev["tally"].count) == cnt_r
    assert abs(float(ev["tally"].nll) - float(nll_r)) <= 1e-5 * float(nll_r)
    ref_loss = tally_loss(nll_r, cnt_r, conf_r, k)
    assert abs(ev["loss"] - ref_loss) <= 1e-5 * ref_loss, (ev["loss"], ref_loss)
    hr, nr = ref_hist(pref, lg, k, t)
    hd = (ev["hist"] - hr).abs().sum(dim=(1, 2)).cpu()
    print(f"3 x flip: histogram L1 {hd.tolist()}, near-edge pairs {nr.tolist()}")
    assert (hd <= 2 * nr).all()
    assert set(ev["curves"]) >= {"auroc", "ap", "macro_auroc", "macro_ap"}
    assert ev["voxels"] == lg.numel() and len(ev["metrics"]) == 9


def test_determinism_group_sizes_and_host_batches(members):
    from innovative3D import models
    xg, lg = _batch(b=12, seed=3)
    ens = models.SpctEnsemble(members[:2], tta="flip")

    def run(x, lab, g):
        out = ens.eval_step((x, lab), return_labels=True, sample_group=g, curves=128)
        return out["labels"], ens.predict_proba(x.cuda(), sample_group=g), out["tally"].confusion, out["hist"]

    first = run(xg, lg, 4)
    again = run(xg, lg, 4)
    for a, b in zip(first, again):
        assert torch.equal(a, b)
    host = run(xg.cpu().pin_memory(), lg.cpu().to(torch.uint8).pin_memory(), 4)
    for a, b in zip(first, host):
        assert torch.equal(a, b)
    other = run(xg, lg, 12)
    near = near_ties(ref_ensemble([m.model for m in members[:2]], xg, (0, 1, 2, 3)))
    diff = other[0] != first[0]
    print(f"group 4 vs 12: {int(diff.sum())} labels differ, {int(near.sum())} near-tie voxels")
    assert not (diff & ~near).any()
    assert (other[1].float() - first[1].float()).abs().max().item() <= 1e-3
    assert int((other[2] - first[2]).abs().sum()) <= 2 * int(diff.sum())


def test_ensemble_memory():
    from innovative3D import config as C
    from innovative3D import models
    torch.manual_seed(42)
    lits = [dict((v[0], v[1]) for v in C.VARIANTS)["SPFF-UNet"]().cuda() for _ in range(3)]
    g = torch.Generator(device="cuda").manual_seed(9)
    x = torch.randn(64, 1, 5, 128, 128, device="cuda", generator=g)
    ens = models.SpctEnsemble(lits, tta="flip")
    lits[0].model.sample_group = 16

    def peak(fn):
        fn()
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        fn()
        torch.cuda.synchronize()
        return torch.cuda.max_memory_allocated() - base

    single = peak(lambda: lits[0].model.predict_labels(x))
    both = peak(lambda: ens.predict_labels(x, sample_group=16))
    per_pos = 16 * 5 * 128 * 128
    bound = per_pos * 64 + per_pos * 4 + 16 * 2**20
    logits = 64 * 13 * 5 * 128 * 128 * 4
    print(f"peak above the resident set: predict_labels {single / 2**20:.1f} MB, 3 x flip ensemble {both / 2**20:.1f} MB; "
          f"bound {bound / 2**20:.1f} MB above the single model; the batch's fp32 logits {logits / 2**20:.0f} MB")
    assert both - single <= bound
    assert both < logits / 2


def test_ensemble_leaves_training_state_untouched():
    """The members' parameters and fused optimizer state are bitwise what they were before the ensemble ran, and equal
    to a control copy that never ran it. The fused training step itself is not bit-reproducible run to run (its
    weight-gradient reductions are not ordered), so the step that follows is compared with the control's to 1 % of the
    Adam step size."""
    import copy

    from innovative3D import config as C
    from innovative3D import models
    from oracle import spff_oracle as O
    torch.manual_seed(42)
    a = dict((v[0], v[1]) for v in C.VARIANTS)["SPFF-UNet"]().cuda()
    x, lab = O.phantom_batch(4, 32, 32, seed=13, ignore_frac=0.02)
    a.fit_step((x.cuda(), lab.cuda()))
    ctrl = copy.deepcopy(a)
    ctrl.load_fused_optimizer_state(a.fused_optimizer_state())
    snap = lambda m: ([p.detach().clone() for p in m.parameters()], m.fused_optimizer_state())
    before = snap(a)
    other = copy.deepcopy(a)
    ens = models.SpctEnsemble([a, other.model], tta="flip")
    ens.evaluate([(x.cuda(), lab.cuda()), (x, lab)], curves=64)
    ens.eval_step((x, lab), per_sample=True, return_labels=True, curves=32)
    ens.predict_proba(x.cuda())
    torch.cuda.synchronize()
    for ref in (before, snap(ctrl)):
        after = snap(a)
        assert all(torch.equal(p, q) for p, q in zip(after[0], ref[0]))
        assert after[1]["step"] == ref[1]["step"] and after[1]["lr"] == ref[1]["lr"]
        assert torch.equal(after[1]["exp_avg"], ref[1]["exp_avg"])
        assert torch.equal(after[1]["exp_avg_sq"], ref[1]["exp_avg_sq"])
    assert all(p.grad is None for p in a.parameters())
    la = float(a.fit_step((x.cuda(), lab.cuda()))["loss"])
    lc = float(ctrl.fit_step((x.cuda(), lab.cuda()))["loss"])
    diff = max((p - q).abs().max().item() for p, q in zip(a.parameters(), ctrl.parameters()))
    print(f"following fit_step: loss {la} vs control {lc}, max |parameter difference| {diff:.2e}")
    assert abs(la - lc) <= 1e-5 * abs(lc)
    assert diff <= 1e-6


def test_native_slices_two_members_flip(members):
    from innovative3D import models
    k = 13
    xg, lg = _batch(b=8, hw=512, seed=21)
    ens = models.SpctEnsemble(members[:2], tta="flip")
    for m in members[:2]:
        m.model.sample_group = 8
    pref = ref_ensemble([m.model for m in members[:2]], xg, (0, 1, 2, 3))
    for m in members[:2]:
        m.model.sample_group = 256
    proba = ens.predict_proba(xg, sample_group=8)
    err = (proba.double() - pref).abs().max().item()
    near = near_ties(pref)
    out = ens.eval_step((xg, lg), return_labels=True, sample_group=8)
    diff = out["labels"].long() != pref.argmax(1)
    print(f"512 x 512: max |proba - ref| {err:.2e}, {int(diff.sum())} labels differ, {int(near.sum())} near ties")
    assert err <= 5e-4
    assert not (diff & ~near).any()
    nll_r, cnt_r, conf_r, _ = ref_tally(pref, lg, k)
    assert int((out["tally"].confusion - conf_r).abs().sum()) <= 2 * int(near.sum())
    assert abs(float(out["tally"].nll) - float(nll_r)) <= 1e-5 * float(nll_r)


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
    ev = ens.evaluate([(x[lo:lo + 1].cuda(), lab[lo:lo + 1].cuda()), (x[lo + 1:lo + 3], lab[lo + 1:lo + 3])], curves=64)
    out[rank] = dict(hist=ev["hist"].cpu(), conf=ev["tally"].confusion.cpu(), loss=ev["loss"], voxels=ev["voxels"])
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_ensemble_equals_single_process():
    world = 2
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    ens, x, lab = _dp_setup()
    batches = [(x[lo:lo + 1].cuda(), lab[lo:lo + 1].cuda()) if i == 0 else (x[lo + 1:lo + 3], lab[lo + 1:lo + 3])
               for lo in (0, 3) for i in (0, 1)]
    ev = ens.evaluate(batches, curves=64)
    for r in range(world):
        assert torch.equal(out[r]["hist"], ev["hist"].cpu())
        assert torch.equal(out[r]["conf"], ev["tally"].confusion.cpu())
        assert out[r]["voxels"] == ev["voxels"]
        assert abs(out[r]["loss"] - ev["loss"]) <= 1e-12 * abs(ev["loss"])
