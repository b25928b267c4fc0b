"""GPU: the ranking statistics of the fused evaluation step. The kernel's softmax histograms (spff_head_eval_hist)
against F.conv3d logits -> fp64 softmax -> bins; evaluate(curves=T) against sklearn's exact AUROC on the weights the
reference trained; sample groups, host batches, the variants, memory, isolation from the training state, and data
parallelism.

Bin edges: the kernel computes p = e_c / se in fp32 from the tensor-core logits (W split into bf16 hi + lo, about 1e-5
from the fp32 logits), the reference in fp64 from fp32 logits. A (voxel, class) pair whose probability lies within
DELTA = 3e-5 of a bin edge i / T may land in either neighbouring bin, and each such pair moves at most one count out of
one bin into another (L1 change 2). So the histograms may differ by at most 2x the number of such pairs, and are
compared exactly everywhere else. DELTA is three times that logit error, carried into p (|dp| <= |dlogit| / 4 at most
for two classes, and p (1 - p) |dlogit| in general)."""
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


def ref_hist(logits, labels, k, t, ignore_index=255):
    """(hist int64 [K,2,T], near-edge pairs per class [K]) from fp32 logits [N,K,...] via an fp64 softmax."""
    p = torch.softmax(logits.double(), dim=1)
    counted = (labels != ignore_index) & (labels >= 0) & (labels < k)
    hist = torch.zeros(k, 2, t, dtype=torch.int64, device=logits.device)
    near = torch.zeros(k, dtype=torch.int64)
    lab = labels[counted]
    for c in range(k):
        pc = p[:, c][counted]
        b = (pc * t).floor().clamp(max=t - 1).long()
        hist[c, 0] = torch.bincount(b[lab == c], minlength=t)
        hist[c, 1] = torch.bincount(b[lab != c], minlength=t)
        near[c] = int(((pc * t - (pc * t).round()).abs() < DELTA * t).sum())
    return hist, near


def assert_hist_close(hist, ref, near, what=""):
    diff = (hist - ref).abs().sum(dim=(1, 2)).cpu()
    print(f"{what}: histogram L1 difference {diff.tolist()}, pairs within {DELTA} of a bin edge {near.tolist()}")
    assert (diff <= 2 * near).all(), (diff.tolist(), near.tolist())


def assert_confusion_identities(hist, confusion):
    assert torch.equal(hist[:, 0].sum(1), confusion.sum(1))                       # positives of c = row c
    assert torch.equal(hist.sum(dim=(1, 2)), confusion.sum().expand(hist.shape[0]))


# --------------------------------------------------------------------------------------------------------------------
# kernel
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,d,h,w,dtype,k,t", [(3, 5, 32, 32, torch.int64, 13, 256), (3, 5, 32, 32, torch.uint8, 13, 1024),
                                               (1, 5, 7, 9, torch.uint8, 5, 16), (2, 5, 12, 12, torch.int64, 16, 1000),
                                               (4, 5, 24, 20, torch.uint8, 16, 16), (2, 5, 40, 24, torch.int64, 5, 1024),
                                               (3, 5, 17, 31, torch.uint8, 13, 1000)])
def test_head_eval_hist(n, d, h, w, dtype, k, t):
    from spff_b200 import ops
    torch.backends.cudnn.allow_tf32 = False
    torch.manual_seed(3 + k + t)
    xb = pm(torch.randn(n, 32, d, h, w, device="cuda"), ld=64)
    wt = torch.randn(k, 32, 1, 1, 1, device="cuda") * 0.5
    b = torch.randn(k, device="cuda") * 0.1
    labels = torch.randint(0, k, (n, d, h, w), device="cuda")
    labels[torch.rand(n, d, h, w, device="cuda") < 0.1] = 255
    labels[torch.rand(n, d, h, w, device="cuda") < 0.02] = 20       # not a class: in nll / count, not in the histogram
    logits = F.conv3d(xb.permute(0, 4, 1, 2, 3).float(), wt, b)
    lab = labels.to(dtype)

    acc, cnt, conf = tally_bufs(k)
    s_acc, s_cnt, s_conf = sample_bufs(n, k)
    out = torch.full((n, d, h, w), 77, dtype=torch.uint8, device="cuda")
    hist = torch.zeros(k, 2, t, dtype=torch.int64, device="cuda")
    s_hist = torch.zeros(n, k, 2, t, dtype=torch.int64, device="cuda")
    ops.head_eval(xb, wt, b, lab, 255, acc, cnt, conf, s_acc, s_cnt, s_conf, out, hist=hist, sample_hist=s_hist)
    ref, near = ref_hist(logits, labels, k, t)
    assert_hist_close(hist, ref, near, f"k {k} T {t}")
    assert_confusion_identities(hist, conf)
    # per sample: rows sum to the batch, and each row is the histogram of that sample alone
    assert torch.equal(s_hist.sum(0), hist)
    for i in range(n):
        a1, c1, f1 = tally_bufs(k)
        h1 = torch.zeros(k, 2, t, dtype=torch.int64, device="cuda")
        ops.head_eval(xb[i:i + 1], wt, b, lab[i:i + 1], 255, a1, c1, f1, hist=h1)
        assert torch.equal(h1, s_hist[i])
    # the histogram leaves every other output as it is
    a0, c0, f0 = tally_bufs(k)
    sa0, sc0, sf0 = sample_bufs(n, k)
    out0 = torch.full((n, d, h, w), 77, dtype=torch.uint8, device="cuda")
    ops.head_eval(xb, wt, b, lab, 255, a0, c0, f0, sa0, sc0, sf0, out0)
    assert torch.equal(c0, cnt) and torch.equal(f0, conf) and torch.equal(out0, out)
    assert torch.equal(sc0, s_cnt) and torch.equal(sf0, s_conf)
    assert abs(float(a0) - float(acc)) <= 1e-12 * abs(float(acc))
    assert torch.allclose(sa0, s_acc, rtol=1e-12, atol=0)
    # accumulation: a second launch adds the same counts
    ops.head_eval(xb, wt, b, lab, 255, a0, c0, f0, hist=hist)
    assert torch.equal(hist, 2 * s_hist.sum(0))


def test_head_eval_hist_rejects_bad_arguments():
    from spff_b200._lib import Shape, call, ptr, stream_ptr
    k = 13
    x = torch.zeros(1, 5, 8, 8, 32, dtype=torch.bfloat16, device="cuda")
    wt, b = torch.zeros(k, 32, device="cuda"), torch.zeros(k, device="cuda")
    lab = torch.zeros(1, 5, 8, 8, dtype=torch.uint8, device="cuda")
    acc, cnt, conf = tally_bufs(k)
    s_acc, s_cnt, s_conf = sample_bufs(1, k)
    hist = torch.zeros(k, 2, 1024, dtype=torch.int64, device="cuda")

    def run(bins, h, per=(None, None, None), sh=None):
        call("spff_head_eval_hist", ptr(x), 32, 32, ptr(wt), ptr(b), ptr(lab), 1, 255, k, Shape(1, 5, 8, 8), ptr(acc),
             ptr(cnt), ptr(conf), *(ptr(p) for p in per), None, bins, ptr(h), ptr(sh), stream_ptr())

    with pytest.raises(RuntimeError, match="bins"):
        run(8, hist)
    with pytest.raises(RuntimeError, match="bins"):
        run(2048, hist)
    with pytest.raises(RuntimeError, match="null histogram"):
        run(256, None)
    with pytest.raises(RuntimeError, match="per-sample histogram"):
        run(256, hist, (s_acc, s_cnt, s_conf), None)
    with pytest.raises(RuntimeError, match="per-sample histogram"):
        run(256, hist, (None, None, None), hist)
    run(1024, hist, (s_acc, s_cnt, s_conf), torch.zeros(1, k, 2, 1024, dtype=torch.int64, device="cuda"))
    torch.cuda.synchronize()
    assert int(hist.sum()) == k * 5 * 8 * 8 and int(cnt) == 5 * 8 * 8


# --------------------------------------------------------------------------------------------------------------------
# model, on the weights the reference trained (loaded as test_eval_gpu.py's `trained` fixture loads them)
# --------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def trained():
    from test_parity_trained import FIX, batch, init_state, trained_weights
    z = np.load(FIX)
    lit = init_state()
    w = trained_weights(z, lit)
    lit = lit.cuda()
    lit.model.materialize(5)
    alias = {k.replace("freq_mask", "_mask"): v for k, v in w.items() if k.endswith("freq_mask")}
    lit.load_state_dict({**w, **alias}, strict=True)
    x, lab = batch()
    xg, lg = x.cuda(), lab.cuda()
    with torch.no_grad():
        logits = lit(xg)
    return lit, x, lab, logits


def test_evaluate_curves_on_reference_trained_weights(trained):
    from sklearn.metrics import average_precision_score, roc_auc_score

    from innovative3D.helpers import curves_from_hist, sample_curves
    lit, x, lab, logits = trained
    k, t = lit.hparams.num_classes, 256
    xg, lg = x.cuda(), lab.cuda()
    ev = lit.evaluate([(xg, lg)], curves=t)
    plain = lit.evaluate([(xg, lg)])
    # the histogram changes nothing else
    assert torch.equal(ev["tally"]._buf[1:], plain["tally"]._buf[1:])
    assert abs(float(ev["tally"].nll) - float(plain["tally"].nll)) <= 1e-12 * float(plain["tally"].nll)
    assert abs(ev["loss"] - plain["loss"]) <= 1e-12 * plain["loss"] and ev["voxels"] == plain["voxels"]
    for a, b in zip(ev["metrics"], plain["metrics"]):
        np.testing.assert_allclose(np.array(a, dtype=float), np.array(b, dtype=float), rtol=1e-12, equal_nan=True)
    hist = ev["hist"]
    assert_confusion_identities(hist, ev["tally"].confusion)
    ref, near = ref_hist(logits, lg, k, t)
    assert_hist_close(hist, ref, near, "trained weights")
    cv = ev["curves"]
    assert set(cv) >= {"fpr", "tpr", "roc_thresholds", "precision", "recall", "pr_thresholds", "auroc", "ap",
                       "auroc_tie_bound", "macro_auroc", "macro_ap"}
    # against sklearn's exact (unbinned) AUROC / AP on the fp64 softmax of model(x)
    p = torch.softmax(logits.double(), 1)
    counted = (lg != 255) & (lg < k)
    y = lg[counted].cpu().numpy()
    h = hist.cpu().numpy().astype(np.float64)
    d = (hist - ref).abs().sum(dim=(1, 2)).cpu().numpy()
    checked = 0
    for c in range(k):
        yc = (y == c).astype(np.int8)
        P, N = int(yc.sum()), int(yc.size - yc.sum())
        if P == 0 or N == 0:
            assert np.isnan(cv["auroc"][c])
            continue
        pc = p[:, c][counted].cpu().numpy()
        exact = roc_auc_score(yc, pc)
        # a pair moved across an edge changes its comparisons with at most one bin of the other kind
        slack = 0.5 * d[c] * max(h[c, 0].max(), h[c, 1].max()) / (P * N)
        err = abs(cv["auroc"][c] - exact)
        ap_err = abs(cv["ap"][c] - average_precision_score(yc, pc))
        print(f"class {c}: AUROC {cv['auroc'][c]:.6f} exact {exact:.6f} |diff| {err:.2e} tie bound "
              f"{cv['auroc_tie_bound'][c]:.2e} slack {slack:.2e}; AP {cv['ap'][c]:.6f} |diff| {ap_err:.2e}")
        assert err <= cv["auroc_tie_bound"][c] + slack + 1e-12
        # AP has no tie bound: the top bin (p >= 255/256) holds most positives with a few negatives, and binning
        # averages the precision over it; 0.05 is a loose ceiling on that effect, the printed value is the measurement
        assert ap_err <= 0.05
        checked += 1
    assert checked >= 2
    # per sample: rows sum to the batch histogram; sample_curves gives one row per case
    out = lit.eval_step((xg, lg), per_sample=True, curves=t)
    assert torch.equal(out["per_sample_hist"].sum(0), out["hist"]) and torch.equal(out["hist"], hist)
    per = sample_curves(out["per_sample_hist"])
    assert len(per) == x.shape[0]
    one = curves_from_hist(out["per_sample_hist"][5])
    np.testing.assert_array_equal(per[5][0], one["auroc"])
    assert lit.eval_step((xg, lg))["hist"] is None


def test_curve_schedule(trained):
    """Equal sample groups: host batches, uint8 labels, the dict form, accumulation and evaluate give the device
    histogram exactly. Across group sizes the activations differ in their last bits (test_eval_gpu), so the histograms
    differ only at pairs near a bin edge: each one is within 2x of the logits path's histogram."""
    lit, x, lab, logits = trained
    k, t = lit.hparams.num_classes, 256
    xg, lg = x.cuda(), lab.cuda()
    g16 = lit.eval_step((xg, lg), sample_group=16, curves=t)["hist"]
    assert torch.equal(lit.eval_step((x.pin_memory(), lab.to(torch.uint8).pin_memory()), sample_group=16, curves=t)["hist"], g16)
    assert torch.equal(lit.eval_step({"image": xg, "label": lg}, sample_group=16, curves=t)["hist"], g16)
    acc = lit.eval_step((xg[:64], lg[:64]), sample_group=16, curves=t)["hist"]
    lit.eval_step((x[64:], lab[64:]), sample_group=16, curves=acc)
    assert torch.equal(acc, g16)
    ev = lit.evaluate([(xg[:64], lg[:64]), (x[64:], lab[64:])], sample_group=16, curves=t)
    assert torch.equal(ev["hist"], g16)
    ref, near = ref_hist(logits, lg, k, t)
    for g in (3, 128):
        hg = lit.eval_step((xg, lg), sample_group=g, curves=t)["hist"]
        assert_hist_close(hg, ref, near, f"sample group {g}")
        assert int((hg - g16).abs().sum()) <= 4 * int(near.sum())
    with pytest.raises(ValueError):
        lit.eval_step((xg[:2], lg[:2]), curves=8)
    with pytest.raises(ValueError):
        lit.eval_step((xg[:2], lg[:2]), curves=torch.zeros(k, 2, 64, dtype=torch.int32, device="cuda"))


# --------------------------------------------------------------------------------------------------------------------
# variants
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("variant,h,w", [("PlainCore_UNet", 32, 32), ("SP_UNet", 24, 40)])
def test_variant_curves(variant, h, w):
    from innovative3D import config as C
    from oracle import spff_oracle as O
    torch.manual_seed(42)
    lit = dict((v[0], v[1]) for v in C.VARIANTS)[variant]().cuda()
    k, t = lit.hparams.num_classes, 128
    x, lab = O.phantom_batch(3, h, w, seed=11, ignore_frac=0.03)
    xg, lg = x.cuda(), lab.cuda()
    with torch.no_grad():
        logits = lit(xg)
    ev = lit.evaluate([(xg, lg)], curves=t)
    hist = ev["hist"]
    # SP_UNet runs on a padded batch; the padding carries ignore_index, so only the input's valid voxels count
    valid = int(((lg != 255) & (lg < k)).sum())
    assert torch.equal(hist.sum(dim=(1, 2)).cpu(), torch.full((k,), valid, dtype=torch.int64))
    assert_confusion_identities(hist, ev["tally"].confusion)
    ref, near = ref_hist(logits, lg, k, t)
    assert_hist_close(hist, ref, near, variant)
    out = lit.eval_step((xg, lg), per_sample=True, curves=t)
    assert tuple(out["per_sample_hist"].shape) == (3, k, 2, t) and torch.equal(out["per_sample_hist"].sum(0), hist)


@pytest.mark.parametrize("mode", ["train", "eval"])
def test_3dunet_curves(mode):
    from innovative3D import config as C
    from oracle import cicek_oracle as CO
    from oracle import spff_oracle as O
    lit = dict((v[0], v[1]) for v in C.VARIANTS)["3DUNet"]().cuda()
    lit.load_state_dict(CO.det_weights(seed=42), strict=True)
    getattr(lit, mode)()
    k, t = lit.hparams.num_classes, 64
    x, lab = O.phantom_batch(2, 32, 32, seed=12, ignore_frac=0.03)
    xg, lg = x.cuda(), lab.cuda()
    with torch.no_grad():
        logits = lit(xg)
    ign = 255 if lit.ignore_index is None else int(lit.ignore_index)
    ev = lit.evaluate([(xg, lg)], curves=t)
    plain = lit.evaluate([(xg, lg)])
    assert torch.equal(ev["tally"]._buf[1:], plain["tally"]._buf[1:])
    assert_confusion_identities(ev["hist"], ev["tally"].confusion)
    ref, near = ref_hist(logits, lg, k, t, ignore_index=ign)
    assert_hist_close(ev["hist"], ref, near, f"3DUNet {mode}")
    out = lit.eval_step((xg, lg), per_sample=True, curves=t)
    assert torch.equal(out["per_sample_hist"].sum(0), out["hist"]) and torch.equal(out["hist"], ev["hist"])


# --------------------------------------------------------------------------------------------------------------------
# memory and isolation
# --------------------------------------------------------------------------------------------------------------------
def test_curves_allocate_nothing_that_scales_with_the_logits():
    from innovative3D import config as C
    torch.manual_seed(42)
    lit = dict((v[0], v[1]) for v in C.VARIANTS)["SPFF-UNet"]().cuda()
    g = torch.Generator(device="cuda").manual_seed(7)
    x = torch.randn(64, 1, 5, 128, 128, device="cuda", generator=g)
    lab = torch.randint(0, 13, (64, 5, 128, 128), device="cuda", generator=g)

    def peak(**kw):
        lit.evaluate([(x, lab)], **kw)          # warm: buffers of this shape are cached by the engine
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        lit.evaluate([(x, lab)], **kw)
        torch.cuda.synchronize()
        return torch.cuda.max_memory_allocated() - base

    plain, curves = peak(), peak(curves=256)
    print(f"peak above the resident set: evaluate() {plain / 2**20:.1f} MB, evaluate(curves=256) {curves / 2**20:.1f} MB "
          f"(the fp32 logits would be {64 * 13 * 5 * 128 * 128 * 4 / 2**20:.0f} MB)")
    assert curves - plain < 16 * 2**20


def test_evaluate_curves_leaves_training_state_untouched():
    from innovative3D import config as C
    from oracle import spff_oracle as O
    torch.manual_seed(42)
    lit = dict((v[0], v[1]) for v in C.VARIANTS)["SPFF-UNet"]().cuda()
    x, lab = O.phantom_batch(4, 32, 32, seed=13, ignore_frac=0.02)
    lit.fit_step((x.cuda(), lab.cuda()))
    lit.fit_step((x.cuda(), lab.cuda()))
    snap = lambda: ([p.detach().clone() for p in lit.parameters()], lit._fused["grad"].clone(), lit._fused["m"].clone(),
                    lit._fused["v"].clone(), lit._fused["step"], float(lit.hparams.lr))
    before = snap()
    ev = lit.evaluate([(x.cuda(), lab.cuda()), (x, lab)], curves=64)
    lit.eval_step((x, lab), per_sample=True, return_labels=True, curves=32)
    torch.cuda.synchronize()
    after = snap()
    assert all(torch.equal(a, b) for a, b in zip(before[0], after[0]))
    for a, b in zip(before[1:4], after[1:4]):
        assert torch.equal(a, b)
    assert before[4:] == after[4:]
    assert all(p.grad is None for p in lit.parameters())
    assert int(ev["hist"].sum()) == 13 * int(((lab != 255) & (lab < 13)).sum()) * 2


# --------------------------------------------------------------------------------------------------------------------
# data parallel (2 ranks over NCCL; skipped on a single-GPU box)
# --------------------------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _dp_batches():
    from oracle import spff_oracle as O
    return O.phantom_batch(6, 32, 32, seed=79, ignore_frac=0.02)


def _worker(rank, world, port, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from innovative3D import config as C
    torch.manual_seed(42)
    lit = dict((v[0], v[1]) for v in C.VARIANTS)["SPFF-UNet"]().cuda()
    x, lab = _dp_batches()
    lo, hi = rank * 3, rank * 3 + 3
    ev = lit.evaluate([(x[lo:lo + 1].cuda(), lab[lo:lo + 1].cuda()), (x[lo + 1:hi], lab[lo + 1:hi])], curves=64)
    out[rank] = dict(hist=ev["hist"].cpu(), auroc=ev["curves"]["auroc"], ap=ev["curves"]["ap"])
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_curves_equal_single_process():
    world = 2
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    from innovative3D import config as C
    torch.manual_seed(42)
    lit = dict((v[0], v[1]) for v in C.VARIANTS)["SPFF-UNet"]().cuda()
    x, lab = _dp_batches()
    # the ranks' batches, concatenated: the same sample groups, so the same activations and exactly the same counts
    batches = [(x[lo:lo + 1].cuda(), lab[lo:lo + 1].cuda()) if i == 0 else (x[lo + 1:lo + 3], lab[lo + 1:lo + 3])
               for lo in (0, 3) for i in (0, 1)]
    ev = lit.evaluate(batches, curves=64)
    for r in range(world):
        assert torch.equal(out[r]["hist"], ev["hist"].cpu())
        np.testing.assert_array_equal(out[r]["auroc"], ev["curves"]["auroc"])
        np.testing.assert_array_equal(out[r]["ap"], ev["curves"]["ap"])
