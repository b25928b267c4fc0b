"""GPU: the fused evaluation step. The kernel (spff_head_eval) against F.conv3d -> cross entropy -> confusion; the model
drivers (eval_step / evaluate) against the logits path of this tree (model(x) -> ce_plus_macro_dice_loss ->
per_class_metrics_3d) and against the reference's stored numbers on the weights the reference trained; sample groups,
host batches, the variants, isolation from the training state, and data parallelism.

Near ties: the fused head computes the logits with tensor cores (W split into bf16 hi + lo) and the logits path with fp32
FMAs, so a voxel whose two largest logits are within 1e-5 of each other (relative, floor 1) may take either arg-max;
such voxels are excluded from the exact comparisons."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

K = 13


def pm(x, ld):  # NCDHW fp32 -> position-major bf16 channel slice of a wider buffer
    n, c, d, h, w = x.shape
    buf = torch.zeros(n, d, h, w, ld, dtype=torch.bfloat16, device=x.device)
    buf[..., :c] = x.permute(0, 2, 3, 4, 1).to(torch.bfloat16)
    return buf[..., :c]


def near_ties(logits):
    top = logits.topk(2, dim=1).values
    return (top[:, 0] - top[:, 1]) <= 1e-5 * top[:, 0].abs().clamp(min=1.0)


def tally_bufs(n, k, dev="cuda"):
    return (torch.zeros(1, dtype=torch.float64, device=dev), torch.zeros(1, dtype=torch.int64, device=dev),
            torch.zeros(k, k, dtype=torch.int64, device=dev))


def sample_bufs(n, k, dev="cuda"):
    return (torch.zeros(n, dtype=torch.float64, device=dev), torch.zeros(n, dtype=torch.int64, device=dev),
            torch.zeros(n, k, k, dtype=torch.int64, device=dev))


# --------------------------------------------------------------------------------------------------------------------
# kernel
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,d,h,w,dtype", [(2, 5, 12, 12, torch.int64), (1, 5, 7, 9, torch.uint8), (3, 5, 32, 32, torch.int64),
                                           (3, 5, 32, 32, torch.uint8), (2, 5, 12, 12, torch.uint8)])
def test_head_eval(n, d, h, w, dtype):
    """head_eval == F.conv3d -> cross entropy (ignore_index 255) -> confusion, per batch and per sample."""
    from oracle import spff_oracle as O
    from spff_b200 import ops
    torch.backends.cudnn.allow_tf32 = False
    torch.manual_seed(2)
    xb = pm(torch.randn(n, 32, d, h, w, device="cuda"), ld=64)
    wt = torch.randn(K, 32, 1, 1, 1, device="cuda") * 0.5
    b = torch.randn(K, device="cuda") * 0.1
    labels = torch.randint(0, K, (n, d, h, w), device="cuda")
    labels[torch.rand(n, d, h, w, device="cuda") < 0.1] = 255
    labels[torch.rand(n, d, h, w, device="cuda") < 0.02] = 20       # not a class: counted in nll / count, not in confusion
    logits = F.conv3d(xb.permute(0, 4, 1, 2, 3).float(), wt, b)
    valid = labels != 255
    inr = valid & (labels < K)
    lse = logits.logsumexp(1)
    picked = logits.gather(1, labels.clamp(max=K - 1).unsqueeze(1))[:, 0]
    nll_ref = torch.where(inr, lse - picked, lse)[valid].double()
    lab = labels.to(dtype)

    acc, cnt, conf = tally_bufs(n, K)
    s_acc, s_cnt, s_conf = sample_bufs(n, K)
    out = torch.full((n, d, h, w), 77, dtype=torch.uint8, device="cuda")
    ops.head_eval(xb, wt, b, lab, 255, acc, cnt, conf, s_acc, s_cnt, s_conf, out)
    ties = near_ties(logits)
    assert int(cnt) == int(valid.sum())
    assert abs(float(acc) / int(cnt) - float(nll_ref.mean())) < 1e-5
    assert (out.long() == logits.argmax(1))[~ties].all()
    assert (conf.cpu().numpy() == O.confusion(out.cpu(), labels.cpu(), K, 255)).all()      # labels_out is what is tallied
    # per sample: sums to the batch, and each row is the tally of that sample alone
    assert torch.equal(s_cnt.sum(), cnt[0]) and torch.equal(s_conf.sum(0), conf)
    assert abs(float(s_acc.sum()) - float(acc)) <= 1e-12 * abs(float(acc))
    for i in range(n):
        a1, c1, f1 = tally_bufs(1, K)
        ops.head_eval(xb[i:i + 1], wt, b, lab[i:i + 1], 255, a1, c1, f1)
        assert int(c1) == int(s_cnt[i]) and torch.equal(f1, s_conf[i])
        assert abs(float(a1) - float(s_acc[i])) <= 1e-5 * abs(float(a1))
    # every optional pointer NULL: the same batch tally
    a2, c2, f2 = tally_bufs(n, K)
    ops.head_eval(xb, wt, b, lab, 255, a2, c2, f2)
    assert torch.equal(c2, cnt) and torch.equal(f2, conf)
    assert abs(float(a2) - float(acc)) <= 1e-12 * abs(float(acc))


def test_head_eval_rejects_partial_per_sample_arrays():
    from spff_b200 import _lib
    from spff_b200._lib import Shape, call, ptr, stream_ptr
    x = torch.zeros(1, 5, 8, 8, 32, dtype=torch.bfloat16, device="cuda")
    wt, b = torch.zeros(K, 32, device="cuda"), torch.zeros(K, device="cuda")
    lab = torch.zeros(1, 5, 8, 8, dtype=torch.uint8, device="cuda")
    acc, cnt, conf = tally_bufs(1, K)
    with pytest.raises(RuntimeError, match="per-sample"):
        call("spff_head_eval", ptr(x), 32, 32, ptr(wt), ptr(b), ptr(lab), 1, 255, K, Shape(1, 5, 8, 8), ptr(acc), ptr(cnt),
             ptr(conf), ptr(acc), None, None, None, stream_ptr())
    assert _lib.lib.spff_version() >= 100


# --------------------------------------------------------------------------------------------------------------------
# model, on the weights the reference trained (as test_parity_trained.py loads them)
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
    return z, lit, x, lab


def _logits_path(lit, x, lab):
    from innovative3D import helpers as H
    with torch.no_grad():
        logits = lit(x)
    loss = float(lit.compute_loss(logits, lab.long()))
    metrics = H.per_class_metrics_3d(logits, lab, K, ignore_index=255)
    return logits, loss, metrics


def _assert_tally_matches_logits(tally, logits, lab, voxels=None):
    """confusion of the fused tally == that of the logits' arg-max, apart from near-tie voxels."""
    from oracle import spff_oracle as O
    cm = tally.confusion.cpu().numpy()
    ref = O.confusion(logits.argmax(1).cpu(), lab.cpu(), K, 255)
    ties = int((near_ties(logits) & (lab != 255)).sum())
    assert int(np.abs(cm - ref).sum()) <= 2 * ties, (int(np.abs(cm - ref).sum()), ties)
    assert int(tally.count) == int((lab != 255).sum())
    return ties


def test_eval_step_on_reference_trained_weights(trained):
    from innovative3D import helpers as H
    z, lit, x, lab = trained
    xg, lg = x.cuda(), lab.cuda()
    logits, ref_loss, ref_m = _logits_path(lit, xg, lg)
    out = lit.eval_step((xg, lg), per_sample=True, return_labels=True)
    loss = float(out["loss"])
    ties = _assert_tally_matches_logits(out["tally"], logits, lg)
    m = H.metrics_from_confusion(out["tally"].confusion.cpu().numpy(), lab.numel())
    print(f"fused eval: loss {loss:.6f} (logits path {ref_loss:.6f}, reference {float(z['loss']):.6f}), macro dice "
          f"{m[3]:.6f} (logits path {ref_m[3]:.6f}, reference {float(z['scalars'][0]):.6f}), near ties {ties}")
    assert abs(loss - ref_loss) <= 1e-5 * abs(ref_loss)
    if ties == 0:
        for a, b in zip(m, ref_m):
            np.testing.assert_allclose(np.array(a, dtype=float), np.array(b, dtype=float), rtol=1e-12, equal_nan=True)
    assert abs(m[3] - ref_m[3]) <= 1e-5
    # the reference's own numbers, at the parity tolerances
    assert abs(loss - float(z["loss"])) <= 1e-3 * max(1.0, float(z["loss"]))
    assert abs(m[3] - float(z["scalars"][0])) <= 1e-3
    # arg-max map
    pred = lit.model.predict_labels(xg)
    assert float((out["labels"] == pred).float().mean()) >= 0.9999
    # per sample: rows sum to the batch; per-case metrics of a few samples equal the logits path on that sample
    nll, cnt, conf = out["per_sample"]
    assert torch.equal(cnt.sum(), out["tally"].count[0]) and torch.equal(conf.sum(0), out["tally"].confusion)
    assert abs(float(nll.sum()) - float(out["tally"].nll)) <= 1e-12 * float(out["tally"].nll)
    per = H.sample_metrics(out["per_sample"], 5 * 64 * 64)
    assert len(per) == 128
    from oracle import spff_oracle as O
    for i in (0, 63, 127):
        if int(near_ties(logits[i:i + 1]).sum()) == 0:
            ref_i = O.metrics_from_confusion(O.confusion(logits[i].argmax(0).cpu(), lab[i], K, 255), 5 * 64 * 64)
            np.testing.assert_allclose(np.array(per[i][3:], dtype=float), np.array(ref_i[3:], dtype=float), rtol=1e-12,
                                       equal_nan=True)


def test_sample_groups_and_host_batches(trained):
    """The tally is exact for the activations it is given. The activations themselves carry the group size in their last
    bits (the InstanceNorm statistics are reduced over work slots that depend on the group's sample count), so across
    group sizes the confusion may differ only where the two arg-max maps differ, and those are near ties (rare)."""
    z, lit, x, lab = trained
    xg, lg = x.cuda(), lab.cuda()
    whole = lit.eval_step((xg, lg), sample_group=128, return_labels=True)
    by3 = lit.eval_step((xg, lg), sample_group=3, return_labels=True)
    valid = lg != 255
    flips = int(((whole["labels"] != by3["labels"]) & valid).sum())
    assert torch.equal(whole["tally"].count, by3["tally"].count)
    assert int((whole["tally"].confusion - by3["tally"].confusion).abs().sum()) <= 2 * flips
    assert flips <= 1e-4 * int(valid.sum())
    assert abs(float(whole["tally"].nll) - float(by3["tally"].nll)) <= 1e-6 * float(whole["tally"].nll)
    # same group size: host batches through StagedBatch, uint8 labels, the dict form, accumulation over two calls and
    # evaluate all give the device tally exactly
    g16 = lit.eval_step((xg, lg), sample_group=16)["tally"]
    same = lambda t: torch.equal(t.count, g16.count) and torch.equal(t.confusion, g16.confusion) and \
        abs(float(t.nll) - float(g16.nll)) <= 1e-12 * float(g16.nll)
    assert same(lit.eval_step((x.pin_memory(), lab.to(torch.uint8).pin_memory()), sample_group=16)["tally"])
    assert same(lit.eval_step({"image": xg, "label": lg}, sample_group=16)["tally"])
    acc = lit.eval_step((xg[:64], lg[:64]), sample_group=16)["tally"]
    lit.eval_step((x[64:], lab[64:]), tally=acc, sample_group=16)
    assert same(acc)
    ev = lit.evaluate([(xg[:64], lg[:64]), (x[64:], lab[64:])], sample_group=16)
    assert same(ev["tally"]) and ev["voxels"] == lab.numel()
    assert abs(ev["loss"] - float(g16.loss())) <= 1e-6 * ev["loss"]


# --------------------------------------------------------------------------------------------------------------------
# variants
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("variant,h,w", [("PlainCore_UNet", 32, 32), ("SP_UNet", 24, 40)])
def test_variants_match_the_logits_path(variant, h, w):
    from innovative3D import config as C
    from oracle import spff_oracle as O
    torch.manual_seed(42)
    lit = dict((v[0], v[1]) for v in C.VARIANTS)[variant]().cuda()
    x, lab = O.phantom_batch(3, h, w, seed=11, ignore_frac=0.03)
    xg, lg = x.cuda(), lab.cuda()
    logits, ref_loss, ref_m = _logits_path(lit, xg, lg)
    assert tuple(logits.shape[2:]) == (5, h, w)
    ev = lit.evaluate([(xg, lg)])
    ties = _assert_tally_matches_logits(ev["tally"], logits, lg)
    assert ev["voxels"] == lab.numel()
    assert abs(ev["loss"] - ref_loss) <= 1e-5 * abs(ref_loss)
    if ties == 0:
        for a, b in zip(ev["metrics"], ref_m):
            np.testing.assert_allclose(np.array(a, dtype=float), np.array(b, dtype=float), rtol=1e-12, equal_nan=True)
    out = lit.eval_step((xg, lg), return_labels=True)
    assert tuple(out["labels"].shape) == (3, 5, h, w)
    assert (out["labels"].long() == logits.argmax(1))[~near_ties(logits)].all()


@pytest.mark.parametrize("mode", ["train", "eval"])
def test_3dunet_matches_loss_and_log(mode):
    from innovative3D import config as C
    from innovative3D import helpers as H
    from oracle import cicek_oracle as CO
    from oracle import spff_oracle as O
    lit = dict((v[0], v[1]) for v in C.VARIANTS)["3DUNet"]().cuda()
    lit.load_state_dict(CO.det_weights(seed=42), strict=True)
    getattr(lit, mode)()
    x, lab = O.phantom_batch(2, 32, 32, seed=12, ignore_frac=0.03)
    xg, lg = x.cuda(), lab.cuda()
    with torch.no_grad():
        logits = lit(xg)
    # _loss_and_log's loss and macro Dice, without its Lightning logging
    ref_loss = float(lit._weighted_softmax_ce(logits, lg) * lit.ce_weight)
    ref_m = H.per_class_metrics_3d(logits, lg, K, ignore_index=lit.ignore_index)
    ev = lit.evaluate([(xg, lg)])
    ties = _assert_tally_matches_logits(ev["tally"], logits, lg)
    assert abs(ev["loss"] - ref_loss) <= 1e-5 * abs(ref_loss)
    if ties == 0:
        assert abs(ev["metrics"][3] - ref_m[3]) <= 1e-12
    out = lit.eval_step((xg, lg), per_sample=True, return_labels=True)
    assert abs(float(out["loss"]) - ref_loss) <= 1e-5 * abs(ref_loss)
    assert tuple(out["labels"].shape) == (2, 5, 32, 32) and torch.equal(out["per_sample"][2].sum(0), out["tally"].confusion)


# --------------------------------------------------------------------------------------------------------------------
# isolation from the training state
# --------------------------------------------------------------------------------------------------------------------
def test_evaluate_leaves_training_state_untouched():
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
    ev = lit.evaluate([(x.cuda(), lab.cuda()), (x, lab)])
    lit.eval_step((x, lab), per_sample=True, return_labels=True)
    torch.cuda.synchronize()
    after = snap()
    assert all(torch.equal(a, b) for a, b in zip(before[0], after[0]))
    for a, b in zip(before[1:4], after[1:4]):
        assert torch.equal(a, b)
    assert before[4:] == after[4:]
    assert all(p.grad is None for p in lit.parameters())
    assert ev["voxels"] == 2 * lab.numel()


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
    ev = lit.evaluate([(x[lo:lo + 1].cuda(), lab[lo:lo + 1].cuda()), (x[lo + 1:hi], lab[lo + 1:hi])])
    out[rank] = dict(buf=ev["tally"]._buf.cpu(), loss=ev["loss"], metrics=ev["metrics"], voxels=ev["voxels"])
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_evaluate_equals_single_process():
    world = 2
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    from innovative3D import config as C
    torch.manual_seed(42)
    lit = dict((v[0], v[1]) for v in C.VARIANTS)["SPFF-UNet"]().cuda()
    x, lab = _dp_batches()
    ev = lit.evaluate([(x.cuda(), lab.cuda())])
    ref = ev["tally"]._buf.cpu()
    for r in range(world):
        buf = out[r]["buf"]
        assert torch.equal(buf[1:], ref[1:])                                      # count, confusion
        nll, nll_ref = float(buf[0:1].view(torch.float64)), float(ref[0:1].view(torch.float64))
        assert abs(nll - nll_ref) <= 1e-9 * abs(nll_ref)
        assert out[r]["voxels"] == lab.numel()
        assert abs(out[r]["loss"] - ev["loss"]) <= 1e-6 * ev["loss"]
        for a, b in zip(out[r]["metrics"], ev["metrics"]):
            np.testing.assert_allclose(np.array(a, dtype=float), np.array(b, dtype=float), rtol=0, atol=0, equal_nan=True)
    assert out[0]["loss"] == out[1]["loss"]
