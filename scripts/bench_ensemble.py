"""Ensembles and mirror test-time augmentation: `SpctEnsemble.predict_labels` and `evaluate(curves=256)` (the softmax
averaged on the device in an fp32 accumulator, no logits in memory) against the unfused torch path one would otherwise
write: per member and flip `member(torch.flip(x))`, softmax, flip back, sum into an fp32 [B,K,F,H,W] buffer, then
arg-max (prediction) or CE, confusion bincount and the per-class probability histogram (evaluation). SPFF-UNet, one
GPU, seeded weights (seeds 42, 123, 999) and inputs.

Configurations: members x tta = 1 x none, 1 x flip, 3 x flip, at the training batch x[1024,1,5,128,128] and the
inference scan x[256,1,5,512,512], resident on the device. All paths run in one process, alternating, after warm-up;
each call is timed whole with CUDA events and ends in a device->host copy of a small result (median of --reps); peak
allocated memory is taken over each call. A separate torch.profiler run times head_prob_accum_kernel and
prob_finalize_kernel inside the fused 3 x flip calls, with their achieved bytes/s against 7.7 TB/s (HBM3e of one B200,
data sheet) from the algorithmic bytes per position: accumulate 64 B of x + 64 B read and 64 B written of the
accumulator (no read at beta = 0), finalize 64 B of the accumulator + the 1-byte label (evaluation) + 1 B of arg-max
(prediction).

    python scripts/bench_ensemble.py --out DIR [--reps 3] [--warmup 1] [--sizes 1024x128,256x512]

Writes DIR/bench_ensemble.json. Fails without a CUDA device."""
import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "spff-unet-spcct_b200"), os.path.join(ROOT, "scripts")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from bench_eval import K, card, inputs, kernel_times, timed  # noqa: E402

BINS = 256
HBM_BYTES_PER_S = 7.7e12
FLIP_DIMS = {0: [], 1: [3], 2: [4], 3: [3, 4]}
CONFIGS = (("1xnone", 1, None), ("1xflip", 1, "flip"), ("3xflip", 3, "flip"))


@torch.no_grad()
def torch_sum_proba(lits, x, flips):
    """Sum over members and flips of flip(softmax(member(flip(x)))), fp32 [B,K,F,H,W]: the unfused path."""
    acc = None
    for lit in lits:
        for f in flips:
            d = FLIP_DIMS[f]
            p = torch.softmax(lit(torch.flip(x, d) if d else x), dim=1)
            p = torch.flip(p, d) if d else p
            if acc is None:
                acc = p
            else:
                acc += p
            del p
    return acc


@torch.no_grad()
def torch_predict(lits, x, flips):
    return torch_sum_proba(lits, x, flips).argmax(1).to(torch.uint8)


@torch.no_grad()
def torch_evaluate(lits, x, lab, flips):
    """The loss of evaluate (CE of the mean probability + 0.5 * (1 - hard macro Dice over classes 1..K-1)), from the
    confusion tally, and the [K,2,BINS] histogram, as evaluate(curves=BINS) has them."""
    pbar = torch_sum_proba(lits, x, flips)
    pbar /= len(lits) * len(flips)
    lab = lab.long()
    valid = lab != 255
    counted = valid & (lab < K)
    arg = pbar.argmax(1)
    y = lab[counted]
    py = pbar.gather(1, lab.clamp(max=K - 1).unsqueeze(1))[:, 0][counted]
    nll = -(py.clamp(min=torch.finfo(torch.float32).tiny).log().double().sum())
    conf = torch.bincount(y * K + arg[counted], minlength=K * K)
    hist = torch.empty(K, 2, BINS, dtype=torch.int64, device=pbar.device)
    for c in range(K):
        b = (pbar[:, c][counted] * BINS).long().clamp_(max=BINS - 1)
        hist[c] = torch.bincount(b + BINS * (y != c), minlength=2 * BINS).view(2, BINS)
    conf = conf.view(K, K).double()
    tp = conf.diagonal()
    dice = (2 * tp + 1e-6) / (conf.sum(0) + conf.sum(1) + 1e-6)     # 2tp + fp + fn = column + row sums
    loss = nll / valid.sum().clamp(min=1) + 0.5 * (1 - dice[1:].mean())
    return float(loss), int(hist.sum())


def kernel_rates(ens, x, lab, passes):
    """Profiler times and achieved bytes/s of the two ensemble kernels in one fused predict_labels and one evaluate."""
    voxels = x.shape[0] * x.shape[2] * x.shape[3] * x.shape[4]
    names = {"accumulate": ("head_prob_accum_kernel",), "finalize": ("prob_finalize_kernel",)}
    acc_bytes = voxels * (128 + (passes - 1) * 192)
    out = {}
    for call, fn, fin_bytes in (("predict_labels", lambda: ens.predict_labels(x), voxels * (64 + 1)),
                                ("evaluate", lambda: ens.evaluate([(x, lab)], curves=BINS), voxels * (64 + 1))):
        fn()
        kt = kernel_times(fn, names)
        res = {}
        for name, nbytes in (("accumulate", acc_bytes), ("finalize", fin_bytes)):
            ms = kt[name]["ms"]
            rate = nbytes / (ms * 1e-3) if ms > 0 else None
            res[name] = {"ms": ms, "launches": kt[name]["launches"], "algorithmic_bytes": nbytes, "bytes_per_s": rate,
                         "fraction_of_7.7TBps": rate / HBM_BYTES_PER_S if rate else None}
        out[call] = res
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--sizes", default="1024x128,256x512", help="BxHW list: batch size x slice size")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_ensemble: no CUDA device: this benchmark measures the GPU and has no CPU mode")
    os.makedirs(args.out, exist_ok=True)
    from innovative3D import config as C
    from innovative3D import models

    lits = []
    for seed in (42, 123, 999):
        torch.manual_seed(seed)
        lits.append(dict((v[0], v[1]) for v in C.VARIANTS)["SPFF-UNet"]().cuda().eval())
    result = {"card": card(), "model": "SPFF-UNet", "seeds": [42, 123, 999], "reps": args.reps, "bins": BINS, "runs": []}
    for spec in args.sizes.split(","):
        b, hw = (int(v) for v in spec.split("x"))
        x, lab = inputs(b, hw)
        voxels = b * 5 * hw * hw
        # every member's engine keeps its own inference buffers on the unfused path (model(x)); at 512 x 512 slices three
        # sets of groups sized for the whole free memory do not fit beside the unfused path's tensors, so both paths run
        # groups of 16 slices there
        group = 256 if hw <= 128 else 16
        for lit in lits:
            lit.model.sample_group = group
        paths = {}
        for cname, m, tta in CONFIGS:
            ens = models.SpctEnsemble(lits[:m], tta=tta)
            members, flips = lits[:m], ens.flips
            paths[f"{cname}/fused_predict"] = lambda ens=ens: int(ens.predict_labels(x)[0, 0, 0, 0])
            paths[f"{cname}/torch_predict"] = lambda mb=members, fl=flips: int(torch_predict(mb, x, fl)[0, 0, 0, 0])
            paths[f"{cname}/fused_evaluate"] = lambda ens=ens: ens.evaluate([(x, lab)], curves=BINS)["loss"]
            paths[f"{cname}/torch_evaluate"] = lambda mb=members, fl=flips: torch_evaluate(mb, x, lab, fl)[0]
        for _ in range(args.warmup):
            for fn in paths.values():
                fn()
        t = {n: [] for n in paths}
        peak, vals = {}, {}
        for _ in range(args.reps):
            for name, fn in paths.items():
                torch.cuda.synchronize()
                base = torch.cuda.memory_allocated()
                ms, mem, r = timed(fn)
                t[name].append(ms)
                peak[name] = max(peak.get(name, 0), mem - base)
                vals[name] = r
        run = {"batch": b, "hw": hw, "voxels": voxels, "sample_group": group, "logits_bytes_per_forward": voxels * K * 4}
        for name in paths:
            run[name] = {"ms_median": statistics.median(t[name]), "ms_all": t[name],
                         "peak_allocated_above_resident_bytes": peak[name], "value": vals[name]}
        for cname, _, _ in CONFIGS:
            for kind in ("predict", "evaluate"):
                f, u = run[f"{cname}/fused_{kind}"], run[f"{cname}/torch_{kind}"]
                run[f"{cname}/{kind}_torch_over_fused_time"] = u["ms_median"] / f["ms_median"]
                run[f"{cname}/{kind}_peak_saved_bytes"] = (u["peak_allocated_above_resident_bytes"]
                                                          - f["peak_allocated_above_resident_bytes"])
        run["loss_fused_minus_torch_3xflip"] = run["3xflip/fused_evaluate"]["value"] - run["3xflip/torch_evaluate"]["value"]
        run["kernels_3xflip"] = kernel_rates(models.SpctEnsemble(lits, tta="flip"), x, lab, passes=12)
        print(json.dumps(run), flush=True)
        result["runs"].append(run)
        del x, lab, paths
        for lit in lits:
            lit.model.engine.release_buffers()
        torch.cuda.empty_cache()
    with open(os.path.join(args.out, "bench_ensemble.json"), "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
