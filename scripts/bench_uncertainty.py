"""Uncertainty maps and calibration of ensembles and mirror test-time augmentation: `SpctEnsemble.predict_uncertainty`
against `predict_labels`, `evaluate(curves=256, calibration=960)` against `evaluate(curves=256)`, and both against the
unfused torch path one would otherwise write: per member and flip `member(torch.flip(x))`, softmax, flip back, fp32 sums
of p and of H(p) over the passes, then H[p̄], the mutual information, the arg-max and a confidence bucketize + bincount.
SPFF-UNet, one GPU, seeded weights (seeds 42, 123, 999) and inputs.

Configurations: members x tta = 1 x none and 3 x flip, at x[1024,1,5,128,128] and x[256,1,5,512,512], resident on the
device. All paths run in one process, alternating, after warm-up; each call is timed whole with CUDA events and ends in
a device->host copy of a small result (median of --reps); peak allocated memory is taken over each call, above the
resident set. A separate torch.profiler run times the two new kernels (head_prob_accum_kernel<ENT = true>,
prob_finalize_kernel<., ., UNC = true>) next to the kernels they extend, with achieved bytes/s against 7.7 TB/s (HBM3e
of one B200, data sheet) from the algorithmic bytes per position: accumulate 64 B of x + 64 B of the accumulator written
(beta = 0) or read and written (beta = 1), plus 4 B of the entropy plane written or 8 B read and written; finalize 64 B
of the accumulator + 1 B of arg-max + 4 B of the entropy plane + 2 x 2 B of fp16 maps (prediction), or + 1 B of label
(evaluation). The card's name, power limit and max SM clock are read in the same run.

    python scripts/bench_uncertainty.py --out DIR [--reps 3] [--warmup 1] [--sizes 1024x128,256x512]

Writes DIR/bench_uncertainty.json. Fails without a CUDA device."""
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

BINS, CAL = 256, 960
HBM_BYTES_PER_S = 7.7e12
FLIP_DIMS = {0: [], 1: [3], 2: [4], 3: [3, 4]}
CONFIGS = (("1xnone", 1, None), ("3xflip", 3, "flip"))
KERNELS = {
    "accumulate": ("head_prob_accum_kernel<false>", "head_prob_accum_kernelILb0EE"),
    "accumulate_ent": ("head_prob_accum_kernel<true>", "head_prob_accum_kernelILb1EE"),
    "finalize": tuple(f"prob_finalize_kernel<{t}, {h}, false, false>" for t in ("unsigned char", "long long")
                      for h in ("false", "true")),
    "finalize_unc": tuple(f"prob_finalize_kernel<{t}, {h}, true, false>" for t in ("unsigned char", "long long")
                          for h in ("false", "true")),
}


def _entropy(p):
    return -(p * torch.where(p > 0, p.log(), torch.zeros_like(p))).sum(1)


@torch.no_grad()
def torch_uncertainty(lits, x, lab, flips):
    """The unfused path: fp32 sums of flip(softmax(member(flip(x)))) and of its entropy over the passes; H[p̄], MI,
    arg-max, and the [3,CAL] confidence histogram of the counted voxels."""
    acc = hsum = None
    for lit in lits:
        for f in flips:
            d = FLIP_DIMS[f]
            p = torch.softmax(lit(torch.flip(x, d) if d else x), dim=1)
            p = torch.flip(p, d) if d else p
            h = _entropy(p)
            if acc is None:
                acc, hsum = p, h
            else:
                acc += p
                hsum += h
            del p, h
    acc /= len(lits) * len(flips)
    hb = _entropy(acc)
    mi = (hb - hsum / (len(lits) * len(flips))).clamp_(min=0)
    conf, arg = acc.max(1)
    del acc
    lab = lab.long()
    counted = (lab != 255) & (lab < K)
    c = conf[counted]
    b = (c * CAL).long().clamp_(max=CAL - 1)
    hist = torch.stack([torch.bincount(b, minlength=CAL), torch.bincount(b[arg[counted] == lab[counted]], minlength=CAL),
                        torch.zeros(CAL, dtype=torch.int64, device=x.device).index_add_(0, b, (c * 2**24).round().long())])
    return float(hb.double().mean()), float(mi.double().mean()), arg.to(torch.uint8), hist


def kernel_rates(ens, x, lab, passes):
    """Profiler times and achieved bytes/s of the accumulate / finalize kernels, with and without uncertainty."""
    v = x.shape[0] * x.shape[2] * x.shape[3] * x.shape[4]
    acc = v * (128 + (passes - 1) * 192)
    acc_ent = acc + v * (4 + (passes - 1) * 8)
    calls = (("predict_labels", lambda: ens.predict_labels(x), {"accumulate": acc, "finalize": v * 65}),
             ("predict_uncertainty", lambda: ens.predict_uncertainty(x),
              {"accumulate_ent": acc_ent, "finalize_unc": v * (65 + 4 + 4)}),
             ("evaluate", lambda: ens.evaluate([(x, lab)], curves=BINS), {"accumulate": acc, "finalize": v * 65}),
             ("evaluate_calibration", lambda: ens.evaluate([(x, lab)], curves=BINS, calibration=CAL),
              {"accumulate_ent": acc_ent, "finalize_unc": v * (65 + 4)}))
    out = {}
    for call, fn, kinds in calls:
        fn()
        kt = kernel_times(fn, {k: KERNELS[k] for k in kinds})
        res = {}
        for name, nbytes in kinds.items():
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
        raise SystemExit("bench_uncertainty: no CUDA device: this benchmark measures the GPU and has no CPU mode")
    os.makedirs(args.out, exist_ok=True)
    from innovative3D import config as C
    from innovative3D import models

    lits = []
    for seed in (42, 123, 999):
        torch.manual_seed(seed)
        lits.append(dict((v[0], v[1]) for v in C.VARIANTS)["SPFF-UNet"]().cuda().eval())
    result = {"card": card(), "model": "SPFF-UNet", "seeds": [42, 123, 999], "reps": args.reps, "bins": BINS,
              "calibration_bins": CAL, "runs": []}
    for spec in args.sizes.split(","):
        b, hw = (int(v) for v in spec.split("x"))
        x, lab = inputs(b, hw)
        voxels = b * 5 * hw * hw
        # as in bench_ensemble: groups of 16 slices at 512 x 512, where three members' buffers sized for the whole free
        # memory do not fit beside the unfused path's tensors
        group = 256 if hw <= 128 else 16
        for lit in lits:
            lit.model.sample_group = group
        paths = {}
        for cname, m, tta in CONFIGS:
            ens = models.SpctEnsemble(lits[:m], tta=tta)
            members, flips = lits[:m], ens.flips
            paths[f"{cname}/predict_labels"] = lambda ens=ens: int(ens.predict_labels(x)[0, 0, 0, 0])
            paths[f"{cname}/predict_uncertainty"] = lambda ens=ens: float(ens.predict_uncertainty(x)["case_entropy"].mean())
            paths[f"{cname}/evaluate"] = lambda ens=ens: ens.evaluate([(x, lab)], curves=BINS)["loss"]
            paths[f"{cname}/evaluate_calibration"] = \
                lambda ens=ens: ens.evaluate([(x, lab)], curves=BINS, calibration=CAL)["calibration"]["ece"]
            paths[f"{cname}/torch_uncertainty"] = lambda mb=members, fl=flips: torch_uncertainty(mb, x, lab, fl)[0]
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
        run = {"batch": b, "hw": hw, "voxels": voxels, "sample_group": group,
               "entropy_plane_bytes_per_group": group * 5 * hw * hw * 4}
        for name in paths:
            run[name] = {"ms_median": statistics.median(t[name]), "ms_all": t[name],
                         "peak_allocated_above_resident_bytes": peak[name], "value": vals[name]}
        for cname, _, _ in CONFIGS:
            r = lambda n: run[f"{cname}/{n}"]["ms_median"]   # noqa: E731
            run[f"{cname}/uncertainty_over_labels_time"] = r("predict_uncertainty") / r("predict_labels")
            run[f"{cname}/calibration_over_evaluate_time"] = r("evaluate_calibration") / r("evaluate")
            run[f"{cname}/torch_over_fused_uncertainty_time"] = r("torch_uncertainty") / r("predict_uncertainty")
        run["case_entropy_fused_vs_torch_3xflip"] = [run["3xflip/predict_uncertainty"]["value"],
                                                     run["3xflip/torch_uncertainty"]["value"]]
        run["kernels_3xflip"] = kernel_rates(models.SpctEnsemble(lits, tta="flip"), x, lab, passes=12)
        print(json.dumps(run), flush=True)
        result["runs"].append(run)
        del x, lab, paths
        for lit in lits:
            lit.model.engine.release_buffers()
        torch.cuda.empty_cache()
    with open(os.path.join(args.out, "bench_uncertainty.json"), "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
