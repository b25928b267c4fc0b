"""Per-class ROC / PR statistics of the fused evaluation step (`evaluate(curves=T)`: the softmax histogram binned inside
the head kernel) against `evaluate()` without them and against what one would otherwise write on the GPU: `model(x)`,
softmax, and per class a bucketize + bincount of the probabilities of the counted voxels. SPFF-UNet, one GPU, seeded
inputs.

All paths run in one process, alternating, after warm-up; each call is timed whole with CUDA events and ends in a
device->host copy of its result (median of --reps). Sizes: the training batch x[1024,1,5,128,128] and the inference
scan x[256,1,5,512,512], with the batch resident on the device and streamed from pinned host memory. Peak allocated
memory is taken over each call. A separate torch.profiler run times head_eval_mma_kernel with and without the histogram
on one sample group of activations, for random logits (probabilities spread over the bins) and for peaked ones (W
scaled, labels = arg-max: almost every negative in bin 0 and every positive in bin T - 1, as with trained weights).

    python scripts/bench_curves.py --out DIR [--reps 5] [--warmup 2] [--sizes 1024x128,256x512]

Writes DIR/bench_curves.json. Fails without a CUDA device."""
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

TORCH_BINS = 256


def torch_hist(lit, x, lab, t=TORCH_BINS):
    """The unfused equivalent of evaluate(curves=t)'s histogram: logits, softmax, per-class bucketize + bincount."""
    with torch.no_grad():
        logits = lit(x)
        p = torch.softmax(logits, dim=1)
        lab = lab.to(p.device, non_blocking=True).long()
        counted = (lab != 255) & (lab < K)
        y = lab[counted]
        hist = torch.empty(K, 2, t, dtype=torch.int64, device=p.device)
        for c in range(K):
            b = (p[:, c][counted] * t).long().clamp_(max=t - 1)
            hist[c] = torch.bincount(b + t * (y != c), minlength=2 * t).view(2, t)
    return hist.cpu()


def head_kernel_times(k, t, launches=20, voxels=32 * 5 * 128 * 128):
    """torch.profiler time of head_eval_mma_kernel with and without the histogram, random and peaked logits."""
    from spff_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(5)
    n = voxels // (5 * 128 * 128)
    x = torch.randn(n, 5, 128, 128, 32, device="cuda", generator=g).to(torch.bfloat16)
    out = {}
    for kind, scale in (("random", 0.5), ("peaked", 4.0)):
        w = torch.randn(k, 32, device="cuda", generator=g) * scale
        b = torch.zeros(k, device="cuda")
        logits = torch.einsum("ndhwc,kc->ndhwk", x.float(), w)
        pmax = torch.softmax(logits, -1).amax(-1)
        lab = logits.argmax(-1).to(torch.uint8) if kind == "peaked" else \
            torch.randint(0, k, x.shape[:4], device="cuda", generator=g, dtype=torch.uint8)
        acc, cnt, conf = (torch.zeros(1, dtype=torch.float64, device="cuda"), torch.zeros(1, dtype=torch.int64, device="cuda"),
                          torch.zeros(k, k, dtype=torch.int64, device="cuda"))
        hist = torch.zeros(k, 2, t, dtype=torch.int64, device="cuda")
        runs = {"plain": lambda: ops.head_eval(x, w, b, lab, 255, acc, cnt, conf),
                "hist": lambda: ops.head_eval(x, w, b, lab, 255, acc, cnt, conf, hist=hist)}
        res = {"voxels": voxels, "frac_max_p_over_0.99": float((pmax > 0.99).float().mean())}
        for name, fn in runs.items():
            for _ in range(3):
                fn()

            def many(fn=fn):
                for _ in range(launches):
                    fn()
            kt = kernel_times(many, {"k": ("head_eval_mma_kernel",)})["k"]
            res[name] = {"ms_per_launch": kt["ms"] / max(kt["launches"], 1), "launches": kt["launches"]}
        res["hist_over_plain"] = res["hist"]["ms_per_launch"] / res["plain"]["ms_per_launch"]
        out[kind] = res
        del logits, pmax, lab
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--sizes", default="1024x128,256x512", help="BxHW list: batch size x slice size")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_curves: no CUDA device: this benchmark measures the GPU and has no CPU mode")
    os.makedirs(args.out, exist_ok=True)
    from innovative3D import config as C
    from innovative3D.helpers import curves_from_hist

    torch.manual_seed(42)
    lit = dict((v[0], v[1]) for v in C.VARIANTS)["SPFF-UNet"]().cuda().eval()
    result = {"card": card(), "model": "SPFF-UNet", "sample_group": lit.model.sample_group, "reps": args.reps,
              "torch_bins": TORCH_BINS, "runs": []}
    paths = {
        "evaluate": lambda x, lab: lit.evaluate([(x, lab)])["loss"],
        "curves256": lambda x, lab: lit.evaluate([(x, lab)], curves=256)["curves"]["macro_auroc"],
        "curves1024": lambda x, lab: lit.evaluate([(x, lab)], curves=1024)["curves"]["macro_auroc"],
        "torch": lambda x, lab: curves_from_hist(torch_hist(lit, x, lab))["macro_auroc"],
    }
    for spec in args.sizes.split(","):
        b, hw = (int(v) for v in spec.split("x"))
        xd, labd = inputs(b, hw)
        voxels = b * 5 * hw * hw
        for mode in ("resident", "host"):
            x, lab = (xd.cpu().pin_memory(), labd.cpu().pin_memory()) if mode == "host" else (xd, labd)
            for _ in range(args.warmup):
                for fn in paths.values():
                    fn(x, lab)
            t = {n: [] for n in paths}
            peak, vals = {}, {}
            for _ in range(args.reps):
                for name, fn in paths.items():
                    ms, mem, r = timed(lambda: fn(x, lab))
                    t[name].append(ms)
                    peak[name] = max(peak.get(name, 0), mem)
                    vals[name] = r
            run = {"batch": b, "hw": hw, "mode": mode, "voxels": voxels, "logits_bytes": voxels * K * 4}
            for name in paths:
                med = statistics.median(t[name])
                run[name] = {"ms_median": med, "ms_all": t[name], "peak_allocated_bytes": peak[name], "value": vals[name]}
            base = run["evaluate"]["ms_median"]
            for name in ("curves256", "curves1024", "torch"):
                run[name]["over_evaluate"] = run[name]["ms_median"] / base
                run[name]["peak_over_evaluate_bytes"] = peak[name] - peak["evaluate"]
            run["macro_auroc_fused256_minus_torch256"] = vals["curves256"] - vals["torch"]
            print(json.dumps(run), flush=True)
            result["runs"].append(run)
            del x, lab
        del xd, labd
        lit.model.engine.release_buffers()
        torch.cuda.empty_cache()
    result["head_kernel"] = {f"T{t}": head_kernel_times(K, t) for t in (256, 1024)}
    print(json.dumps(result["head_kernel"]), flush=True)
    with open(os.path.join(args.out, "bench_curves.json"), "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
