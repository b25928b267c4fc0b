"""Temperature scaling of ensembles and mirror test-time augmentation: `SpctEnsemble.fit_temperature` against
`evaluate(calibration=960)` on the same data (one pass each), against `evaluate(calibration=960)` at the fitted
temperature, and against the unfused torch path one would otherwise write: per member and flip `member(torch.flip(x))`,
softmax, flip back, the fp32 p̄ of the whole set kept in memory, then `torch.optim.LBFGS` on β = 1/T of
cross_entropy(β log p̄, y). SPFF-UNet, one GPU, seeded weights (seeds 42, 123, 999) and inputs. The labels are the first
member's arg-max with 30 % of the voxels replaced by a random class and 1 % ignored, so that the nll has its minimum at
a finite temperature (against random labels the seeded random members are best at T -> infinity).

Configurations: members x tta = 1 x none and 3 x flip, at x[1024,1,5,128,128] and x[256,1,5,512,512] (groups of 16
slices at 512 x 512), resident on the device. All paths run in one process, alternating, after warm-up; each call is
timed whole with CUDA events and ends in a device->host copy of a small result (median of --reps); peak allocated memory
is taken over each call, above the resident set. A separate torch.profiler run times the fit kernel
(prob_temp_fit_kernel + its reduction) and the finishing pass with and without the temperature
(prob_finalize_kernel<., ., UNC = true, TEMP>) inside the 3 x flip calls, and sets the fit kernel against one forward
(the fit call's time over its member x flip passes). The card's name, power limit and max SM clock are read in the
same run.

    python scripts/bench_temperature.py --out DIR [--reps 3] [--warmup 1] [--sizes 1024x128,256x512]

Writes DIR/bench_temperature.json. Fails without a CUDA device."""
import argparse
import json
import os
import statistics
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "spff-unet-spcct_b200"), os.path.join(ROOT, "scripts")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from bench_eval import card, inputs, kernel_times, timed  # noqa: E402

CAL = 960
FLIP_DIMS = {0: [], 1: [3], 2: [4], 3: [3, 4]}
CONFIGS = (("1xnone", 1, None), ("3xflip", 3, "flip"))
KERNELS = {
    "fit": ("prob_temp_fit_kernel", "prob_temp_fit_reduce_kernel"),
    "finalize_unc": tuple(f"prob_finalize_kernel<{t}, {h}, true, false>" for t in ("unsigned char", "long long")
                          for h in ("false", "true")),
    "finalize_unc_tempered": tuple(f"prob_finalize_kernel<{t}, {h}, true, true>" for t in ("unsigned char", "long long")
                                   for h in ("false", "true")),
    "accumulate": ("head_prob_accum_kernel",),
}


@torch.no_grad()
def torch_pbar(lits, x, flips):
    """fp32 p̄ of the whole set: the sum of flip(softmax(member(flip(x)))) over the passes, divided by their number."""
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
    return acc.div_(len(lits) * len(flips))


def torch_fit(lits, x, lab, flips, chunk=16):
    """The unfused fit: p̄ kept, then LBFGS (strong Wolfe) on β of the mean tempered nll; returns T. The objective and
    its gradient are summed over chunks of `chunk` samples: at x[256,1,5,512,512] the logits tensor has 4.4e9 elements,
    and cross_entropy over all of it at once ends in an illegal memory access (32-bit indexing inside the torch kernel)."""
    logp = torch_pbar(lits, x, flips).clamp_(min=torch.finfo(torch.float32).tiny).log_()
    y = lab.long()
    counted = int((y != 255).sum())
    beta = torch.ones(1, device=x.device, requires_grad=True)
    opt = torch.optim.LBFGS([beta], lr=1.0, max_iter=50, line_search_fn="strong_wolfe", tolerance_grad=1e-9,
                            tolerance_change=1e-12)

    def closure():
        opt.zero_grad()
        total = torch.zeros((), device=x.device)
        for lo in range(0, logp.shape[0], chunk):
            loss = F.cross_entropy(beta * logp[lo:lo + chunk], y[lo:lo + chunk], ignore_index=255,
                                   reduction="sum") / counted
            loss.backward()
            total += loss.detach()
        return total
    opt.step(closure)
    return 1.0 / float(beta.detach())


def kernel_rates(ens, x, lab, t_fit):
    """Profiler times of the fit kernel in fit_temperature and of the finishing pass in evaluate(calibration=960) at
    T = 1 and at the fitted T, next to the accumulate kernel of the same calls."""
    out = {}
    calls = (("fit_temperature", lambda: ens.fit_temperature([(x, lab)], apply=False), ("fit", "accumulate")),
             ("evaluate_calibration", lambda: ens.evaluate([(x, lab)], calibration=CAL),
              ("finalize_unc", "accumulate")),
             ("evaluate_calibration_tempered",
              lambda: tempered(ens, t_fit, lambda: ens.evaluate([(x, lab)], calibration=CAL)),
              ("finalize_unc_tempered", "accumulate")))
    for name, fn, kinds in calls:
        fn()
        kt = kernel_times(fn, {k: KERNELS[k] for k in kinds})
        out[name] = {k: kt[k] for k in kinds}
    return out


def tempered(ens, t, fn):
    ens.temperature = t
    try:
        return fn()
    finally:
        ens.temperature = 1.0


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--sizes", default="1024x128,256x512", help="BxHW list: batch size x slice size")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_temperature: no CUDA device: this benchmark measures the GPU and has no CPU mode")
    os.makedirs(args.out, exist_ok=True)
    from innovative3D import config as C
    from innovative3D import models

    lits = []
    for seed in (42, 123, 999):
        torch.manual_seed(seed)
        lits.append(dict((v[0], v[1]) for v in C.VARIANTS)["SPFF-UNet"]().cuda().eval())
    result = {"card": card(), "model": "SPFF-UNet", "seeds": [42, 123, 999], "reps": args.reps,
              "calibration_bins": CAL, "grid": {"t_max": 8.0, "points": 33}, "runs": []}
    for spec in args.sizes.split(","):
        b, hw = (int(v) for v in spec.split("x"))
        x, lab = inputs(b, hw)
        group = 256 if hw <= 128 else 16
        for lit in lits:
            lit.model.sample_group = group
        ens = {c: models.SpctEnsemble(lits[:m], tta=tta) for c, m, tta in CONFIGS}
        g = torch.Generator(device="cuda").manual_seed(77)
        noisy = torch.rand(lab.shape, device="cuda", generator=g) < 0.3
        lab = torch.where(noisy, lab, ens["1xnone"].predict_labels(x))
        lab[torch.rand(lab.shape, device="cuda", generator=g) < 0.01] = 255
        t_fit = {c: e.fit_temperature([(x, lab)], apply=False)["temperature"] for c, e in ens.items()}
        paths = {}
        for cname, m, _ in CONFIGS:
            e = ens[cname]
            paths[f"{cname}/fit_temperature"] = lambda e=e: e.fit_temperature([(x, lab)], apply=False)["temperature"]
            paths[f"{cname}/evaluate_calibration"] = \
                lambda e=e: e.evaluate([(x, lab)], calibration=CAL)["calibration"]["ece"]
            paths[f"{cname}/evaluate_calibration_tempered"] = lambda e=e, t=t_fit[cname]: tempered(
                e, t, lambda: e.evaluate([(x, lab)], calibration=CAL)["calibration"]["ece"])
            paths[f"{cname}/torch_lbfgs"] = lambda mb=lits[:m], fl=e.flips: torch_fit(mb, x, lab, fl)
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
        run = {"batch": b, "hw": hw, "voxels": b * 5 * hw * hw, "sample_group": group}
        for name in paths:
            run[name] = {"ms_median": statistics.median(t[name]), "ms_all": t[name],
                         "peak_allocated_above_resident_bytes": peak[name], "value": vals[name]}
        for cname, m, _ in CONFIGS:
            r = lambda n: run[f"{cname}/{n}"]["ms_median"]   # noqa: E731
            run[f"{cname}/fit_over_evaluate_time"] = r("fit_temperature") / r("evaluate_calibration")
            run[f"{cname}/tempered_over_evaluate_time"] = r("evaluate_calibration_tempered") / r("evaluate_calibration")
            run[f"{cname}/torch_over_fit_time"] = r("torch_lbfgs") / r("fit_temperature")
            run[f"{cname}/temperature_fused_vs_torch"] = [run[f"{cname}/fit_temperature"]["value"],
                                                         run[f"{cname}/torch_lbfgs"]["value"]]
        kr = kernel_rates(ens["3xflip"], x, lab, t_fit["3xflip"])
        passes = 3 * 4
        kr["fit_kernel_over_one_forward"] = \
            kr["fit_temperature"]["fit"]["ms"] / (run["3xflip/fit_temperature"]["ms_median"] / passes)
        run["kernels_3xflip"] = kr
        print(json.dumps(run), flush=True)
        result["runs"].append(run)
        del x, lab, paths, ens
        for lit in lits:
            lit.model.engine.release_buffers()
        torch.cuda.empty_cache()
    with open(os.path.join(args.out, "bench_temperature.json"), "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
