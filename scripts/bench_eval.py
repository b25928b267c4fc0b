"""Fused evaluation step (`evaluate`: forward + fused head/CE/confusion, no logits) against the logits path
(`model(x)` + `ce_plus_macro_dice_loss` + `per_class_metrics_3d`) on one GPU, SPFF-UNet, same seeded inputs.

Both paths run in one process, alternating, after warm-up; each call is timed whole with CUDA events (both end in a
device->host copy of the metrics). Sizes: the training batch x[1024,1,5,128,128] and the inference scan
x[256,1,5,512,512], with the batch resident on the device and streamed from pinned host memory. A separate
torch.profiler run gives the time of the fused head kernel and of the two kernels it replaces (head_fwd + ce); the head
kernel's algorithmic bytes are 64 B of bf16 activations + the label per voxel (the 1-byte arg-max map is not written
here). HBM fraction = those bytes / kernel time / 7.7 TB/s (HGX B200 data sheet, one GPU).

    python scripts/bench_eval.py --out DIR [--reps 5] [--warmup 2] [--sizes 1024x128,256x512]

Writes DIR/bench_eval.json. Fails without a CUDA device."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "spff-unet-spcct_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

HBM_BYTES_PER_S = 7.7e12
K = 13


def card():
    """Name, power limit and max SM clock of GPU 0 (read-only query)."""
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60, check=True).stdout.strip()
        name, power, clock = [s.strip() for s in q.split(",")]
        info.update(smi_name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:  # the numbers stay meaningful without it; say why it is missing
        info["smi_error"] = repr(e)
    return info


def inputs(b, hw, seed=1234):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(b, 1, 5, hw, hw, device="cuda", generator=g)
    lab = torch.randint(0, K, (b, 5, hw, hw), device="cuda", generator=g, dtype=torch.int64).to(torch.uint8)
    lab[torch.rand(b, 5, hw, hw, device="cuda", generator=g) < 0.01] = 255
    return x, lab


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    e0.record()
    r = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), torch.cuda.max_memory_allocated(), r


def kernel_times(fn, names):
    """{name: {ms, launches}} over one call of fn, for CUDA kernels matching any of the alternatives of each name (the
    demangled and the mangled spelling)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {n: {"ms": 0.0, "launches": 0} for n in names}
    for ev in prof.events():
        if ev.device_type.name != "CUDA":
            continue
        for n, alts in names.items():
            if any(a in ev.name for a in alts):
                out[n]["ms"] += ev.time_range.elapsed_us() / 1e3
                out[n]["launches"] += 1
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--sizes", default="1024x128,256x512", help="BxHW list: batch size x slice size")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_eval: no CUDA device: this benchmark measures the GPU and has no CPU mode")
    os.makedirs(args.out, exist_ok=True)
    from innovative3D import config as C
    from innovative3D import helpers as H

    torch.manual_seed(42)
    lit = dict((v[0], v[1]) for v in C.VARIANTS)["SPFF-UNet"]().cuda().eval()
    result = {"card": card(), "model": "SPFF-UNet", "sample_group": lit.model.sample_group, "reps": args.reps, "runs": []}

    def logits_path(x, lab):
        with torch.no_grad():
            logits = lit(x)
            loss = lit.compute_loss(logits, lab)
            m = H.per_class_metrics_3d(logits, lab, K, ignore_index=255)
        return float(loss), m[3]

    def fused_path(x, lab):
        ev = lit.evaluate([(x, lab)])
        return ev["loss"], ev["metrics"][3]

    for spec in args.sizes.split(","):
        b, hw = (int(v) for v in spec.split("x"))
        xd, labd = inputs(b, hw)
        voxels = b * 5 * hw * hw
        for mode in ("resident", "host"):
            if mode == "host":
                x, lab = xd.cpu().pin_memory(), labd.cpu().pin_memory()
            else:
                x, lab = xd, labd
            for _ in range(args.warmup):
                fused_path(x, lab)
                logits_path(x, lab)
            t = {"fused": [], "logits": []}
            peak = {}
            vals = {}
            for _ in range(args.reps):
                for name, fn in (("fused", fused_path), ("logits", logits_path)):
                    ms, mem, r = timed(lambda: fn(x, lab))
                    t[name].append(ms)
                    peak[name] = max(peak.get(name, 0), mem)
                    vals[name] = r
            run = {"batch": b, "hw": hw, "mode": mode, "voxels": voxels, "logits_bytes": voxels * K * 4}
            for name in ("fused", "logits"):
                med = statistics.median(t[name])
                run[name] = {"ms_median": med, "ms_all": t[name], "voxels_per_s": voxels / (med * 1e-3),
                             "peak_allocated_bytes": peak[name], "loss": vals[name][0], "macro_dice": vals[name][1]}
            run["speedup"] = run["logits"]["ms_median"] / run["fused"]["ms_median"]
            run["peak_saving_bytes"] = peak["logits"] - peak["fused"]
            run["loss_rel_diff"] = abs(vals["fused"][0] - vals["logits"][0]) / abs(vals["logits"][0])
            if mode == "resident":
                kt = kernel_times(lambda: fused_path(x, lab), {"head_eval_mma_kernel": ("head_eval_mma_kernel",)})
                kl = kernel_times(lambda: logits_path(x, lab), {"head_fwd_kernel": ("head_fwd_kernel",),
                                                                 "ce_kernel": ("::ce_kernel<", "10ce_kernelI")})
                k_ms = kt["head_eval_mma_kernel"]["ms"]
                nbytes = voxels * (64 + lab.element_size())
                run["kernels"] = {"fused": kt, "logits": kl, "head_eval_bytes": nbytes,
                                  "head_eval_bytes_per_s": nbytes / (k_ms * 1e-3) if k_ms else None,
                                  "head_eval_hbm_fraction": nbytes / (k_ms * 1e-3) / HBM_BYTES_PER_S if k_ms else None}
            print(json.dumps(run), flush=True)
            result["runs"].append(run)
            del x, lab
        del xd, labd
        lit.model.engine.release_buffers()
        torch.cuda.empty_cache()
    with open(os.path.join(args.out, "bench_eval.json"), "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
