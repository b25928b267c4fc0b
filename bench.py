#!/usr/bin/env python
"""Headline benchmark: SPFF-UNet bf16 training step, voxels/s (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[1], SURVEY.md §8d "C2"): per GPU a synthetic batch 8x5x128^3 presented
the way the reference's data pipeline presents a scan, one z-slice per sample: x [1024,1,5,128,128]
fp32, labels [1024,5,128,128] int64 in 0..12 -> 83 886 080 voxels per GPU per step. One step =
forward + ce_plus_macro_dice_loss + backward (+ NCCL gradient all-reduce for N > 1) + Adam step, through
`LitSPCT_EFiLM_FourierGate.fit_step` (the reference-facing plugin surface of this tree).

  value     voxels/s with the batch already resident in HBM (device-timed, CUDA events, max over ranks)
  e2e       the same step fed from pinned HOST buffers (H2D of images + labels and D2H of the loss
            inside the timed region)
  roofline  the dominant kernel family (conv3 fprop kernel: forward + dgrad launches): algorithmic
            FLOPs / CUDA-event time of those launches inside the timed steps, vs the measured
            sustained bf16 peak in MEASURED_PEAKS.json
  cpu_baseline / --impl reference   the CPU restatement of the reference's path (oracle/, the same
            torch CPU fp32 operator sequence the reference dispatches) timed on the host cores on
            a bounded sample of the same workload
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "spff-unet-spcct_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "SPFF-UNet train voxels/s"
FLOP_PER_VOXEL_TRAIN = 2_448_192          # SURVEY.md §8d: fwd + dgrad + wgrad dense contractions
SAMPLES, FRAMES, H, W = 1024, 5, 128, 128  # per GPU
NUM_CLASSES = 13


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return p, "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


# --------------------------------------------------------------------------------------------------
# CPU arm: the reference itself (staged copy under baseline/_ref), else the oracle port, on the host cores
# --------------------------------------------------------------------------------------------------
REF_STAGED = os.path.join(ROOT, "baseline", "_ref")
REF_SLICES_MAX = 32      # 32 slices [1,5,128,128] = 2 621 440 voxels = the voxel count of BASELINE configs[0] (12 GB RSS)


def _cpu_inputs(samples: int):
    import torch
    g = torch.Generator().manual_seed(42)
    x = torch.randn(samples, 1, FRAMES, H, W, generator=g)
    lab = torch.randint(0, NUM_CLASSES, (samples, FRAMES, H, W), generator=g)
    return x, lab


def _reference_stepper():
    """(step(x, lab), kind): fwd + ce_plus_macro_dice_loss + backward of SPFF-UNet on the CPU in fp32.
    kind "reference": the UNMODIFIED reference modules (`config.VARIANTS["SPFF-UNet"]` of baseline/_ref, the git-ignored
    copy of /root/reference that __graft_entry__.build() stages and gpurun ships), imported under inert stubs for the
    plotting / Lightning packages this image lacks - none of this repo's package is on that path. kind "port": the
    oracle restatement (oracle/spff_oracle.py, pinned to the reference by tests/golden) when no staged copy exists."""
    import torch
    if os.path.isfile(os.path.join(REF_STAGED, "innovative3D", "models.py")):
        pkg = os.path.join(ROOT, "spff-unet-spcct_b200")
        sys.path[:] = [p for p in sys.path if os.path.abspath(p) != pkg]      # this repo's `innovative3D` must not shadow it
        for k in [k for k in sys.modules if k == "innovative3D" or k.startswith("innovative3D.")]:
            del sys.modules[k]
        from oracle.make_golden import install_stubs
        install_stubs()
        os.environ.setdefault("CHECKPOINT_DIR", os.path.join(tempfile.gettempdir(), "spff_ref_ckpt"))
        os.environ.setdefault("LOG_DIR", os.path.join(tempfile.gettempdir(), "spff_ref_logs"))
        from pathlib import Path
        _mkdir = Path.mkdir

        def safe_mkdir(self, *a, **k):      # config.py:15-19 creates directories under a hard-coded home path
            try:
                return _mkdir(self, *a, **k)
            except OSError:
                return None

        Path.mkdir = safe_mkdir
        sys.path.insert(0, REF_STAGED)
        try:
            import innovative3D.config as RC
        finally:
            Path.mkdir = _mkdir
        assert os.path.abspath(RC.__file__).startswith(REF_STAGED), RC.__file__
        torch.manual_seed(42)
        lit = dict((v[0], v[1]) for v in RC.VARIANTS)["SPFF-UNet"]()
        lit.train()

        def step(x, lab):
            lit.zero_grad(set_to_none=True)
            loss = lit.compute_loss(lit(x), lab)
            loss.backward()
            return float(loss)
        return step, "reference"
    from oracle import spff_oracle as O
    torch.manual_seed(42)
    p = O.det_weights(O.param_shapes("SPFF-UNet"), seed=42)
    return (lambda x, lab: O.loss_and_grads(p, x, lab, "SPFF-UNet")[0]), "port"


def cpu_step_time(samples: int, reps: int, warmup: int, budget_s: float = 1e9):
    """Times `reps` steps (fwd + loss + bwd, CPU fp32, all host threads) on `samples` slices of the bench shape;
    returns (seconds per step list, threads, kind)."""
    import torch
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    step, kind = _reference_stepper()
    x, lab = _cpu_inputs(samples)
    times = []
    t_start = time.perf_counter()
    for i in range(warmup + reps):
        t0 = time.perf_counter()
        step(x, lab)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
        if time.perf_counter() - t_start > budget_s and times:
            break
    return times, threads, kind


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the host cores, all threads. Rank 0 only; a
    step is a bounded sample of the workload: as many slices (8..32) as keep the whole --steps/--warmup run under ~4
    minutes, found with one calibration step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    step, kind = _reference_stepper()
    x8, l8 = _cpu_inputs(8)
    step(x8[:2], l8[:2])                               # first-call set-up (lazy parameters, oneDNN primitives)
    t0 = time.perf_counter()
    step(x8, l8)
    per_slice = (time.perf_counter() - t0) / 8
    n_steps = args.steps + args.warmup
    samples = REF_SLICES_MAX
    while samples > 8 and per_slice * samples * n_steps > 240.0:
        samples //= 2
    samples = int(os.environ.get("SPFF_REF_SLICES", samples))
    x, lab = _cpu_inputs(samples)
    times = []
    for i in range(n_steps):
        t0 = time.perf_counter()
        step(x, lab)
        if i >= args.warmup:
            times.append(time.perf_counter() - t0)
    vox = samples * FRAMES * H * W
    sec = sum(times) / len(times)
    value = vox / sec
    sample = (f"{samples} of the {SAMPLES} slices [1,5,{H},{W}] per step ({vox} voxels), fp32 fwd+loss+bwd, {threads} threads, "
              f"{'the reference modules themselves (baseline/_ref)' if kind == 'reference' else 'oracle port'}")
    cfg = workload_config(args.gpus)
    cfg["workload"] += f" - CPU arm: a bounded sample of {samples} slices per step"
    cfg["samples_per_step_timed"] = samples
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "voxels/s", "n_gpus": args.gpus,
        "steps": len(times), "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": value, "unit": "voxels/s", "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "voxels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(n_gpus: int, variant: str = "SPFF-UNet", samples: int = SAMPLES):
    if variant != "SPFF-UNet":   # BASELINE.json configs[3]: the ablation controls through the same kernels
        opt = "SGD(momentum)" if variant == "3DUNet" else "Adam"
        return {
            "workload": f"{variant} bf16 training step (control, BASELINE.json configs[3]), synthetic x[{samples},1,{FRAMES},{H},{W}] per GPU"
                        + (" (16 planes inside the depth adapter; whole batch resident: BatchNorm)" if variant == "3DUNet" else ""),
            "samples_per_gpu": samples, "voxels_per_gpu_step": samples * FRAMES * H * W, "num_classes": NUM_CLASSES,
            "step": f"fwd + loss + bwd + grad all-reduce + {opt}", "parallelism": f"dp{n_gpus}",
            "l2": "working set >> 126 MB L2 (inputs larger than L2; no flush needed)",
        }
    return {
        "workload": f"SPFF-UNet bf16 training step, synthetic batch 8x5x128^3 per GPU = x[{SAMPLES},1,{FRAMES},{H},{W}] "
                    f"(BASELINE.json configs[1]; configs[2] for N>1)",
        "samples_per_gpu": SAMPLES, "voxels_per_gpu_step": SAMPLES * FRAMES * H * W, "num_classes": NUM_CLASSES,
        "step": "fwd + CE/Dice loss + bwd + grad all-reduce + Adam", "parallelism": f"dp{n_gpus}",
        "l2": "working set per sample group >> 126 MB L2 (inputs larger than L2; no flush needed)",
    }


DUMP_MAX_ELEMS = 6_000_000      # per array: SPFF-UNet's parameters and gradients fit whole; 3DUNet's are sampled


def dump_outputs(path: str, lit, out) -> None:
    """What one training step hands its caller, as <path>/<name>.npy: the loss and the loss / metric tally fit_step
    returns, and the parameters (state_dict order) and gradients (fused_grads order) the step leaves behind, each
    flattened. An array longer than DUMP_MAX_ELEMS keeps the entries at fixed positions (a seeded permutation), so
    two builds of the project compare entry for entry. The step is not bit-reproducible: two runs of one build
    (`--steps 5 --warmup 3`, one B200 at a 1000 W power limit) differed by 3e-6 in the loss and, as rel-L2, by 1.4e-3
    in the parameters and 1e-2 in the gradients."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    t = out["tally"]
    arrays = {"loss": out["loss"].double(), "tally_nll": t.nll.double(), "tally_count": t.count.double(),
              "confusion": t.confusion.double()}
    for name, parts in (("params", lit.state_dict().values()), ("grads", lit.fused_grads().values())):
        v = torch.cat([p.detach().reshape(-1).float() for p in parts])
        if v.numel() > DUMP_MAX_ELEMS:
            idx = torch.randperm(v.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_MAX_ELEMS].sort().values
            v = v[idx.to(v.device)]
        arrays[name] = v
    for name, v in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), v.cpu().numpy())


def conv_traffic():
    """Mean DRAM bytes (read + write) per conv3_fprop_kernel launch from the committed ncu capture
    (profiles/r01f_conv_traffic.json: every conv launch of `SPFF_BENCH_SAMPLES=256 bench.py`, i.e. the same 256-slice
    launches as the default sample group). None when the capture is absent."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_conv_traffic.json")) as f:
            k = json.load(f)["kernels"]
        rows = [v for name, v in k.items() if "conv3_fprop_kernel" in name or "conv3_halo_kernel" in name]
        n = sum(v["launches"] for v in rows)
        return sum(v["launches"] * (v["dram_read_bytes_per_launch"] + v["dram_write_bytes_per_launch"]) for v in rows) / n
    except Exception:
        return None


# --------------------------------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                       "-i", str(self.index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for line in self.f.read().splitlines():
            c = [t.strip() for t in line.split(",")]
            if len(c) < 8:
                continue
            try:
                sm.append(float(c[1]))
                mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.f.name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist

    from innovative3D import config as C
    from spff_b200 import _lib

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("bench.py --gpus N > 1 must be launched with torch.distributed.run (one process per GPU)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    variant = args.variant
    samples = int(os.environ.get("SPFF_BENCH_SAMPLES", 256 if variant == "3DUNet" else SAMPLES))
    torch.manual_seed(42)
    lit = dict((v[0], v[1]) for v in C.VARIANTS)[variant]().to(dev)
    if variant == "3DUNet":
        lit.train()
    g = torch.Generator().manual_seed(1234 + rank)
    x_host = torch.randn(samples, 1, FRAMES, H, W, generator=g).pin_memory()
    lab_host = torch.randint(0, NUM_CLASSES, (samples, FRAMES, H, W), generator=g).pin_memory()
    x_dev = x_host.to(dev)
    lab_dev = lab_host.to(dev)
    vox = samples * FRAMES * H * W
    loss_host = torch.zeros(1).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    per_rank = {}

    def timed(fn, steps, tag=None):
        barrier()
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            if tag is not None:      # every rank's own time: which rank is the slow one, and by how much
                allt = [torch.zeros_like(t) for _ in range(world)]
                dist.all_gather(allt, t)
                per_rank[tag] = [float(v) / steps for v in allt]
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t) * 1e-3

    last = {}

    def step_resident():
        last["out"] = lit.fit_step((x_dev, lab_dev))

    def step_e2e():
        out = lit.fit_step((x_host, lab_host))            # H2D of images + labels inside
        loss_host.copy_(out["loss"].reshape(1), non_blocking=True)
        torch.cuda.current_stream().synchronize()         # the loss is on the host when the step ends

    for _ in range(max(args.warmup, 3)):
        step_resident()
    # ---- device-resident steps, with CUDA events around the conv3 launches (roofline) ----
    clocks = ClockSampler(local)
    clocks.start()
    conv_names = {"spff_conv3d_k3_fwd", "spff_conv3d_k3_fwd_stats", "spff_conv3d_k3_dgrad", "spff_conv3d_k3_dgrad_stats",
                  "spff_conv3d_k3_wgrad"}
    prof = _lib.Profile(select=lambda n: n in conv_names)
    calls0 = _lib.CALLS
    _lib.PROFILE = prof
    from spff_b200 import dp as _dp
    _dp.EXPOSED = [] if world > 1 else None
    sec = timed(step_resident, args.steps, tag="ms_per_step")
    exposed_ms = None
    if world > 1:      # all-reduce time NOT hidden behind the backward (compute stream: backward enqueued -> every range reduced)
        torch.cuda.synchronize()
        mine = sum(a.elapsed_time(b) for a, b in _dp.EXPOSED) / max(1, len(_dp.EXPOSED))
        t = torch.tensor([mine], device=dev, dtype=torch.float64)
        allt = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        exposed_ms = [float(v) for v in allt]
        _dp.EXPOSED = None
    _lib.PROFILE = None
    launches = _lib.CALLS - calls0
    clk = clocks.stop()
    conv = prof.summary()
    if args.dump_outputs and rank == 0:      # before the e2e steps below move the weights on
        dump_outputs(args.dump_outputs, lit, last["out"])
    # ---- end-to-end steps from pinned host memory ----
    step_e2e()
    sec_e2e = timed(step_e2e, args.steps, tag="e2e_ms_per_step")
    # ---- one extra step with every call timed: breakdown by entry point ----
    full = _lib.Profile()
    _lib.PROFILE = full
    step_resident()
    _lib.PROFILE = None
    brk = full.summary()
    final_loss = float(loss_host[0])

    if rank == 0:
        peaks, peak_kind = load_peaks()
        n_f, ms_f, fl_f = [a + b for a, b in zip(conv.get("spff_conv3d_k3_fwd", (0, 0.0, 0.0)),
                                                 conv.get("spff_conv3d_k3_fwd_stats", (0, 0.0, 0.0)))]
        n_d, ms_d, fl_d = [a + b for a, b in zip(conv.get("spff_conv3d_k3_dgrad", (0, 0.0, 0.0)),
                                                 conv.get("spff_conv3d_k3_dgrad_stats", (0, 0.0, 0.0)))]
        n_w, ms_w, fl_w = conv.get("spff_conv3d_k3_wgrad", (0, 0.0, 0.0))
        ach = (fl_f + fl_d) / max(ms_f + ms_d, 1e-9) * 1e3 / 1e12
        peak = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1400.0)))
        value = world * vox * args.steps / sec
        total_ms = sum(v[1] for v in brk.values())
        line = {
            "metric": METRIC if variant == "SPFF-UNet" else f"{variant} train voxels/s", "value": value, "unit": "voxels/s",
            "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": sec / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": workload_config(world, variant, samples),
            "clocks": clk,
            "e2e": {"value": world * vox * args.steps / sec_e2e, "unit": "voxels/s",
                    "h2d_bytes_per_step": x_host.numel() * 4 + lab_host.numel() * 8, "d2h_bytes_per_step": 4,
                    "ms_per_step": sec_e2e / args.steps * 1e3},
            "gpu_launches": launches,
            "roofline": {"bound": "tensor", "kernel": "conv3_fprop_kernel (3x3x3 conv forward + dgrad launches)",
                         "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                         "traffic": conv_traffic() if variant == "SPFF-UNet" else None,
                         "traffic_note": "mean DRAM bytes per launch over all conv3_fprop launches (ncu, 256-slice sample group); "
                                         "algorithmic (activations in + out, bf16): 1.426e9 B per launch",
                         "peak_kind": f"{peak_kind} sustained bf16 (kernel timed inside a long step)",
                         "launches": n_f + n_d, "ms_per_step": (ms_f + ms_d) / args.steps,
                         "wgrad": {"achieved": fl_w / max(ms_w, 1e-9) * 1e3 / 1e12, "ms_per_step": ms_w / args.steps,
                                   "launches": n_w},
                         "step_tensor_frac": (value / world * FLOP_PER_VOXEL_TRAIN / 1e12 / peak if variant != "3DUNet" else
                                              (fl_f + fl_d + fl_w) / sec * 1e-12 / peak)},
            "breakdown_ms": {k: round(v[1], 3) for k, v in sorted(brk.items(), key=lambda kv: -kv[1][1])},
            "breakdown_total_ms": round(total_ms, 3),
            "final_loss": final_loss,
        }
        if world > 1:
            line["per_rank"] = {**per_rank, "allreduce_exposed_ms": exposed_ms,
                                "note": "per-rank device time per step (the line's ms_per_step is their max) and the part of the "
                                        "gradient all-reduce that is not hidden behind the backward"}
        if not args.no_extras and world == 1 and variant == "SPFF-UNet":
            # BASELINE.json configs[3] (the controls) and configs[4] (inference scan), measured in this same process so that
            # the driver's record holds them; each is the full line `--variant X` / `--mode infer` prints, fewer steps
            del x_dev, lab_dev
            lit.model.engine.release_buffers()
            torch.cuda.empty_cache()
            line["extra"] = run_extras(args)
        if not args.no_cpu and world == 1 and variant == "SPFF-UNet":
            # the reference's CPU path on this box's host cores: a separate process (this one holds this repo's
            # `innovative3D`; the reference's package of the same name cannot be imported beside it)
            try:
                out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "2", "--warmup", "0"],
                                     capture_output=True, text=True, timeout=600, env={**os.environ, "SPFF_REF_SLICES": "8"})
                ref = json.loads(out.stdout.strip().splitlines()[-1])
                line["cpu_baseline"] = ref["cpu_baseline"]
            except Exception as e:      # the GPU numbers stand on their own
                line["cpu_baseline"] = {"value": None, "unit": "voxels/s", "cores": os.cpu_count(), "kind": "unavailable",
                                        "sample": f"reference leg failed: {e!r}"[:300]}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_extras(args):
    """PlainCore_UNet / 3DUNet training steps and the inference scan, as sub-lines of the default run."""
    import copy
    import io
    from contextlib import redirect_stdout
    out = {}
    for key, mode, variant in (("plaincore", "train", "PlainCore_UNet"), ("unet3d", "train", "3DUNet"), ("infer", "infer", "SPFF-UNet")):
        a = copy.copy(args)
        a.variant, a.mode, a.no_cpu, a.no_extras, a.dump_outputs = variant, mode, True, True, None
        a.steps, a.warmup = min(args.steps, 3), 3
        buf = io.StringIO()
        try:
            with redirect_stdout(buf):
                (run_infer if mode == "infer" else run_b200)(a)
            d = json.loads(buf.getvalue().strip().splitlines()[-1])
            out[key] = {k: d[k] for k in ("metric", "value", "unit", "ms_per_step", "steps", "config", "e2e", "roofline", "gpu_launches")
                        if k in d}
        except Exception as e:
            out[key] = {"error": repr(e)[:300]}
        import torch
        torch.cuda.empty_cache()
    return out


def run_infer(args):
    """--mode infer: BASELINE.json configs[4] — SPFF-UNet inference over a synthetic 5x512x512x256 scan = x[256,1,5,512,512],
    whole z-slices sharded over the ranks with no collective (SURVEY.md §8e); output: the uint8 label map (argmax fused
    into the head kernel). A "step" is one pass over the rank's shard. Not the headline metric: an extra line."""
    import torch
    import torch.distributed as dist

    from innovative3D import config as C
    from spff_b200 import _lib, dp

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    slices, hh, ww = int(os.environ.get("SPFF_INFER_SLICES", 256)), 512, 512
    lo, hi = dp.shard_range(slices, rank, world)
    torch.manual_seed(42)
    lit = dict((v[0], v[1]) for v in C.VARIANTS)["SPFF-UNet"]().to(dev).eval()
    g = torch.Generator().manual_seed(99 + rank)
    x_host = torch.randn(hi - lo, 1, FRAMES, hh, ww, generator=g).pin_memory()
    x_dev = x_host.to(dev)
    out_host = torch.empty(hi - lo, FRAMES, hh, ww, dtype=torch.uint8).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t) * 1e-3

    def step_resident():
        return lit.model.predict_labels(x_dev)

    def step_e2e():      # images streamed in and label maps streamed out group by group; complete on return
        lit.model.predict_labels_streamed(x_host, out_host)

    for _ in range(max(args.warmup, 3)):
        step_resident()
    clocks = ClockSampler(local)
    clocks.start()
    calls0 = _lib.CALLS
    sec = timed(step_resident, args.steps)
    launches = _lib.CALLS - calls0
    clk = clocks.stop()
    step_e2e()
    sec_e2e = timed(step_e2e, args.steps)
    if rank == 0:
        vox = slices * FRAMES * hh * ww
        peaks, peak_kind = load_peaks()
        peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
        fwd_flop = 816_640     # SURVEY.md §8d: forward FLOP per voxel
        print(json.dumps({
            "metric": "SPFF-UNet inference voxels/s", "value": vox * args.steps / sec, "unit": "voxels/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": sec / args.steps * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"SPFF-UNet inference, synthetic scan 5x512x512x{slices} = x[{slices},1,5,512,512] "
                                   f"(BASELINE.json configs[4]), whole z-slices sharded over {world} rank(s), no collective",
                       "slices_per_gpu": hi - lo, "output": "uint8 label map (argmax fused into the head kernel)",
                       "l2": "inputs larger than L2"},
            "clocks": clk,
            "e2e": {"value": vox * args.steps / sec_e2e, "unit": "voxels/s", "h2d_bytes_per_step": x_host.numel() * 4,
                    "d2h_bytes_per_step": out_host.numel(), "ms_per_step": sec_e2e / args.steps * 1e3},
            "gpu_launches": launches,
            "roofline": {"bound": "tensor", "kernel": "whole forward (816 640 FLOP/voxel dense)",
                         "achieved": vox / world * args.steps / sec * fwd_flop / 1e12, "peak": peak, "unit": "TFLOP/s",
                         "frac": vox / world * args.steps / sec * fwd_flop / 1e12 / peak, "traffic": None,
                         "peak_kind": f"{peak_kind} sustained bf16"},
        }), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extras", action="store_true", help="skip the configs[3] / configs[4] sub-lines of the default run")
    ap.add_argument("--variant", default="SPFF-UNet",
                    choices=["SPFF-UNet", "E_SP_UNet", "FG_SP_UNet", "SP_UNet", "PlainCore_UNet", "3DUNet"],
                    help="SPFF-UNet is the headline (BASELINE.json configs[1]); the others are the controls of configs[3]")
    ap.add_argument("--mode", default="train", choices=["train", "infer"],
                    help="train: the headline step (default); infer: BASELINE.json configs[4], an extra line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed training step's loss, tally, parameters and gradients as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.mode != "train"):
        ap.error("--dump-outputs writes the outputs of the training step (--impl b200 --mode train)")
    if args.impl == "reference":
        run_reference(args)
    elif args.mode == "infer":
        run_infer(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
