#!/usr/bin/env python
"""bench.py -- headline benchmark of the multi-view RL deconvolution hot path.

    python bench.py --gpus N --steps K --warmup W          # this build (sm_100a)
    python bench.py --impl reference --steps K --warmup W  # CPU restatement of the reference path
    torchrun ... bench.py --gpus N ...                     # one rank per GPU, weak scaling

Workload (BASELINE.json config 3): 6 views, 512x512x256 float32, 41^3 PSFs,
50 iterations, Tikhonov lambda = 0.006, minValue 1e-4.  One "step" = one whole
50-iteration deconvolution of that volume.  Metric: G voxel*view*iteration / s.

  value  device-resident: views, weights, PSF spectra and psi already in HBM, the
         loop timed with CUDA events on the library's stream (max over ranks);
  e2e    the reference-facing C-ABI call inplace_gpu_deconvolve(psi, workspace, device)
         with pinned HOST buffers: uploads, spectrum precompute, loop and download
         all inside the timed region.

N > 1: independent volumes (blocks) sharded one per rank, no collective on the
data path (SURVEY.md §8e) -- "weak" scaling.

--dump-outputs DIR (rank 0) writes what the last timed step of each timed path handed back, so that two builds can
be compared output for output on the same seeded inputs:
  psi.npy             psi of the device-resident loop after the last timed step
  e2e_psi.npy         psi returned by the last timed e2e call with pageable host buffers
  e2e_pinned_psi.npy  the same with page-locked host buffers
float32, each the whole volume when it has at most DUMP_VOXELS voxels, else the voxels at DUMP_SEED's fixed sample of
flat indices (sorted); at most 3 x 16 MiB in all.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DIMS = (512, 512, 256)  # {z, y, x}, ref: bench/bench_gpu_deconvolve.cu:72-74
VIEWS = 6
KERNEL = 41
ITERATIONS = 50
LAMBDA = 0.006
MIN_VALUE = 1e-4
METRIC = "rl_deconv_gvoxel_view_iter_per_s"
UNIT = "Gvoxel*view*iter/s"
DUMP_VOXELS = 1 << 22
DUMP_SEED = 20240607


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--dims", type=str, default=None, help="z,y,x override (debug only; invalidates the metric)")
    ap.add_argument("--iterations", type=int, default=ITERATIONS)
    ap.add_argument("--views", type=int, default=VIEWS)
    ap.add_argument("--kernel", type=int, default=KERNEL)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--strategy", default="auto", choices=["auto", "generic", "fused"])
    ap.add_argument("--workload", default="deconv", choices=["deconv", "conv_sweep", "blocks", "volume"],
                    help="deconv = config 3 (the headline, default); conv_sweep = config 2; blocks = config 4; volume = config 5")
    ap.add_argument("--blocks", type=int, default=64)
    ap.add_argument("--no-extra", action="store_true",
                    help="skip the config-4 / config-5 sub-records of the default run (blocks batch, 1024^3 volume)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (native deconv workload only)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and (args.impl != "native" or args.workload != "deconv"):
        ap.error("--dump-outputs needs --impl native and --workload deconv")
    return args


def dump_sample(a):
    """`a` itself when it is small enough, else its voxels at a fixed seeded sample of flat indices."""
    flat = np.ascontiguousarray(a).reshape(-1)
    if flat.size <= DUMP_VOXELS:
        return np.array(a, copy=True)
    idx = np.sort(np.random.default_rng(DUMP_SEED).choice(flat.size, DUMP_VOXELS, replace=False))
    return flat[idx]


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def fast_views(dims, num_views, ksize, seed, workers):
    """Config-3 style inputs (SURVEY.md §8d), see libmultiviewnative_b200.synthetic.make_views_fast."""
    from libmultiviewnative_b200.synthetic import make_views_fast

    return make_views_fast(dims, num_views, ksize, seed, workers)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        def pump():
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, power = [], [], set(), []
        for r in self.rows:
            try:
                sm.append(float(r[1])); smax.append(float(r[2])); power.append(float(r[3]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(smax)), "power_w_max": max(power),
                "samples": len(sm), "reasons": sorted(reasons)}


def cpu_reference_sample(data, dims, views_per_step, steps, warmup, threads):
    """Times the CPU restatement of inplace_cpu_deconvolve -- the oracle's checked torch/MKL twin
    (oracle.mvn_oracle.inplace_cpu_deconvolve_torch, the function the full-size parity test compares the GPU
    with) -- on a bounded sample: `views_per_step` consecutive (view, iteration) units of the same workload
    per step, psi carried from step to step.  The PSF spectra are built before the clock starts (in the full
    workload they are 12 of 1212 transforms); the result is normalised per unit, so it reads in the same
    G voxel*view*iteration/s as the whole 300-unit job."""
    from oracle import mvn_oracle as orc  # checker code, allowed here (cpu_baseline / reference leg)

    nv = len(data["views"])
    nvox = int(np.prod(dims))
    khats = (orc.torch_forwarded_kernels(data["kernels1"], dims, threads),
             orc.torch_forwarded_kernels(data["kernels2"], dims, threads))
    its = -(-views_per_step // nv)
    psi = data["psi0"]

    def step(psi):
        return orc.inplace_cpu_deconvolve_torch(psi, data["views"], None, None, data["weights"], its, LAMBDA, MIN_VALUE,
                                                nthreads=threads, max_units=views_per_step, khats=khats)

    for _ in range(warmup):
        psi = step(psi)
    t0 = time.perf_counter()
    for _ in range(steps):
        psi = step(psi)
    dt = time.perf_counter() - t0
    return dt, nvox * views_per_step * steps


def config_of(args, dims, workload):
    """The workload description, identical in both arms (native and --impl reference)."""
    return {"workload": workload, "dims_zyx": list(dims), "views": args.views, "kernel": args.kernel,
            "iterations_per_step": args.iterations, "lambda": LAMBDA, "min_value": MIN_VALUE,
            "l2": "inputs larger than L2: the working set of one step is > 7 GiB per GPU against 126 MB of L2, no flush needed",
            "parallelism": "independent volumes, one per GPU, no collective",
            "reference_arm": "times a bounded sample of consecutive (view, iteration) units of THIS workload on the host "
                             "cores and reports it in the same unit (units / s); the native arm times all of them"}


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dims = tuple(int(x) for x in args.dims.split(",")) if args.dims else DIMS
    nvox = int(np.prod(dims))
    workers = max(1, (os.cpu_count() or 1) // max(1, world))
    workload = "%d-view %dx%dx%d f32, %d^3 PSFs, %d iterations, lambda=%g" % (
        args.views, dims[0], dims[1], dims[2], args.kernel, args.iterations, LAMBDA)

    # ------------------------------------------------------------------ reference arm
    if args.impl == "reference":
        if rank != 0:
            return 0
        threads = os.cpu_count() or 1
        data = fast_views(dims, args.views, args.kernel, 20240607, threads)
        # probe one (view, iteration) to bound the sample
        dt1, _ = cpu_reference_sample(data, dims, 1, 1, 1, threads)
        budget = 150.0 / max(1, args.steps + args.warmup)
        vps = int(max(1, min(args.views, budget // max(dt1, 1e-3))))
        dt, units = cpu_reference_sample(data, dims, vps, args.steps, args.warmup, threads)
        value = units / dt / 1e9
        sample = ("%d consecutive (view,iteration) units of the workload per step (of its %d per step), through "
                  "oracle.mvn_oracle.inplace_cpu_deconvolve_torch (torch/MKL restatement of inplace_cpu_deconvolve, all "
                  "host cores; the FFTW reference is not buildable here)" % (vps, args.views * args.iterations))
        line = {
            "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_of(args, dims, workload),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ native arm
    import torch

    from libmultiviewnative_b200 import capi, load

    if not torch.cuda.is_available():
        print("bench.py: no CUDA device -- the native arm has no CPU fallback", file=sys.stderr)
        return 2
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    device = local_rank if world > 1 else 0
    lib = load()
    lib.set_default_strategy({"auto": 0, "generic": 1, "fused": 2}[args.strategy])

    def barrier():
        torch.cuda.synchronize(device)
        if dist is not None:
            dist.barrier()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda:%d" % device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    if args.workload != "deconv":
        from tools import workloads

        peak, peak_src = peaks()
        if args.workload == "conv_sweep":
            line = workloads.conv_sweep(args, lib, torch, peak, peak_src, device) if rank == 0 else None
        elif args.workload == "blocks":
            line = workloads.blocks(args, lib, torch, dist, rank, world, device, fast_views, barrier, max_over_ranks)
        else:
            line = workloads.volume(args, lib, torch, dist, rank, world, device, barrier, max_over_ranks, peak, peak_src)
        if rank == 0:
            print(json.dumps(line))
        if dist is not None:
            dist.destroy_process_group()
        return 0

    data = fast_views(dims, args.views, args.kernel, 20240607 + 100 * rank, workers)

    # pinned host buffers: the e2e call copies straight from them
    def pin(a):
        t = torch.from_numpy(a).pin_memory()
        return t, t.numpy()
    keep = []
    for key in ("views", "weights"):
        for i, a in enumerate(data[key]):
            tt, data[key][i] = pin(a)
            keep.append(tt)
    tt, psi_host = pin(data["psi0"].copy())
    keep.append(tt)

    plan = lib.plan(dims, args.views, device)
    for v in range(args.views):
        plan.set_view(v, data["views"][v], data["weights"][v], data["kernels1"][v], data["kernels2"][v])
    plan.set_psi(data["psi0"])
    plan.synchronize()
    info = plan.info()

    for _ in range(args.warmup):
        plan.iterate(args.iterations, LAMBDA, MIN_VALUE)
    sampler = ClockSampler(device)
    barrier()
    sampler.start()
    t_wall0 = time.perf_counter()
    dev_ms = 0.0
    for _ in range(args.steps):
        dev_ms += plan.iterate(args.iterations, LAMBDA, MIN_VALUE)
    barrier()
    wall_ms = (time.perf_counter() - t_wall0) * 1e3
    clocks = sampler.stop()
    outputs = {}
    if args.dump_outputs and rank == 0:
        outputs["psi"] = dump_sample(plan.get_psi())
    dev_ms = max_over_ranks(dev_ms)
    units_per_rank = nvox * args.views * args.iterations * args.steps
    value = world * units_per_rank / (dev_ms * 1e-3) / 1e9

    # per-launch profile -> roofline of the dominant kernel (rank 0)
    prof = plan.profile(LAMBDA, MIN_VALUE)
    agg = {}
    for name, ms, nbytes in prof:
        a = agg.setdefault(name, [0.0, 0, 0])
        a[0] += ms; a[1] += nbytes; a[2] += 1
    step_ms = sum(a[0] for a in agg.values())
    top = max(agg.items(), key=lambda kv: kv[1][0])
    peak, peak_src = peaks()
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get(top[0])
        except Exception:
            traffic = None
    top_ms = top[1][0] / top[1][2]
    top_bytes = top[1][1] / top[1][2]
    achieved = top_bytes / (top_ms * 1e-3) / 1e9
    roofline = {
        "bound": "hbm", "kernel": top[0], "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
        "traffic": traffic, "peak_source": peak_src, "alg_bytes_per_launch": top_bytes, "ms_per_launch": top_ms,
        "share_of_step": top[1][0] / step_ms,
        "whole_step": {"alg_bytes_per_view_iteration": int(info.alg_bytes_per_view_iteration),
                       "achieved": info.alg_bytes_per_view_iteration * args.views * args.iterations * args.steps / (dev_ms * 1e-3) / 1e9,
                       "frac": info.alg_bytes_per_view_iteration * args.views * args.iterations * args.steps / (dev_ms * 1e-3) / 1e9 / peak},
        "kernels": {k: {"ms": v[0] / v[2], "launches_per_view_iteration": v[2], "alg_GBps": v[1] / v[2] / (v[0] / v[2] * 1e-3) / 1e9}
                    for k, v in agg.items()},
    }
    plan.close()

    # ---- e2e through the reference-facing C-ABI call, host buffers ----
    # headline: PAGEABLE numpy buffers, which is what a JNA caller hands over (the library stages them through its
    # pinned ring); the same call with pinned buffers is reported beside it
    e2e = None
    if not args.no_e2e:
        ksz = sum(k.size for k in data["kernels1"]) + sum(k.size for k in data["kernels2"])

        def measure(views, weights, psi_buf):
            def call():
                np.copyto(psi_buf, data["psi0"])  # fresh psi for every call; host-side reset, not part of the call
                t0 = time.perf_counter()
                lib.inplace_gpu_deconvolve(psi_buf, views, data["kernels1"], data["kernels2"], weights,
                                           args.iterations, LAMBDA, MIN_VALUE, device)
                return time.perf_counter() - t0  # the call returns after psi has been copied back (synchronous)
            call()  # warm-up (plan store, allocator)
            barrier()
            sec = 0.0
            for _ in range(args.steps):
                sec += call()
            barrier()
            return max_over_ranks(sec)

        pinned_s = measure(data["views"], data["weights"], psi_host)
        pageable_views = [np.array(a, copy=True) for a in data["views"]]      # plain malloc'ed numpy memory
        pageable_weights = [np.array(a, copy=True) for a in data["weights"]]
        pageable_psi = np.array(data["psi0"], copy=True)
        pageable_s = measure(pageable_views, pageable_weights, pageable_psi)
        del pageable_views, pageable_weights
        if args.dump_outputs and rank == 0:
            outputs["e2e_psi"] = dump_sample(pageable_psi)
            outputs["e2e_pinned_psi"] = dump_sample(psi_host)
        e2e = {"value": world * units_per_rank / pageable_s / 1e9, "unit": UNIT,
               "h2d_bytes_per_step": int((2 * args.views + 1) * nvox * 4 + ksz * 4), "d2h_bytes_per_step": int(nvox * 4),
               "ms_per_step": pageable_s / args.steps * 1e3,
               "api": "inplace_gpu_deconvolve(psi, workspace, device) with PAGEABLE host buffers (numpy arrays, like JNA's)",
               "pinned": {"value": world * units_per_rank / pinned_s / 1e9, "ms_per_step": pinned_s / args.steps * 1e3,
                          "api": "the same call with page-locked host buffers"}}

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        dt1, _ = cpu_reference_sample(data, dims, 1, 1, 0, threads)
        vps = int(max(1, min(args.views, 20.0 // max(dt1, 1e-3))))
        dt, units = cpu_reference_sample(data, dims, vps, 1, 0, threads)
        cpu_baseline = {"value": units / dt / 1e9, "unit": UNIT, "cores": threads, "kind": "port",
                        "sample": "%d consecutive (view,iteration) units of the same workload through "
                                  "oracle.mvn_oracle.inplace_cpu_deconvolve_torch (torch/MKL restatement of "
                                  "inplace_cpu_deconvolve; FFTW reference not buildable here)" % vps}

    # ---- configs 4 and 5 as sub-records (every N; N = 1 gives the single-GPU baselines) ----
    config4 = config5 = None
    if not args.no_extra and not args.dims:
        from tools import workloads

        del data["views"][:], data["weights"][:]
        keep.clear()
        lib.release_cached_memory()
        try:
            config4 = workloads.blocks_record(lib, torch, dist, rank, world, device, barrier, max_over_ranks,
                                              n_blocks=args.blocks)
        except Exception as exc:  # a sub-record must not take the headline down
            config4 = {"error": repr(exc)} if rank == 0 else None
        lib.release_cached_memory()
        try:
            config5 = workloads.volume_record(lib, torch, dist, rank, world, device, barrier, max_over_ranks, peaks()[0])
        except Exception as exc:
            config5 = {"error": repr(exc)} if rank == 0 else None
        lib.release_cached_memory()

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": config_of(args, dims, workload),
            "engine": {"strategy": {1: "generic (5 launches/conv)", 2: "fast power-of-two path (%d launches/conv)" % (info.launches_per_view_iteration // 2)}.get(info.strategy, "?"),
                       "arena_GiB": info.arena_bytes / 2**30},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(info.launches_per_view_iteration * args.views * args.iterations * args.steps),
            "wall_ms_timed_region": wall_ms, "roofline": roofline, "cpu_baseline": cpu_baseline,
            "config4": config4, "config5": config5,
        }
        if args.dump_outputs and rank == 0:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in outputs.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
