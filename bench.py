#!/usr/bin/env python3
"""Benchmark of the per-view acquisition pipeline (BASELINE.json: simulated voxels/s and views/s,
achieved HBM GB/s vs peak).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg3|cfg1|small] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch: the 6 views of BASELINE config 3
(1024x1024x512 float32 ground truth, 6 views 60 deg apart (+15), one 128^3 PSF per view, delta 0.01,
every 5th slice, Poisson SNR 25).  With N > 1 (torchrun, one rank per GPU) every rank simulates its
own batch of 6 views (weak scaling, no data-path collective; views are independent units).

`value`  : voxels/s, inputs resident in HBM, CUDA-event timed on the stream the kernels run on.
`e2e`    : same metric through the host-buffer C-ABI call (mvsim_simulate_views) from pinned host
           memory, ground truth H2D + results D2H inside the timed region.
`roofline`: the dominant kernel (fused z pass) timed live with CUDA events inside the timed region.
`cpu_baseline`: the CPU oracle (restatement of the reference; no JVM in this image) on a bounded sample.

--dump-outputs DIR writes what the last timed step of the device-resident arm returned to its caller on rank 0 (every view's
acquired volume and its PSF, normalised in place; for cfg5 the convolved z slab) as DIR/<name>.npy in float32, so that two builds
can be compared output for output on identical seeded inputs.  --steps sets the timed steps of every arm (each caller thread of
the pipelined end-to-end mode runs that many).
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (shape_zyx, kshape_zyx, sigma_zyx, degrees, inc, snr)
    "cfg3": ((512, 1024, 1024), (128, 128, 128), (17.5, 5.5, 5.0), [15, 75, 135, 195, 255, 315], 5, 25.0),
    "cfg1": ((256, 512, 512), (51, 51, 51), (7.0, 2.2, 2.0), [15, 105, 195, 285], 3, 25.0),
    "cfg4": ((512, 512, 512), (51, 51, 51), (7.0, 2.2, 2.0), [15, 105, 195, 285], 3, 25.0),      # bead-volume shape: 576-point z lines, inc 3
    "small": ((64, 128, 128), (16, 16, 16), (3.0, 1.2, 1.1), [15, 75, 135, 195, 255, 315], 5, 25.0),
}
CPU_SAMPLE = {"cfg3": ((128, 256, 256), (32, 32, 32), (4.4, 1.4, 1.25)), "cfg1": ((64, 128, 128), (25, 25, 25), (3.5, 1.1, 1.0)),
              "cfg4": ((128, 128, 128), (25, 25, 25), (3.5, 1.1, 1.0)),
              "small": ((32, 64, 64), (8, 8, 8), (1.5, 0.8, 0.8))}


def _periodic_sphere_tile(t, n_spheres, rng):
    """t^3 tile of max-composited spheres, radius U{1..20}/2 px, intensity U(0,1), periodic wrap."""
    tile = np.zeros((t, t, t), dtype=np.float32)
    ax = np.arange(t, dtype=np.float32)
    for _ in range(n_spheres):
        c = rng.uniform(0, t, 3)
        r = rng.integers(1, 21) / 2.0
        v = np.float32(rng.random())
        d = [np.minimum(np.abs(ax - c[i]), t - np.abs(ax - c[i])) ** 2 for i in range(3)]
        m = (d[0][:, None, None] + d[1][None, :, None] + d[2][None, None, :]) <= r * r
        tile[m] = np.maximum(tile[m], v)
    return tile


def make_ground_truth(shape, seed=464232194):
    """Sphere-phantom statistics of the reference's simulate() (S/SimulateMultiViewDataset.java:366-522):
    a centred body with semi-axes 0.337*dim (16 % of the volume, background exactly 0) filled with small
    max-composited random spheres of intensity U(0,1).  Own generator: one periodic 64^3 tile repeated
    over the volume (cheap for 0.5 G voxels), masked by the body."""
    z, y, x = shape
    t = 64
    tile = _periodic_sphere_tile(t, 80, np.random.default_rng(seed))
    reps = (math.ceil(z / t), math.ceil(y / t), math.ceil(x / t))
    vol = np.tile(tile, reps)[:z, :y, :x]
    zz = ((np.arange(z, dtype=np.float32) - (z - 1) / 2.0) / (0.337 * z)) ** 2
    yy = ((np.arange(y, dtype=np.float32) - (y - 1) / 2.0) / (0.337 * y)) ** 2
    xx = ((np.arange(x, dtype=np.float32) - (x - 1) / 2.0) / (0.337 * x)) ** 2
    out = np.empty(shape, dtype=np.float32)
    for k in range(z):          # slab-wise to keep the temporary small
        out[k] = vol[k] * ((zz[k] + yy[:, None] + xx[None, :]) <= 1.0)
    return out


DUMP_BYTES = 60 << 20          # --dump-outputs writes at most this much array data in all (< 64 MB)


def dump_indices(size, n):
    """The fixed sample of --dump-outputs: n sorted distinct flat indices out of `size`, from a seeded generator, so that runs of
    the same workload write the same voxels."""
    return np.sort(np.random.default_rng(20261020).choice(size, n, replace=False))


def dump_outputs(out_dir, arrays):
    """Writes every array of {name: array} as out_dir/<name>.npy in float32.  An array larger than its even share of DUMP_BYTES
    is replaced by its values at dump_indices()."""
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // (4 * len(arrays))
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float32)
        if a.size > share:
            a = a.reshape(-1)[dump_indices(a.size, share)]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def make_psfs(kshape, sigma, n):
    from helpers import gaussian_psf
    return [gaussian_psf(kshape, (sigma[0] * (1 + 0.03 * v), sigma[1] * (1 - 0.02 * v), sigma[2] * (1 + 0.01 * v)), threshold=1e-3)
            for v in range(n)]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []          # (arrival time, csv line)
        self.t_start = None
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def mark_start(self):
        """The timed region starts now: only samples that arrive from here on are reported (the sampler itself is started
        before the warm-up, so that nvidia-smi's start-up does not eat a timed region of a few hundred ms)."""
        self.t_start = time.perf_counter()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        rows = list(self.rows)
        inside = [r for t, r in rows if self.t_start is None or t >= self.t_start]
        note = None
        if not inside and rows:
            inside = [rows[-1][1]]      # region shorter than the sampling period: the last sample before it (warm-up, same load)
            note = "timed region shorter than the 100 ms sampling period: last warm-up sample"
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in inside:
            f = [c.strip() for c in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); power.append(float(f[2]))
            except ValueError:
                continue
            for nme, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nme)
        out = {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
               "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}
        if note:
            out["note"] = note
        return out


def host_link_probe(torch, n=1 << 28):
    """Pinned-memory copy rates of this GPU's host link right now: each direction alone and both at once (GB/s)."""
    h_in = torch.empty(n, dtype=torch.float32).pin_memory()
    h_out = torch.empty(n, dtype=torch.float32).pin_memory()
    d_a = torch.empty(n, dtype=torch.float32, device="cuda")
    d_b = torch.ones(n, dtype=torch.float32, device="cuda")
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    gb = n * 4 / 1e9

    def up():
        with torch.cuda.stream(s1):
            d_a.copy_(h_in, non_blocking=True)

    def down():
        with torch.cuda.stream(s2):
            h_out.copy_(d_b, non_blocking=True)

    def timed(fns):
        best = float("inf")
        for _ in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for f in fns:
                f()
            torch.cuda.synchronize()
            best = min(best, time.perf_counter() - t0)
        return gb / best
    r = {"h2d_alone_GBps": timed([up]), "d2h_alone_GBps": timed([down])}
    both = timed([up, down])
    r["h2d_concurrent_GBps"] = r["d2h_concurrent_GBps"] = both
    return r


def nvlink_counters(index):
    """Cumulative NVLink data bytes (tx, rx) of one GPU summed over its links, from NVML's throughput field values (KiB); None when
    NVML or the counters are unavailable."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        out = []
        for fid in (pynvml.NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_TX, pynvml.NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_RX):
            vals = pynvml.nvmlDeviceGetFieldValues(h, [(fid, link) for link in range(pynvml.NVML_NVLINK_MAX_LINKS)])
            good = [int(v.value.ullVal) for v in vals if v.nvmlReturn == 0]
            if not good:
                return None
            out.append(sum(good) * 1024)
        return tuple(out)
    except Exception:
        return None


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def _cpu_view(shape, kshape, sigma, degrees, inc, snr, mode, cores):
    """One view of the loop body S/SimulateMultiViewDataset.java:570-585 through the C oracle.
    mode "reference-shaped": rotate / attenuate / adjust / extract+Poisson on ONE thread (the reference's cursor loops are
    single-threaded), FFT lines on `cores` threads (its ExecutorService), ONE sequential java.util.Random for the Poisson loop.
    mode "best-effort": every stage on `cores` threads, the Poisson loop split over slices (one generator per slice)."""
    from helpers import gaussian_psf
    from oracle import oracle as orc
    gt = make_ground_truth(shape)
    psf = gaussian_psf(kshape, sigma, threshold=1e-3)
    best = mode == "best-effort"
    t0 = time.perf_counter()
    _, _, st = orc.simulate_view(gt, psf, degrees=degrees, inc=inc, snr=snr, use_fft=True, fft_threads=cores,
                                 stage_threads=cores if best else 1, poisson_threads=cores if best else 0, want_conv=False)
    dt = time.perf_counter() - t0
    return dt, dict(zip(["rotate", "attenuate", "convolve", "adjust", "extract_poisson"], [float(v) for v in st]))


def host_cores():
    """Processors of this process -- not OMP_NUM_THREADS (torchrun exports 1)."""
    from oracle import oracle as orc
    return orc.host_threads()


def cpu_baseline_sample(workload):
    """`cpu_baseline` of the default run: the C oracle (kind "port": no JVM on the box, profiles/r02_box_probe.txt) on a BOUNDED
    sample -- one view of a sub-volume -- in both shapes BASELINE.md section 4.2 names."""
    shape, kshape, sigma = CPU_SAMPLE[workload]
    _, _, _, degrees, inc, snr = WORKLOADS[workload]
    cores = host_cores()
    vox = int(np.prod(shape))
    dt_ref, st_ref = _cpu_view(shape, kshape, sigma, degrees[1 % len(degrees)], inc, snr, "reference-shaped", cores)
    dt_best, st_best = _cpu_view(shape, kshape, sigma, degrees[1 % len(degrees)], inc, snr, "best-effort", cores)
    return {"value": vox / dt_ref, "unit": "voxels/s", "cores": cores, "kind": "port",
            "sample": (f"NOT the bench workload: 1 view of a {shape[2]}x{shape[1]}x{shape[0]} sub-volume with a {kshape[2]}^3 PSF (1/64 of the voxels), "
                       f"inc {inc}, SNR {snr}; C oracle of the reference (no JVM on the box); `value` is reference-shaped: stages on 1 thread, "
                       f"FFT lines on {cores} threads, sequential O(lambda) Poisson loop; `best_effort` runs every stage on {cores} threads. "
                       f"`bench.py --impl reference` times the FULL-SIZE view"),
            "sample_volume_xyz": [shape[2], shape[1], shape[0]], "sample_psf_xyz": [kshape[2], kshape[1], kshape[0]],
            "seconds_per_view": dt_ref, "views_per_s": 1.0 / dt_ref, "stage_seconds": st_ref,
            "best_effort": {"value": vox / dt_best, "unit": "voxels/s", "seconds_per_view": dt_best, "stage_seconds": st_best}}


def run_reference(args, rank, world):
    """Reference arm: the reference's CPU implementation of the path (C oracle port; the Java original cannot run: no JVM here
    or on the box) on the SAME config as our arm -- one FULL-SIZE view of the workload, every stage on all host threads.
    One view takes minutes, so a step is ONE view and steps_effective = 1 whatever --steps says; rank 0 alone runs it."""
    if rank != 0:
        return
    shape, kshape, sigma, degrees, inc, snr = WORKLOADS[args.workload]
    cores = host_cores()
    dt, st = _cpu_view(shape, kshape, sigma, degrees[1 % len(degrees)], inc, snr, "best-effort", cores)
    vox = int(np.prod(shape))
    cfg = workload_config(args.workload)
    cfg["views_per_step_timed"] = 1
    base = {"value": vox / dt, "unit": "voxels/s", "cores": cores, "kind": "port",
            "sample": (f"1 full-size view of the workload ({shape[2]}x{shape[1]}x{shape[0]}, PSF {kshape[2]}x{kshape[1]}x{kshape[0]}, inc {inc}, SNR {snr}, "
                       f"{degrees[1 % len(degrees)]} degrees) through the C oracle of the reference, EVERY stage on {cores} host threads (best effort: the "
                       f"reference itself runs rotate / attenuate / adjust / Poisson on one thread), float32 FFT convolution like FFTConvolution, "
                       f"O(lambda) Poisson loop of PoissonGenerator split over slices; voxels/s does not depend on the number of views"),
            "seconds_per_view": dt, "views_per_s": 1.0 / dt, "stage_seconds": st}
    line = {"impl": "reference", "metric": "simulated voxels/s (per-view acquisition pipeline)", "value": base["value"], "unit": "voxels/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "steps_effective": 1, "warmup_effective": 0,
            "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg, "views_per_s": base["views_per_s"], "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": "voxels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def workload_config(name):
    shape, kshape, _, degrees, inc, snr = WORKLOADS[name]
    return {"workload": f"BASELINE config 3 (configs[2])" if name == "cfg3" else name,
            "volume_xyz": [shape[2], shape[1], shape[0]], "psf_xyz": [kshape[2], kshape[1], kshape[0]],
            "views_per_gpu_per_step": len(degrees), "degrees": degrees, "axis": 0, "delta": 0.01, "inc": inc, "snr": snr,
            "l2": "inputs exceed L2 (2.1 GB ground truth, 2.4-3.4 GB spectra per pass vs 126 MB L2)",
            "parallelism": "view-sharded, one batch of views per GPU, no collective"}


def run_ours(args, rank, world, local_rank):
    import torch
    import mvsim_b200 as mv
    from mvsim_b200._lib import check
    import ctypes as C

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the CUDA path is the only implementation (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    grp = mv.Group("nccl", device=torch.device("cuda", local_rank))     # control plane only: barrier, max, sum

    shape, kshape, sigma, degrees, inc, snr = WORKLOADS[args.workload]
    degrees = [d + 7 * rank for d in degrees]          # every rank owns different views
    nv = len(degrees)
    vox_per_view = int(np.prod(shape))
    oshape = ((shape[0] - 1) // inc + 1, shape[1], shape[2])

    stream = torch.cuda.Stream()            # a real (non-default) stream shared by torch's events and the library's kernels
    torch.cuda.set_stream(stream)
    ctx = mv.Context(local_rank, cuda_stream=stream.cuda_stream)
    lib = ctx._lib

    # ---- inputs: pinned host buffers (e2e) and device-resident volumes (value) ----------------------
    gt_pin = mv.PinnedBuffer(shape)
    gt_pin.array[...] = make_ground_truth(shape)
    psf_raw = make_psfs(kshape, sigma, nv)
    psf_pin = [mv.PinnedBuffer(kshape) for _ in range(nv)]
    out_pin = [mv.PinnedBuffer(oshape) for _ in range(nv)]
    d_gt = mv.DeviceVolume(ctx, shape, gt_pin.array)
    d_psf = [mv.DeviceVolume(ctx, kshape, p) for p in psf_raw]
    d_out = [mv.DeviceVolume(ctx, oshape) for _ in range(nv)]
    params = [mv.make_view_params(shape, kshape, 0, degrees[v], 0.01, 0.0001, 1.0, inc, snr, seed=464232194, stream=rank * nv + v)
              for v in range(nv)]

    def step_device():
        for v in range(nv):
            check(lib.mvsim_dev_simulate_view(ctx.h, C.byref(params[v]), d_gt.h, d_psf[v].h, d_out[v].h), ctx.h)

    def barrier():
        torch.cuda.synchronize()
        grp.barrier()
        torch.cuda.synchronize()

    max_over_ranks = grp.max

    # ---- device-resident arm -------------------------------------------------------------------------
    clocks = ClockSampler(local_rank) if rank == 0 else None      # started early; samples are counted from mark_start() on
    for _ in range(args.warmup):
        step_device()
    barrier()
    ctx.profile(True)
    launches0 = ctx.kernel_launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if clocks:
        clocks.mark_start()
    e0.record(stream)
    for _ in range(args.steps):
        step_device()
    e1.record(stream)
    barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    clk = clocks.stop() if clocks else None
    launches = ctx.kernel_launches - launches0
    stage = ctx.stage_times()
    ctx.profile(False)
    launches = grp.sum(launches)
    ms_step = ms_total / args.steps
    value = world * nv * vox_per_view / (ms_step * 1e-3)           # COLD: every view rebuilds its PSF spectrum like the reference (:257)
    if args.dump_outputs and rank == 0:        # before the arms below overwrite d_out; out_pin is free until the e2e arm
        dump = {}
        for v in range(nv):
            dump[f"acquired_view{v}"] = d_out[v].download(out_pin[v].array)
            dump[f"psf_view{v}"] = d_psf[v].download()
        dump_outputs(args.dump_outputs, dump)

    # the same step with the PSF-spectrum cache on (SURVEY C6): the six PSFs repeat from step to step, so every view hits
    ctx.psf_cache(8 << 30)
    step_device()
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        step_device()
    e1.record(stream)
    barrier()
    warm_ms_step = max_over_ranks(e0.elapsed_time(e1)) / args.steps
    cache_stats = ctx.psf_cache_stats()
    ctx.psf_cache(0)

    # ---- end-to-end arm: host buffers through the C ABI ------------------------------------------------
    # Serial: one caller thread, one context: every step = ground truth H2D, 6 views, results D2H (downloads overlap the
    # next view inside the call).  Pipelined: THREE caller threads with one context each (the calling pattern of the
    # reference's own S/SimulateTileStitching.java:85-117), each running --steps steps; the library's per-device upload / compute gates line the
    # callers up so that the H2D of one step runs under the kernels of another and the D2H tail of a third (PCIe is full duplex).  Every step still moves all of its bytes inside the timed region.
    S = mv.SimulateMultiViewDataset
    e2e_steps = args.steps
    kvox, ovox = int(np.prod(kshape)), int(np.prod(oshape))

    def step_e2e(c=ctx, psfs=psf_pin, outs=out_pin):
        for v in range(nv):
            psfs[v].array[...] = psf_raw[v]          # the call normalises the PSF in place
        S.simulateViews(gt_pin.array, [p.array for p in psfs], degrees, inc=inc, poissonSNR=snr, rnd=464232194, ctx=c,
                        outs=[o.array for o in outs], first_stream=rank * nv)

    # the same protocol at every N: up to three caller threads per rank (pinned host memory permitting), the same step counts
    callers = [(ctx, psf_pin, out_pin)]
    per_caller = nv * (4 * ovox + 4 * kvox + 2 * ovox)          # pinned outputs + PSFs + uint16 staging
    for _ in range(2):
        try:
            import psutil
            if psutil.virtual_memory().available < 3 * world * per_caller:      # never drive the box towards its memory limit
                break
        except ImportError:
            pass
        try:
            callers.append((mv.Context(local_rank), [mv.PinnedBuffer(kshape) for _ in range(nv)], [mv.PinnedBuffer(oshape) for _ in range(nv)]))
        except (MemoryError, mv.MvsimError):
            break                           # pinned host memory exhausted: fewer callers
    n_callers = int(grp.min(len(callers)))      # the same number on every rank
    callers = callers[:n_callers]
    pipe_steps = n_callers * args.steps         # every caller thread runs --steps steps
    gt_tensor = torch.empty(shape, dtype=torch.float32, device=torch.device("cuda", local_rank)) if world > 1 else None
    gt_tensor_b = torch.empty_like(gt_tensor) if world > 1 else None

    def caller_loop(i, n):
        for _ in range(n):
            step_e2e(*callers[i])

    def step_bcast():
        for v in range(nv):
            psf_pin[v].array[...] = psf_raw[v]
        vol, _ = grp.broadcast_ground_truth(ctx, shape, host=gt_pin.array if rank == 0 else None, tensor=gt_tensor)
        S.simulateViews(vol, [p.array for p in psf_pin], degrees, inc=inc, poissonSNR=snr, rnd=464232194, ctx=ctx,
                        outs=[o.array for o in out_pin], first_stream=rank * nv)
        vol.free()

    def checksum(outs):
        return float(outs[0].array[::7, ::31, ::29].astype(np.float64).mean())

    def run_modes(uint16, host_threads=0):
        """All e2e modes with one count transport; returns {mode: ms per step (max over ranks)} and the result checksum."""
        for c, _, _ in callers:
            c.count_transport(uint16, host_threads=host_threads)
        res = {}
        for i in range(n_callers):           # warm every context (workspaces, staging buffers)
            caller_loop(i, 1)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            step_e2e()
        barrier()
        res["serial"] = max_over_ranks((time.perf_counter() - t0) * 1e3 / e2e_steps)
        chk = checksum(out_pin)
        if n_callers > 1:
            barrier()
            threads = [threading.Thread(target=caller_loop, args=(i, pipe_steps // n_callers)) for i in range(n_callers)]
            t0 = time.perf_counter()
            for t in threads:
                t.start()
            for t in threads:
                t.join()                        # every call returns only after its results are in the host buffers
            torch.cuda.synchronize()
            res["pipelined"] = max_over_ranks((time.perf_counter() - t0) * 1e3 / pipe_steps)
            barrier()
            if checksum(callers[-1][2]) != chk:
                raise SystemExit("bench.py: concurrent callers changed the result")
        if world > 1:
            step_bcast()
            barrier()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                step_bcast()
            barrier()
            res["broadcast"] = max_over_ranks((time.perf_counter() - t0) * 1e3 / e2e_steps)
            if checksum(out_pin) != chk:
                raise SystemExit("bench.py: broadcast ground truth changed the result")
            # the same, with the NEXT dataset's ground truth uploaded (rank 0) and broadcast on a side stream while the current one is
            # simulated and its results drain: the host link is full duplex and the results' direction is the busy one
            bufs = [gt_tensor, gt_tensor_b]
            side = torch.cuda.Stream()

            def issue(i):
                with torch.cuda.stream(side):
                    if rank == 0:
                        bufs[i].copy_(torch.from_numpy(gt_pin.array), non_blocking=True)
                    return grp.dist.broadcast(bufs[i], src=0, async_op=True)

            def run_prefetched(n):
                w = issue(0)
                for k in range(n):
                    w.wait()
                    side.synchronize()
                    torch.cuda.current_stream().synchronize()
                    cur = bufs[k % 2]
                    w = issue((k + 1) % 2)              # every step issues one upload + broadcast (the last one is waited for below)
                    for v in range(nv):
                        psf_pin[v].array[...] = psf_raw[v]
                    vol = mv.DeviceVolume.wrap(ctx, shape, cur.data_ptr(), keepalive=cur)
                    S.simulateViews(vol, [p.array for p in psf_pin], degrees, inc=inc, poissonSNR=snr, rnd=464232194, ctx=ctx,
                                    outs=[o.array for o in out_pin], first_stream=rank * nv)
                    vol.free()
                w.wait()
                side.synchronize()
                torch.cuda.current_stream().synchronize()
            run_prefetched(1)
            barrier()
            t0 = time.perf_counter()
            run_prefetched(e2e_steps)
            barrier()
            # n steps contain n + 1 uploads, the first of them not overlapped: a conservative figure
            res["broadcast_prefetch"] = max_over_ranks((time.perf_counter() - t0) * 1e3 / e2e_steps)
            if checksum(out_pin) != chk:
                raise SystemExit("bench.py: prefetched broadcast changed the result")
        return res, chk

    MODE_TEXT = {"serial": "1 caller thread per rank, ground truth uploaded by every rank",
                 "pipelined": f"{n_callers} caller threads x 1 context each per rank, --steps steps each (H2D of one step runs under the kernels and D2H of the others)",
                 "broadcast": "views of one dataset sharded over the ranks: ground truth uploaded once by rank 0 and NCCL-broadcast over NVLink, 1 caller per rank",
                 "broadcast_prefetch": ("views of one dataset sharded over the ranks, one dataset per step: the next dataset's ground truth is uploaded by rank 0 and "
                                        "NCCL-broadcast on a side stream while the current one is simulated and its results drain, 1 caller per rank")}
    modes_f32, chk_f32 = run_modes(False)
    modes_u16, result_checksum = run_modes(True, args.widen_threads)
    widen_sweep = {}
    for t in (args.widen_sweep or []):          # investigation only: other widening thread counts
        widen_sweep[str(t)], _ = run_modes(True, t)
    if chk_f32 != result_checksum:
        raise SystemExit(f"bench.py: the uint16 count transport changed the result ({result_checksum} vs {chk_f32})")
    # headline: the fastest (mode, transport) pair; every other pair is printed beside it
    best_u16, best_f32 = min(modes_u16, key=modes_u16.get), min(modes_f32, key=modes_f32.get)
    use_u16 = modes_u16[best_u16] < modes_f32[best_f32]
    e2e_key = best_u16 if use_u16 else best_f32
    e2e_ms = (modes_u16 if use_u16 else modes_f32)[e2e_key]
    e2e_mode = MODE_TEXT[e2e_key]
    h2d = (4 * vox_per_view // world if e2e_key.startswith("broadcast") else 4 * vox_per_view) + nv * 4 * kvox      # per rank (broadcast: one upload for all)
    d2h_u16 = nv * (2 * ovox + 4 * kvox + 4)        # uint16 counts + the normalised PSFs + the overflow flags
    d2h_f32 = nv * 4 * (ovox + kvox)
    d2h = d2h_u16 if use_u16 else d2h_f32
    barrier()
    link = host_link_probe(torch)            # every rank at the same time: the rates a GPU gets while its neighbours use the host too
    barrier()

    if rank != 0:
        grp.close()
        return

    # ---- roofline of the dominant kernel ------------------------------------------------------------------
    nfft = (C.c_int64 * 3)()
    check(lib.mvsim_conv_padded_dims(mv._lib.dims3(shape), mv._lib.dims3(kshape), nfft))
    kxc, ny, nz = nfft[0] // 2, nfft[1], nfft[2]
    z_ms, z_n = stage["fft_zfused"]
    planes_out = oshape[0] + 1 if (inc > 1 and oshape[0] + 1 <= shape[0]) else shape[0]
    # algorithmic bytes of the fused z pass per launch (= per view): SURVEY section 8(d) counts 3S for it (read S, read the
    # PSF spectrum S, write S; S = 8 (Nx/2+1) Ny Nz).  The pruned kernel must move less: read Z planes + H (Nz planes) +
    # write the kept planes and one sum plane; that figure and the ncu DRAM traffic are reported beside it.
    S_model = 8 * (nfft[0] // 2 + 1) * ny * nz
    bytes_model = 3 * S_model
    otf = not os.environ.get("MVSIM_H_MATERIALIZE")
    bytes_pruned = 8 * kxc * ny * (shape[0] + (kshape[0] if otf else nz) + planes_out)   # U2 planes + PSF partial spectrum (or H) + kept planes
    peak, peak_src = measured_peak_gbs()
    per_launch_ms = z_ms / max(z_n, 1)
    # PRIMARY figure: the bytes the pruned kernel MUST move once per launch (read Z planes of U2 + the PSF partial spectrum,
    # write the kept planes + the sum plane) / its CUDA-event time.  ncu's dram bytes of the same kernel (`traffic`, from the
    # committed profile named in `traffic_source`) equal this figure, i.e. there are no wasted re-reads.  The 3S figure SURVEY 8(d)
    # books for a z pass that reads and writes the whole padded spectrum plus a materialised PSF spectrum is a MODEL-EQUIVALENT
    # throughput (what an unpruned pass would have to sustain to be as fast), not achieved bandwidth: reported as *_model_3S.
    achieved = bytes_pruned / (per_launch_ms * 1e-3) / 1e9
    achieved_model = bytes_model / (per_launch_ms * 1e-3) / 1e9
    traffic, traffic_src = None, None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if args.workload == "cfg3":
            traffic, traffic_src = tj["fft_zfused"]["bytes"], tj["fft_zfused"].get("source")
    except Exception:
        pass
    fft_passes = {k: stage[k][0] / max(stage[k][1], 1) for k in ("fft_xfwd", "fft_yfwd", "fft_zfused", "fft_yinv", "fft_xinv")}
    N = vox_per_view
    O = int(np.prod(oshape))
    b_fused_model = 8 * N + 9 * S_model + 8 * O
    b_stage_model = 32 * N + 11 * S_model + 8 * O
    view_ms = ms_step / nv
    roofline = {"bound": "hbm", "kernel": ("fft_zfused (ZFusedPoly at config 3: the kept planes as inc cyclic convolutions of Nz / inc points -- forward transforms of the image and "
                           "PSF phases, multiply-add, one inverse -- plus the sum plane, in place)"),
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": peak_src, "bytes_per_launch": bytes_pruned,
                "bytes_basis": ("compulsory bytes of the pruned pass per view: 8 B x KXc x Ny x (Z planes read + KZ planes of the PSF partial spectrum read "
                                "+ kept planes and one sum plane written); equals the ncu dram bytes. The kernel is FP32-issue bound, not HBM bound "
                                "(ten 128-point forward transforms and one inverse per line on 4 B of traffic per point; DESIGN.md section 4.1)"),
                "bytes_per_launch_model_3S": bytes_model, "achieved_model_3S": achieved_model, "frac_model_3S": achieved_model / peak,
                "model_3S_basis": "SURVEY 8(d): read S + PSF spectrum S + write S for an unpruned fused z pass; model-equivalent throughput, not bandwidth",
                "ms_per_launch": per_launch_ms, "launches_timed": z_n,
                "whole_view": {"ms": view_ms, "B_fused_model_GB": b_fused_model / 1e9, "B_stage_model_GB": b_stage_model / 1e9,
                               "frac_of_peak_fused_model": b_fused_model / (view_ms * 1e-3) / 1e9 / peak,
                               "frac_of_peak_stage_model": b_stage_model / (view_ms * 1e-3) / 1e9 / peak}}
    stages_ms = {k: {"ms_per_view": v[0] / (args.steps * nv), "launches": v[1]} for k, v in stage.items() if v[1]}
    # every pass against the same peak: compulsory bytes of the pruned pass (what it must read + write once) / its CUDA-event time
    try:
        X, Y, Z = shape[2], shape[1], shape[0]
        u1, u2 = 8 * kxc * Y * Z, 8 * kxc * ny * Z
        per_pass_bytes = {"rotate": 8 * N, "fft_xfwd": 4 * N + u1, "fft_yfwd": u1 + u2, "fft_zfused": bytes_pruned,
                          "fft_yinv": planes_out * 8 * kxc * (ny + Y), "fft_xinv": planes_out * Y * (8 * kxc + 4 * X), "sample": 8 * O}
        roofline["passes"] = {k: {"GB": b / 1e9, "GBps": b / (stages_ms[k]["ms_per_view"] * 1e-3) / 1e9,
                                  "frac": b / (stages_ms[k]["ms_per_view"] * 1e-3) / 1e9 / peak}
                              for k, b in per_pass_bytes.items() if k in stages_ms and stages_ms[k]["ms_per_view"] > 0}
        moved = sum(per_pass_bytes.values())
        roofline["whole_view"]["compulsory_GB"] = moved / 1e9
        roofline["whole_view"]["frac_of_peak_compulsory"] = moved / (view_ms * 1e-3) / 1e9 / peak
    except Exception as e:      # reporting only
        roofline["passes"] = {"error": str(e)}

    cpu = cpu_baseline_sample(args.workload) if not args.no_cpu else {"value": None, "unit": "voxels/s", "cores": 0, "kind": "port", "sample": "skipped"}

    line = {"metric": "simulated voxels/s (per-view acquisition pipeline)", "value": value, "unit": "voxels/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args.workload),
            "views_per_s": world * nv / (ms_step * 1e-3), "ms_per_view": view_ms,
            "value_is": "cold: PSF-spectrum cache off, every view rebuilds its PSF spectrum like the reference (S/SimulateMultiViewDataset.java:257)",
            "psf_cache_warm": {"value": world * nv * vox_per_view / (warm_ms_step * 1e-3), "unit": "voxels/s", "ms_per_step": warm_ms_step,
                               "ms_per_view": warm_ms_step / nv, "hits": cache_stats["hits"], "misses": cache_stats["misses"],
                               "bytes_held": cache_stats["bytes"],
                               "note": "mvsim_psf_cache_configure(8 GiB): repeated PSFs skip their x / y transforms; not the headline"},
            "e2e": {"value": world * nv * vox_per_view / (e2e_ms * 1e-3), "unit": "voxels/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms, "views_per_s": world * nv / (e2e_ms * 1e-3),
                    "api": "mvsim_simulate_views / mvsim_dev_simulate_views (pinned host buffers in, float32 volumes out)",
                    "steps": pipe_steps if e2e_key == "pipelined" else e2e_steps, "mode": e2e_mode, "mode_key": e2e_key, "callers": n_callers,
                    "count_transport": "uint16" if use_u16 else "float32",
                    "count_transport_note": ("uint16 = opt-in MVSIM_OPT_COUNT_TRANSPORT: Poisson counts cross the host link as uint16 and host threads widen "
                                             "them to the caller's float32 buffers inside the timed call (bit-identical results, half the D2H bytes, but "
                                             "3x the host-memory traffic of the results); both transports are timed in every mode, the headline is the fastest pair"),
                    "ms_per_step_by_mode_uint16_transport": modes_u16, "ms_per_step_by_mode_float32_transport": modes_f32,
                    "d2h_bytes_per_step_uint16_transport": d2h_u16, "d2h_bytes_per_step_float32_transport": d2h_f32,
                    "widen_threads": args.widen_threads, "widen_sweep_ms_per_step": widen_sweep or None,
                    "host_link": link,
                    "frac_of_host_link": (max(h2d / link["h2d_concurrent_GBps"], d2h / link["d2h_concurrent_GBps"]) / 1e9 / (e2e_ms * 1e-3)) if link else None,
                    "frac_of_host_link_basis": ("time the busier direction needs at rank 0's rate with both directions active and all N GPUs copying at once "
                                                "/ e2e time per step"),
                    "result_checksum": result_checksum},
            "gpu_launches": launches, "roofline": roofline, "stages": stages_ms, "fft_ms_per_launch": fft_passes,
            "fft_padded_xyz": [int(nfft[0]), int(ny), int(nz)], "cpu_baseline": cpu, "clocks": clk}
    print(json.dumps(line), flush=True)
    grp.close()


def run_slab(args, rank, world, local_rank):
    """BASELINE config 5 (configs[4]): ONE 2048x2048x1024 volume, PSF 256^3, convolve stage only, z slabs over the
    N GPUs with two NCCL all-to-all transposes per y block (strong scaling).  Not the default bench line."""
    import torch
    import mvsim_b200 as mv
    from helpers import gaussian_psf
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    grp = mv.Group("nccl", device=dev)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = mv.Context(local_rank, cuda_stream=stream.cuda_stream)
    shape, kshape = ((1024, 2048, 2048), (256, 256, 256)) if args.workload == "cfg5" else ((256, 512, 512), (64, 64, 64))
    sc = mv.SlabConvolution(ctx, shape, kshape, grp.rank, grp.world, grp.dist, p2p=not os.environ.get("MVSIM_SLAB_NCCL"))
    g = torch.Generator(device=dev)
    g.manual_seed(1234 + rank)
    img = torch.rand((sc.z_local,) + shape[1:], generator=g, device=dev, dtype=torch.float32)     # generated on device, slab-wise
    psf = gaussian_psf(kshape, (kshape[0] / 7.3, kshape[1] / 23.0, kshape[2] / 25.0), threshold=1e-3)
    d_psf = torch.from_numpy(psf).to(dev)
    d_psf /= d_psf.double().sum().float()
    out = torch.empty_like(img)

    def barrier():
        torch.cuda.synchronize()
        grp.barrier()
        torch.cuda.synchronize()
    for _ in range(args.warmup):
        sc.convolve(img, d_psf, out)
    nv0 = nvlink_counters(local_rank)       # (NVML queries take milliseconds: before the barrier, so that no rank enters the timed loop late)
    barrier()
    ctx.profile(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        sc.convolve(img, d_psf, out)
    e1.record(stream)
    barrier()
    nv1 = nvlink_counters(local_rank)
    ms = grp.max(e0.elapsed_time(e1)) / args.steps
    nvlink = None
    if nv0 and nv1:
        tx, rx = (nv1[0] - nv0[0]) / args.steps, (nv1[1] - nv0[1]) / args.steps
        nvlink = {"tx_bytes_per_step": tx, "rx_bytes_per_step": rx, "tx_GBps_over_the_step": tx / (ms * 1e-3) / 1e9, "rx_GBps_over_the_step": rx / (ms * 1e-3) / 1e9,
                  "peak_GBps_per_direction": 900.0, "source": "NVML NVLINK_THROUGHPUT_DATA_TX/RX of rank 0's GPU, all links, around the timed region"}
    stage = {k: round(v[0] / args.steps, 3) for k, v in ctx.stage_times().items() if v[1]}
    chk = float(out[::max(1, sc.z_local // 4), ::97, ::89].double().mean().item())
    if args.dump_outputs and rank == 0:        # rank 0's slab, sampled on the device (16 GB at config 5 on one GPU)
        res, share = out, DUMP_BYTES // 4
        if out.numel() > share:
            res = out.reshape(-1)[torch.from_numpy(dump_indices(out.numel(), share)).to(dev)]
        dump_outputs(args.dump_outputs, {"convolved_slab_rank0": res.cpu().numpy()})
    if rank == 0:
        vox = int(np.prod(shape))
        print(json.dumps({"metric": "convolved voxels/s (slab-decomposed FFT convolution)", "value": vox / (ms * 1e-3), "unit": "voxels/s",
                          "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
                          "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                          "config": {"workload": "BASELINE config 5 (configs[4])" if args.workload == "cfg5" else args.workload,
                                     "volume_xyz": list(shape[::-1]), "psf_xyz": list(kshape[::-1]), "fft_padded_xyz": list(sc.nfft),
                                     "y_blocks": sc.y_blocks, "parallelism": (f"z slabs x{world}, exchanges fused into the y and z kernels as NVLink peer stores" if sc.p2p else
                                                     f"z slabs x{world}, NCCL all_to_all_single x{2 * sc.y_blocks}")},
                          "nvlink_bytes_sent_per_rank_per_step": sc.exchange_bytes_per_rank(), "nvlink_counters_rank0": nvlink,
                          "rank0_kernel_ms_per_step": stage,
                          "rank0_kernel_ms_total": round(sum(stage.values()), 3), "result_checksum": chk}), flush=True)
    sc.close()
    grp.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS) + ["cfg5", "cfg5small"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--widen-threads", type=int, default=0, help="host threads per context that widen uint16 counts (0 = library default)")
    ap.add_argument("--widen-sweep", type=int, nargs="*", help="also time the uint16 transport with these widening thread counts")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy (float32, sampled to "
                                                          "at most 60 MiB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU path (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world == 1 and args.gpus > 1:
        # plain `python bench.py --gpus N`: relaunch under torchrun, one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", str(29500 + os.getpid() % 1000), os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    if args.workload.startswith("cfg5"):
        run_slab(args, rank, world, local_rank)
        return
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
