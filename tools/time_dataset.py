#!/usr/bin/env python3
"""Measurements of main()'s post-acquisition chain in one device call (DESIGN.md section 8, row 8f-5).

    python tools/time_dataset.py [out.json] [--skip-wall]

1. CUDA-event milliseconds per view of the two new kernels at config 3 (1024 x 1024 x 512, inc 5: acq 103 planes, aligned 511
   planes; 6 views), with the rate on their compulsory bytes and its fraction of the project's measured 6534 GB/s copy peak, and
   timed reference variants that bound them: a store-only fill of the aligned view's bytes, the existing rotate kernel on an
   isotropic volume (the second of the two stages align_view replaces) and a device copy.
2. Wall seconds per view, outputs in host memory: run_main (stage entry points, one host round trip per stage) against
   simulate_dataset at 289^3 x 7 views, and the same two chains at config 3 x 6 views, with output equality checked in the run.
The card name and power limit are read in the same run."""
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
import mvsim_b200 as mv  # noqa: E402

COPY_PEAK_GBS = 6534.0          # device-to-device copy peak measured for this project on a B200 (BASELINE.md)
S = mv.SimulateMultiViewDataset
res = {}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def event_ms(fn, reps=20, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def kernels():
    ctx = mv.Context(0, cuda_stream=torch.cuda.current_stream().cuda_stream)
    X, Y, Z, inc = 1024, 1024, 512, 5
    za = (Z - 1) // inc + 1
    ziso = (za - 1) * inc + 1
    acq = mv.DeviceVolume(ctx, (za, Y, X), np.random.default_rng(1).random((za, Y, X), dtype=np.float32) * 200)
    out = mv.DeviceVolume(ctx, (ziso, Y, X))
    angles = [0, 60, 120, 180, 240, 300]
    r = {}
    b_align = 4 * X * Y * (ziso + za)
    t = event_ms(lambda: acq.alignView(inc, -60, out=out))
    r["align_view"] = {"ms": t, "compulsory_GB": b_align / 1e9, "GB_s": b_align / t / 1e6, "of_copy_peak": b_align / t / 1e6 / COPY_PEAK_GBS}
    w = mv.DeviceVolume(ctx, (Z, Y, X))
    lib, i32 = ctx._lib, C.c_int32
    al = (i32 * 6)(*[-a for a in angles])
    one = (i32 * 1)(1)
    oarr = (C.c_void_p * 1)(w.h.value)
    dims = mv._lib.dims3((Z, Y, X))

    def weights():
        mv._lib.check(lib.mvsim_dev_aligned_weights(ctx.h, dims, 6, al, 3.0, 1, one, oarr, None), ctx.h)
    b_w = 4 * X * Y * Z
    t = event_ms(weights)
    r["aligned_weights"] = {"ms": t, "compulsory_GB": b_w / 1e9, "GB_s": b_w / t / 1e6, "of_copy_peak": b_w / t / 1e6 / COPY_PEAK_GBS}
    # bounds: stores alone (the aligned view's output bytes), a copy, and the existing rotate kernel over an isotropic volume
    buf = torch.empty(X * Y * ziso, dtype=torch.float32, device="cuda")
    t = event_ms(lambda: buf.fill_(1.0))
    r["variant_store_only_fill_aligned_bytes"] = {"ms": t, "GB_s": 4 * X * Y * ziso / t / 1e6}
    src = torch.rand(X * Y * ziso // 2, device="cuda")
    dst = torch.empty_like(src)
    t = event_ms(lambda: dst.copy_(src))
    r["variant_copy"] = {"ms": t, "GB_s": 2 * 4 * src.numel() / t / 1e6}
    iso = mv.DeviceVolume(ctx, (ziso, Y, X))
    mv._lib.check(lib.mvsim_dev_align_view(ctx.h, acq.h, inc, 0, iso.h), ctx.h)
    t = event_ms(lambda: mv._lib.check(lib.mvsim_dev_rotate_axis(ctx.h, iso.h, out.h, 0, -60), ctx.h))
    r["variant_existing_rotate_on_iso_volume"] = {"ms": t, "GB_s": 2 * 4 * X * Y * ziso / t / 1e6}
    for v in (acq, out, w, iso):
        v.free()
    del buf, src, dst
    ctx.close()
    return r


def chain_main(ctx, gt, psf, angles, inc, snr, osem, offset=15, delta=0.01):
    """run_main's view loop body (:567-663) through the stage entry points for an arbitrary ground truth; outputs in host memory."""
    rnd = mv.JavaRandom(S.seed)
    out = {"acq": [], "view": [], "psf": [], "weights": []}
    for v, angle in enumerate(angles):
        rot = S.rotateAroundAxis(gt, 0, angle + offset, ctx=ctx)
        att = S.attenuate3d(rot, delta, ctx=ctx)
        w = S.computeWeightImage(rot, delta, ctx=ctx)
        del rot
        k = psf.copy()
        con = S.convolve(att, k, None, ctx=ctx)
        del att
        mv.Tools.adjustImage(con, S.minValue, S.avgIntensity, ctx=ctx)
        acq = S.extractSlices(con, inc, snr, rnd=rnd, ctx=ctx, stream=v)
        del con
        out["view"].append(S.rotateAroundAxis(S.makeIsotropic(acq, inc, ctx=ctx), 0, -angle, ctx=ctx))
        out["weights"].append(S.rotateAroundAxis(w, 0, -angle, ctx=ctx))
        out["psf"].append(S.rotateAroundAxis(k, 0, -angle, ctx=ctx))
        out["acq"].append(acq)
    out["sum_weights"] = S.normalizeWeights(out["weights"], osem, ctx=ctx)
    return out


def compare(a, b):
    """fraction of equal voxels per output kind (acq: Poisson counts of two paths that differ by rounding before the sampler)"""
    r = {}
    for key in ("acq", "view", "psf", "weights"):
        r[key] = min(float(np.mean(x == y)) for x, y in zip(a[key], b[key]))
    r["sum_weights"] = float(np.mean(a["sum_weights"] == b["sum_weights"]))
    return r


def walls():
    r = {}
    ctx = mv.Context(0)
    psf = mv.default_psf()
    quiet = dict(log=lambda *_: None, keep=("acq", "view", "weights", "psf"), ctx=ctx, psf=psf)
    mv.simulate_dataset(None, size=121, angle_increment=120, **quiet)            # warm up: module load, plans, pools
    mv.run_main(None, size=121, angle_increment=120, **quiet)
    t0 = time.perf_counter()
    a = mv.run_main(None, size=289, angle_increment=52, **quiet)
    t1 = time.perf_counter()
    b = mv.simulate_dataset(None, size=289, angle_increment=52, **quiet)
    t2 = time.perf_counter()
    n = len(a["angles"])
    r["289^3_x7"] = {"views": n, "run_main_s_per_view": (t1 - t0) / n, "simulate_dataset_s_per_view": (t2 - t1) / n,
                     "equal_fraction": compare(a, b)}
    del a, b
    shape, kshape, sigma, _, inc, snr = bench.WORKLOADS["cfg3"]
    small = bench.make_ground_truth((shape[0] // 8, shape[1], shape[2]))
    gt = np.concatenate([small] * 8, axis=0)
    k = bench.make_psfs(kshape, sigma, 1)[0]
    angles = [0, 60, 120, 180, 240, 300]
    t0 = time.perf_counter()
    a = chain_main(ctx, gt, k, angles, inc, snr, 3.0)
    t1 = time.perf_counter()
    d = S.simulateDataset(gt, [k.copy() for _ in angles], angles, inc=inc, poissonSNR=snr, osem=3.0, ctx=ctx)
    t2 = time.perf_counter()
    b = {"acq": d["acq"], "view": d["aligned"], "psf": d["aligned_psf"], "weights": d["weights"], "sum_weights": d["sum_weights"]}
    r["cfg3_x6"] = {"dims": list(shape[::-1]), "inc": inc, "snr": snr, "views": 6, "run_main_chain_s_per_view": (t1 - t0) / 6,
                    "simulate_dataset_s_per_view": (t2 - t1) / 6, "equal_fraction": compare(a, b)}
    ctx.close()
    return r


if __name__ == "__main__":
    out_path = next((p for p in sys.argv[1:] if not p.startswith("--")), None)
    res["card"] = card()
    res["kernels_cfg3"] = kernels()
    print(json.dumps(res, indent=1), flush=True)
    if "--skip-wall" not in sys.argv:
        res["wall_host_outputs"] = walls()
    print(json.dumps(res, indent=1))
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as f:
            json.dump(res, f, indent=1)
