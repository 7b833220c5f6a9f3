#!/usr/bin/env python3
"""Measurements of the tile-stitching pair generator on the device (DESIGN.md section 8, mvsim_dev_extract_interval).

    python tools/time_tile_pairs.py [out.json]

1. CUDA-event milliseconds of mvsim_dev_extract_interval (the tile read in place from its parent) against
   mvsim_dev_extract_slices on the materialised tile with the same output dims, at snr = -1 (copy) and snr = 25 (Poisson), inc 3:
   the 289^3 pair's tile 1 (174^3 voxels at min = 115, rows not 4-aligned) and a 1024 x 1024 x 512 parent with a 0.6-size tile.
   Every timed launch reads another copy of its input, so the working set of a timed loop exceeds the 126 MB L2.
2. Wall milliseconds of SimulateTileStitching.getNextPair: the former driver path (two threads, a new context each, numpy cut,
   host-buffer extractSlices) rebuilt here, against the driver's device path, at size 289 and 512, with the two results
   checked equal in the run.
The card name and power limit are read in the same run.  Needs a CUDA device; fails without one."""
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import mvsim_b200 as mv  # noqa: E402
from mvsim_b200._lib import check  # noqa: E402

S = mv.SimulateMultiViewDataset
L2_BYTES = 126 << 20
INC = 3


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def event_ms(fns, reps, warmup=3):
    """mean milliseconds of one call, cycling over fns (one per input copy)"""
    for i in range(warmup * len(fns)):
        fns[i % len(fns)]()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(reps):
        fns[i % len(fns)]()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def kernel_case(ctx, name, parent_zyx, mn, mx):
    lib = ctx._lib
    i3 = C.c_int64 * 3
    b = [mx[d] - mn[d] + 1 for d in range(3)]
    out_zyx = ((b[2] - 1) // INC + 1, b[1], b[0])
    read_bytes = 4 * out_zyx[0] * out_zyx[1] * out_zyx[2]
    copies = max(2, -(-3 * L2_BYTES // read_bytes))
    g = torch.Generator(device="cuda").manual_seed(3)
    parents = [torch.rand(parent_zyx, device="cuda", generator=g) * 2 for _ in range(copies)]
    tiles = [p[mn[2]:mx[2] + 1, mn[1]:mx[1] + 1, mn[0]:mx[0] + 1].contiguous() for p in parents]
    torch.cuda.synchronize()
    pv = [mv.DeviceVolume.wrap(ctx, p.shape, p.data_ptr(), keepalive=p) for p in parents]
    tv = [mv.DeviceVolume.wrap(ctx, t.shape, t.data_ptr(), keepalive=t) for t in tiles]
    out = mv.DeviceVolume(ctx, out_zyx)
    r = {"parent_xyz": parent_zyx[::-1], "min": list(mn), "max": list(mx), "out_xyz": list(out_zyx[::-1]), "input_copies": copies}
    for snr in (-1.0, 25.0):
        def interval(v):
            return lambda: check(lib.mvsim_dev_extract_interval(ctx.h, v.h, i3(*mn), i3(*mx), INC, snr, 7, 1, out.h), ctx.h)

        def dense(v):
            return lambda: check(lib.mvsim_dev_extract_slices(ctx.h, v.h, INC, snr, 7, 1, out.h), ctx.h)
        fi, fd = [interval(v) for v in pv], [dense(v) for v in tv]
        reps = max(20, 4 * copies)
        ti, td = [], []
        for _ in range(3):                       # alternated, three rounds each
            ti.append(event_ms(fi, reps))
            td.append(event_ms(fd, reps))
        a = mv.DeviceVolume(ctx, out_zyx)
        ref = mv.DeviceVolume(ctx, out_zyx)
        pv[0].extractSlices(INC, snr, rnd=7, stream=1, interval=(mn, mx), out=a)
        tv[0].extractSlices(INC, snr, rnd=7, stream=1, out=ref)
        same = bool(np.array_equal(a.download().view(np.uint32), ref.download().view(np.uint32)))
        a.free()
        ref.free()
        key = "snr_m1" if snr < 0 else "snr_25"
        r[key] = {"interval_ms": [round(v, 4) for v in ti], "dense_tile_ms": [round(v, 4) for v in td],
                  "interval_over_dense_median": round(statistics.median(ti) / statistics.median(td), 3),
                  "interval_read_gbs_median": round(read_bytes * 2 / statistics.median(ti) / 1e6, 1),   # kept-plane reads + tile writes
                  "bit_identical": same}
        print(name, key, r[key], flush=True)
    out.free()
    for v in pv + tv:
        v.free()
    del parents, tiles
    torch.cuda.empty_cache()
    return r


def old_pair(sts, src, snr, rnd):
    """the driver's getNextPair before the device path: one thread and a new context per tile, numpy cut, host-buffer extractSlices"""
    seeds = [rnd.nextInt(), rnd.nextInt()]
    out = [None, None]

    def task(i):
        ctx = mv.Context(0)
        mn, mx = sts.getInterval(i)
        cut = np.ascontiguousarray(src[i][mn[2]:mx[2] + 1, mn[1]:mx[1] + 1, mn[0]:mx[0] + 1])
        out[i] = S.extractSlices(cut, INC, snr, rnd=mv.JavaRandom(seeds[i]), ctx=ctx, stream=i)
        ctx.close()
    threads = [threading.Thread(target=task, args=(i,)) for i in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    return out


def wall_case(size, rounds=5):
    psf = mv.default_psf()
    t0 = time.perf_counter()
    sts = mv.SimulateTileStitching(None, True, (0.2, 0.2, 0.2), psf=psf, size=size)
    init_s = time.perf_counter() - t0
    src = [sts.con, sts.conHalfPixel]
    r = {"size": size, "init_s_device_path": round(init_s, 3), "tile_xyz": [sts.getInterval(1)[1][d] - sts.getInterval(1)[0][d] + 1 for d in range(3)]}
    for snr in (-1.0, 25.0):
        rnd_old, sts.rnd = mv.JavaRandom(77), mv.JavaRandom(77)
        old, new = [], []
        same = True
        for k in range(rounds + 2):                # two warm-up pairs each, then alternated
            a = time.perf_counter()
            o = old_pair(sts, src, snr, rnd_old)
            b = time.perf_counter()
            n = sts.getNextPair(snr)
            c = time.perf_counter()
            same &= all(np.array_equal(x.view(np.uint32), y.view(np.uint32)) for x, y in zip(o, n))
            if k >= 2:
                old.append((b - a) * 1e3)
                new.append((c - b) * 1e3)
        key = "snr_m1" if snr < 0 else "snr_25"
        r[key] = {"former_path_ms": [round(v, 2) for v in old], "device_path_ms": [round(v, 2) for v in new],
                  "speedup_median": round(statistics.median(old) / statistics.median(new), 2), "bit_identical": bool(same)}
        print("pair", size, key, r[key], flush=True)
    sts.close()
    return r


def main():
    if not torch.cuda.is_available():
        raise SystemExit("time_tile_pairs.py needs a CUDA device")
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    res = {"card": card(), "torch_device": torch.cuda.get_device_name(0), "inc": INC}
    ctx = mv.Context(0, cuda_stream=torch.cuda.current_stream().cuda_stream)
    res["kernels"] = {
        "pair_289": kernel_case(ctx, "pair_289", (289, 289, 289), (115, 115, 115), (288, 288, 288)),
        "parent_1024x1024x512": kernel_case(ctx, "parent_1024x1024x512", (512, 1024, 1024), (205, 205, 102), (818, 818, 408)),
    }
    ctx.close()
    res["pairs"] = [wall_case(289), wall_case(512)]
    res["card_after"] = card()
    text = json.dumps(res, indent=1)
    print(text)
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
