"""The two callers of the acquisition path inside the reference, mirrored on top of the CUDA library.

    run_main(...)            SimulateMultiViewDataset.main()     S/SimulateMultiViewDataset.java:524-665
    SimulateTileStitching    S/SimulateTileStitching.java:58-258

Both are host-side drivers (the reference's are single `main()` / constructor bodies); every stage they call goes
through the C ABI (api.py).  They exist so that a user of the reference finds the same entry points and file names,
and they double as integration tests of the boundary: the tile-stitching driver runs two pipelines from two threads
with one context each and re-samples one convolved volume at many SNRs, exactly the calling pattern the boundary must
support (SURVEY section 3.2).

    simulate_dataset(...)    main() with the view loop in one device call (acquisition + aligned outputs)

    python -m mvsim_b200.drivers --out /tmp/sim [--size 289] [--angles 7] [--psf-dir DIR] [--fused [--rank R --world W]]
"""
import argparse
import ctypes as C
import os
import threading
import time

import numpy as np

from . import tiff
from ._lib import check
from .api import Context, DeviceVolume, JavaRandom, SimulateMultiViewDataset as S, Tools

# main(): angleIncrement -> osem factor (:536-546)
OSEM = {60: 3.0, 52: 3.0, 45: 4.0}


def open_psf(path, square=True, ctx=None):
    """Tools.open(file, square) (S/Tools.java:297-307) for the reference's float32 TIFF stacks."""
    psf = tiff.read_float_stack(path)
    return Tools.makeSquare(psf, ctx=ctx) if square else psf


def default_psf(shape=(51, 51, 51), sigma=(7.0, 2.2, 2.0)):
    """Stand-in for the reference's measured PSF fixtures (src/main/resources/Angle*.tif: 51^3, peak 0.99 at the centre,
    sigma ~ (2.0, 2.2, 7.0) px in x, y, z, ~4 % support) when those files are not at hand."""
    z, y, x = shape
    zz, yy, xx = np.mgrid[0:z, 0:y, 0:x].astype(np.float64)
    g = 0.99 * np.exp(-((zz - z // 2) ** 2 / (2 * sigma[0] ** 2) + (yy - y // 2) ** 2 / (2 * sigma[1] ** 2) +
                         (xx - x // 2) ** 2 / (2 * sigma[2] ** 2)))
    g[g < 1e-3] = 0
    return np.ascontiguousarray(g, dtype=np.float32)


def run_main(out_dir=None, size=289, angle_increment=52, osem=None, poissonSNR=25.0, lightsheetSpacing=3, attenuation=0.01,
             angleOffset=15, psf_dir=None, psf=None, ctx=None, log=print, keep=("acq", "view", "weights")):
    """main() (:524-665).  Renders the phantom, then per angle: rotate, attenuate, weights, convolve, adjustImage,
    extractSlices, makeIsotropic, rotate view / weights / PSF back, and finally the cross-view weight normalisation.
    Saves the reference's file names into out_dir (when given) and returns a dict of the volumes named in `keep`
    (plus 'rendered', 'groundtruth', 'angles', 'sum_weights', 'seconds')."""
    ctx = ctx or Context(0)
    osem = OSEM.get(angle_increment, 3.0) if osem is None else osem
    t_start = time.perf_counter()

    def save(vol, name):
        if out_dir:
            tiff.write_float_stack(os.path.join(out_dir, name), vol)

    if out_dir:
        os.makedirs(out_dir, exist_ok=True)
    log("rendering basis for ground truth")
    rendered = S.simulate(size=size, ctx=ctx)                                           # :554
    log("computing ground truth")
    obj = S.rotateAroundAxis(rendered, 0, angleOffset, ctx=ctx)                         # :557
    save(rendered, "rendered.tif")
    save(obj, "groundtruth.tif")
    res = {"rendered": rendered, "groundtruth": obj, "angles": [], "acq": [], "view": [], "weights": [], "psf": [], "con": []}
    weights = []
    rnd = JavaRandom(S.seed)        # the class-static generator extractSlices(img, inc, snr) draws from (:76, :183)
    for angle in range(0, 360, angle_increment):                                        # :567
        log(f"angle {angle}: rotate, attenuate, weights")
        rot = S.rotateAroundAxis(rendered, 0, angle + angleOffset, ctx=ctx)             # :570
        att = S.attenuate3d(rot, attenuation, ctx=ctx)                                  # :573
        w = S.computeWeightImage(rot, attenuation, ctx=ctx)                             # :576
        if psf is not None:
            k = np.array(psf, dtype=np.float32, order="C", copy=True)
        elif psf_dir and os.path.exists(os.path.join(psf_dir, f"Angle{angle}.tif")):
            k = open_psf(os.path.join(psf_dir, f"Angle{angle}.tif"), True, ctx=ctx)     # :579
        else:
            k = default_psf()
        log(f"angle {angle}: convolve")
        con = S.convolve(att, k, None, ctx=ctx)                                         # :580 (normalises k in place)
        Tools.adjustImage(con, S.minValue, S.avgIntensity, ctx=ctx)                     # :582
        log(f"angle {angle}: extract slices, make isotropic, rotate back")
        acq = S.extractSlices(con, lightsheetSpacing, poissonSNR, rnd=rnd, ctx=ctx, stream=len(weights))   # :585
        iso = S.makeIsotropic(acq, lightsheetSpacing, ctx=ctx)                          # :588
        view = S.rotateAroundAxis(iso, 0, -angle, ctx=ctx)                              # :591
        view_weights = S.rotateAroundAxis(w, 0, -angle, ctx=ctx)                        # :592
        view_psf = S.rotateAroundAxis(k, 0, -angle, ctx=ctx)                            # :593
        for vol, name in ((rot, "rot_view_"), (att, "att_view_"), (con, "con_view_"), (acq, "acq_view_"), (iso, "iso_view_"),
                          (view, "aligned_view_"), (view_psf, "aligned_view_psf_")):
            save(vol, f"{name}{angle}.tif")                                             # :598-604
        weights.append(view_weights)
        res["angles"].append(angle)
        for key, vol in (("acq", acq), ("view", view), ("psf", view_psf), ("con", con)):
            if key in keep:
                res[key].append(vol)
    log("normalising weights")
    sum_weights = S.normalizeWeights(weights, osem, ctx=ctx)                            # :615-661
    for i, wv in enumerate(weights):
        save(wv, f"aligned_view_weights{i * angle_increment}.tif")                      # :642-646
    save(sum_weights, "sum_weights.tif")                                                # :663
    if "weights" in keep:
        res["weights"] = weights
    res["sum_weights"] = sum_weights
    res["seconds"] = time.perf_counter() - t_start
    log("done")
    return res


def simulate_dataset(out_dir=None, size=289, angle_increment=52, osem=None, poissonSNR=25.0, lightsheetSpacing=3, attenuation=0.01,
                     angleOffset=15, psf_dir=None, psf=None, ctx=None, log=print, keep=("acq", "view", "weights"), rank=0, world=1):
    """main() (:524-665) with its view loop in one device call (SimulateMultiViewDataset.simulateDataset): the phantom is rendered
    on the device and stays there; per view the library runs the whole-view acquisition, the aligned view, the view's normalised
    weights and the rotated-back PSF, and only those outputs cross the host link.  Writes run_main's file names for what it
    produces (acq_view_, aligned_view_, aligned_view_psf_, aligned_view_weights, sum_weights, rendered, groundtruth); the
    intermediate rot / att / con / iso volumes exist only in run_main.

    rank / world: this process simulates the views v with v % world == rank (sharding.views_for_rank).  The normalised weights
    depend on the angles alone, so no rank needs another's data: there is no collective.  Rank 0 also writes rendered,
    groundtruth and sum_weights.  Returns run_main's dict for this rank's views ('angles' lists them)."""
    from .api import DeviceVolume
    from .sharding import views_for_rank
    ctx = ctx or Context(0)
    osem = OSEM.get(angle_increment, 3.0) if osem is None else osem
    t_start = time.perf_counter()

    def save(vol, name):
        if out_dir:
            tiff.write_float_stack(os.path.join(out_dir, name), vol)

    if out_dir:
        os.makedirs(out_dir, exist_ok=True)
    angles = list(range(0, 360, angle_increment))                                       # :567
    mine = views_for_rank(len(angles), rank, world)
    log("rendering basis for ground truth")
    gt = DeviceVolume(ctx, (size, size, size))
    n_small = C.c_int64(0)
    check(ctx._lib.mvsim_dev_simulate_phantom(ctx.h, size, 0, S.seed, gt.h, C.byref(n_small)), ctx.h)   # :554
    res = {"angles": [angles[v] for v in mine], "acq": [], "view": [], "weights": [], "psf": [], "sum_weights": None}
    if rank == 0:
        log("computing ground truth")
        obj = DeviceVolume(ctx, gt.shape)
        check(ctx._lib.mvsim_dev_rotate_axis(ctx.h, gt.h, obj.h, 0, angleOffset), ctx.h)   # :557
        res["rendered"], res["groundtruth"] = gt.download(), obj.download()
        obj.free()
        save(res["rendered"], "rendered.tif")
        save(res["groundtruth"], "groundtruth.tif")
    psfs = []
    for v in mine:
        angle = angles[v]
        if psf is not None:
            psfs.append(np.array(psf, dtype=np.float32, order="C", copy=True))
        elif psf_dir and os.path.exists(os.path.join(psf_dir, f"Angle{angle}.tif")):
            psfs.append(open_psf(os.path.join(psf_dir, f"Angle{angle}.tif"), True, ctx=ctx))   # :579
        else:
            psfs.append(default_psf())
    log(f"views {[angles[v] for v in mine]}: acquire, align, weights")
    r = S.simulateDataset(gt, psfs, angles, angleOffset, attenuation, lightsheetSpacing, poissonSNR, osem, JavaRandom(S.seed),
                          views=mine, ctx=ctx, sum_weights=rank == 0)
    gt.free()
    for i, v in enumerate(mine):
        angle = angles[v]
        save(r["acq"][i], f"acq_view_{angle}.tif")                                      # :598-604
        save(r["aligned"][i], f"aligned_view_{angle}.tif")
        save(r["aligned_psf"][i], f"aligned_view_psf_{angle}.tif")
        save(r["weights"][i], f"aligned_view_weights{v * angle_increment}.tif")         # :642-646
    if rank == 0:
        save(r["sum_weights"], "sum_weights.tif")                                       # :663
        res["sum_weights"] = r["sum_weights"]
    for key, src in (("acq", "acq"), ("view", "aligned"), ("psf", "aligned_psf"), ("weights", "weights")):
        if key in keep:
            res[key] = r[src]
    res["seconds"] = time.perf_counter() - t_start
    log("done")
    return res


class SimulateTileStitching:
    """S/SimulateTileStitching.java:58-258: two convolved phantoms (with and without a half-pixel shift) are built by two
    threads, then pairs of overlapping tiles are cut out of them and sampled (every 3rd slice + Poisson noise) at any SNR.

    Both convolved volumes stay on the device, each with the context of the thread that built it: a pair samples its two
    tiles straight from them (DeviceVolume.extractSlices over the tile's interval) and only the tiles cross the host link.
    `con` / `conHalfPixel` download the volumes on first access.  close() frees the volumes and the contexts."""

    lightsheetSpacing = 3           # :52
    attenuation = 0.01              # :53

    def __init__(self, rnd=None, halfPixelOffset=False, overlapRatio=(0.2, 0.2, 0.2), service=None, psf=None, size=289, device=0):
        self.rnd = JavaRandom(464232194) if rnd is None else (rnd if isinstance(rnd, JavaRandom) else JavaRandom(rnd))   # :65-68
        self.psf = default_psf() if psf is None else np.array(psf, dtype=np.float32, order="C", copy=True)              # :71
        self.size = size
        self.device = device
        self._ctx, self._vol, self._host, self._tiles = {}, {}, {}, []
        self.init(overlapRatio, halfPixelOffset)

    def init(self, overlapRatio, halfPixelOffset):
        self.close()
        self._host = {}
        self.halfPixelOffset = halfPixelOffset
        seed = self.rnd.nextInt()                                                       # :83, same phantom for both
        raw = self.psf.copy()
        errors = []

        def task(half, key):                                                            # :85-114: one pipeline per thread
            shape = (self.size,) * 3
            tmp = []
            try:
                ctx = self._ctx[key] = Context(self.device)
                for shp, host in ((shape, None), (shape, None), (raw.shape, raw)):
                    tmp.append(DeviceVolume(ctx, shp, host))
                gt, att, psf = tmp
                con = self._vol[key] = DeviceVolume(ctx, shape)
                check(ctx._lib.mvsim_dev_simulate_phantom(ctx.h, self.size, int(half), seed, gt.h, C.byref(C.c_int64())), ctx.h)
                check(ctx._lib.mvsim_dev_attenuate(ctx.h, gt.h, att.h, self.attenuation, 1), ctx.h)
                check(ctx._lib.mvsim_dev_psf_normalize(ctx.h, psf.h, None), ctx.h)
                check(ctx._lib.mvsim_dev_convolve(ctx.h, att.h, psf.h, con.h), ctx.h)
                check(ctx._lib.mvsim_dev_adjust(ctx.h, con.h, S.minValue, S.avgIntensity, None), ctx.h)
                if key == "con":
                    psf.download(self.psf)                                              # convolve normalises its PSF in place (:255)
                ctx.synchronize()
            except Exception as e:
                errors.append(e)
            finally:
                for v in tmp:
                    v.free()
        threads = [threading.Thread(target=task, args=(False, "con")), threading.Thread(target=task, args=(True, "conHalfPixel"))]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        if errors:
            self.close()
            raise errors[0]
        dims = self._dims()
        self.overlap = [int(np.floor(dims[d] * overlapRatio[d] / 2 + 0.5)) for d in range(3)]   # Math.round, :121
        # the two tiles' device outputs, on the context of the volume each is cut from; reused by every pair
        for i, vol in enumerate(self._sources()):
            mn, mx = self.getInterval(i)
            self._tiles.append(DeviceVolume(vol.ctx, ((mx[2] - mn[2]) // self.lightsheetSpacing + 1, mx[1] - mn[1] + 1, mx[0] - mn[0] + 1)))

    def _dims(self):
        return self._vol["con"].shape[::-1]                                             # x, y, z

    def _sources(self):
        return [self._vol["con"], self._vol["conHalfPixel" if self.halfPixelOffset else "con"]]

    def _host_volume(self, key):
        if key not in self._host:
            self._host[key] = self._vol[key].download()
        return self._host[key]

    @property
    def con(self):
        return self._host_volume("con")

    @property
    def conHalfPixel(self):
        return self._host_volume("conHalfPixel")

    def getInterval(self, tile):
        """(:214-233) -> (min_xyz, max_xyz), inclusive.  Tile 1 starts at dimension(0)/2 - overlap in EVERY dimension, as written."""
        dims = self._dims()
        mn, mx = [0, 0, 0], [d - 1 for d in dims]
        if tile == 0:
            mx = [dims[d] // 2 + self.overlap[d] for d in range(3)]
        else:
            mn = [dims[0] // 2 - self.overlap[d] for d in range(3)]
        return mn, mx

    def getNextPair(self, snr):
        """(:131-189): two tiles, each with its own seed and Philox stream, sampled from Views.zeroMin(Views.interval(...)) of the
        resident volumes without a dense copy; the results equal extractSlices of the numpy cuts, bit for bit."""
        seeds = [self.rnd.nextInt(), self.rnd.nextInt()]
        for i, vol in enumerate(self._sources()):       # asynchronous on the volumes' contexts: the two samplers may overlap
            vol.extractSlices(self.lightsheetSpacing, snr, rnd=JavaRandom(seeds[i]), stream=i, interval=self.getInterval(i), out=self._tiles[i])
        return self._tiles[0].download(), self._tiles[1].download()

    def getCorrectTranslation(self):
        """(:191-212)"""
        mn, _ = self.getInterval(1)
        t = [float(v) for v in mn]
        if self.halfPixelOffset:
            t[0] -= 0.5
            t[1] -= 0.5
        t[2] /= self.lightsheetSpacing
        return t

    def close(self):
        """Frees the resident volumes and the two contexts (downloaded `con` / `conHalfPixel` arrays stay valid)."""
        for v in self._tiles + list(self._vol.values()):
            v.free()
        for ctx in self._ctx.values():
            ctx.close()
        self._tiles, self._vol, self._ctx = [], {}, {}


def _cli():
    ap = argparse.ArgumentParser(description="SimulateMultiViewDataset.main() on the GPU")
    ap.add_argument("--out", required=True)
    ap.add_argument("--size", type=int, default=289)
    ap.add_argument("--angle-increment", type=int, default=52)
    ap.add_argument("--snr", type=float, default=25.0)
    ap.add_argument("--psf-dir", default=None, help="directory with the reference's Angle<angle>.tif PSFs")
    ap.add_argument("--fused", action="store_true", help="the whole view loop in one device call (simulate_dataset); "
                    "writes no rot / att / con / iso volumes")
    ap.add_argument("--rank", type=int, default=0, help="with --fused: simulate the views v %% world == rank")
    ap.add_argument("--world", type=int, default=1)
    a = ap.parse_args()
    if a.fused:
        r = simulate_dataset(a.out, size=a.size, angle_increment=a.angle_increment, poissonSNR=a.snr, psf_dir=a.psf_dir, keep=(),
                             rank=a.rank, world=a.world)
    else:
        r = run_main(a.out, size=a.size, angle_increment=a.angle_increment, poissonSNR=a.snr, psf_dir=a.psf_dir, keep=())
    print(f"{len(r['angles'])} views of {a.size}^3 in {r['seconds']:.2f} s -> {a.out}")


if __name__ == "__main__":
    _cli()
