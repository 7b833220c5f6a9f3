"""The batch calls (mvsim_simulate_views, mvsim_simulate_dataset) under concurrent callers and after a failure in the middle of a
batch, and the per-thread error state every entry point starts from."""
import threading

import numpy as np
import pytest

from helpers import gaussian_psf, sphere_phantom

pytestmark = pytest.mark.gpu
DEGREES = [15, 105, 195, 285]
ANGLES = [0, 90, 180, 270]
TIMEOUT_S = 600          # a gate left locked shows as a caller that never returns


@pytest.fixture(scope="module")
def mv():
    import mvsim_b200
    return mvsim_b200


def _same(a, b):
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def _in_threads(fns):
    """Runs fns concurrently, each on its own thread; returns their results in order (an exception is re-raised)."""
    out, start = [None] * len(fns), threading.Barrier(len(fns))

    def run(i):
        try:
            start.wait()
            out[i] = ("ok", fns[i]())
        except BaseException as e:          # noqa: B036 -- handed to the test thread
            out[i] = ("error", e)
    threads = [threading.Thread(target=run, args=(i,), daemon=True) for i in range(len(fns))]
    for t in threads:
        t.start()
    for t in threads:
        t.join(TIMEOUT_S)
    assert not any(t.is_alive() for t in threads), "a batch call did not return"
    for kind, val in out:
        if kind == "error":
            raise val
    return [val for _, val in out]


def _views_float32(mv, ctx, gt, psfs):
    ctx.count_transport(False)
    p = [q.copy() for q in psfs]
    return mv.SimulateMultiViewDataset.simulateViews(gt, p, DEGREES, inc=3, poissonSNR=4.0, rnd=5, ctx=ctx) + p


def _views_uint16_resident(mv, ctx, gt, psfs):
    ctx.count_transport(True)
    vol = mv.DeviceVolume(ctx, gt.shape, gt)
    try:
        p = [q.copy() for q in psfs]
        return mv.SimulateMultiViewDataset.simulateViews(vol, p, DEGREES, inc=3, poissonSNR=4.0, rnd=7, ctx=ctx) + p
    finally:
        vol.free()


def _dataset(mv, ctx, gt, psfs):
    p = [q.copy() for q in psfs]
    r = mv.SimulateMultiViewDataset.simulateDataset(gt, p, ANGLES, inc=3, poissonSNR=4.0, rnd=11, ctx=ctx)
    return r["acq"] + r["aligned"] + r["aligned_psf"] + r["weights"] + [r["sum_weights"]] + p


def test_concurrent_batch_callers_match_serial_calls(mv):
    """Three callers with a context each share the device's upload and compute gates; each runs its call twice."""
    gt = sphere_phantom((64, 128, 120), n_spheres=200)
    psfs = [gaussian_psf((11, 9, 7), (2.0 + 0.2 * v, 1.2, 1.0), threshold=1e-3) for v in range(4)]
    jobs = [_views_float32, _views_uint16_resident, _dataset]
    serial = mv.Context(0)
    ref = [job(mv, serial, gt, psfs) for job in jobs]
    serial.close()

    def caller(job):
        def run():
            ctx = mv.Context(0)
            try:
                return [job(mv, ctx, gt, psfs) for _ in range(2)]
            finally:
                ctx.close()
        return run
    got = _in_threads([caller(job) for job in jobs])
    for job, expect, runs in zip(jobs, ref, got):
        for res in runs:
            assert len(res) == len(expect)
            assert all(_same(a, b) for a, b in zip(res, expect)), job.__name__


@pytest.mark.parametrize("call", ["views_float32", "views_uint16", "dataset"])
def test_failure_in_the_middle_of_a_batch(mv, call):
    """View 1's PSF is too long for the planner (Z + KZ - 1 > 1600): the call fails after view 0 ran, and releases its gates."""
    S = mv.SimulateMultiViewDataset
    gt = sphere_phantom((32, 40, 40), n_spheres=60)
    good = [gaussian_psf((7, 7, 7), (1.5, 1.1, 1.0), threshold=1e-3), gaussian_psf((9, 7, 7), (2.0, 1.1, 1.0), threshold=1e-3)]
    bad = [good[0], np.full((1600, 1, 1), 1.0 / 1600, dtype=np.float32)]

    def batch(ctx, psfs):
        p = [q.copy() for q in psfs]
        if call == "dataset":
            r = S.simulateDataset(gt, p, [0, 180], inc=3, poissonSNR=4.0, rnd=3, ctx=ctx)
            return r["acq"] + r["aligned"] + r["aligned_psf"] + r["weights"] + [r["sum_weights"]] + p
        ctx.count_transport(call == "views_uint16")
        return S.simulateViews(gt, p, [15, 195], inc=3, poissonSNR=4.0, rnd=3, ctx=ctx) + p

    def fresh():
        ctx = mv.Context(0)
        try:
            return batch(ctx, good)
        finally:
            ctx.close()
    expect = fresh()
    ctx = mv.Context(0)
    with pytest.raises(mv.MvsimError) as e:
        batch(ctx, bad)
    assert e.value.status == mv._lib.MVSIM_EUNSUPPORTED
    again = batch(ctx, good)
    other, = _in_threads([fresh])
    ctx.close()
    for res in (again, other):
        assert len(res) == len(expect) and all(_same(a, b) for a, b in zip(res, expect))


def test_an_earlier_failure_is_not_reported_by_a_later_call(mv):
    """A failed allocation leaves the CUDA runtime's last error set on this thread; the slab convolution's launch checks read
    that error, so the next entry point must start from a clean state instead of reporting the allocation as its own failure."""
    import torch
    rng = np.random.default_rng(21)
    vol = rng.random((24, 40, 56), dtype=np.float32)
    psf = rng.random((5, 7, 9), dtype=np.float32)
    psf /= psf.sum(dtype=np.float64)
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        ctx = mv.Context(0, cuda_stream=stream.cuda_stream)
        sc = mv.SlabConvolution(ctx, vol.shape, psf.shape)
        img, k = torch.from_numpy(vol).cuda(), torch.from_numpy(psf).cuda()
        out = torch.empty_like(img)
        sc.convolve(img, k, out)
        stream.synchronize()
        first = out.cpu().numpy()
        with pytest.raises(mv.MvsimError) as e:
            mv.DeviceVolume(ctx, (10, 100000, 100000))            # 400 GB: more than the device holds, nothing is allocated
        assert e.value.status == mv._lib.MVSIM_ENOMEM
        out.zero_()
        sc.convolve(img, k, out)
        stream.synchronize()
        assert _same(out.cpu().numpy(), first)
        sc.close()
        ctx.close()
