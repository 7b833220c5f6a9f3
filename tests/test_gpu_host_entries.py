"""The host-buffer entry points of the C ABI: each gives what its mvsim_dev_* twin gives on the same inputs, bit for bit, records
the same per-stage launches as before their staging was written once, and fails an allocation the device cannot hold before it
copies anything."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SHAPE = (24, 56, 40)         # (Z, Y, X); X <= Y, as the reference's attenuation loop needs
KSHAPE = (5, 7, 9)
BEADS = ((0, 0, 0), (28, 40, 32))
MIN_VALUE, TARGET_AVG = 0.0001, 1.0


@pytest.fixture(scope="module")
def mv():
    import mvsim_b200
    return mvsim_b200


def _inputs():
    rng = np.random.default_rng(17)
    gt = rng.random(SHAPE, dtype=np.float32)
    psf = rng.random(KSHAPE, dtype=np.float32) + 0.05
    return gt, psf


def _same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()


def _bead_points(mv):
    return mv.SimulateBeads.randomPoints(40, BEADS)


# ---- every host entry against its device twin ------------------------------------------------------------------------
def _host_and_dev(mv, ctx, op, keep):
    """(outputs of the host entry, outputs of the mvsim_dev_* twin) of `op` on the same inputs."""
    from mvsim_b200._lib import check, dims3, fptr
    S, L, h = mv.SimulateMultiViewDataset, ctx._lib, ctx.h
    gt, psf = _inputs()
    i3, d3 = C.c_int64 * 3, C.c_double * 3

    def vol(host=None, shape=None):
        v = mv.DeviceVolume(ctx, host.shape if shape is None else shape, host)
        keep.append(v)
        return v

    if op == "rotate":
        o = vol(shape=SHAPE)
        check(L.mvsim_dev_rotate_axis(h, vol(gt).h, o.h, 1, 30), h)
        return [S.rotateAroundAxis(gt, 1, 30, ctx=ctx)], [o.download()]
    if op == "attenuate":
        o = vol(shape=SHAPE)
        check(L.mvsim_dev_attenuate(h, vol(gt).h, o.h, 0.01, 1), h)
        return [S.attenuate3d(gt, 0.01, ctx=ctx)], [o.download()]
    if op == "psf_normalize":
        k, s_host, s_dev = vol(psf), C.c_double(), C.c_double()
        check(L.mvsim_dev_psf_normalize(h, k.h, C.byref(s_dev)), h)
        p = psf.copy()
        check(L.mvsim_psf_normalize(h, fptr(p), dims3(KSHAPE), C.byref(s_host)), h)
        return [p, s_host.value], [k.download(), s_dev.value]
    if op == "convolve":
        p = psf.copy()
        host = S.convolve(gt, p, ctx=ctx)                 # normalises p in place; the device twin takes it normalised
        o = vol(shape=SHAPE)
        check(L.mvsim_dev_convolve(h, vol(gt).h, vol(p).h, o.h), h)
        return [host], [o.download()]
    if op == "adjust":
        img = gt.copy()
        c = mv.Tools.adjustImage(img, MIN_VALUE, TARGET_AVG, ctx=ctx)
        v, c_dev = vol(gt), C.c_double()
        check(L.mvsim_dev_adjust(h, v.h, MIN_VALUE, TARGET_AVG, C.byref(c_dev)), h)
        return [img, c], [v.download(), c_dev.value]
    if op == "extract_slices":
        o = vol(gt).extractSlices(3, 10.0, rnd=5)
        keep.append(o)
        return [S.extractSlices(gt, 3, 10.0, rnd=5, ctx=ctx)], [o.download()]
    if op == "simulate_view":
        p = psf.copy()
        host = S.simulateView(gt, p, 15, inc=3, poissonSNR=10.0, rnd=5, ctx=ctx)
        params = mv.make_view_params(SHAPE, KSHAPE, 0, 15, 0.01, MIN_VALUE, TARGET_AVG, 3, 10.0, seed=5)
        k, o = vol(psf), vol(shape=host.shape)
        check(L.mvsim_dev_simulate_view(h, C.byref(params), vol(gt).h, k.h, o.h), h)
        return [host, p], [o.download(), k.download()]
    if op == "render_beads":
        pts = _bead_points(mv)
        host = mv.SimulateBeads.renderPoints([pts], BEADS, (1.0, 1.0, 3.0), ctx=ctx)[0]
        o = vol(shape=host.shape)
        check(L.mvsim_dev_render_beads(h, pts.ctypes.data_as(C.POINTER(C.c_double)), len(pts), d3(1.0, 1.0, 3.0), i3(*BEADS[0]),
                                       i3(*BEADS[1]), o.h), h)
        return [host], [o.download()]
    if op == "simulate_phantom":
        size, n_host, n_dev = 121, C.c_int64(), C.c_int64()
        host = np.empty((size,) * 3, dtype=np.float32)
        check(L.mvsim_simulate_phantom(h, size, 0, 7, fptr(host), C.byref(n_host)), h)
        o = vol(shape=host.shape)
        check(L.mvsim_dev_simulate_phantom(h, size, 0, 7, o.h, C.byref(n_dev)), h)
        return [host, n_host.value], [o.download(), n_dev.value]
    raise AssertionError(op)


@pytest.mark.parametrize("op", ["rotate", "attenuate", "psf_normalize", "convolve", "adjust", "extract_slices", "simulate_view",
                                "render_beads", "simulate_phantom"])
def test_host_entry_equals_its_device_twin(mv, op):
    ctx, keep = mv.Context(0), []
    try:
        host, dev = _host_and_dev(mv, ctx, op, keep)
    finally:
        for v in keep:
            v.free()
        ctx.close()
    assert len(host) == len(dev)
    for i, (a, b) in enumerate(zip(host, dev)):
        assert _same(a, b), (op, i)


# ---- launches per stage ------------------------------------------------------------------------------------------------
def _call_host_entry(mv, ctx, entry):
    S, T, B = mv.SimulateMultiViewDataset, mv.Tools, mv.SimulateBeads
    gt, psf = _inputs()
    calls = {
        "rotate_axis": lambda: S.rotateAroundAxis(gt, 1, 30, ctx=ctx),
        "attenuate": lambda: S.attenuate3d(gt, 0.01, ctx=ctx),
        "psf_normalize": lambda: T.normImage(psf.copy(), ctx=ctx),
        "convolve": lambda: S.convolve(gt, psf.copy(), ctx=ctx),
        "adjust": lambda: T.adjustImage(gt.copy(), MIN_VALUE, TARGET_AVG, ctx=ctx),
        "extract_slices": lambda: S.extractSlices(gt, 3, 10.0, rnd=5, ctx=ctx),
        "poisson": lambda: T.poissonProcess(gt.copy(), 10.0, 5, ctx=ctx),
        "simulate_view": lambda: S.simulateView(gt, psf.copy(), 15, inc=3, poissonSNR=10.0, rnd=5, ctx=ctx),
        # about y: the fused rotate + attenuate kernel does not apply and the view falls back to the two kernels
        "simulate_view_axis1": lambda: S.simulateView(gt, psf.copy(), 15, axis=1, inc=3, poissonSNR=10.0, rnd=5, ctx=ctx),
        "make_isotropic": lambda: S.makeIsotropic(np.ascontiguousarray(gt[::3]), 3, ctx=ctx),
        "weight_image": lambda: S.computeWeightImage(SHAPE, ctx=ctx),
        "normalize_weights": lambda: S.normalizeWeights([gt.copy(), gt[::-1].copy(), gt[:, ::-1].copy()], 3.0, ctx=ctx),
        "render_beads": lambda: B.renderPoints([_bead_points(mv)], BEADS, (1.0, 1.0, 3.0), ctx=ctx),
        "draw_spheres": lambda: S.drawSpheres((120, 120, 120), scale=1, rnd=7, ctx=ctx),
        "downsample2x": lambda: S.downSample2x(gt, ctx=ctx),
        "simulate_phantom": lambda: S.simulate(False, 7, size=121, ctx=ctx),
        "make_square": lambda: T.makeSquare(gt, ctx=ctx),
    }
    calls[entry]()


def stage_launches(mv, entry):
    """{stage: launches} (non-zero stages) and the kernel launches of one call of `entry` on a fresh context."""
    ctx = mv.Context(0)
    try:
        ctx.profile(True)
        k0 = ctx.kernel_launches
        _call_host_entry(mv, ctx, entry)
        stages = {k: n for k, (_, n) in ctx.stage_times().items() if n}
        return stages, ctx.kernel_launches - k0
    finally:
        ctx.close()


# {entry: ({stage: launches}, kernel launches)}, recorded with stage_launches() on a B200 with the library as it was before the
# host entries shared one staging helper (HostCall in csrc/capi.cu), when each entry wrote its allocations, copies and
# synchronisation out by hand.  A change to the staging must not add, drop or move a timed stage or a kernel launch.
PARENT_LAUNCHES = {
    "adjust": ({"h2d": 1, "adjust": 1, "d2h": 1}, 4),
    "attenuate": ({"h2d": 1, "attenuate": 1, "d2h": 1}, 1),
    "convolve": ({"h2d": 2, "psf": 4, "fft_xfwd": 1, "fft_yfwd": 1, "fft_zfused": 1, "fft_yinv": 1, "fft_xinv": 1, "d2h": 2}, 10),
    "downsample2x": ({"h2d": 1, "d2h": 1}, 1),
    "draw_spheres": ({"d2h": 1}, 1),
    "extract_slices": ({"h2d": 1, "sample": 1, "d2h": 1}, 1),
    "make_isotropic": ({"h2d": 1, "d2h": 1}, 1),
    "make_square": ({"h2d": 1, "d2h": 1}, 2),
    "normalize_weights": ({"h2d": 3, "d2h": 4}, 1),
    "poisson": ({"h2d": 1, "sample": 1, "d2h": 1}, 1),
    "psf_normalize": ({"h2d": 1, "psf": 1, "d2h": 1}, 3),
    "render_beads": ({"d2h": 1}, 1),
    "rotate_axis": ({"h2d": 1, "rotate": 1, "d2h": 1}, 1),
    "simulate_phantom": ({"d2h": 1}, 2),
    "simulate_view": ({"h2d": 2, "rotate": 1, "psf": 4, "fft_xfwd": 1, "fft_yfwd": 1, "fft_zfused": 1, "fft_yinv": 1, "fft_xinv": 1,
                       "adjust": 2, "sample": 1, "d2h": 2}, 15),
    "simulate_view_axis1": ({"h2d": 2, "rotate": 2, "attenuate": 1, "psf": 4, "fft_xfwd": 1, "fft_yfwd": 1, "fft_zfused": 1, "fft_yinv": 1,
                             "fft_xinv": 1, "adjust": 2, "sample": 1, "d2h": 2}, 15),
    "weight_image": ({"d2h": 1}, 1),
}


@pytest.mark.parametrize("entry", sorted(PARENT_LAUNCHES))
def test_host_entry_launches_per_stage(mv, entry):
    assert stage_launches(mv, entry) == PARENT_LAUNCHES[entry]


# ---- a failed allocation -----------------------------------------------------------------------------------------------
def _small_chain(mv, ctx):
    S = mv.SimulateMultiViewDataset
    gt, psf = _inputs()
    return [S.makeIsotropic(np.ascontiguousarray(gt[::3]), 3, ctx=ctx),
            S.simulateView(gt, psf.copy(), 15, inc=3, poissonSNR=10.0, rnd=5, ctx=ctx)]


def test_failed_allocation_returns_enomem_before_any_copy(mv):
    """makeIsotropic of a 400 MB volume whose result would take about 400 GB: the second allocation fails, the call returns
    MVSIM_ENOMEM without a copy in either direction, and the context then computes what a fresh one does."""
    import torch
    from mvsim_b200._lib import MVSIM_ENOMEM, dims3, fptr
    shape, inc = (100, 1000, 1000), 1000
    out_bytes = 4 * shape[1] * shape[2] * ((shape[0] - 1) * inc + 1)
    if out_bytes <= torch.cuda.get_device_properties(0).total_memory:
        pytest.skip("the device could hold the result: the call would copy it into the one-element buffer")
    src = np.zeros(shape, dtype=np.float32)
    one = np.zeros(1, dtype=np.float32)         # never written: nothing is copied after a failed allocation
    ctx = mv.Context(0)
    try:
        ctx.profile(True)
        assert ctx._lib.mvsim_make_isotropic(ctx.h, fptr(src), dims3(shape), inc, fptr(one)) == MVSIM_ENOMEM
        times = ctx.stage_times()
        assert times["h2d"][1] == 0 and times["d2h"][1] == 0
        assert one[0] == 0
        again = _small_chain(mv, ctx)
    finally:
        ctx.close()
    fresh = mv.Context(0)
    try:
        expect = _small_chain(mv, fresh)
    finally:
        fresh.close()
    assert all(_same(a, b) for a, b in zip(again, expect))
