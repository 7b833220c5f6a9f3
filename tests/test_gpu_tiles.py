"""extractSlices over an interval of a resident volume (mvsim_dev_extract_interval, DeviceVolume.extractSlices(interval=...)) and
the tile-stitching pair generator built on it (drivers.SimulateTileStitching): bit for bit against extractSlices of the dense cut
and against the host-buffer stage chain the driver used before."""
import ctypes as C

import numpy as np
import pytest

from helpers import gaussian_psf

pytestmark = pytest.mark.gpu
SNRS = [-1.0, 0.5, 25.0, 1e4]          # copy; inversion (lambda < 10); PTRS (lambda >= 10); normal limit (lambda > 1e7)


@pytest.fixture(scope="module")
def mv():
    import mvsim_b200
    return mvsim_b200


@pytest.fixture(scope="module")
def ctx(mv):
    c = mv.Context(0)
    yield c
    c.close()


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _parent(shape_zyx, seed):
    # values up to 3: with SNR 25 every lambda >= 10 voxel meets the PTRS path, with 1e4 the normal limit
    return (np.random.default_rng(seed).random(shape_zyx, dtype=np.float32) * 3).astype(np.float32)


@pytest.mark.parametrize("X", [181, 180])                          # X % 4 != 0 and X % 4 == 0
@pytest.mark.parametrize("width,x0", [(1, 3), (3, 1), (4, 5), (7, 0), (174, 5)])
@pytest.mark.parametrize("inc", [1, 3, 5])
def test_interval_equals_extract_of_dense_cut(mv, ctx, X, width, x0, inc):
    S = mv.SimulateMultiViewDataset
    host = _parent((23, 19, X), seed=X + width)
    vol = mv.DeviceVolume(ctx, host.shape, host)
    mn, mx = (x0, 2, 1), (x0 + width - 1, 16, 21)
    cut = np.ascontiguousarray(host[mn[2]:mx[2] + 1, mn[1]:mx[1] + 1, mn[0]:mx[0] + 1])
    dense = mv.DeviceVolume(ctx, cut.shape, cut)
    try:
        for snr in SNRS:
            got = vol.extractSlices(inc, snr, rnd=12345 + inc, stream=7, interval=(mn, mx))
            ref = dense.extractSlices(inc, snr, rnd=12345 + inc, stream=7)
            assert got.shape == ref.shape == ((mx[2] - mn[2]) // inc + 1, mx[1] - mn[1] + 1, width)
            g, r = got.download(), ref.download()
            got.free()
            ref.free()
            assert np.array_equal(_bits(g), _bits(r)), snr
            # the host-buffer entry point on the numpy cut (what SimulateTileStitching.getNextPair ran before)
            assert np.array_equal(_bits(g), _bits(S.extractSlices(cut, inc, snr, rnd=12345 + inc, ctx=ctx, stream=7))), snr
            if snr < 0:
                assert np.array_equal(_bits(g), _bits(cut[::inc]))
    finally:
        vol.free()
        dense.free()


@pytest.mark.parametrize("X", [181, 180])
@pytest.mark.parametrize("inc", [1, 3])
def test_whole_volume_interval_equals_extract_slices(mv, ctx, X, inc):
    host = _parent((17, 13, X), seed=3)
    vol = mv.DeviceVolume(ctx, host.shape, host)
    for snr in SNRS:
        a = vol.extractSlices(inc, snr, rnd=99, stream=2, interval=((0, 0, 0), (X - 1, 12, 16)))
        b = vol.extractSlices(inc, snr, rnd=99, stream=2)             # mvsim_dev_extract_slices
        assert np.array_equal(_bits(a.download()), _bits(b.download())), snr
        a.free()
        b.free()
    vol.free()


def test_interval_rejects_bad_arguments(mv, ctx):
    from mvsim_b200._lib import check
    lib = ctx._lib
    vol = mv.DeviceVolume(ctx, (9, 8, 7))            # X, Y, Z = 7, 8, 9
    out = mv.DeviceVolume(ctx, (3, 4, 5))            # interval (1, 2, 0) .. (5, 5, 6), inc 3
    i3 = C.c_int64 * 3

    def call(mn=(1, 2, 0), mx=(5, 5, 6), inc=3, src=vol, dst=out, c=ctx.h):
        check(lib.mvsim_dev_extract_interval(c, src.h if src else None, i3(*mn) if mn else None, i3(*mx) if mx else None, inc,
                                             -1.0, 1, 0, dst.h if dst else None), ctx.h)

    call()                                           # valid
    ctx.synchronize()
    bad = [dict(src=None), dict(dst=None), dict(mn=None), dict(mx=None), dict(c=None),
           dict(inc=0), dict(inc=-2),
           dict(mn=(-1, 2, 0)), dict(mn=(1, -1, 0)), dict(mn=(1, 2, -1)),
           dict(mx=(7, 5, 6)), dict(mx=(5, 8, 6)), dict(mx=(5, 5, 9)),
           dict(mn=(6, 2, 0), mx=(5, 5, 6)), dict(mn=(1, 6, 0)), dict(mn=(1, 2, 7), mx=(5, 5, 6)),
           dict(mx=(4, 5, 6)), dict(mx=(5, 4, 6)), dict(mx=(5, 5, 3)), dict(inc=2)]
    for kw in bad:
        with pytest.raises(mv.MvsimError) as e:
            call(**kw)
        assert e.value.status == 1, kw                 # MVSIM_EINVAL
    square = mv.DeviceVolume(ctx, (9, 8, 7))
    with pytest.raises(mv.MvsimError):               # in == out (same dims, so only the aliasing is wrong)
        check(lib.mvsim_dev_extract_interval(ctx.h, square.h, i3(0, 0, 0), i3(6, 7, 8), 1, -1.0, 0, 0, square.h), ctx.h)
    with pytest.raises(mv.MvsimError):
        vol.extractSlices(0, -1.0, interval=((0, 0, 0), (6, 7, 8)))
    for v in (vol, out, square):
        v.free()


def _host_chain(mv, ctx, half, seed, size, psf):
    """The driver's former init(): S.simulate -> S.attenuate3d -> S.convolve -> Tools.adjustImage through host buffers."""
    S = mv.SimulateMultiViewDataset
    gt = S.simulate(half, seed, size=size, ctx=ctx)
    att = S.attenuate3d(gt, 0.01, ctx=ctx)
    con = S.convolve(att, psf.copy(), None, ctx=ctx)
    mv.Tools.adjustImage(con, S.minValue, S.avgIntensity, ctx=ctx)
    return con


@pytest.mark.parametrize("half", [True, False])
def test_tile_stitching_matches_host_chain(mv, ctx, monkeypatch, half):
    S = mv.SimulateMultiViewDataset
    size, inc = 97, 3
    psf = gaussian_psf((9, 7, 7), (2.0, 1.0, 1.0), threshold=1e-3)
    sts = mv.SimulateTileStitching(None, half, (0.2, 0.3, 0.25), psf=psf, size=size)
    try:
        rnd = mv.JavaRandom(464232194)
        seed = rnd.nextInt()
        con, con_half = _host_chain(mv, ctx, False, seed, size, psf), _host_chain(mv, ctx, True, seed, size, psf)
        assert np.array_equal(_bits(sts.con), _bits(con))
        assert np.array_equal(_bits(sts.conHalfPixel), _bits(con_half))
        src = [con, con_half if half else con]
        for snr in (-1.0, 1.0, 4.0, 16.0, 64.0):
            seeds = [rnd.nextInt(), rnd.nextInt()]
            ref = []
            for i in range(2):
                mn, mx = sts.getInterval(i)
                cut = np.ascontiguousarray(src[i][mn[2]:mx[2] + 1, mn[1]:mx[1] + 1, mn[0]:mx[0] + 1])
                ref.append(S.extractSlices(cut, inc, snr, rnd=mv.JavaRandom(seeds[i]), ctx=ctx, stream=i))
            # a pair runs on the object's two contexts: no new context, no upload, one sampler launch per tile
            monkeypatch.setattr(mv.drivers, "Context", None)
            monkeypatch.setattr(mv.DeviceVolume, "upload", None)
            before = sum(c.kernel_launches for c in sts._ctx.values())
            t0, t1 = sts.getNextPair(snr)
            assert sum(c.kernel_launches for c in sts._ctx.values()) - before == 2
            monkeypatch.undo()
            assert np.array_equal(_bits(t0), _bits(ref[0])), snr
            assert np.array_equal(_bits(t1), _bits(ref[1])), snr
    finally:
        sts.close()
    assert sts._ctx == {} and sts._vol == {}


def test_large_parent_interval(mv, ctx):
    """A parent of more than 2^31 voxels (8.7 GB) and a tile whose rows start at min0 % 4 == 3, far out in z: 64-bit parent
    offsets throughout.  The parent and the dense cut live in torch tensors on the device."""
    import torch
    X, Y, Z = 2048, 1024, 1040
    g = torch.Generator(device="cuda").manual_seed(11)
    parent = torch.rand((Z, Y, X), device="cuda", generator=g) * 3
    mn, mx = (1027, 301, 700), (1027 + 614, 301 + 600, 1039)
    cut = parent[mn[2]:mx[2] + 1, mn[1]:mx[1] + 1, mn[0]:mx[0] + 1].contiguous()
    torch.cuda.synchronize()
    pv = mv.DeviceVolume.wrap(ctx, parent.shape, parent.data_ptr(), keepalive=parent)
    cv = mv.DeviceVolume.wrap(ctx, cut.shape, cut.data_ptr(), keepalive=cut)
    for snr in (-1.0, 25.0):
        a = pv.extractSlices(3, snr, rnd=5, stream=1, interval=(mn, mx))
        b = cv.extractSlices(3, snr, rnd=5, stream=1)
        ha, hb = a.download(), b.download()
        assert np.array_equal(_bits(ha), _bits(hb)), snr
        if snr < 0:
            assert np.array_equal(_bits(ha), _bits(cut[::3].cpu().numpy()))
        a.free()
        b.free()
    pv.free()
    cv.free()
    del parent, cut
    torch.cuda.empty_cache()
