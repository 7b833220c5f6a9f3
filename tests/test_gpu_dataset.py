"""main()'s view loop with its post-acquisition chain in one device call (mvsim_simulate_dataset) and its two new primitives:
the aligned view gathered straight from the acquired planes (mvsim_dev_align_view) and the analytic normalised weights
(mvsim_dev_aligned_weights), against the library's existing stage entry points (bit for bit) and the oracle."""
import os

import numpy as np
import pytest

from helpers import gaussian_psf, rel_err

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def mv():
    import mvsim_b200
    return mvsim_b200


@pytest.fixture(scope="module")
def ctx(mv):
    c = mv.Context(0)
    yield c
    c.close()


def _align(mv, ctx, acq, inc, degrees):
    vol = mv.DeviceVolume(ctx, acq.shape, acq)
    out = vol.alignView(inc, degrees)
    res = out.download()
    vol.free()
    out.free()
    return res


@pytest.mark.parametrize("z,inc", [(31, 1), (31, 3), (32, 3), (31, 5), (29, 5)])
@pytest.mark.parametrize("x", [24, 21])
@pytest.mark.parametrize("degrees", [0, 52, -52, 90, 180, 315])
def test_align_view_bit_identical_to_stages(mv, ctx, z, inc, x, degrees):
    """(Z-1) % inc zero and non-zero; X % 4 == 0 (float4 kernel) and not (scalar kernel)."""
    S = mv.SimulateMultiViewDataset
    za = (z - 1) // inc + 1
    acq = np.random.default_rng(z * 100 + inc).standard_normal((za, 19, x)).astype(np.float32)
    acq[0, 3, :5] = -0.0                          # a -0 tap: the second plane decides the sign of the blend
    acq[-1, 7, 2:9] = 0.0
    got = _align(mv, ctx, acq, inc, degrees)
    ref = S.rotateAroundAxis(S.makeIsotropic(acq, inc, ctx=ctx), 0, degrees, ctx=ctx)
    assert got.shape == ((za - 1) * inc + 1, 19, x)
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))


def test_align_view_rejects_bad_shapes(mv, ctx):
    acq = mv.DeviceVolume(ctx, (5, 8, 8))
    wrong = mv.DeviceVolume(ctx, (12, 8, 8))
    with pytest.raises(mv.MvsimError):
        acq.alignView(3, 30, out=wrong)               # needs 13 planes
    with pytest.raises(mv.MvsimError):
        acq.alignView(0, 30)
    acq.free()
    wrong.free()


def _composed_weights(S, ctx, shape, align_degrees, osem):
    ws = [S.rotateAroundAxis(S.computeWeightImage(shape, ctx=ctx), 0, d, ctx=ctx) for d in align_degrees]
    s = S.normalizeWeights(ws, osem, ctx=ctx)
    return ws, s


@pytest.mark.parametrize("n_all", [1, 3, 7, 16])
def test_aligned_weights_bit_identical_to_stages(mv, ctx, n_all):
    S = mv.SimulateMultiViewDataset
    shape = (37, 121, 10)
    align = [-(k * (360 // n_all)) for k in range(n_all)]
    ws, s = _composed_weights(S, ctx, shape, align, 3.0)
    vols = mv.DeviceVolume.alignedWeights(ctx, shape, align, 3.0, sum_weights=True)
    got = [v.download() for v in vols]
    for v in vols:
        v.free()
    for a, b in zip(got[:-1], ws):
        assert np.array_equal(a, b)
    assert np.array_equal(got[-1], s)
    # a subset gives exactly the corresponding volumes of the full set
    subset = [n_all - 1, 0] if n_all > 1 else [0]
    part = mv.DeviceVolume.alignedWeights(ctx, shape, align, 3.0, views=subset)
    for v, k in zip(part, subset):
        assert np.array_equal(v.download(), ws[k])
        v.free()


def test_aligned_weights_scalar_kernel_and_limits(mv, ctx):
    S = mv.SimulateMultiViewDataset
    shape = (9, 97, 7)                                # X % 4 != 0
    align = [0, -52, -104]
    ws, s = _composed_weights(S, ctx, shape, align, 4.0)
    vols = mv.DeviceVolume.alignedWeights(ctx, shape, align, 4.0, sum_weights=True)
    assert all(np.array_equal(v.download(), r) for v, r in zip(vols, ws + [s]))
    for v in vols:
        v.free()
    with pytest.raises(mv.MvsimError):
        mv.DeviceVolume.alignedWeights(ctx, shape, list(range(17)), 3.0)       # MVSIM_MAX_WEIGHT_VIEWS = 16
    with pytest.raises(mv.MvsimError):
        mv.DeviceVolume.alignedWeights(ctx, shape, align, 3.0, views=[1, 1])  # repeated view
    with pytest.raises(mv.MvsimError):
        mv.DeviceVolume.alignedWeights(ctx, shape, align, 3.0, views=[3])     # out of range


@pytest.fixture(scope="module")
def psf():
    return gaussian_psf((15, 9, 9), (3.0, 1.2, 1.1), threshold=1e-3)


@pytest.mark.parametrize("size", [121, 110])          # (Z-1) % 3 == 0 and == 1
def test_simulate_dataset_noise_free(mv, ctx, oracle, psf, size):
    S = mv.SimulateMultiViewDataset
    angles = [0, 120, 240]
    main = mv.run_main(None, size=size, angle_increment=120, poissonSNR=-1.0, psf=psf, log=lambda *_: None,
                       keep=("acq", "view", "weights", "psf"), ctx=ctx)
    gt = main["rendered"]
    psfs = [psf.copy() for _ in angles]
    r = S.simulateDataset(gt, psfs, angles, inc=3, poissonSNR=-1.0, osem=3.0, ctx=ctx)
    assert r["views"] == [0, 1, 2]
    for i, angle in enumerate(angles):
        ref_acq, _, _ = oracle.simulate_view(gt, psf, degrees=angle + 15, inc=3, snr=-1.0, use_fft=True)
        assert r["acq"][i].shape == ((size - 1) // 3 + 1, size, size)
        assert rel_err(r["acq"][i], ref_acq) <= 1e-4
        # psfs normalised in place, exactly like the stage path's normImage
        norm = psf.copy()
        mv.Tools.normImage(norm, ctx=ctx)
        assert np.array_equal(psfs[i], norm)
        # run_main's chain (:588-593) applied to the returned acq / normalised PSF
        iso = S.makeIsotropic(r["acq"][i], 3, ctx=ctx)
        assert np.array_equal(r["aligned"][i], S.rotateAroundAxis(iso, 0, -angle, ctx=ctx))
        assert np.array_equal(r["aligned_psf"][i], S.rotateAroundAxis(psfs[i], 0, -angle, ctx=ctx))
        assert np.array_equal(r["aligned_psf"][i], main["psf"][i])
        assert np.array_equal(r["weights"][i], main["weights"][i])
    assert np.array_equal(r["sum_weights"], main["sum_weights"])
    # ground truth already on the device: identical
    dgt = mv.DeviceVolume(ctx, gt.shape, gt)
    r2 = S.simulateDataset(dgt, [psf.copy() for _ in angles], angles, inc=3, poissonSNR=-1.0, osem=3.0, ctx=ctx)
    dgt.free()
    for key in ("acq", "aligned", "aligned_psf", "weights"):
        assert all(np.array_equal(a, b) for a, b in zip(r[key], r2[key]))
    assert np.array_equal(r["sum_weights"], r2["sum_weights"])
    # outputs not asked for are not produced; the rest is unchanged; a subset of views gives the same volumes
    r3 = S.simulateDataset(gt, [psf.copy()], angles, inc=3, poissonSNR=-1.0, osem=3.0, ctx=ctx, views=[2], outputs=("aligned",),
                           sum_weights=False)
    assert r3["acq"] == [None] and r3["weights"] == [None] and r3["aligned_psf"] == [None] and r3["sum_weights"] is None
    assert np.array_equal(r3["aligned"][0], r["aligned"][2])


def test_simulate_dataset_rejects_bad_arguments(mv, ctx, psf):
    S = mv.SimulateMultiViewDataset
    gt = np.zeros((20, 24, 24), dtype=np.float32)
    with pytest.raises(mv.MvsimError):
        S.simulateDataset(gt, [psf.copy()], list(range(0, 340, 20)), poissonSNR=-1.0, ctx=ctx, views=[0])    # 17 views
    with pytest.raises(mv.MvsimError):
        S.simulateDataset(gt, [psf.copy(), psf.copy()], [0, 90], poissonSNR=-1.0, ctx=ctx, views=[1, 1])  # repeated
    with pytest.raises(mv.MvsimError):
        S.simulateDataset(gt, [psf.copy()], [0, 90], poissonSNR=-1.0, ctx=ctx, views=[2])                 # out of range


def test_simulate_dataset_with_noise(mv, ctx, psf, tmp_path):
    S = mv.SimulateMultiViewDataset
    angles = [0, 120, 240]
    main = mv.run_main(None, size=121, angle_increment=120, poissonSNR=25.0, psf=psf, log=lambda *_: None, keep=("acq",), ctx=ctx)
    gt = main["rendered"]
    a = S.simulateDataset(gt, [psf.copy() for _ in angles], angles, inc=3, poissonSNR=25.0, ctx=ctx, outputs=("acq",))
    b = S.simulateDataset(gt, [psf.copy() for _ in angles], angles, inc=3, poissonSNR=25.0, ctx=ctx, outputs=("acq",))
    for i in range(3):
        assert np.array_equal(a["acq"][i], b["acq"][i])
        assert np.array_equal(a["acq"][i], np.floor(a["acq"][i]))
        # same seeds and streams as run_main; the whole-view path differs from the stage path only by rounding
        assert np.mean(a["acq"][i] == main["acq"][i]) >= 0.999
    # sharded over two ranks (called in turn, no collective): the same files as one rank
    one, two = tmp_path / "w1", tmp_path / "w2"
    kw = dict(size=121, angle_increment=120, poissonSNR=25.0, psf=psf, log=lambda *_: None, keep=(), ctx=ctx)
    mv.simulate_dataset(str(one), **kw)
    for rank in (0, 1):
        mv.simulate_dataset(str(two), rank=rank, world=2, **kw)
    names = sorted(os.listdir(one))
    assert names == sorted(os.listdir(two))
    for stem in ("acq_view_", "aligned_view_", "aligned_view_psf_", "aligned_view_weights"):
        for angle in angles:
            assert f"{stem}{angle}.tif" in names
    assert {"rendered.tif", "groundtruth.tif", "sum_weights.tif"} <= set(names)
    for name in names:
        assert (one / name).read_bytes() == (two / name).read_bytes(), name
    back = mv.tiff.read_float_stack(str(one / "acq_view_120.tif"))
    assert np.array_equal(back, a["acq"][1])


def test_simulate_dataset_config3_dims(mv, ctx):
    """1024 x 1024 x 512, inc 5, PSF 128^3, two of six views: aligned view and weights against the composed existing kernels."""
    S = mv.SimulateMultiViewDataset
    gt = np.random.default_rng(5).random((512, 1024, 1024), dtype=np.float32)
    k = gaussian_psf((128, 128, 128), (6.0, 2.2, 2.0), threshold=1e-3)
    angles = [0, 60, 120, 180, 240, 300]
    views = [1, 4]
    r = S.simulateDataset(gt, [k.copy(), k.copy()], angles, inc=5, poissonSNR=-1.0, osem=3.0, ctx=ctx, views=views,
                          outputs=("acq", "aligned", "weights"), sum_weights=False)
    del gt
    for i, v in enumerate(views):
        assert r["aligned"][i].shape == (511, 1024, 1024)
        ref = S.rotateAroundAxis(S.makeIsotropic(r["acq"][i], 5, ctx=ctx), 0, -angles[v], ctx=ctx)
        assert np.array_equal(r["aligned"][i], ref)
        del ref
        r["aligned"][i] = None
    ws, _ = _composed_weights(S, ctx, (512, 1024, 1024), [-a for a in angles], 3.0)
    for i, v in enumerate(views):
        assert np.array_equal(r["weights"][i], ws[v])
