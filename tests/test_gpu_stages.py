"""Parity of every CUDA stage with the CPU oracle, through the C ABI (ctypes) -- run with -m gpu on a B200.

Tolerances (BASELINE.json north_star): max|a-b| / max|b| <= 1e-4 for rotation, attenuation,
convolution and adjust; bit exact for voxel indexing / slice selection; Poisson by mean/variance and
a two-sample KS test against the oracle's replay of the reference sampler."""
import ctypes as C
import math

import numpy as np
import pytest

from helpers import gaussian_psf, rel_err, sphere_phantom

pytestmark = pytest.mark.gpu

TOL = 1e-4


@pytest.fixture(scope="module")
def mv():
    import mvsim_b200
    return mvsim_b200


@pytest.fixture(scope="module")
def S(mv):
    return mv.SimulateMultiViewDataset


# ---- rotate ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(24, 32, 40), (17, 23, 31), (9, 40, 12)])
@pytest.mark.parametrize("degrees", [0, 15, 60, 90, 135, 330, -52])
def test_rotate_axis0_matches_oracle(S, oracle, shape, degrees):
    v = np.random.default_rng(1).random(shape, dtype=np.float32)
    got = S.rotateAroundAxis(v, 0, degrees)
    ref = oracle.rotate(v, 0, degrees)
    assert got.shape == v.shape
    assert rel_err(got, ref) <= 1e-6
    if degrees == 0:
        assert np.array_equal(got, v)


@pytest.mark.parametrize("axis", [1, 2])
@pytest.mark.parametrize("degrees", [0, 33, 90, 200])
def test_rotate_other_axes_match_oracle(S, oracle, axis, degrees):
    v = np.random.default_rng(2).random((14, 19, 22), dtype=np.float32)
    assert rel_err(S.rotateAroundAxis(v, axis, degrees), oracle.rotate(v, axis, degrees)) <= 1e-6


def test_rotate_phantom_within_tolerance(S, oracle):
    v = sphere_phantom((48, 64, 64), n_spheres=60)
    for deg in (15, 75):
        assert rel_err(S.rotateAroundAxis(v, 0, deg), oracle.rotate(v, 0, deg)) <= TOL


# ---- attenuate ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(5, 16, 16), (7, 33, 20), (3, 9, 9), (2, 1, 1)])
def test_attenuate_matches_oracle_bitwise(S, oracle, shape):
    v = np.random.default_rng(3).random(shape, dtype=np.float32) * 3
    got = S.attenuate3d(v, 0.01)
    ref = oracle.attenuate(v, 0.01, strict=True)
    assert np.array_equal(got, ref)
    assert np.array_equal(S.attenuate3d(v, 0.5, strict_reference=False), oracle.attenuate(v, 0.5, strict=False))


def test_attenuate_strict_rejects_x_greater_y(mv, S):
    with pytest.raises(mv.MvsimError) as e:
        S.attenuate3d(np.ones((2, 4, 8), dtype=np.float32), 0.01)
    assert e.value.status == 1
    S.attenuate3d(np.ones((2, 4, 8), dtype=np.float32), 0.01, strict_reference=False)


# ---- fused rotate + attenuate ------------------------------------------------------------------------
# one shape per march kernel: X % 4 == 0 (offset table), X % 4 == 2 (float2), odd X (scalar); the phantom is non-negative, the
# condition under which the offset table's out-of-volume taps give exactly the bounds-tested result
@pytest.mark.parametrize("shape", [(24, 40, 32), (17, 34, 30), (9, 40, 13)])
@pytest.mark.parametrize("strict,delta", [(True, 0.01), (False, 0.01), (False, 0.5)])
def test_fused_rotate_attenuate_equals_rotate_then_attenuate_bitwise(mv, shape, strict, delta):
    from mvsim_b200._lib import check, dims3
    ctx = mv.Context(0)
    lib = ctx._lib
    gt, rot, att, fused = (mv.DeviceVolume(ctx, shape) for _ in range(4))
    gt.upload(sphere_phantom(shape, n_spheres=20) * 3)
    for deg in (0, 15, 60, 90, 135, 200, -52):
        check(lib.mvsim_dev_rotate_axis(ctx.h, gt.h, rot.h, 0, deg), ctx.h)
        check(lib.mvsim_dev_attenuate(ctx.h, rot.h, att.h, delta, int(strict)), ctx.h)
        check(lib.mvsim_slab_rotate_attenuate(ctx.h, C.c_void_p(gt.device_ptr), dims3(shape), 0, deg, delta, int(strict), 0, shape[0],
                                              C.c_void_p(fused.device_ptr)), ctx.h)
        assert np.array_equal(fused.download().view(np.uint32), att.download().view(np.uint32)), deg
    for v in (gt, rot, att, fused):
        v.free()
    ctx.close()


# ---- normImage / convolve ----------------------------------------------------------------------------
def test_norm_image_in_place(mv, oracle):
    psf = gaussian_psf((11, 9, 13), (2.0, 1.5, 2.5))
    ref = psf.copy()
    oracle.norm_image(ref)
    mv.Tools.normImage(psf)
    assert rel_err(psf, ref) <= 1e-6
    assert float(psf.astype(np.float64).sum()) == pytest.approx(1.0, abs=1e-6)


@pytest.mark.parametrize("shape,kshape", [
    ((12, 14, 20), (5, 7, 9)), ((9, 10, 11), (4, 6, 8)), ((3, 4, 1), (7, 9, 4)), ((1, 1, 1), (3, 3, 3)),
    ((30, 17, 40), (1, 1, 1)), ((20, 33, 50), (9, 3, 13)), ((40, 48, 56), (13, 11, 15)),
])
def test_convolve_matches_direct_sum(S, oracle, shape, kshape):
    rng = np.random.default_rng(4)
    v = rng.random(shape, dtype=np.float32)
    psf = rng.random(kshape, dtype=np.float32)
    psf_ref = psf.copy()
    ref = oracle.convolve(v, psf_ref, "direct")
    got = S.convolve(v, psf)
    assert rel_err(got, ref) <= 1e-5
    assert rel_err(psf, psf_ref) <= 1e-6             # caller's PSF normalised in place (:255)


def test_convolve_medium_phantom_vs_both_oracle_paths(S, oracle):
    v = sphere_phantom((64, 96, 96), n_spheres=80)
    psf = gaussian_psf((17, 9, 9), (3.5, 1.1, 1.0), threshold=1e-3)
    ref_d = oracle.convolve(v, psf.copy(), "direct")
    ref_f = oracle.convolve(v, psf.copy(), "fft")
    got = S.convolve(v, psf.copy())
    assert rel_err(got, ref_d) <= TOL and rel_err(got, ref_f) <= TOL
    assert rel_err(got, ref_d) <= 1e-5


def test_convolve_large_lines_exercise_every_size_group(S, oracle):
    # padded lines 2*160 / 432 / 1152: groups 1, 2 and 4 of the size table
    rng = np.random.default_rng(5)
    v = rng.random((1100, 400, 300), dtype=np.float32)
    psf = np.zeros((40, 20, 15), dtype=np.float32)
    taps = [(0, 0, 0), (39, 19, 14), (20, 10, 7), (5, 17, 2)]
    for i, t in enumerate(taps):
        psf[t] = i + 1.0
    got = S.convolve(v, psf)
    w = psf[[t[0] for t in taps], [t[1] for t in taps], [t[2] for t in taps]].astype(np.float64)
    # sparse kernel: direct evaluation at a sample of voxels (mirror-single border)
    def mir(i, n):
        p = 2 * (n - 1); j = i % p
        return p - j if j >= n else j
    for (z, y, x) in [(0, 0, 0), (1099, 399, 299), (500, 200, 150), (3, 398, 1), (1090, 2, 297)]:
        exp = sum(w[i] * v[mir(z - (t[0] - 20), 1100), mir(y - (t[1] - 10), 400), mir(x - (t[2] - 7), 300)] for i, t in enumerate(taps))
        assert got[z, y, x] == pytest.approx(exp, rel=2e-5)


# ---- adjustImage -------------------------------------------------------------------------------------
def test_adjust_matches_oracle(mv, oracle):
    v = sphere_phantom((20, 24, 28), n_spheres=30)
    ref = v.copy()
    c_ref = oracle.adjust(ref, 0.0001, 1.0)
    c = mv.Tools.adjustImage(v, 0.0001, 1.0)
    assert c == pytest.approx(c_ref, rel=1e-12)
    assert rel_err(v, ref) <= 1e-6
    assert float(np.mean(v != ref)) < 1e-3
    assert float(v.astype(np.float64).mean()) == pytest.approx(1.0, rel=1e-6)


# ---- extractSlices -----------------------------------------------------------------------------------
@pytest.mark.parametrize("z,inc", [(10, 3), (9, 3), (1, 5), (103, 5), (7, 1), (4, 9)])
def test_extract_slices_bit_exact(S, oracle, z, inc):
    v = np.random.default_rng(6).random((z, 6, 10), dtype=np.float32)
    got = S.extractSlices(v, inc, -1.0)
    assert got.shape == ((z - 1) // inc + 1, 6, 10)
    assert np.array_equal(got, v[::inc])
    assert np.array_equal(got, oracle.extract_slices(v, inc, -1.0))


def test_extract_slices_rejects_bad_inc(mv, S):
    with pytest.raises(mv.MvsimError):
        S.extractSlices(np.ones((3, 3, 3), dtype=np.float32), 0, -1.0)


# ---- Poisson -------------------------------------------------------------------------------------------
def _ks_two_sample(a, b):
    from scipy import stats
    return stats.ks_2samp(a, b).pvalue


@pytest.mark.parametrize("lam", [0.01, 0.5, 3.0, 30.0, 300.0, 3000.0])
def test_poisson_matches_reference_sampler_statistically(mv, oracle, lam):
    snr = 10.0
    mul = (snr / math.sqrt(5)) ** 2
    v = np.float32(lam / mul)
    lam_eff = float(v) * mul
    n = 200000 if lam <= 30 else 60000
    a = np.full(n, v, dtype=np.float32)
    mv.Tools.poissonProcess(a, snr, mv.JavaRandom(77))
    assert np.array_equal(a, np.round(a)) and a.min() >= 0
    se = math.sqrt(lam_eff / n)
    assert abs(a.mean() - lam_eff) < 5 * se
    assert abs(a.var() - lam_eff) < 6 * lam_eff * math.sqrt(2.0 / n) + 6 * se
    m = 20000 if lam <= 300 else 4000
    b = np.full(m, v, dtype=np.float32)
    oracle.poisson(b, snr, oracle.JavaRandom(5))
    # two-sample KS against the oracle's replay of the reference sampler, p > 0.01 as SURVEY 8c asks (the CPU emulation of
    # the same sampler code gives p = 0.70 .. 1.0 for these seeds)
    assert _ks_two_sample(a[:m * 3], b) > 0.01


def test_poisson_zero_negative_and_snr0(mv):
    a = np.array([0.0, -1.0, 5.0, np.nan], dtype=np.float32)
    b = a.copy()
    mv.Tools.poissonProcess(b, 25.0, 1)
    assert b[0] == 0 and b[1] == 0 and b[3] == 0 and b[2] > 0
    c = np.full(1000, 5.0, dtype=np.float32)
    mv.Tools.poissonProcess(c, 0.0, 1)
    assert np.all(c == 0)


def test_poisson_is_counter_based(mv, S):
    v = np.random.default_rng(7).random((6, 16, 16), dtype=np.float32) * 4
    a = S.extractSlices(v, 2, 10.0, rnd=123, stream=3)
    b = S.extractSlices(v, 2, 10.0, rnd=123, stream=3)
    c = S.extractSlices(v, 2, 10.0, rnd=123, stream=4)
    d = S.extractSlices(v, 2, 10.0, rnd=124, stream=3)
    assert np.array_equal(a, b)
    assert not np.array_equal(a, c) and not np.array_equal(a, d)
    # the facade draws exactly one nextLong() from the caller's generator
    r = mv.JavaRandom(9)
    e = S.extractSlices(v, 2, 10.0, rnd=r)
    assert np.array_equal(e, S.extractSlices(v, 2, 10.0, rnd=mv.JavaRandom(9).nextLong()))
    r2 = mv.JavaRandom(9)
    r2.nextLong()
    assert r.nextInt() == r2.nextInt()


# ---- the whole view -------------------------------------------------------------------------------------
def test_simulate_view_equals_stage_by_stage_and_oracle(mv, S, oracle):
    gt = sphere_phantom((40, 48, 48), n_spheres=50)
    psf = gaussian_psf((13, 7, 7), (2.5, 1.0, 0.9), threshold=1e-3)
    rot = S.rotateAroundAxis(gt, 0, 67)
    att = S.attenuate3d(rot, 0.01)
    con = S.convolve(att, psf.copy())
    mv.Tools.adjustImage(con, S.minValue, S.avgIntensity)
    acq = S.extractSlices(con, 3, -1.0)
    fused = S.simulateView(gt, psf.copy(), 67, inc=3, poissonSNR=-1.0)
    assert rel_err(fused, acq) <= 1e-6
    ref, ref_con, _ = oracle.simulate_view(gt, psf, degrees=67, inc=3, snr=-1.0, use_fft=False)
    assert rel_err(con, ref_con) <= TOL
    assert rel_err(fused, ref) <= TOL
    # noisy: same noise-free intensity => same per-voxel mean; check the global statistics
    noisy = S.simulateView(gt, psf.copy(), 67, inc=3, poissonSNR=25.0, rnd=5)
    lam = acq.astype(np.float64) * (25.0 / math.sqrt(5)) ** 2
    m = lam > 5        # the z-score of tiny-lambda background voxels is too heavy tailed for a tight bound
    z = (noisy[m] - lam[m]) / np.sqrt(lam[m])
    assert m.sum() > 2000 and abs(z.mean()) < 5 / math.sqrt(m.sum()) and abs(z.std() - 1.0) < 0.05
    assert noisy[lam < 0.05].mean() == pytest.approx(lam[lam < 0.05].mean(), rel=0.3)


def test_views_do_not_depend_on_context_or_order(mv, S):
    gt = sphere_phantom((24, 32, 32), n_spheres=30)
    psf = gaussian_psf((9, 5, 5), (2.0, 0.9, 0.9))
    c1, c2 = mv.Context(0), mv.Context(0)
    views = [(d, i) for i, d in enumerate((15, 75, 135))]
    a = {i: S.simulateView(gt, psf.copy(), d, inc=2, poissonSNR=10.0, rnd=42, ctx=c1, stream=i) for d, i in views}
    b = {i: S.simulateView(gt, psf.copy(), d, inc=2, poissonSNR=10.0, rnd=42, ctx=c2, stream=i) for d, i in reversed(views)}
    for i in a:
        assert np.array_equal(a[i], b[i])
    c1.close(); c2.close()


def test_device_resident_snr_sweep(mv, S):
    ctx = mv.Context(0)
    gt = sphere_phantom((16, 24, 24), n_spheres=20) + 0.5
    vol = mv.DeviceVolume(ctx, gt.shape, gt)
    out = mv.DeviceVolume(ctx, (6, 24, 24))
    from mvsim_b200._lib import check
    means = []
    for snr in (2.0, 8.0, 32.0):
        check(ctx._lib.mvsim_dev_extract_slices(ctx.h, vol.h, 3, snr, 11, 0, out.h), ctx.h)
        o = out.download()
        means.append(o.mean() / (snr ** 2 / 5))
    assert all(abs(m - gt[::3].mean()) < 0.05 for m in means)
    vol.free(); out.free(); ctx.close()


def test_unsupported_and_invalid_shapes(mv, S):
    with pytest.raises(mv.MvsimError) as e:
        S.convolve(np.ones((2, 2, 3300), dtype=np.float32), np.ones((1, 1, 3), dtype=np.float32))
    assert e.value.status == 5
    with pytest.raises(ValueError):
        S.convolve(np.ones((2, 2), dtype=np.float32), np.ones((1, 1, 3), dtype=np.float32))


def test_two_threads_with_their_own_contexts(mv, S):
    """The reference calls the path from two pool threads at once (S/SimulateTileStitching.java:85-117): contexts are
    independent (own stream, own workspaces), results must equal the serial ones."""
    import threading
    gt = sphere_phantom((32, 40, 40), n_spheres=60)
    psf = gaussian_psf((9, 7, 7), (2.0, 1.0, 1.0))
    jobs = [(15, 3), (75, 4), (135, 5), (195, 6)]
    serial = {d: S.simulateView(gt, psf.copy(), d, inc=2, poissonSNR=12.0, rnd=99, stream=st) for d, st in jobs}
    out, errs = {}, []

    def work(sub):
        try:
            ctx = mv.Context(0)
            for _ in range(3):
                for d, st in sub:
                    out[d] = S.simulateView(gt, psf.copy(), d, inc=2, poissonSNR=12.0, rnd=99, ctx=ctx, stream=st)
            ctx.close()
        except Exception as e:      # pragma: no cover
            errs.append(e)
    ts = [threading.Thread(target=work, args=(jobs[:2],)), threading.Thread(target=work, args=(jobs[2:],))]
    [t.start() for t in ts]
    [t.join() for t in ts]
    assert not errs, errs
    for d, _ in jobs:
        assert np.array_equal(out[d], serial[d])


def test_cooperative_and_per_thread_sampler_paths_agree_bit_for_bit(mv, S):
    """extractSlices finishes the PTRS voxels cooperatively (compacted in shared memory), Tools.poissonProcess thread by thread:
    a voxel's count depends on (seed, stream, voxel index) only, so both must return the same volume."""
    rng = np.random.default_rng(31)
    v = (rng.random((5, 37, 52), dtype=np.float32) * 3).astype(np.float32)      # lambda 0 .. 375 at SNR 25: every regime, ragged size
    v[0, :5] = 0
    a = S.extractSlices(v, 1, 25.0, rnd=99, stream=6)
    b = v.copy()
    mv.Tools.poissonProcess(b, 25.0, 99, stream=6)
    assert np.array_equal(a, b)
