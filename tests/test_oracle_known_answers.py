"""Known-answer pins for the CPU oracle (SURVEY.md section 4): every expectation here follows from
the cited reference source semantics alone; the reference ships no tests of its own."""
import math

import numpy as np
import pytest

from helpers import gaussian_psf, rel_err, sphere_phantom


# ---- java.util.Random (JDK spec) -------------------------------------------------------------
def test_java_random_known_values(oracle):
    # new Random(42).nextInt() == -1170105035, 234785527 ; new Random(0).nextDouble()=0.730967787376657
    r = oracle.JavaRandom(42)
    assert r.next_int() == -1170105035
    assert r.next_int() == 234785527
    assert oracle.JavaRandom(0).next_double() == pytest.approx(0.730967787376657, abs=1e-15)
    assert oracle.JavaRandom(0).next_long() == -4962768465676381896


# ---- a1 axisRotation ---------------------------------------------------------------------------
def test_axis_rotation_centre_is_integer_division(oracle):
    m = oracle.axis_rotation((1024, 1024, 512), 0, 0)
    assert np.allclose(m, np.hstack([np.eye(3), np.zeros((3, 1))]))
    m = oracle.axis_rotation((1024, 1024, 512), 0, 90)
    # centre (1023//2, 511//2) = (511, 255) is a fixed point
    p = m[:, :3] @ np.array([7.0, 511.0, 255.0]) + m[:, 3]
    assert np.allclose(p, [7.0, 511.0, 255.0], atol=1e-9)


def test_axis_rotation_float_rounded_angle(oracle):
    m = oracle.axis_rotation((289, 289, 289), 0, 90)
    th = float(np.float32(math.radians(90)))
    assert m[1, 1] == pytest.approx(math.cos(th), abs=1e-15)   # -4.371139e-08, not 0
    assert abs(m[1, 1] + 4.371139e-08) < 1e-12
    assert m[1, 2] == pytest.approx(-math.sin(th))
    assert m[2, 1] == pytest.approx(math.sin(th))
    inv = oracle.affine_invert(m)
    assert np.allclose(inv[:, :3] @ m[:, :3], np.eye(3), atol=1e-12)


# ---- a2 rotateAroundAxis -----------------------------------------------------------------------
def test_rotate_zero_degrees_is_copy(oracle):
    v = np.random.default_rng(1).random((9, 11, 13), dtype=np.float32)
    for axis in range(3):
        assert np.array_equal(oracle.rotate(v, axis, 0), v)


def test_rotate_90_axis0_is_permutation_on_odd_cube(oracle):
    n = 15
    v = np.random.default_rng(2).random((n, n, n), dtype=np.float32)
    out = oracle.rotate(v, 0, 90)
    # inverse map (axis 0): y_src = c*(y-cy) + s*(z-cz) + cy ; z_src = -s*(y-cy) + c*(z-cz) + cz, s=1,c~0
    c = (n - 1) // 2
    exp = np.zeros_like(v)
    for z in range(n):
        for y in range(n):
            ys, zs = (z - c) + c, -(y - c) + c
            exp[z, y, :] = v[zs, ys, :]
    assert rel_err(out, exp) < 1e-5


def test_rotate_outside_is_zero_and_dims_kept(oracle):
    v = np.ones((8, 20, 6), dtype=np.float32)           # (Z,Y,X) = non cubic
    out = oracle.rotate(v, 0, 45)
    assert out.shape == v.shape
    assert out[7, 0, 0] == 0.0                           # maps to z_src = 12.2: outside -> extendZero
    assert out.max() <= 1.0 + 1e-6
    cz, cy = (8 - 1) // 2, (20 - 1) // 2
    assert out[cz, cy, 3] == pytest.approx(1.0, abs=1e-6)


def test_rotate_axis0_keeps_x(oracle):
    v = np.zeros((11, 11, 7), dtype=np.float32)
    v[:, :, 3] = 1.0
    out = oracle.rotate(v, 0, 33)
    assert np.all(out[:, :, [0, 1, 2, 4, 5, 6]] == 0)
    assert out[5, 5, 3] == pytest.approx(1.0, abs=1e-6)


# ---- a3 attenuate3d -----------------------------------------------------------------------------
def test_attenuate_constant_volume_closed_form(oracle):
    n, v, delta = 16, np.float32(0.7), 0.01
    vol = np.full((5, n, n), v, dtype=np.float32)
    out = oracle.attenuate(vol, delta)
    for k in range(n):                                   # k-th voxel from the top (y = n-1-k)
        exp = np.float32(float(v) * (1 - delta * float(v)) ** (k + 1))
        assert out[2, n - 1 - k, 3] == pytest.approx(exp, rel=2e-7)


def test_attenuate_clamps_to_zero(oracle):
    vol = np.full((2, 8, 8), 3.0, dtype=np.float32)
    out = oracle.attenuate(vol, 0.5)                     # v*delta = 1.5 > 1  -> n = 0 from the first voxel on
    assert np.all(out == 0)


def test_attenuate_light_enters_at_top_y(oracle):
    vol = np.zeros((1, 6, 6), dtype=np.float32)
    vol[0, 5, :] = 1.0
    vol[0, 0, :] = 1.0
    out = oracle.attenuate(vol, 0.1)
    assert out[0, 5, 0] == pytest.approx(0.9)
    assert out[0, 0, 0] == pytest.approx(0.81)


def test_attenuate_strict_uses_dimension0_loop_bound(oracle):
    vol = np.ones((2, 10, 6), dtype=np.float32)          # X=6 < Y=10
    out = oracle.attenuate(vol, 0.01, strict=True)
    assert np.all(out[:, :4, :] == 0) and np.all(out[:, 4:, :] > 0)
    out2 = oracle.attenuate(vol, 0.01, strict=False)
    assert np.all(out2 > 0)
    with pytest.raises(ValueError):
        oracle.attenuate(np.ones((2, 6, 10), dtype=np.float32), 0.01, strict=True)


# ---- a4/a5 normImage + convolve -------------------------------------------------------------------
def test_norm_image_in_place(oracle):
    psf = gaussian_psf((7, 5, 9), (1.5, 1.0, 2.0))
    s = float(psf.astype(np.float64).sum())
    ret = oracle.norm_image(psf)
    assert ret == pytest.approx(s, rel=1e-12)
    assert float(psf.astype(np.float64).sum()) == pytest.approx(1.0, abs=1e-6)


@pytest.mark.parametrize("method", ["direct", "fft"])
def test_convolve_constant_image_stays_constant(oracle, method):
    vol = np.full((10, 12, 14), 2.5, dtype=np.float32)
    psf = gaussian_psf((5, 7, 6), (1.0, 1.5, 1.2))
    out = oracle.convolve(vol, psf, method)
    assert rel_err(out, vol) < 2e-6
    assert float(psf.astype(np.float64).sum()) == pytest.approx(1.0, abs=1e-6)   # side effect :255


@pytest.mark.parametrize("kshape", [(5, 7, 9), (4, 6, 8)])
@pytest.mark.parametrize("method", ["direct", "fft"])
def test_convolve_impulse_gives_unflipped_psf_centred_at_kdim_half(oracle, method, kshape):
    vol = np.zeros((20, 22, 24), dtype=np.float32)
    p = (10, 11, 12)
    vol[p] = 1.0
    psf = np.random.default_rng(3).random(kshape, dtype=np.float32)
    out = oracle.convolve(vol, psf, method)              # psf now normalised
    kz, ky, kx = kshape
    for dz in range(kz):
        for dy in range(ky):
            for dx in range(kx):
                # out[x] = psfN[x - p + c], c = kdim/2
                o = out[p[0] + dz - kz // 2, p[1] + dy - ky // 2, p[2] + dx - kx // 2]
                assert o == pytest.approx(psf[dz, dy, dx], abs=2e-7)


def test_convolve_fft_matches_direct_with_mirror_border(oracle):
    rng = np.random.default_rng(4)
    vol = rng.random((13, 17, 19), dtype=np.float32)
    psf = rng.random((6, 5, 9), dtype=np.float32)
    a = oracle.convolve(vol, psf.copy(), "direct")
    b = oracle.convolve(vol, psf.copy(), "fft")
    assert rel_err(b, a) < 2e-6
    # independent second opinion: numpy mirror pad + float64 FFT
    k = psf.astype(np.float64) / psf.astype(np.float64).sum()
    pads = [(ks - 1 - ks // 2, ks // 2) for ks in k.shape]
    padded = np.pad(vol.astype(np.float64), pads, mode="reflect")
    full = np.fft.irfftn(np.fft.rfftn(padded) * np.fft.rfftn(k, padded.shape), padded.shape)
    crop = full[k.shape[0] - 1:, k.shape[1] - 1:, k.shape[2] - 1:][:13, :17, :19]
    assert rel_err(a, crop) < 1e-6


def test_convolve_kernel_larger_than_image(oracle):
    rng = np.random.default_rng(5)
    vol = rng.random((3, 4, 1), dtype=np.float32)
    psf = rng.random((7, 9, 4), dtype=np.float32)
    a = oracle.convolve(vol, psf.copy(), "direct")
    b = oracle.convolve(vol, psf.copy(), "fft")
    assert rel_err(b, a) < 2e-6


# ---- a6 adjustImage ---------------------------------------------------------------------------------
def test_adjust_mean_min_and_correction(oracle):
    vol = sphere_phantom((12, 14, 16), n_spheres=12)
    before_avg = float(vol.astype(np.float64).mean())
    corr = oracle.adjust(vol, 0.0001, 1.0)
    assert corr == pytest.approx(float(np.float32(1.0) - np.float32(0.0001)) / before_avg, rel=1e-12)
    assert float(vol.astype(np.float64).mean()) == pytest.approx(1.0, rel=1e-6)
    assert vol.min() >= np.float32(0.0001)


def test_adjust_rounds_twice(oracle):
    vol = np.random.default_rng(6).random((4, 5, 6), dtype=np.float32)
    src = vol.copy()
    corr = oracle.adjust(vol, 0.0001, 1.0)
    exp = (src.astype(np.float64) * corr).astype(np.float32) + np.float32(0.0001)
    assert np.array_equal(vol, exp)


# ---- a7 extractSlices ---------------------------------------------------------------------------------
@pytest.mark.parametrize("z,inc", [(10, 3), (9, 3), (1, 5), (512, 5), (7, 1)])
def test_extract_slices_bit_exact_selection(oracle, z, inc):
    vol = np.random.default_rng(7).random((z, 3, 4), dtype=np.float32)
    out = oracle.extract_slices(vol, inc, -1.0)
    assert out.shape[0] == (z - 1) // inc + 1
    assert np.array_equal(out, vol[::inc])


# ---- a8 Poisson ---------------------------------------------------------------------------------------
def test_poisson_snr0_gives_zero_and_integer_output(oracle):
    vol = np.random.default_rng(8).random((4, 8, 8), dtype=np.float32)
    assert np.all(oracle.extract_slices(vol, 1, 0.0) == 0)
    out = oracle.extract_slices(vol * 5, 1, 10.0)
    assert np.array_equal(out, np.round(out))


@pytest.mark.parametrize("v,snr", [(0.05, 2.0), (1.0, 5.0), (6.0, 25.0)])
def test_poisson_mean_equals_variance_equals_lambda(oracle, v, snr):
    n = 40000
    a = np.full(n, v, dtype=np.float32)
    oracle.poisson(a, snr, oracle.JavaRandom(123))
    lam = float(np.float32(v)) * (snr / math.sqrt(5)) ** 2
    se = math.sqrt(lam / n)
    assert abs(a.mean() - lam) < 5 * se
    assert abs(a.var() - lam) < 5 * lam * math.sqrt(2.0 / n) + 5 * se


def test_poisson_is_deterministic_in_the_seed_and_consumes_the_stream_in_flat_order(oracle):
    a = np.full(100, 2.0, dtype=np.float32)
    b = a.copy()
    oracle.poisson(a, 5.0, oracle.JavaRandom(9))
    r = oracle.JavaRandom(9)
    oracle.poisson(b[:50], 5.0, r)
    oracle.poisson(b[50:], 5.0, r)
    assert np.array_equal(a, b)


# ---- fixtures of the reference (inputs only) ------------------------------------------------------------
def test_reference_psf_fixture_statistics():
    """Angle0.tif of the reference, through its lossless copy in tests/golden/psf_angle0.npz."""
    from test_golden import load_psf
    psf = load_psf()
    assert psf.shape == (51, 51, 51) and psf.dtype == np.float32
    assert psf.max() == pytest.approx(0.99, abs=1e-6) and psf.min() == 0
    assert np.unravel_index(psf.argmax(), psf.shape) == (25, 25, 25)
    assert float(psf.astype(np.float64).sum()) == pytest.approx(265.355, abs=2e-3)   # SURVEY appendix B
