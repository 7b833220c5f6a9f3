"""Parity at the shapes of BASELINE.json's configs (scaled where the CPU oracle would take minutes):
config 0 (reference default: odd cube, 51^3 fixture-like PSF, 7 views at 52 deg + 15), config 1 stage by
stage (attenuate + convolve only, anisotropic PSF), config 3's view loop through mvsim_simulate_views, and
config 3's bead volume with an SNR sweep on a device-resident convolved view."""
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


def fixture_like_psf(n=51, sigma=(7.0, 2.2, 2.0)):
    """Statistics of src/main/resources/Angle*.tif (SURVEY appendix B): 51^3, peak 0.99 at the centre,
    elongated in z, thresholded to a few percent support."""
    return gaussian_psf((n, n, n), sigma, threshold=0.01)


def test_reference_default_shape_stage_by_stage(mv, oracle):
    S = mv.SimulateMultiViewDataset
    gt = sphere_phantom((145, 145, 145), n_spheres=400)          # odd cube: centre (dim-1)/2 is exact, like 289
    psf = fixture_like_psf()
    for angle in (0, 52, 208):                                   # 7 views at 52 deg steps, +15 offset (:540,548,567)
        rot = S.rotateAroundAxis(gt, 0, angle + 15)
        assert rel_err(rot, oracle.rotate(gt, 0, angle + 15)) <= 1e-6
        att = S.attenuate3d(rot, 0.01)
        assert np.array_equal(att, oracle.attenuate(rot, 0.01))
        p1, p2 = psf.copy(), psf.copy()
        con = S.convolve(att, p1)
        ref = oracle.convolve(att, p2, "fft")
        assert rel_err(con, ref) <= 1e-5 and rel_err(p1, p2) <= 1e-6
        c_ref = oracle.adjust(ref, 0.0001, 1.0)
        c = mv.Tools.adjustImage(con, 0.0001, 1.0)
        assert c == pytest.approx(c_ref, rel=1e-5) and rel_err(con, ref) <= TOL
        acq = S.extractSlices(con, 3, -1.0)
        assert acq.shape[0] == 49 and np.array_equal(acq, con[::3])
        fused = S.simulateView(gt, psf.copy(), angle + 15, inc=3, poissonSNR=-1.0)
        assert rel_err(fused, acq) <= 1e-5


def test_config1_attenuate_and_convolve_only(mv, oracle):
    S = mv.SimulateMultiViewDataset
    gt = sphere_phantom((256, 256, 256), n_spheres=600)
    psf = gaussian_psf((64, 32, 32), (7.0 * 64 / 51, 2.2 * 32 / 51, 2.0 * 32 / 51), threshold=0.01)   # 64x64x128 scaled by 1/2
    att = S.attenuate3d(gt, 0.01)
    assert np.array_equal(att, oracle.attenuate(gt, 0.01))
    con = S.convolve(att, psf.copy())
    ref = oracle.convolve(att, psf.copy(), "fft")
    assert rel_err(con, ref) <= 1e-5
    # per-voxel relative error where the signal is significant (SURVEY section 7 "defining relative error")
    m = np.abs(ref) > 1e-3 * np.abs(ref).max()
    assert np.max(np.abs(con[m] - ref[m]) / np.abs(ref[m])) <= 1e-3


def test_view_loop_api_equals_single_view_calls(mv):
    S = mv.SimulateMultiViewDataset
    gt = sphere_phantom((40, 64, 64), n_spheres=60)
    degrees = [15, 75, 135, 195, 255, 315]
    psfs = [gaussian_psf((16, 16, 16), (3.0 + 0.1 * v, 1.2, 1.1), threshold=1e-3) for v in range(6)]
    a = S.simulateViews(gt, [p.copy() for p in psfs], degrees, inc=5, poissonSNR=25.0, rnd=7, first_stream=10)
    for v, d in enumerate(degrees):
        b = S.simulateView(gt, psfs[v].copy(), d, inc=5, poissonSNR=25.0, rnd=7, stream=10 + v)
        assert np.array_equal(a[v], b)
    # the PSFs handed to the loop were normalised in place (:255)
    q = [p.copy() for p in psfs]
    S.simulateViews(gt, q, degrees, inc=5, poissonSNR=-1.0)
    assert all(abs(float(p.astype(np.float64).sum()) - 1.0) < 1e-5 for p in q)


def bead_volume(shape, n_beads, sigma=(0.5, 0.5, 0.5), seed=535):
    """Sub-resolution beads: 1000 * exp(-sum d^2 / 2 sigma^2) (S/SimulateBeads.java:168-205), own generator."""
    rng = np.random.default_rng(seed)
    vol = np.zeros(shape, dtype=np.float32)
    for _ in range(n_beads):
        c = rng.uniform(4, np.array(shape) - 5)
        lo = np.floor(c).astype(int) - 3
        zz, yy, xx = np.mgrid[lo[0]:lo[0] + 8, lo[1]:lo[1] + 8, lo[2]:lo[2] + 8]
        g = 1000.0 * np.exp(-(((zz - c[0]) / sigma[0]) ** 2 + ((yy - c[1]) / sigma[1]) ** 2 + ((xx - c[2]) / sigma[2]) ** 2) / 2)
        vol[lo[0]:lo[0] + 8, lo[1]:lo[1] + 8, lo[2]:lo[2] + 8] += g.astype(np.float32)
    return vol


def test_bead_volume_snr_sweep_on_device_resident_view(mv):
    from mvsim_b200._lib import check
    S = mv.SimulateMultiViewDataset
    ctx = mv.Context(0)
    shape = (96, 128, 128)
    gt = bead_volume(shape, 250)
    psf = fixture_like_psf(25, (3.5, 1.1, 1.0))
    d_gt, d_rot, d_att, d_con = (mv.DeviceVolume(ctx, shape) for _ in range(4))
    d_gt.upload(gt)
    d_psf = mv.DeviceVolume(ctx, psf.shape, psf)
    d_out = mv.DeviceVolume(ctx, (32, 128, 128))
    lib = ctx._lib
    check(lib.mvsim_dev_psf_normalize(ctx.h, d_psf.h, None), ctx.h)
    for view, deg in enumerate((0, 45, 90)):                       # 8 views at 45 deg: three of them
        check(lib.mvsim_dev_rotate_axis(ctx.h, d_gt.h, d_rot.h, 0, deg), ctx.h)
        check(lib.mvsim_dev_attenuate(ctx.h, d_rot.h, d_att.h, 0.01, 1), ctx.h)
        check(lib.mvsim_dev_convolve(ctx.h, d_att.h, d_psf.h, d_con.h), ctx.h)
        corr = C.c_double()
        check(lib.mvsim_dev_adjust(ctx.h, d_con.h, 0.0001, 1.0, C.byref(corr)), ctx.h)
        con = d_con.download()
        assert float(con.astype(np.float64).mean()) == pytest.approx(1.0, rel=1e-5)
        clean = con[::3]
        for snr in (1, 2, 4, 8, 16, 25, 50, 100):                  # one convolved volume re-sampled at many SNRs
            check(lib.mvsim_dev_extract_slices(ctx.h, d_con.h, 3, float(snr), 99, view, d_out.h), ctx.h)
            noisy = d_out.download()
            mul = snr ** 2 / 5.0
            lam = clean.astype(np.float64) * mul
            assert noisy.sum() == pytest.approx(lam.sum(), rel=6 / math.sqrt(lam.sum()) + 1e-6)
            hot = lam > 20
            if hot.sum() > 500:
                z = (noisy[hot] - lam[hot]) / np.sqrt(lam[hot])
                assert abs(z.std() - 1) < 0.1
    for v in (d_gt, d_rot, d_att, d_con, d_psf, d_out):
        v.free()
    ctx.close()


def test_view_loop_on_resident_and_wrapped_ground_truth(mv):
    """mvsim_dev_simulate_views: the view loop on a ground truth that is already in HBM (uploaded once / broadcast over
    NVLink when views are sharded), through an owned volume and through a non-owning mvsim_volume_wrap handle."""
    S = mv.SimulateMultiViewDataset
    ctx = mv.Context(0)
    gt = sphere_phantom((24, 40, 40), n_spheres=60)
    psfs = [gaussian_psf((9, 7, 7), (2.0 + 0.1 * v, 1.0, 1.1), threshold=1e-3) for v in range(3)]
    degrees = [15, 135, 255]
    ref = S.simulateViews(gt, [p.copy() for p in psfs], degrees, inc=3, poissonSNR=25.0, rnd=7, ctx=ctx)
    vol = mv.DeviceVolume(ctx, gt.shape, gt)
    got = S.simulateViews(vol, [p.copy() for p in psfs], degrees, inc=3, poissonSNR=25.0, rnd=7, ctx=ctx)
    alias = mv.DeviceVolume.wrap(ctx, gt.shape, vol.device_ptr, keepalive=vol)
    got2 = S.simulateViews(alias, [p.copy() for p in psfs], degrees, inc=3, poissonSNR=25.0, rnd=7, ctx=ctx)
    for a, b, c in zip(ref, got, got2):
        assert np.array_equal(a, b) and np.array_equal(a, c)
    alias.free()                                   # frees the handle only
    assert np.array_equal(vol.download(), gt)      # the memory is still the owner's
    with pytest.raises(ValueError):
        S.simulateViews(mv.DeviceVolume(ctx, (24, 40, 44)), [p.copy() for p in psfs], degrees, inc=3, ctx=ctx,
                        outs=[np.empty((8, 40, 40), dtype=np.float32) for _ in range(3)])
    vol.free()
    ctx.close()


@pytest.mark.parametrize("shape,kshape,inc,distinct", [
    ((330, 48, 40), (31, 9, 7), 3, 3),       # z line 360: polyphase (3 x 120), decimated inverse (18 | 3) and full spectral kernel
    ((330, 40, 24), (31, 7, 5), 5, 2),       # 360 at inc 5: polyphase (5 x 72); no decimated kernel for this split -> full spectral
    ((512, 32, 24), (128, 9, 5), 5, 3),      # BASELINE config 3's z line: 640 = 5 x 128
    # other line lengths the polyphase kernel is built for
    ((300, 24, 16), (25, 5, 3), 3, 3),       # 324 = 3 x 108 (9 x 12), 36 groups
    ((360, 24, 16), (25, 5, 3), 3, 2),       # 384 = 3 x 128 (8 x 16), 24 groups, two rounds of level-1 items; no decimated kernel (3 does not divide 16)
    ((380, 24, 16), (21, 5, 3), 5, 3),       # 400 = 5 x 80 (8 x 10), 40 groups, two rounds
    ((400, 24, 16), (33, 5, 3), 3, 3),       # 432 = 3 x 144 (12 x 12), 36 groups
    ((450, 24, 16), (31, 5, 3), 3, 2),       # 480 = 3 x 160 (10 x 16), 30 groups, two rounds; no decimated kernel
])
def test_fused_z_kernel_variants_agree(mv, shape, kshape, inc, distinct):
    """MVSIM_OPT_Z_KERNEL: the polyphase, decimated-inverse and full spectral fused z kernels compute the same view (kept planes AND,
    through adjustImage's mean, the sum of the dropped planes) to float32 rounding -- and are really different kernels.  Every built
    instantiation against the direct-sum oracle: tests/test_gpu_fft_sizes.py::test_every_built_whole_view_kernel."""
    S = mv.SimulateMultiViewDataset
    rng = np.random.default_rng(31)
    gt = rng.random(shape, dtype=np.float32)
    psf = gaussian_psf(kshape, (kshape[0] / 6.0, 1.5, 1.2), threshold=0.0) + 1e-3 * rng.random(kshape, dtype=np.float32)
    outs = []
    for which in (3, 1, 2):
        ctx = mv.Context(0).z_kernel(which)
        outs.append(S.simulateView(gt, psf.copy(), 40, inc=inc, poissonSNR=-1.0, ctx=ctx))
    for o in outs[1:]:
        assert rel_err(outs[0], o) < 2e-6
        assert float(o.astype(np.float64).mean()) == pytest.approx(float(outs[0].astype(np.float64).mean()), rel=2e-6)
    assert len({o.tobytes() for o in outs}) == distinct
