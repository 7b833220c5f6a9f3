"""CPU emulation of the CUDA FFT-convolution kernels (tests/emu/emu_conv.cpp runs the kernels' own
__host__ __device__ phase functions thread by thread) against the oracle's direct-sum convolution.
Covers the host-side plan logic, the padded/pruned indexing and the fold+twist real transform."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import fft_cases
from helpers import rel_err

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(ROOT, "multiview-simulation_b200", "csrc")


@pytest.fixture(scope="module")
def emu():
    return fft_cases.build_emu(full=False)


@pytest.fixture(autouse=True, params=["materialised-H", "on-the-fly"])
def psf_spectrum_mode(request, monkeypatch):
    """Every test runs with both fused z kernels: ZFused (PSF spectrum H materialised by a z pass) and ZFusedOTF (the
    library's default: the PSF line is transformed inside the fused z pass)."""
    if request.param == "on-the-fly":
        monkeypatch.setenv("MVSIM_EMU_OTF", "1")
    else:
        monkeypatch.delenv("MVSIM_EMU_OTF", raising=False)


def _run(emu, vol, psfn, keep_inc=1, planes=None, world=1, max_line=0, p2p=0):
    z, y, x = vol.shape
    kz, ky, kx = psfn.shape
    out = np.empty_like(vol) if planes is None else np.empty((planes, y, x), dtype=np.float32)
    s = C.c_double(0)
    fp = C.POINTER(C.c_float)
    err = emu.emu_convolve(vol.ctypes.data_as(fp), (C.c_int64 * 3)(x, y, z), psfn.ctypes.data_as(fp),
                           (C.c_int64 * 3)(kx, ky, kz), out.ctypes.data_as(fp), C.byref(s), keep_inc, world, max_line, p2p)
    assert err == 0
    return out, s.value


@pytest.mark.parametrize("shape,kshape", [
    ((12, 14, 20), (5, 7, 9)),      # odd kernel
    ((9, 10, 11), (4, 6, 8)),       # even kernel (centre kdim/2)
    ((3, 4, 1), (7, 9, 4)),         # kernel larger than the image: multiple mirror folds, X = 1
    ((1, 1, 1), (3, 3, 3)),
    ((30, 17, 40), (1, 1, 1)),      # identity kernel
    ((20, 33, 50), (9, 3, 13)),     # several row blocks
    ((6, 7, 30), (3, 2, 8)),        # 20 complex columns: partial last kx tile of the tile-major layout
])
def test_emulated_kernels_match_direct_convolution(emu, oracle, shape, kshape):
    rng = np.random.default_rng(11)
    vol = rng.random(shape, dtype=np.float32)
    psf = rng.random(kshape, dtype=np.float32)
    ref = oracle.convolve(vol, psf, "direct")        # normalises psf in place
    out, s = _run(emu, vol, psf)
    assert rel_err(out, ref) < 5e-6
    assert s == pytest.approx(float(out.astype(np.float64).sum()), rel=1e-6)


def test_plan_sizes_cover_dim_plus_kdim_minus_one(emu):
    out = (C.c_int * 11)()
    for dims, kdims in [((1024, 1024, 512), (128, 128, 128)), ((289, 289, 289), (51, 51, 51)),
                        ((512, 512, 512), (64, 64, 128)), ((1, 1, 1), (1, 1, 1))]:
        err = emu.emu_plan((C.c_int64 * 3)(*dims), (C.c_int64 * 3)(*kdims), out, 0)
        if err == 5:        # the emulator's size table ends at 640 points
            continue
        assert err == 0
        assert 2 * out[0] >= dims[0] + kdims[0] - 1
        # y lines beyond the table are convolved in out[9] overlap-save blocks of out[10] rows each
        assert out[1] >= out[10] + kdims[1] - 1 and out[9] * out[10] >= dims[1] and out[2] >= dims[2] + kdims[2] - 1
        assert out[3] * out[4] == out[0] and out[5] * out[6] == out[1] and out[7] * out[8] == out[2]


@pytest.mark.parametrize("shape,kshape,inc", [((12, 14, 20), (5, 7, 9), 3), ((9, 10, 11), (4, 6, 8), 5), ((7, 6, 9), (3, 3, 3), 2),
                                              ((10, 5, 8), (2, 3, 3), 9)])
def test_kept_slices_and_sum_plane(emu, oracle, shape, kshape, inc):
    """Whole-view path: only every inc-th slice is carried through the inverse passes, plus one plane with
    the sum of the dropped slices; the total sum (adjustImage's mean) must not change."""
    rng = np.random.default_rng(12)
    vol = rng.random(shape, dtype=np.float32)
    psf = rng.random(kshape, dtype=np.float32)
    ref = oracle.convolve(vol, psf, "direct")
    kept = ref[::inc]
    nk = kept.shape[0]
    out, s = _run(emu, vol, psf, keep_inc=inc, planes=nk + 1)
    assert rel_err(out[:nk], kept) < 5e-6
    dropped = ref.astype(np.float64).sum(axis=0) - kept.astype(np.float64).sum(axis=0)
    assert rel_err(out[nk], dropped.astype(np.float32)) < 2e-5
    assert s == pytest.approx(float(ref.astype(np.float64).sum()), rel=2e-6)


@pytest.mark.parametrize("shape,kshape,max_line", [((6, 50, 12), (3, 7, 5), 24), ((4, 33, 9), (2, 4, 3), 16), ((5, 70, 8), (3, 9, 3), 30)])
def test_overlap_save_blocks_along_y(emu, oracle, shape, kshape, max_line):
    """y lines longer than the size table are convolved in overlap-save blocks (the 2048+255 rows of the
    largest single volume); max_line forces the same code path at test sizes."""
    out = (C.c_int * 11)()
    z, y, x = shape
    kz, ky, kx = kshape
    assert emu.emu_plan((C.c_int64 * 3)(x, y, z), (C.c_int64 * 3)(kx, ky, kz), out, max_line) == 0
    assert out[9] >= 2 and out[1] <= max_line and out[9] * out[10] >= y
    rng = np.random.default_rng(13)
    vol = rng.random(shape, dtype=np.float32)
    psf = rng.random(kshape, dtype=np.float32)
    ref = oracle.convolve(vol, psf, "direct")
    got, s = _run(emu, vol, psf, max_line=max_line)
    assert rel_err(got, ref) < 5e-6
    assert s == pytest.approx(float(ref.astype(np.float64).sum()), rel=2e-6)
    kept, _ = _run(emu, vol, psf, keep_inc=2, planes=(z - 1) // 2 + 2, max_line=max_line)
    assert rel_err(kept[:(z - 1) // 2 + 1], ref[::2]) < 5e-6


@pytest.mark.parametrize("world", [2, 4])
@pytest.mark.parametrize("shape,kshape,max_line", [((8, 14, 110), (3, 5, 9), 0), ((4, 40, 120), (5, 7, 3), 24)])
def test_slab_decomposed_convolution_with_host_all_to_all(emu, oracle, world, shape, kshape, max_line):
    """Largest-single-volume path (SURVEY section 8e): z slabs for the x/y passes, kx tiles for the z pass, two
    all-to-all transposes (done on the host here).  Must equal the undecomposed result."""
    rng = np.random.default_rng(14)
    vol = rng.random(shape, dtype=np.float32)
    psf = rng.random(kshape, dtype=np.float32)
    ref = oracle.convolve(vol, psf, "direct")
    got, s = _run(emu, vol, psf, world=world, max_line=max_line)
    assert rel_err(got, ref) < 5e-6
    one, _ = _run(emu, vol, psf, world=1, max_line=max_line)
    assert np.array_equal(got, one)          # the decomposition does not change a single bit
    assert s == pytest.approx(float(ref.astype(np.float64).sum()), rel=2e-6)
    # peer-to-peer variant: no exchange pass, the y and z passes store into the owners' buffers
    p2p, _ = _run(emu, vol, psf, world=world, max_line=max_line, p2p=1)
    assert np.array_equal(p2p, one)


def test_pruned_sub_transforms_match_the_full_ones(emu):
    """RegFFTPZ<N> (forward transform of a zero-extended line: inputs x[K..N) are never read) for every generated size."""
    emu.emu_check_pruned_ffts.restype = C.c_double
    assert emu.emu_check_pruned_ffts() < 2e-6


def test_zero_extended_psf_line_takes_the_pruned_path(emu, oracle):
    """PSF no longer than a fifth of the padded z line: the fused z pass transforms it with the pruned sub-transform."""
    rng = np.random.default_rng(5)
    vol = rng.random((26, 9, 10), dtype=np.float32)          # z = 26, kz = 5 -> 30 = 5 x 6 points, K * B = 6 >= 5
    psf = rng.random((5, 3, 4), dtype=np.float32)
    ref = oracle.convolve(vol, psf, "direct")
    out, _ = _run(emu, vol, psf)
    assert rel_err(out, ref) < 5e-6


def test_generated_butterflies_are_in_sync_with_the_generator(tmp_path):
    """fft/regfft_gen*.cuh are generated files: regenerating them must reproduce the committed text."""
    import sys
    a, b = tmp_path / "regfft_gen.cuh", tmp_path / "regfft_gen_packed.cuh"
    subprocess.check_call([sys.executable, os.path.join(ROOT, "tools", "gen_regfft.py"), str(a), str(b)])
    assert a.read_text() == open(os.path.join(CSRC, "fft", "regfft_gen.cuh")).read()
    assert b.read_text() == open(os.path.join(CSRC, "fft", "regfft_gen_packed.cuh")).read()


@pytest.mark.parametrize("shape,kshape,inc", [
    ((30, 6, 9), (7, 3, 4), 3),        # z line 36 = 6 x 6 -> ZFusedDec<6, 6, T, 3>, r = crop0 mod 3 = 0
    ((45, 5, 8), (10, 2, 3), 3),       # 54 = 6 x 9 -> ZFusedDec<9, 6, T, 3>, even kernel: r = 0 (crop0 = 9)
    ((46, 5, 8), (8, 2, 3), 3),        # 54 again with crop0 = 7: r = 1
    ((80, 4, 9), (21, 3, 2), 5),       # 100 = 10 x 10 -> ZFusedDec<10, 10, T, 5>, crop0 = 20: r = 0
    ((100, 3, 10), (19, 2, 3), 5),     # 120 = 10 x 12 -> ZFusedDec<12, 10, T, 5>, crop0 = 18: r = 3
    ((101, 3, 20), (17, 1, 2), 5),     # 120, crop0 = 16: r = 1; partial last kx tile
    ((599, 2, 3), (42, 1, 2), 5),      # 640 = 20 x 32 (BASELINE config 3's z line) -> ZFusedDec<32, 20, T, 5>: second inverse half split 4 x 8, two threads per (column, m); r = 1
    ((344, 2, 3), (17, 1, 2), 3),      # 360 = 18 x 20 (config 1 / 4 z lines at inc 3) -> ZFusedDec<20, 18, T, 3>: split 2 x 10
    ((560, 1, 3), (17, 1, 1), 3),      # 576 = 24 x 24 -> ZFusedDec<24, 24, T, 3>: split 3 x 8, every thread of a line busy
])
def test_decimated_inverse_of_the_fused_z_pass(emu, oracle, monkeypatch, psf_spectrum_mode, request, shape, kshape, inc):
    """ZFusedDec (the whole-view default where the split allows it): kept planes = whole columns of the exchange, pruned first
    inverse half, second inverse half for the kept columns only, sum plane from a dot product with the crop's Dirichlet table."""
    monkeypatch.setenv("MVSIM_EMU_DECIMATE", "1")
    emu.emu_decimated_launches.restype = C.c_int
    before = emu.emu_decimated_launches()
    rng = np.random.default_rng(21)
    vol = rng.random(shape, dtype=np.float32)
    psf = rng.random(kshape, dtype=np.float32)
    ref = oracle.convolve(vol, psf, "direct")
    kept = ref[::inc]
    nk = kept.shape[0]
    out, s = _run(emu, vol, psf, keep_inc=inc, planes=nk + 1)
    if "on-the-fly" in request.node.name:
        assert emu.emu_decimated_launches() == before + 1       # the decimated kernel really ran
    assert rel_err(out[:nk], kept) < 5e-6
    dropped = ref.astype(np.float64).sum(axis=0) - kept.astype(np.float64).sum(axis=0)
    assert rel_err(out[nk], dropped.astype(np.float32)) < 3e-5
    assert s == pytest.approx(float(ref.astype(np.float64).sum()), rel=3e-6)


@pytest.mark.parametrize("shape,kshape,inc", [
    ((599, 2, 3), (42, 1, 2), 5),      # 640 = 5 x 128 (BASELINE config 3's z line): 5 phases of 8 x 16 points, top == N exactly
    ((580, 1, 3), (42, 2, 1), 5),      # 640 with padding samples beyond the last tap's reach
    ((271, 1, 2), (90, 1, 1), 3),      # 360 = 3 x 120, PSF phases longer than the pruned sub-transform reads: full level 1
    ((261, 1, 2), (100, 1, 1), 5),     # 360 = 5 x 72, the same
    ((513, 1, 20), (128, 1, 2), 5),    # 640 = 513 + 128 - 1, even kernel, partial last kx tile
    ((344, 2, 3), (17, 1, 2), 3),      # 360 = 3 x 120 (config 1 / 4 z lines at inc 3): 10 x 12
    ((344, 1, 3), (17, 2, 1), 5),      # 360 = 5 x 72: 8 x 9, 40 groups, two rounds of level-1 items (5 in the second)
    ((330, 2, 3), (30, 1, 2), 3),      # 360 = 3 x 120 with an even kernel (crop0 = 29), one padding sample
    ((330, 1, 2), (1, 1, 1), 3),       # identity kernel: crop0 = 0 < inc - 1 (negative phase offsets wrap)
    ((350, 1, 2), (2, 1, 1), 5),       # two taps
])
def test_polyphase_fused_z_pass(emu, oracle, monkeypatch, psf_spectrum_mode, request, shape, kshape, inc):
    """ZFusedPoly: inc cyclic convolutions of n / inc points for the kept planes, sum of the dropped planes from the time domain
    (PSF prefix sums against the border samples of the image line)."""
    monkeypatch.setenv("MVSIM_EMU_POLY", "1")
    emu.emu_polyphase_launches.restype = C.c_int
    before = emu.emu_polyphase_launches()
    rng = np.random.default_rng(22)
    vol = rng.random(shape, dtype=np.float32)
    psf = rng.random(kshape, dtype=np.float32)
    ref = oracle.convolve(vol, psf, "direct")
    kept = ref[::inc]
    nk = kept.shape[0]
    out, s = _run(emu, vol, psf, keep_inc=inc, planes=nk + 1)
    assert rel_err(out[:nk], kept) < 5e-6
    total = ref.astype(np.float64).sum(axis=0)
    if "on-the-fly" in request.node.name:
        assert emu.emu_polyphase_launches() == before + 1       # the polyphase kernel really ran
        assert emu.emu_last_sum_plane_is_total() == 1            # ... and its extra plane is the sum of ALL cropped planes
        assert rel_err(out[nk], total.astype(np.float32)) < 3e-5
    else:
        assert emu.emu_last_sum_plane_is_total() == 0
        assert rel_err(out[nk], (total - kept.astype(np.float64).sum(axis=0)).astype(np.float32)) < 3e-5
    assert s == pytest.approx(float(ref.astype(np.float64).sum()), rel=3e-6)


def test_polyphase_kernel_is_vetoed_for_long_psf_lines(emu, oracle, monkeypatch):
    """More PSF taps than the border groups hold in registers (4 per group): the launcher falls back to the spectral kernels."""
    monkeypatch.setenv("MVSIM_EMU_POLY", "1")
    monkeypatch.setenv("MVSIM_EMU_OTF", "1")
    emu.emu_polyphase_launches.restype = C.c_int
    before = emu.emu_polyphase_launches()
    rng = np.random.default_rng(23)
    vol = rng.random((441, 1, 2), dtype=np.float32)
    psf = rng.random((200, 1, 1), dtype=np.float32)
    ref = oracle.convolve(vol, psf, "direct")
    out, _ = _run(emu, vol, psf, keep_inc=5, planes=(441 - 1) // 5 + 2)
    assert emu.emu_polyphase_launches() == before
    assert rel_err(out[:-1], ref[::5]) < 5e-6


def test_polyphase_kernel_applicability_table(emu):
    """zfused_poly_ok: inc in {3, 5} divides the line, n / inc is a table size of >= 64 points, at most 40 groups of 8 lanes, no
    split whose two gathered items per group would spill (measured slower than the decimated kernel at 576 points, inc 3)."""
    emu.emu_poly_ok.restype = C.c_int
    emu.emu_poly_ok.argtypes = [C.c_int, C.c_int]
    ok = {(n, inc): emu.emu_poly_ok(n, inc) for n in (320, 324, 360, 384, 400, 432, 480, 512, 540, 576, 600, 625, 640, 648) for inc in (2, 3, 5)}
    # BASELINE config 3: 640-point z lines at inc 5 -> 5 phases of 128 = 8 x 16 points, 40 groups, 4 taps x 32 border groups >= 128
    assert ok[(640, 5)] == 128
    assert ok[(360, 3)] > 0 and ok[(360, 5)] > 0 and ok[(320, 5)] > 0 and ok[(400, 5)] > 0
    assert ok[(576, 3)] == 0 and ok[(648, 3)] == 0 and ok[(540, 3)] == 0      # two 12-sample items per group: spills, excluded
    assert ok[(512, 5)] == 0 and ok[(625, 5)] == 0                            # 5 does not divide 512; 125 points is not a table size
    assert all(v == 0 for (n, inc), v in ok.items() if inc == 2)


def test_polyphase_pass_with_overlap_save_blocks_along_y(emu, oracle, monkeypatch):
    """Every y block runs its own fused z pass; with the polyphase kernel each block's extra plane is the sum of ALL cropped planes
    of its rows, and the inverse x pass counts that plane alone: the total must still be the sum of the whole convolved volume."""
    monkeypatch.setenv("MVSIM_EMU_POLY", "1")
    monkeypatch.setenv("MVSIM_EMU_OTF", "1")
    emu.emu_polyphase_launches.restype = C.c_int
    out = (C.c_int * 11)()
    shape, kshape, inc, max_line = (344, 33, 3), (17, 4, 2), 3, 16
    z, y, x = shape
    kz, ky, kx = kshape
    assert emu.emu_plan((C.c_int64 * 3)(x, y, z), (C.c_int64 * 3)(kx, ky, kz), out, max_line) == 0 and out[9] >= 2 and out[2] == 360
    before = emu.emu_polyphase_launches()
    rng = np.random.default_rng(24)
    vol = rng.random(shape, dtype=np.float32)
    psf = rng.random(kshape, dtype=np.float32)
    ref = oracle.convolve(vol, psf, "direct")
    nk = (z - 1) // inc + 1
    got, s = _run(emu, vol, psf, keep_inc=inc, planes=nk + 1, max_line=max_line)
    assert emu.emu_polyphase_launches() == before + out[9]          # one launch per y block
    assert emu.emu_last_sum_plane_is_total() == 1
    assert rel_err(got[:nk], ref[::inc]) < 5e-6
    assert rel_err(got[nk], ref.astype(np.float64).sum(axis=0).astype(np.float32)) < 3e-5
    assert s == pytest.approx(float(ref.astype(np.float64).sum()), rel=3e-6)
