"""Every FFT line length and every whole-view fused z kernel the library ships, in the CPU emulation (tests/emu/emu_conv.cpp built
with the full size table: the kernels' own phase functions, thread by thread), against the oracle's float64 direct sum.  Plus
every generated in-register sub-transform against a float64 DFT.  The cases come from fft_cases.py (read from conv_plan.h)."""
import ctypes as C
import importlib.util
import os

import numpy as np
import pytest

import fft_cases
from helpers import rel_err

CASES = fft_cases.cases()
CASE_IDS = [c.id for c in CASES]
_refs = {}


@pytest.fixture(scope="module")
def emu():
    return fft_cases.build_emu(full=True)


def _ref(oracle, case):
    if case.id not in _refs:
        vol, psf = case.arrays()
        _refs[case.id] = fft_cases.reference(oracle, vol, psf)
    return _refs[case.id]


def _plan(emu, shape, kshape):
    out = (C.c_int * 11)()
    z, y, x = shape
    kz, ky, kx = kshape
    assert emu.emu_plan((C.c_int64 * 3)(x, y, z), (C.c_int64 * 3)(kx, ky, kz), out, 0) == 0
    return {"x": 2 * out[0], "y": out[1], "z": out[2]}, out[9]


def _run(emu, oracle, vol, psf, keep_inc=1, planes=None):
    """emu_convolve with a normalised copy of psf (the library normalises in place before it convolves)"""
    psf = psf.copy()
    oracle.norm_image(psf)
    z, y, x = vol.shape
    kz, ky, kx = psf.shape
    out = np.empty_like(vol) if planes is None else np.empty((planes, y, x), dtype=np.float32)
    s = C.c_double(0)
    fp = C.POINTER(C.c_float)
    err = emu.emu_convolve(vol.ctypes.data_as(fp), (C.c_int64 * 3)(x, y, z), psf.ctypes.data_as(fp), (C.c_int64 * 3)(kx, ky, kz),
                           out.ctypes.data_as(fp), C.byref(s), keep_inc, 1, 0, 0)
    assert err == 0
    return out, s.value


def test_the_sweep_names_every_length_of_the_table():
    table = fft_cases.size_table()
    assert len(table) == 57 and all(n == a * b and a <= 40 and b <= 40 for n, a, b in table)
    assert [n for n, _, _ in table] == sorted({n for n, _, _ in table})
    assert {c.n for c in CASES} == {n for n, _, _ in table}
    assert len(CASES) == 3 * (2 * len(table) + sum(1 for n, _, _ in table if n % 8 == 0)) == 462
    for c in CASES:
        assert c.axis != "x" or c.kind != "a" or c.shape[2] % 4 == 0          # the x passes' X % 4 == 0 branch ...
        assert c.axis != "x" or c.kind != "b" or c.shape[2] % 2 == 1          # ... and the other one


@pytest.mark.parametrize("mode", ["materialised-H", "on-the-fly"])
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_every_line_length_along_every_axis(emu, oracle, monkeypatch, case, mode):
    """Stand-alone convolution: the planner picks the case's length, and the emulated passes (x forward / inverse, strided y, fused
    z with the PSF spectrum materialised (ZFused) or built on the fly (ZFusedOTF)) match the float64 direct sum."""
    if mode == "on-the-fly":
        monkeypatch.setenv("MVSIM_EMU_OTF", "1")
    else:
        monkeypatch.delenv("MVSIM_EMU_OTF", raising=False)
    lines, y_blocks = _plan(emu, case.shape, case.kshape)
    assert lines[case.axis] == case.line and y_blocks == 1
    vol, psf = case.arrays()
    ref = _ref(oracle, case)
    out, s = _run(emu, oracle, vol, psf)
    assert rel_err(out, ref) < 5e-6
    assert s == pytest.approx(float(ref.astype(np.float64).sum()), rel=2e-6)


Z_CASES = [c for c in CASES if c.axis == "z"]


@pytest.mark.parametrize("mode", ["materialised-H", "on-the-fly"])
@pytest.mark.parametrize("inc", [2, 3, 5])
@pytest.mark.parametrize("case", Z_CASES, ids=[c.id for c in Z_CASES])
def test_keep_and_sum_store_at_every_z_length(emu, oracle, monkeypatch, case, inc, mode):
    """Whole-view convolution with the spectral fused z kernels (ZFused / ZFusedOTF, no whole-view kernel requested): only every
    inc-th plane is carried through the inverse passes, plus one plane with the sum of the dropped ones."""
    monkeypatch.delenv("MVSIM_EMU_POLY", raising=False)
    monkeypatch.delenv("MVSIM_EMU_DECIMATE", raising=False)
    if mode == "on-the-fly":
        monkeypatch.setenv("MVSIM_EMU_OTF", "1")
    else:
        monkeypatch.delenv("MVSIM_EMU_OTF", raising=False)
    vol, psf = case.arrays()
    ref = _ref(oracle, case)
    kept = ref[::inc]
    nk = kept.shape[0]
    out, s = _run(emu, oracle, vol, psf, keep_inc=inc, planes=nk + 1)
    assert emu.emu_last_sum_plane_is_total() == 0
    assert rel_err(out[:nk], kept) < 5e-6
    dropped = ref.astype(np.float64).sum(axis=0) - kept.astype(np.float64).sum(axis=0)
    if nk < case.shape[0]:
        assert rel_err(out[nk], dropped.astype(np.float32)) < 3e-5
    assert s == pytest.approx(float(ref.astype(np.float64).sum()), rel=3e-6)


def test_built_whole_view_kernels_are_the_ones_fft_group_instantiates(emu):
    """emu_poly_ok / emu_dec_ok apply the built range kDecMinLine..kDecMaxLine like fft_group.cu; the pairs are pinned so that a
    change of either predicate shows up in review."""
    pairs = fft_cases.built_z_pairs(emu)
    poly = sorted(p for p, (ok, _) in pairs.items() if ok)
    dec = sorted(p for p, (_, ok) in pairs.items() if ok)
    assert poly == [(320, 5), (324, 3), (360, 3), (360, 5), (384, 3), (400, 5), (432, 3), (480, 3), (640, 5)]
    assert dec == [(324, 3), (360, 3), (400, 5), (432, 3), (480, 5), (540, 5), (576, 3), (600, 3), (625, 5), (640, 5), (648, 3)]
    assert len(pairs) == 15 and all(n in fft_cases.whole_view_lengths() for n, _ in pairs)
    assert emu.emu_poly_ok(120, 3) == 0 and emu.emu_dec_ok(120, 5) == 0      # emulated with the small table, but not built


@pytest.mark.parametrize("mode", ["materialised-H", "on-the-fly"])
@pytest.mark.parametrize("inc", [3, 5])
@pytest.mark.parametrize("n", fft_cases.whole_view_lengths())
def test_every_built_whole_view_kernel(emu, oracle, monkeypatch, n, inc, mode):
    """Every z length of the built range at inc 3 and 5: each whole-view kernel fft_group.cu builds for the pair (ZFusedPoly,
    ZFusedDec) and the spectral keep-and-sum store, kept planes and sum plane against the direct sum, and the launch counters say
    the intended kernel ran.  The whole-view kernels need the PSF spectrum on the fly; with H materialised every request runs
    ZFused's keep-and-sum store."""
    poly_ok, dec_ok = emu.emu_poly_ok(n, inc) > 0, emu.emu_dec_ok(n, inc) > 0
    otf = mode == "on-the-fly"
    if otf:
        monkeypatch.setenv("MVSIM_EMU_OTF", "1")
    else:
        monkeypatch.delenv("MVSIM_EMU_OTF", raising=False)
    case = fft_cases.whole_view_case(n)
    assert _plan(emu, case.shape, case.kshape)[0]["z"] == n
    vol, psf = case.arrays()
    ref = _ref(oracle, case)
    kept = ref[::inc]
    nk = kept.shape[0]
    total = ref.astype(np.float64).sum(axis=0)
    for kernel, env in (("polyphase", "MVSIM_EMU_POLY"), ("decimated", "MVSIM_EMU_DECIMATE"), ("spectral", None)):
        monkeypatch.delenv("MVSIM_EMU_POLY", raising=False)
        monkeypatch.delenv("MVSIM_EMU_DECIMATE", raising=False)
        if env:
            monkeypatch.setenv(env, "1")
        ran_poly = otf and kernel == "polyphase" and poly_ok
        ran_dec = otf and kernel == "decimated" and dec_ok
        before = (emu.emu_polyphase_launches(), emu.emu_decimated_launches())
        out, s = _run(emu, oracle, vol, psf, keep_inc=inc, planes=nk + 1)
        assert (emu.emu_polyphase_launches() - before[0], emu.emu_decimated_launches() - before[1]) == (int(ran_poly), int(ran_dec)), kernel
        assert rel_err(out[:nk], kept) < 5e-6, kernel
        is_total = emu.emu_last_sum_plane_is_total() == 1
        assert is_total == ran_poly
        want = total if is_total else total - kept.astype(np.float64).sum(axis=0)
        assert rel_err(out[nk], want.astype(np.float32)) < 3e-5, kernel
        assert s == pytest.approx(float(total.sum()), rel=3e-6), kernel


# ---- the generated sub-transforms (tools/gen_regfft.py) against a float64 DFT --------------------------------------------------
def _generator():
    spec = importlib.util.spec_from_file_location("gen_regfft", os.path.join(fft_cases.ROOT, "tools", "gen_regfft.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


GEN = _generator()
FAMILIES = ([pytest.param(0, n, d, 0, id=f"RegFFT<{n},{d:+d}>") for n in GEN.SIZES for d in (-1, 1)] +
            [pytest.param(1, n, d, 0, id=f"RegFFTP<{n},{d:+d}>") for n in GEN.SIZES for d in (-1, 1)] +
            [pytest.param(2, n, -1, 0, id=f"RegFFTPZ<{n}>") for n in GEN.SIZES] +
            [pytest.param(3, n, inc, r, id=f"RegFFTPD<{n},{inc},{r}>") for n, inc in GEN.DECIM for r in range(inc)])
BUTTERFLY_TOL = 1e-6       # worst seen on the CPU over 20 inputs per variant: 2.4e-7 (RegFFTPD), 1.8e-7 (RegFFTP)


def _dft(x, sign):
    n = len(x)
    k = np.arange(n)
    return np.exp(sign * 2j * np.pi * np.outer(k, k) / n) @ x


@pytest.mark.parametrize("family,n,d,r", FAMILIES)
def test_generated_sub_transform_against_a_float64_dft(emu, family, n, d, r):
    """RegFFT / RegFFTP: DIR = -1 forward exp(-2 pi i nk / N), +1 inverse, unscaled, natural order.  RegFFTPZ: the forward
    transform of x[0..K) zero-extended (x[K..N) holds garbage it must not read).  RegFFTPD<N, INC, R>: o[j] = inverse X[R + INC j]."""
    rng = np.random.default_rng(1000 * n + 10 * family + r + (d > 0))
    z = (rng.random(n) - 0.5) + 1j * (rng.random(n) - 0.5)
    x = z.astype(np.complex64)
    src = np.ascontiguousarray(x.view(np.float32))
    ref_in = x.astype(np.complex128)
    if family == 2:
        k = emu.emu_regfft_pz_k(n)
        assert k == (n + 4) // 5
        ref_in[k:] = 0
        src = src.copy()
        src[2 * k:] = 7.77e5            # must not be read
    sign = 1 if (family == 3 or d > 0) else -1
    ref = _dft(ref_in, sign)
    if family == 3:
        ref = ref[r::d]
    got = np.empty(2 * n, dtype=np.float32)
    fp = C.POINTER(C.c_float)
    assert emu.emu_regfft(family, n, d, r, src.ctypes.data_as(fp), got.ctypes.data_as(fp)) == 0
    out = got.view(np.complex64)[:len(ref)].astype(np.complex128)
    err = np.abs(out - ref).max() / np.abs(ref).max()
    assert err < BUTTERFLY_TOL, f"max |error| / max |X| = {err:.3g}"
