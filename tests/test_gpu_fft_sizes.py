"""Every FFT line length and every whole-view fused z kernel the library ships, run on the GPU against the oracle's float64 direct
sum.  The cases come from fft_cases.py, which reads the size table from conv_plan.h: a length added there is covered here.

- stand-alone sweep: 3 cases per length and axis (462), the planned lengths confirmed through mvsim_slabconv_info;
- whole-view sweep: simulateView at 0 deg for every z case and inc 2, 3, 5 (ZFusedOTF's keep-and-sum store outside the built
  range of the whole-view kernels, the automatic kernel choice inside it);
- every built whole-view instantiation: MVSIM_OPT_Z_KERNEL 3 / 1 / 2 at every z length of the built range, each against the
  reference, and as many distinct outputs as kernels built for the pair (which proves each of them ran);
- the process-wide knobs MVSIM_H_MATERIALIZE (ZFused and the strided pass that builds H) and MVSIM_NO_TMA (the cp.async PSF tile,
  the spectral fallback of the polyphase kernel) in a worker process each."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import fft_cases
from helpers import rel_err

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))

CASES = fft_cases.cases()
CASE_IDS = [c.id for c in CASES]
Z_CASES = [c for c in CASES if c.axis == "z"]
# tolerances: 10x the worst rel_err of the CPU emulation (4.6e-7 stand-alone) and of the whole view against its oracle chain
TOL_CONV, TOL_VIEW = 5e-6, 1e-5

_refs, _view_refs = {}, {}
_worst = {}         # (test, pass) -> largest rel_err seen, printed at the end of the module (pytest -s)


def _note(what, err):
    _worst[what] = max(_worst.get(what, 0.0), err)


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for k in sorted(_worst):
        print(f"largest rel_err {k}: {_worst[k]:.3g}")


@pytest.fixture(scope="module")
def mv():
    import mvsim_b200
    return mvsim_b200


@pytest.fixture(scope="module")
def ctx(mv):
    c = mv.Context(0)
    yield c
    c.close()


def _ref(oracle, case):
    if case.id not in _refs:
        vol, psf = case.arrays()
        _refs[case.id] = fft_cases.reference(oracle, vol, psf)
    return _refs[case.id]


def _view_ref(oracle, case, inc):
    key = (case.id, inc)
    if key not in _view_refs:
        vol, psf = case.arrays()
        _view_refs[key] = fft_cases.whole_view_reference(oracle, vol, psf, inc)
    return _view_refs[key]


def _planned_lines(ctx, case):
    """(2 * sx.n, sy.n, sz.n) of the library's own plan (one rank)"""
    from mvsim_b200._lib import check, dims3
    lib = ctx._lib
    h = C.c_void_p()
    check(lib.mvsim_slabconv_create(ctx.h, dims3(case.shape), dims3(case.kshape), 0, 1, C.byref(h)), ctx.h)
    try:
        info = (C.c_int64 * 8)()
        check(lib.mvsim_slabconv_info(h, info))
        return {"x": int(info[4]), "y": int(info[5]), "z": int(info[6])}, int(info[2])
    finally:
        lib.mvsim_slabconv_destroy(ctx.h, h)


@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_every_line_length_along_every_axis(mv, ctx, oracle, case):
    lines, y_blocks = _planned_lines(ctx, case)
    assert lines[case.axis] == case.line and y_blocks == 1
    vol, psf = case.arrays()
    got = mv.SimulateMultiViewDataset.convolve(vol, psf, ctx=ctx)
    err = rel_err(got, _ref(oracle, case))
    _note(f"stand-alone {case.axis}", err)
    assert err <= TOL_CONV


@pytest.mark.parametrize("inc", [2, 3, 5])
@pytest.mark.parametrize("case", Z_CASES, ids=[c.id for c in Z_CASES])
def test_whole_view_at_every_z_length(mv, ctx, oracle, case, inc):
    vol, psf = case.arrays()
    got = mv.SimulateMultiViewDataset.simulateView(vol, psf.copy(), 0, inc=inc, poissonSNR=-1.0, ctx=ctx, strict_reference=False)
    err = rel_err(got, _view_ref(oracle, case, inc))
    _note("whole view (automatic kernel)", err)
    assert err <= TOL_VIEW


@pytest.fixture(scope="module")
def emu():
    """the CPU emulator's predicates: which whole-view kernels fft_group.cu builds for a (length, inc) pair"""
    return fft_cases.build_emu(full=False)


@pytest.mark.parametrize("inc", [3, 5])
@pytest.mark.parametrize("n", fft_cases.whole_view_lengths())
def test_every_built_whole_view_kernel(mv, oracle, emu, n, inc):
    """MVSIM_OPT_Z_KERNEL 3 (polyphase where built), 1 (decimated inverse where built) and 2 (full spectral kernel): each against the
    reference; the number of distinct outputs is 1 + the kernels built for the pair, so each built kernel really ran."""
    poly_ok, dec_ok = emu.emu_poly_ok(n, inc) > 0, emu.emu_dec_ok(n, inc) > 0
    case = fft_cases.whole_view_case(n)
    vol, psf = case.arrays()
    ref = _view_ref(oracle, case, inc)
    outs = []
    for which, name in ((3, "polyphase"), (1, "decimated"), (2, "spectral")):
        ctx = mv.Context(0).z_kernel(which)
        outs.append(mv.SimulateMultiViewDataset.simulateView(vol, psf.copy(), 0, inc=inc, poissonSNR=-1.0, ctx=ctx,
                                                             strict_reference=False))
        ctx.close()
        err = rel_err(outs[-1], ref)
        _note(f"whole view (MVSIM_OPT_Z_KERNEL {which}, {name} where built)", err)
        assert err <= TOL_VIEW, which
    assert len({o.tobytes() for o in outs}) == 1 + int(poly_ok) + int(dec_ok)


@pytest.mark.parametrize("knob", ["MVSIM_H_MATERIALIZE", "MVSIM_NO_TMA"])
def test_process_wide_knobs(oracle, tmp_path, knob):
    """The stand-alone sweep and the whole-view call at every z length of the built range, in a process with the knob set."""
    out = tmp_path / "out.npz"
    env = dict(os.environ, **{knob: "1"})
    r = subprocess.run([sys.executable, os.path.join(HERE, "fft_sizes_worker.py"), str(out)], env=env, capture_output=True, text=True,
                       timeout=1800)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    got = np.load(out)
    bad = []
    for case in CASES:
        err = rel_err(got["conv_" + case.id], _ref(oracle, case))
        _note(f"{knob} stand-alone {case.axis}", err)
        if err > TOL_CONV:
            bad.append((case.id, err))
    for n in fft_cases.whole_view_lengths():
        case = fft_cases.whole_view_case(n)
        for inc in (3, 5):
            err = rel_err(got[f"view_{case.id}_{inc}"], _view_ref(oracle, case, inc))
            _note(f"{knob} whole view", err)
            if err > TOL_VIEW:
                bad.append((f"view {case.id} inc {inc}", err))
    assert not bad, bad
