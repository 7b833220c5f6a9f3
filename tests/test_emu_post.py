"""The row / tap arithmetic of the aligned outputs (csrc/post.cuh, __host__ __device__) evaluated on the CPU against the oracle's
stage chain: rotate(make_isotropic(acq, inc), 0, d) for the aligned view, normalize_weights(rotate(weight_image(dims), 0, d_v))
for the aligned weights."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(os.path.dirname(HERE), "multiview-simulation_b200", "csrc")
SO = os.path.join(HERE, "emu", "libemu_post.so")
SRC = os.path.join(HERE, "emu", "emu_post.cpp")
_fp = C.POINTER(C.c_float)
_dp = C.POINTER(C.c_double)


@pytest.fixture(scope="module")
def emu():
    deps = [SRC, os.path.join(CSRC, "post.cuh"), os.path.join(CSRC, "fft", "fft_defs.cuh")]
    if not os.path.exists(SO) or os.path.getmtime(SO) < max(os.path.getmtime(d) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-fno-gnu-unique", "-Wl,-Bsymbolic", "-I", CSRC, SRC, "-o", SO])
    L = C.CDLL(SO)
    L.emu_align_view.argtypes = [_fp, C.c_int, C.c_int, C.c_int, C.c_int, _dp, _fp]
    L.emu_aligned_weights.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, _dp, C.c_float, C.POINTER(_fp), _fp]
    return L


def _inverse(oracle, shape_zyx, degrees):
    z, y, x = shape_zyx
    return np.ascontiguousarray(oracle.affine_invert(oracle.axis_rotation((x, y, z), 0, degrees)), dtype=np.float64)


def _err(a, b):
    return float(np.max(np.abs(a.astype(np.float64) - b)) / max(1e-30, float(np.max(np.abs(b)))))


@pytest.mark.parametrize("shape,inc", [((7, 13, 6), 3), ((5, 9, 5), 5), ((6, 11, 4), 1), ((1, 8, 3), 3), ((4, 10, 7), 4)])
@pytest.mark.parametrize("degrees", [0, 52, -52, 90, 180, 315])
def test_align_view_matches_oracle_chain(emu, oracle, shape, inc, degrees):
    acq = np.random.default_rng(41).random(shape, dtype=np.float32)
    za, y, x = shape
    iso_shape = ((za - 1) * inc + 1, y, x)
    out = np.empty(iso_shape, dtype=np.float32)
    inv = _inverse(oracle, iso_shape, degrees)
    emu.emu_align_view(acq.ctypes.data_as(_fp), x, y, za, inc, inv.ctypes.data_as(_dp), out.ctypes.data_as(_fp))
    ref = oracle.rotate(oracle.make_isotropic(acq, inc), 0, degrees)
    assert _err(out, ref) <= 1e-6


@pytest.mark.parametrize("n_all", [1, 3, 7, 16])
def test_aligned_weights_match_oracle_chain(emu, oracle, n_all):
    shape = (23, 101, 3)                     # Y > 2 * 40: the taper and both flat parts are present
    angles = [-(k * (360 // n_all)) for k in range(n_all)]
    z, y, x = shape
    inv = np.concatenate([_inverse(oracle, shape, d).reshape(-1) for d in angles])
    outs = [np.empty(shape, dtype=np.float32) for _ in range(n_all)]
    s = np.empty(shape, dtype=np.float32)
    emu.emu_aligned_weights(x, y, z, n_all, inv.ctypes.data_as(_dp), 3.0, (_fp * n_all)(*[o.ctypes.data_as(_fp) for o in outs]),
                            s.ctypes.data_as(_fp))
    ref = [oracle.rotate(oracle.weight_image(shape), 0, d) for d in angles]
    s_ref = oracle.normalize_weights(ref, 3.0)
    for a, b in zip(outs, ref):
        assert _err(a, b) <= 1e-6
    assert _err(s, s_ref) <= 1e-6
    assert np.all(outs[0] == outs[0][:, :, :1])          # constant along x
