"""The row / tap arithmetic of the rotation about x, the attenuation and the aligned outputs (csrc/post.cuh, __host__ __device__)
evaluated on the CPU against the oracle's stage chain: rotate(v, 0, d) for the bounds-tested rotation, attenuate(rotate(v, 0, d))
for the offset-table march of the whole-view call, rotate(make_isotropic(acq, inc), 0, d) for the aligned view and
normalize_weights(rotate(weight_image(dims), 0, d_v)) for the aligned weights."""
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
    L.emu_rotate_axis0.argtypes = [_fp, C.c_int, C.c_int, C.c_int, _dp, _fp]
    L.emu_rotate_attenuate_off.argtypes = [_fp, C.c_int, C.c_int, C.c_int, _dp, C.c_double, C.c_int, _fp]
    L.emu_align_view.argtypes = [_fp, C.c_int, C.c_int, C.c_int, C.c_int, _dp, _fp]
    L.emu_aligned_weights.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, _dp, C.c_float, C.POINTER(_fp), _fp]
    return L


def _inverse(oracle, shape_zyx, degrees):
    z, y, x = shape_zyx
    return np.ascontiguousarray(oracle.affine_invert(oracle.axis_rotation((x, y, z), 0, degrees)), dtype=np.float64)


def _err(a, b):
    return float(np.max(np.abs(a.astype(np.float64) - b)) / max(1e-30, float(np.max(np.abs(b)))))


def _emu_rotate(emu, oracle, v, degrees):
    z, y, x = v.shape
    out = np.empty_like(v)
    emu.emu_rotate_axis0(v.ctypes.data_as(_fp), x, y, z, _inverse(oracle, v.shape, degrees).ctypes.data_as(_dp), out.ctypes.data_as(_fp))
    return out


SHAPES = [(7, 13, 6), (5, 9, 5), (6, 11, 4), (1, 8, 3), (4, 10, 7)]     # (Z, Y, X) with X <= Y: strict attenuation applies
ANGLES = [0, 52, -52, 90, 180, 315]


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("degrees", ANGLES)
def test_rotate_axis0_matches_oracle(emu, oracle, shape, degrees):
    v = np.random.default_rng(43).random(shape, dtype=np.float32)
    assert _err(_emu_rotate(emu, oracle, v, degrees), oracle.rotate(v, 0, degrees)) <= 1e-6


# the offset table reads row (0, 0) for out-of-volume taps with weight 0: bit-identical to the bounds-tested rotation followed by
# attenuate for non-negative data
@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("degrees", ANGLES)
@pytest.mark.parametrize("strict,delta", [(True, 0.01), (False, 0.01), (True, 0.5), (False, 0.5)])
def test_offset_table_march_equals_rotate_then_attenuate(emu, oracle, shape, degrees, strict, delta):
    v = np.random.default_rng(47).random(shape, dtype=np.float32) * 3
    z, y, x = shape
    got = np.empty_like(v)
    emu.emu_rotate_attenuate_off(v.ctypes.data_as(_fp), x, y, z, _inverse(oracle, shape, degrees).ctypes.data_as(_dp), delta,
                                 x if strict else y, got.ctypes.data_as(_fp))
    ref = oracle.attenuate(_emu_rotate(emu, oracle, v, degrees), delta, strict=strict)
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))


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
