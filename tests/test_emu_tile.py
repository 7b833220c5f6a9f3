"""The interval addressing of the sampler (csrc/tile.cuh, __host__ __device__) evaluated on the CPU: the parent offsets it gives
the tile's output voxels equal numpy's slicing parent[z0:z1+1:inc, y0:y1+1, x0:x1+1] -- extractSlices of
Views.zeroMin(Views.interval(parent, min, max)) -- for odd widths, unaligned row starts, every face of the parent, and parents
and tiles beyond 32-bit indices."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(os.path.dirname(HERE), "multiview-simulation_b200", "csrc")
SO = os.path.join(HERE, "emu", "libemu_tile.so")
SRC = os.path.join(HERE, "emu", "emu_tile.cpp")
_i64p = C.POINTER(C.c_int64)


@pytest.fixture(scope="module")
def emu():
    deps = [SRC, os.path.join(CSRC, "tile.cuh"), os.path.join(CSRC, "sampler.cuh"), os.path.join(CSRC, "fft", "fft_defs.cuh")]
    if not os.path.exists(SO) or os.path.getmtime(SO) < max(os.path.getmtime(d) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-fno-gnu-unique", "-Wl,-Bsymbolic", "-I", CSRC, SRC, "-o", SO])
    L = C.CDLL(SO)
    L.emu_tile_offsets.argtypes = [_i64p, _i64p, _i64p, C.c_int, C.POINTER(C.c_uint64), C.c_longlong, _i64p]
    return L


def _offsets(emu, dims, mn, mx, inc, i0s):
    i3 = C.c_int64 * 3
    i0s = np.ascontiguousarray(i0s, dtype=np.uint64)
    off = np.empty(4 * len(i0s), dtype=np.int64)
    emu.emu_tile_offsets(i3(*dims), i3(*mn), i3(*mx), inc, i0s.ctypes.data_as(C.POINTER(C.c_uint64)), len(i0s), off.ctypes.data_as(_i64p))
    return off


def _check_tile(emu, dims, mn, mx, inc):
    x, y, z = dims
    idx = np.arange(x * y * z, dtype=np.int64).reshape(z, y, x)
    want = idx[mn[2]:mx[2] + 1:inc, mn[1]:mx[1] + 1, mn[0]:mx[0] + 1].ravel()
    got = _offsets(emu, dims, mn, mx, inc, np.arange(0, want.size, 4))[:want.size]    # voxels past the end are not read
    assert np.array_equal(got, want), (dims, mn, mx, inc)


PARENTS = [(13, 11, 17), (16, 9, 12), (9, 5, 7)]       # (X, Y, Z): X % 4 != 0 and X % 4 == 0


@pytest.mark.parametrize("dims", PARENTS)
@pytest.mark.parametrize("inc", [1, 3, 5])
def test_interval_offsets_match_numpy_slicing(emu, dims, inc):
    X, Y, Z = dims
    for x0 in (0, 1, 3, 5):
        for w in sorted({1, 3, 4, 7, X - x0}):
            if x0 + w > X:
                continue
            # y / z ranges: the whole axis (both faces), an inner range, a range at the far face, a single plane at each face
            for y0, y1 in ((0, Y - 1), (1, Y - 2), (Y - 2, Y - 1), (0, 0), (Y - 1, Y - 1)):
                for z0, z1 in ((0, Z - 1), (2, Z - 3), (Z - 1, Z - 1), (0, 0), (Z - 4, Z - 1)):
                    _check_tile(emu, dims, (x0, y0, z0), (x0 + w - 1, y1, z1), inc)


def _formula(dims, mn, mx, inc, i):
    X, Y, _ = dims
    bx, by = mx[0] - mn[0] + 1, mx[1] - mn[1] + 1
    k, r = divmod(int(i), bx * by)
    yy, xx = divmod(r, bx)
    return mn[0] + xx + X * (mn[1] + yy + Y * (mn[2] + k * inc))


@pytest.mark.parametrize("dims,mn,mx,inc", [
    # a parent of 2^31 voxels and more, tile at its far corner, min0 % 4 == 3
    ((2051, 1031, 1100), (1027, 800, 600), (2050, 1030, 1099), 3),
    # tile plane 2^32 - 1 (the largest accepted) and 4 * (2^32 - 1) output voxels: the quotient by the plane needs 64 bits
    ((65540, 65540, 7), (3, 5, 0), (65539, 65539, 6), 2),
    # one-voxel rows and planes of a long z axis
    ((3, 2, 1 << 20), (2, 1, 5), (2, 1, (1 << 20) - 1), 1),
])
def test_interval_offsets_beyond_32_bits(emu, dims, mn, mx, inc):
    bx, by = mx[0] - mn[0] + 1, mx[1] - mn[1] + 1
    n_out = bx * by * ((mx[2] - mn[2]) // inc + 1)
    plane = bx * by
    rng = np.random.default_rng(5)
    starts = {0, (n_out - 1) // 4 * 4}
    for k in range(0, n_out // plane + 1, max(1, n_out // plane // 7)):
        for d in range(-8, 9):              # groups around every sampled plane boundary (straddling two planes when plane % 4 != 0)
            starts.add((k * plane + d) // 4 * 4)
    starts.update(int(v) // 4 * 4 for v in rng.integers(0, n_out, 2000, dtype=np.int64))
    starts = sorted(s for s in starts if 0 <= s < n_out)
    got = _offsets(emu, dims, mn, mx, inc, starts).reshape(-1, 4)
    for s, row in zip(starts, got):
        for j in range(4):
            if s + j < n_out:
                assert row[j] == _formula(dims, mn, mx, inc, s + j), (s, j)
