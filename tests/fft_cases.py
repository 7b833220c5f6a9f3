"""Convolution cases that make the planner pick every FFT line length the library ships, along every axis that length serves.

The size table is read from the text of multiview-simulation_b200/csrc/fft/conv_plan.h (the X(n, a, b) entries of the
MVSIM_FFT_SIZES_* lists), so a length added there is covered without editing a test.  Shared by the CPU emulation sweep
(test_emu_fft_sizes.py) and the GPU sweep (test_gpu_fft_sizes.py), together with the build of the CPU emulator (also used by
test_emu_conv.py).

For a length n and an axis (x only for n % 8 == 0: the x pass folds a real line of 2n points into n complex ones), with
L = n (2n on x) and P = the previous length the planner could pick on that axis (0 for the first), three cases:
  a  long image, even short kernel (8 taps)
  b  long image, odd short kernel (7 taps)
  c  5 voxels along the axis, a kernel of L - 4 taps: the mirror extension folds many times and the PSF line is longer
     than the pruned sub-transform reads
where image dim + kernel dim - 1 lies in (P, L], so the planner picks exactly n.  On x, (a) has X % 4 == 0 and (b) odd X
(the x passes take an L2-prefetch branch on X % 4).  The two other axes are small (5 / 3 voxels or so, 3- and 2-tap kernels)
and chosen so that the x pass's row count is not a multiple of its rows per CTA.
"""
import ctypes as C
import os
import re
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(ROOT, "multiview-simulation_b200", "csrc")
PLAN_H = os.path.join(CSRC, "fft", "conv_plan.h")
EMU_SRC = os.path.join(HERE, "emu", "emu_conv.cpp")

AXES = ("z", "y", "x")                  # index into a (Z, Y, X) shape
KINDS = ("a", "b", "c")
X_THREADS_FWD, X_THREADS_INV = 144, 192     # kXThreadsFwd / kXThreadsInv of conv_plan.h


def size_table(path=PLAN_H):
    """[(n, a, b)] ascending: every entry of the MVSIM_FFT_SIZES_* lists (the full table the library is built with)."""
    text = open(path).read().replace("\\\n", " ")
    out = set()
    for m in re.finditer(r"^#define MVSIM_FFT_SIZES_\w+\(X\)(.*)$", text, re.M):
        out.update((int(n), int(a), int(b)) for n, a, b in re.findall(r"X\((\d+),\s*(\d+),\s*(\d+)\)", m.group(1)))
    return sorted(out)


def whole_view_range(path=PLAN_H):
    """(kDecMinLine, kDecMaxLine): the z line lengths for which the decimated and polyphase fused z kernels are built"""
    m = re.search(r"kDecMinLine\s*=\s*(\d+),\s*kDecMaxLine\s*=\s*(\d+)", open(path).read())
    return int(m.group(1)), int(m.group(2))


def whole_view_lengths(table=None):
    lo, hi = whole_view_range()
    return [n for n, _, _ in (table or size_table()) if lo <= n <= hi]


def _rows_per_cta(split, inverse):
    a, b = split
    return max((X_THREADS_INV if inverse else X_THREADS_FWD) // max(a, b), 1)


class Case:
    def __init__(self, axis, n, kind, shape, kshape, seed):
        self.axis, self.n, self.kind, self.shape, self.kshape, self.seed = axis, n, kind, shape, kshape, seed

    @property
    def id(self):
        return f"{self.axis}{self.n}{self.kind}"

    @property
    def line(self):
        """the padded line the planner must pick along the case's axis: 2n real points on x, n otherwise"""
        return 2 * self.n if self.axis == "x" else self.n

    def arrays(self):
        """seeded random positive image and PSF (float32, (Z, Y, X))"""
        rng = np.random.default_rng(self.seed)
        vol = (0.25 + rng.random(self.shape)).astype(np.float32)
        psf = (0.25 + rng.random(self.kshape)).astype(np.float32)
        return vol, psf

    def __repr__(self):
        return f"Case({self.id}, shape={self.shape}, kshape={self.kshape})"


# small dims of the two other axes, (5, 3) first, then by voxel count; kernels 3 and 2 taps
_SMALL = [(5, 3)] + sorted(((p, q) for p in range(3, 10) for q in range(3, 8)), key=lambda t: (t[0] * t[1], t))


def cases(table=None):
    """Every (axis, n, kind) case: 3 per length along y and z, 3 per multiple-of-8 length along x."""
    table = table or size_table()
    out = []
    for ai, axis in enumerate(AXES):
        lens = [t for t in table if axis != "x" or t[0] % 8 == 0]
        prev = 0
        for n, a, b in lens:
            L = 2 * n if axis == "x" else n
            P = 2 * prev if axis == "x" else prev
            if axis == "x":
                long = {"a": (L - 8, 8), "b": (L - 7, 7)}            # X + KX - 1 = L - 1: X % 4 == 0 resp. X odd
            else:
                long = {"a": (L - 7, 8), "b": (L - 6 if L - 1 > P else L - 7, 7)}     # (b) one point of padding where possible
            long["c"] = (5, L - 4)
            for ki, kind in enumerate(KINDS):
                d0, k = long[kind]
                # x split of the case: the x-axis length itself, else the smallest multiple-of-8 length (X <= 9 here)
                xsplit = (a, b) if axis == "x" else next((ta, tb) for tn, ta, tb in table if tn % 8 == 0)
                rf, ri = _rows_per_cta(xsplit, False), _rows_per_cta(xsplit, True)
                found = None
                # the preferred long dim first; on y / z a neighbour when no small dims avoid a whole number of CTAs
                for d in [d0] + ([] if axis == "x" or kind == "c" else [d0 - 1, d0 + 1]):
                    if not P < d + k - 1 <= L:
                        continue
                    for s1, s2 in _SMALL:
                        shape, kshape = [0, 0, 0], [0, 0, 0]
                        shape[ai], kshape[ai] = d, k
                        others = [i for i in range(3) if i != ai]
                        shape[others[0]], kshape[others[0]] = s1, 3
                        shape[others[1]], kshape[others[1]] = s2, 2
                        rows = shape[0] * shape[1]                   # x pass rows: Z * Y
                        if rows % rf and rows % ri:
                            found = (tuple(shape), tuple(kshape))
                            break
                    if found:
                        break
                assert found, f"no dims for {axis}{n}{kind}"
                out.append(Case(axis, n, kind, found[0], found[1], seed=100000 + 1000 * ai + 3 * n + ki))
            prev = n
    return out


def z_cases(table=None):
    return [c for c in cases(table) if c.axis == "z"]


def whole_view_case(n):
    """Long image along z (the (a) case of length n): short kernel, single mirror fold, image line longer than the PSF line --
    every whole-view fused z kernel built for n accepts it."""
    return next(c for c in z_cases() if c.n == n and c.kind == "a")


def reference(oracle, vol, psf):
    """float64 direct sum (the oracle's direct path); normalises a copy of psf"""
    return oracle.convolve(vol, psf.copy(), "direct")


def whole_view_reference(oracle, vol, psf, inc):
    """simulateView(vol, psf, 0, inc, poissonSNR=-1, strict_reference=False): 0 deg rotation is the identity, corrected
    attenuation, convolution, adjustImage, every inc-th plane"""
    c = oracle.convolve(oracle.attenuate(vol, 0.01, strict=False), psf.copy(), "direct")
    oracle.adjust(c)
    return np.ascontiguousarray(c[::inc])


# ---- the CPU emulator (tests/emu/emu_conv.cpp) -----------------------------------------------------------------------------
def build_emu(full):
    """libemu_conv.so (small size table) or libemu_conv_full.so (-DMVSIM_EMU_FULL_TABLE: the library's table), rebuilt when a
    source is newer."""
    so = os.path.join(HERE, "emu", "libemu_conv_full.so" if full else "libemu_conv.so")
    deps = [EMU_SRC] + [os.path.join(CSRC, "fft", f) for f in os.listdir(os.path.join(CSRC, "fft"))]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps):
        # -fno-gnu-unique / -Bsymbolic: the emulator's inline statics (size table) must not become process-wide unique symbols
        # that libmvsim.so (loaded later in the same pytest process) or the other emulator build would bind to
        tmp = f"{so}.{os.getpid()}.tmp"
        try:
            subprocess.check_call(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-fno-gnu-unique", "-Wl,-Bsymbolic"] +
                                  (["-DMVSIM_EMU_FULL_TABLE=1"] if full else []) + ["-I", CSRC, EMU_SRC, "-o", tmp])
            os.replace(tmp, so)
        finally:
            if os.path.exists(tmp):
                os.remove(tmp)
    L = C.CDLL(so)
    i64p, fp = C.POINTER(C.c_int64), C.POINTER(C.c_float)
    L.emu_convolve.argtypes = [fp, i64p, fp, i64p, fp, C.POINTER(C.c_double), C.c_int, C.c_int, C.c_int, C.c_int]
    L.emu_plan.argtypes = [i64p, i64p, C.POINTER(C.c_int), C.c_int]
    for f in ("emu_poly_ok", "emu_dec_ok"):
        getattr(L, f).argtypes = [C.c_int, C.c_int]
        getattr(L, f).restype = C.c_int
    L.emu_regfft.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, fp, fp]
    L.emu_regfft_pz_k.argtypes = [C.c_int]
    for f in ("emu_decimated_launches", "emu_polyphase_launches", "emu_last_sum_plane_is_total"):
        getattr(L, f).restype = C.c_int
    return L


def built_z_pairs(emu, table=None):
    """{(n, inc): (poly_ok, dec_ok)} for every pair for which fft_group.cu builds a polyphase or a decimated fused z kernel"""
    table = table or size_table()
    out = {}
    for n, _, _ in table:
        for inc in (2, 3, 5):
            p, d = emu.emu_poly_ok(n, inc) > 0, emu.emu_dec_ok(n, inc) > 0
            if p or d:
                out[(n, inc)] = (p, d)
    return out
