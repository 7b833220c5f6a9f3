"""Host-side mirror of the reference's public static methods for the per-view acquisition path.

Same names, argument meaning and side effects as the Java originals (S = src/main/java/net/
preibisch/simulation), over numpy float32 volumes of shape (Z, Y, X) -- the ArrayImg float[] in
x-fastest order.  Every body is a call through the C ABI of libmvsim.so (include/mvsim.h), exactly
what the JNI facade in INTEGRATION.md does on the Java side.  There is no CPU implementation here.

    SimulateMultiViewDataset.axisRotation      S/SimulateMultiViewDataset.java:80
    SimulateMultiViewDataset.rotateAroundAxis  S/SimulateMultiViewDataset.java:104
    SimulateMultiViewDataset.attenuate3d       S/SimulateMultiViewDataset.java:318
    SimulateMultiViewDataset.convolve          S/SimulateMultiViewDataset.java:253
    SimulateMultiViewDataset.extractSlices     S/SimulateMultiViewDataset.java:181,195
    SimulateMultiViewDataset.poissonProcess    S/SimulateMultiViewDataset.java:233
    Tools.normImage / adjustImage / poissonProcess   S/Tools.java:112,143,73
Input generators either side of the path (SURVEY section 8f):
    SimulateMultiViewDataset.simulate / drawSpheres / downSample2x   S/SimulateMultiViewDataset.java:366-522
    SimulateBeads.randomPoints / transformPoints / renderPoints      S/SimulateBeads.java:97-205
    Tools.makeSquare                                                 S/Tools.java:315
"""
import ctypes as C
import threading

import numpy as np

from . import _lib
from ._lib import DatasetOutputs, MvsimError, ViewParams, check, dims3, fptr


class JavaRandom:
    """java.util.Random (JDK specification): the RNG type the reference's signatures take.  The GPU
    sampler is counter based (Philox); like the Java facade, the mirror only draws ONE nextLong()
    from the caller's generator to key it, so results stay reproducible from the caller's seed."""

    def __init__(self, seed):
        self._s = (int(seed) ^ 0x5DEECE66D) & ((1 << 48) - 1)

    def _next(self, bits):
        self._s = (self._s * 0x5DEECE66D + 0xB) & ((1 << 48) - 1)
        v = self._s >> (48 - bits)
        return v - (1 << bits) if v >= (1 << (bits - 1)) else v

    def nextInt(self):
        return self._next(32)

    def nextLong(self):
        v = (self._next(32) << 32) + self._next(32)
        v &= (1 << 64) - 1
        return v - (1 << 64) if v >= (1 << 63) else v

    def nextDouble(self):
        return ((self._next(26) % (1 << 26) << 27) + (self._next(27) % (1 << 27))) * 2.0 ** -53


class Context:
    """One CUDA device + stream + cached workspaces (mvsim_ctx).  Not shared between threads."""

    def __init__(self, device=0, cuda_stream=None):
        """cuda_stream: None = own stream; an int cudaStream_t handle (0 = legacy default stream) = enqueue there."""
        self._lib = _lib.load()
        h = C.c_void_p()
        if cuda_stream is None:
            check(self._lib.mvsim_ctx_create(device, C.byref(h)))
        else:
            check(self._lib.mvsim_ctx_create_on_stream(device, C.c_void_p(cuda_stream), C.byref(h)))
        self.h = h
        self.device = device

    def close(self):
        if self.h:
            self._lib.mvsim_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def synchronize(self):
        check(self._lib.mvsim_ctx_synchronize(self.h), self.h)

    def profile(self, on=True):
        check(self._lib.mvsim_profile_enable(self.h, int(on)), self.h)
        check(self._lib.mvsim_profile_reset(self.h), self.h)

    def stage_times(self):
        ms = (C.c_double * _lib.NSTAGES)()
        n = (C.c_int64 * _lib.NSTAGES)()
        check(self._lib.mvsim_stage_times(self.h, ms, n), self.h)
        return {k: (ms[i], n[i]) for i, k in enumerate(_lib.STAGE_NAMES)}

    @property
    def kernel_launches(self):
        return int(self._lib.mvsim_kernel_launches(self.h))

    def count_transport(self, uint16=True, host_threads=0):
        """Batch calls (simulateViews): move the Poisson counts over the host link as uint16 and widen them to float32 on host
        threads inside the call (mvsim_ctx_set_option MVSIM_OPT_COUNT_TRANSPORT).  Bit-identical results, half the D2H bytes."""
        check(self._lib.mvsim_ctx_set_option(self.h, _lib.OPT_HOST_THREADS, int(host_threads)), self.h)
        check(self._lib.mvsim_ctx_set_option(self.h, _lib.OPT_COUNT_TRANSPORT, int(bool(uint16))), self.h)
        return self

    def z_kernel(self, which=0):
        """Fused z pass of the whole-view calls (mvsim_ctx_set_option MVSIM_OPT_Z_KERNEL): 0 = the kernel measured fastest for the
        shape, 1 = decimated inverse / full spectral (no polyphase kernel), 2 = full spectral kernel only, 3 = polyphase kernel."""
        check(self._lib.mvsim_ctx_set_option(self.h, _lib.OPT_Z_KERNEL, int(which)), self.h)
        return self

    def psf_cache(self, max_bytes):
        """PSF-spectrum cache of this context (mvsim_psf_cache_configure): keep the spectra of repeated PSFs in up to
        `max_bytes` of HBM (0 = off, the library default: the reference rebuilds the kernel FFT per call, :257)."""
        check(self._lib.mvsim_psf_cache_configure(self.h, int(max_bytes)), self.h)
        return self

    def psf_cache_stats(self):
        st = (C.c_int64 * 4)()
        check(self._lib.mvsim_psf_cache_stats(self.h, st), self.h)
        return {"hits": int(st[0]), "misses": int(st[1]), "entries": int(st[2]), "bytes": int(st[3])}


_tls = threading.local()


def default_context():
    """Per-thread context on device 0 (the reference's callers invoke the path from 2 threads)."""
    ctx = getattr(_tls, "ctx", None)
    if ctx is None:
        ctx = _tls.ctx = Context(0)
    return ctx


def _vol(a, name="img"):
    a = np.ascontiguousarray(a, dtype=np.float32)
    if a.ndim != 3:
        raise ValueError(f"{name}: expected a 3-D (Z, Y, X) volume")
    return a


def _inplace(a, name):
    if not (isinstance(a, np.ndarray) and a.dtype == np.float32 and a.flags.c_contiguous and a.flags.writeable):
        raise ValueError(f"{name}: in-place argument must be a writable C-contiguous float32 ndarray")
    return a


def _seed_from(rnd):
    if rnd is None:
        rnd = SimulateMultiViewDataset.rnd
    if isinstance(rnd, (int, np.integer)):
        return int(rnd) & ((1 << 64) - 1)
    draw = getattr(rnd, "nextLong", None) or getattr(rnd, "next_long")
    return int(draw()) & ((1 << 64) - 1)


class PinnedBuffer:
    """Pinned off-heap float buffer (mvsim_alloc_pinned) exposed as a numpy array."""

    def __init__(self, shape):
        self.shape = tuple(int(s) for s in shape)
        n = int(np.prod(self.shape))
        self._p = C.c_void_p()
        check(_lib.load().mvsim_alloc_pinned(max(n, 1) * 4, C.byref(self._p)))
        self.array = np.ctypeslib.as_array(C.cast(self._p, C.POINTER(C.c_float)), shape=(max(n, 1),))[:n].reshape(self.shape)

    def free(self):
        if self._p:
            self.array = None
            _lib.load().mvsim_free_pinned(self._p)
            self._p = None


class DeviceVolume:
    """Device-resident float32 volume (mvsim_volume): keeps a convolved view in HBM for SNR sweeps
    like S/SimulateTileStitching.java:131-189."""

    def __init__(self, ctx, shape_zyx, host=None):
        self.ctx = ctx
        self.shape = tuple(int(s) for s in shape_zyx)
        self.h = C.c_void_p()
        check(ctx._lib.mvsim_volume_create(ctx.h, dims3(self.shape), C.byref(self.h)), ctx.h)
        if host is not None:
            self.upload(host)

    @classmethod
    def wrap(cls, ctx, shape_zyx, device_ptr, keepalive=None):
        """Non-owning handle over device memory of the caller (mvsim_volume_wrap), e.g. `tensor.data_ptr()` of a torch tensor
        that an NCCL broadcast fills; `keepalive` holds the owner."""
        self = cls.__new__(cls)
        self.ctx = ctx
        self.shape = tuple(int(s) for s in shape_zyx)
        self.h = C.c_void_p()
        self._keepalive = keepalive
        check(ctx._lib.mvsim_volume_wrap(ctx.h, dims3(self.shape), C.c_void_p(int(device_ptr)), C.byref(self.h)), ctx.h)
        return self

    def upload(self, host):
        host = _vol(host)
        if host.shape != self.shape:
            raise ValueError("shape mismatch")
        check(self.ctx._lib.mvsim_volume_upload(self.ctx.h, self.h, fptr(host)), self.ctx.h)
        self.ctx.synchronize()      # host may be pageable / temporary
        return self

    def download(self, out=None):
        out = np.empty(self.shape, dtype=np.float32) if out is None else out
        check(self.ctx._lib.mvsim_volume_download(self.ctx.h, self.h, fptr(out)), self.ctx.h)
        self.ctx.synchronize()
        return out

    @property
    def device_ptr(self):
        return self.ctx._lib.mvsim_volume_device_ptr(self.h)

    def free(self):
        if self.h:
            self.ctx._lib.mvsim_volume_free(self.ctx.h, self.h)
            self.h = None

    def extractSlices(self, inc, poissonSNR, rnd=None, stream=0, interval=None, out=None):
        """extractSlices (:195-231) on the device: every inc-th plane, Poisson noise when poissonSNR >= 0.  interval = (min_xyz,
        max_xyz), inclusive (SimulateTileStitching.getInterval's form), samples Views.zeroMin(Views.interval(self, min, max))
        (S/SimulateTileStitching.java:152-153,174) in place, without a dense copy of the tile (mvsim_dev_extract_interval); the
        result equals extractSlices of the dense cut, bit for bit.  None = the whole volume (mvsim_dev_extract_slices).  The seed
        is drawn like SimulateMultiViewDataset.extractSlices.  Returns `out` or a new DeviceVolume of ((bz-1)//inc+1, by, bx)."""
        if inc < 1:
            raise MvsimError(_lib.MVSIM_EINVAL, "inc must be >= 1")
        seed = _seed_from(rnd) if poissonSNR >= 0 else 0
        if interval is None:
            z, y, x = self.shape
            out = DeviceVolume(self.ctx, ((z - 1) // inc + 1, y, x)) if out is None else out
            check(self.ctx._lib.mvsim_dev_extract_slices(self.ctx.h, self.h, int(inc), float(poissonSNR), seed, int(stream), out.h),
                  self.ctx.h)
            return out
        mn, mx = (tuple(int(v) for v in t) for t in interval)
        new = out is None
        if new:
            out = DeviceVolume(self.ctx, ((mx[2] - mn[2]) // inc + 1, mx[1] - mn[1] + 1, mx[0] - mn[0] + 1))
        i3 = C.c_int64 * 3
        try:
            check(self.ctx._lib.mvsim_dev_extract_interval(self.ctx.h, self.h, i3(*mn), i3(*mx), int(inc), float(poissonSNR), seed,
                                                           int(stream), out.h), self.ctx.h)
        except MvsimError:
            if new:
                out.free()
            raise
        return out

    def alignView(self, inc, degrees, out=None):
        """rotateAroundAxis(makeIsotropic(self, inc), 0, degrees) (:588, :591) of this acquired view, gathered on the device
        without the isotropic volume (mvsim_dev_align_view); returns `out` or a new DeviceVolume of ((Za-1)*inc+1, Y, X)."""
        za, y, x = self.shape
        out = DeviceVolume(self.ctx, ((za - 1) * inc + 1, y, x)) if out is None else out
        check(self.ctx._lib.mvsim_dev_align_view(self.ctx.h, self.h, int(inc), int(degrees), out.h), self.ctx.h)
        return out

    @staticmethod
    def alignedWeights(ctx, shape_zyx, align_degrees, osem, views=None, sum_weights=False):
        """The normalised rotate-back weight images of a dataset whose views are rotated back by `align_degrees` (all of them:
        the normalisation needs every angle), computed from the dims alone (mvsim_dev_aligned_weights).  Returns the DeviceVolumes
        of `views` (default: all) and, with sum_weights=True, the sum image as a last element."""
        n_all = len(align_degrees)
        views = list(range(n_all)) if views is None else [int(v) for v in views]
        outs = [DeviceVolume(ctx, shape_zyx) for _ in views]
        s = DeviceVolume(ctx, shape_zyx) if sum_weights else None
        i32 = C.c_int32
        oarr = (C.c_void_p * max(len(outs), 1))(*[o.h.value for o in outs])
        check(ctx._lib.mvsim_dev_aligned_weights(ctx.h, dims3(shape_zyx), n_all, (i32 * n_all)(*[int(d) for d in align_degrees]), float(osem),
                                                 len(views), (i32 * max(len(views), 1))(*views), oarr, s.h if s else None), ctx.h)
        return outs + ([s] if s else [])


def make_view_params(shape_zyx, kshape_zyx, axis=0, degrees=15, delta=0.01, min_value=0.0001, target_avg=1.0, inc=3,
                     snr=25.0, seed=0, stream=0, strict_reference=True):
    p = ViewParams()
    p.dims = dims3(shape_zyx)
    p.kdims = dims3(kshape_zyx)
    p.axis, p.degrees, p.delta = axis, degrees, delta
    p.min_value, p.target_avg, p.inc, p.snr = min_value, target_avg, inc, snr
    p.seed, p.stream = seed & ((1 << 64) - 1), stream
    p.strict_reference = int(strict_reference)
    return p


class Tools:
    @staticmethod
    def normImage(img, ctx=None):
        """In place: sum becomes 1 (S/Tools.java:112-118).  Returns None like the reference."""
        ctx = ctx or default_context()
        _inplace(img, "img")
        s = C.c_double()
        shape = img.shape if img.ndim == 3 else (1, 1, img.size)
        check(ctx._lib.mvsim_psf_normalize(ctx.h, fptr(img), dims3(shape), C.byref(s)), ctx.h)

    @staticmethod
    def adjustImage(image, minValue, targetAverage, ctx=None):
        """In place; returns the factor all intensities were multiplied with (S/Tools.java:143-159)."""
        ctx = ctx or default_context()
        _inplace(image, "image")
        c = C.c_double()
        shape = image.shape if image.ndim == 3 else (1, 1, image.size)
        check(ctx._lib.mvsim_adjust(ctx.h, fptr(image), dims3(shape), minValue, targetAverage, C.byref(c)), ctx.h)
        return c.value

    @staticmethod
    def poissonProcess(img, SNR, rnd, ctx=None, stream=0):
        """In place Poisson noise, lambda = v * (SNR/sqrt 5)^2, raw counts (S/Tools.java:73-86)."""
        ctx = ctx or default_context()
        _inplace(img, "img")
        check(ctx._lib.mvsim_poisson(ctx.h, fptr(img), img.size, float(SNR), _seed_from(rnd), stream), ctx.h)


def _phantom_seed(rnd):
    """Seed whose fresh java.util.Random equals the caller's generator: an int is a seed, a JavaRandom contributes its
    current state (the replay then continues the caller's stream; the caller's object itself is not advanced)."""
    if rnd is None:
        return 464232194                 # the class-static generator (:76), as on the first call of simulate()
    if isinstance(rnd, JavaRandom):
        return rnd._s ^ 0x5DEECE66D
    return int(rnd)


def _tools_make_square(img, ctx=None):
    """Tools.makeSquare (S/Tools.java:315-349): centre-pad to the cube of the largest dimension with the minimum."""
    ctx = ctx or default_context()
    img = _vol(img)
    m = max(img.shape)
    out = np.empty((m, m, m), dtype=np.float32)
    check(ctx._lib.mvsim_make_square(ctx.h, fptr(img), dims3(img.shape), fptr(out)), ctx.h)
    return out


Tools.makeSquare = staticmethod(_tools_make_square)


class SimulateMultiViewDataset:
    seed = 464232194
    rnd = JavaRandom(seed)          # static generator of the reference (:76)
    minValue = 0.0001               # :77
    avgIntensity = 1.0              # :78

    @staticmethod
    def axisRotation(shape_zyx, axis, degrees):
        """3x4 forward model T(+c) R T(-c), c = (dim-1)//2 (:80-102).  Returns (forward, inverse)."""
        fwd, inv = (C.c_double * 12)(), (C.c_double * 12)()
        check(_lib.load().mvsim_axis_rotation(dims3(shape_zyx), axis, degrees, fwd, inv))
        return np.array(fwd[:]).reshape(3, 4), np.array(inv[:]).reshape(3, 4)

    @staticmethod
    def rotateAroundAxis(img, axis, degrees, ctx=None):
        ctx = ctx or default_context()
        img = _vol(img)
        out = np.empty_like(img)
        check(ctx._lib.mvsim_rotate_axis(ctx.h, fptr(img), fptr(out), dims3(img.shape), axis, int(degrees)), ctx.h)
        return out

    @staticmethod
    def attenuate3d(img, delta, ctx=None, strict_reference=True):
        ctx = ctx or default_context()
        img = _vol(img)
        out = np.empty_like(img)
        check(ctx._lib.mvsim_attenuate(ctx.h, fptr(img), fptr(out), dims3(img.shape), float(delta), int(strict_reference)), ctx.h)
        return out

    @staticmethod
    def convolve(img, psf, service=None, ctx=None):
        """`psf` is normalised IN PLACE (:255); `service` (the ExecutorService) is accepted and ignored."""
        ctx = ctx or default_context()
        img = _vol(img)
        _inplace(psf, "psf")
        if psf.ndim != 3:
            raise ValueError("psf: expected a 3-D volume")
        out = np.empty_like(img)
        check(ctx._lib.mvsim_convolve(ctx.h, fptr(img), dims3(img.shape), fptr(psf), dims3(psf.shape), fptr(out)), ctx.h)
        return out

    @staticmethod
    def extractSlices(img, inc, poissonSNR, rnd=None, ctx=None, stream=0):
        ctx = ctx or default_context()
        img = _vol(img)
        if inc < 1:
            raise MvsimError(_lib.MVSIM_EINVAL, "inc must be >= 1")
        z, y, x = img.shape
        out = np.empty(((z - 1) // inc + 1, y, x), dtype=np.float32)
        seed = _seed_from(rnd) if poissonSNR >= 0 else 0
        check(ctx._lib.mvsim_extract_slices(ctx.h, fptr(img), dims3(img.shape), inc, poissonSNR, seed, stream, fptr(out)), ctx.h)
        return out

    @staticmethod
    def poissonProcess(img, poissonSNR, rnd, ctx=None, stream=0):
        """Returns a noisy copy (:233-251)."""
        out = np.array(img, dtype=np.float32, order="C", copy=True)
        Tools.poissonProcess(out, poissonSNR, rnd, ctx=ctx, stream=stream)
        return out

    @staticmethod
    def simulateView(gt, psf, degrees, axis=0, delta=0.01, inc=3, poissonSNR=25.0, rnd=None, ctx=None, stream=0,
                     strict_reference=True):
        """Fused loop body :570-585 (rotate, attenuate, convolve, adjustImage, extractSlices) with all
        intermediates resident on the device.  `psf` is normalised in place."""
        ctx = ctx or default_context()
        gt = _vol(gt, "gt")
        _inplace(psf, "psf")
        z, y, x = gt.shape
        out = np.empty(((z - 1) // inc + 1, y, x), dtype=np.float32)
        p = make_view_params(gt.shape, psf.shape, axis, int(degrees), delta, SimulateMultiViewDataset.minValue,
                             SimulateMultiViewDataset.avgIntensity, inc, poissonSNR,
                             _seed_from(rnd) if poissonSNR >= 0 else 0, stream, strict_reference)
        check(ctx._lib.mvsim_simulate_view(ctx.h, C.byref(p), fptr(gt), fptr(psf), fptr(out)), ctx.h)
        return out

    @staticmethod
    def makeIsotropic(img, inc, ctx=None):
        """Linear z up-sampling by `inc` over the mirror-single extension (:144-171)."""
        ctx = ctx or default_context()
        img = _vol(img)
        z, y, x = img.shape
        out = np.empty(((z - 1) * inc + 1, y, x), dtype=np.float32)
        check(ctx._lib.mvsim_make_isotropic(ctx.h, fptr(img), dims3(img.shape), inc, fptr(out)), ctx.h)
        return out

    @staticmethod
    def computeWeightImage(img_or_shape, delta=None, ctx=None):
        """Cosine-taper weight image along y with the dims of the argument (:280-316); `delta` is ignored like in the reference."""
        ctx = ctx or default_context()
        shape = tuple(img_or_shape.shape) if hasattr(img_or_shape, "shape") else tuple(img_or_shape)
        out = np.empty(shape, dtype=np.float32)
        check(ctx._lib.mvsim_weight_image(ctx.h, dims3(shape), fptr(out)), ctx.h)
        return out

    @staticmethod
    def normalizeWeights(weights, osem, ctx=None):
        """The cross-view weight normalisation at the end of main() (:615-661), in place; returns the sum image."""
        ctx = ctx or default_context()
        for w in weights:
            _inplace(w, "weight")
        fpp = C.POINTER(C.c_float)
        arr = (fpp * len(weights))(*[fptr(w) for w in weights])
        s = np.empty_like(weights[0])
        check(ctx._lib.mvsim_normalize_weights(ctx.h, arr, len(weights), dims3(weights[0].shape), osem, fptr(s)), ctx.h)
        return s

    @staticmethod
    def simulate(halfPixelOffset=False, rnd=None, size=289, ctx=None):
        """The sphere-phantom ground truth (:366-392): drawSpheres at 2x, then downSample2x, on the device.  `rnd` is the
        seed of the java.util.Random the reference passes (class-static generator: 464232194, :76); its draws are replayed
        bit-exactly.  `size` is the reference's hard-coded 289."""
        ctx = ctx or default_context()
        seed = _phantom_seed(rnd)
        out = np.empty((size, size, size), dtype=np.float32)
        n = C.c_int64(0)
        check(ctx._lib.mvsim_simulate_phantom(ctx.h, size, int(bool(halfPixelOffset)), seed, fptr(out), C.byref(n)), ctx.h)
        return out

    @staticmethod
    def drawSpheres(shape_zyx, minValue=0.0, maxValue=1.0, scale=2, halfPixelOffset=False, rnd=None, ctx=None, return_count=False):
        """drawSpheres (:436-522) into a new zero volume of `shape_zyx` (the reference draws into its argument)."""
        ctx = ctx or default_context()
        seed = _phantom_seed(rnd)
        out = np.empty(tuple(shape_zyx), dtype=np.float32)
        n = C.c_int64(0)
        check(ctx._lib.mvsim_draw_spheres(ctx.h, dims3(out.shape), minValue, maxValue, scale, int(bool(halfPixelOffset)), seed,
                                          fptr(out), C.byref(n)), ctx.h)
        return (out, n.value) if return_count else out

    @staticmethod
    def downSample2x(img, ctx=None):
        """downSample2x (:394-423): dims/2 - 1, n-linear at 2l + 0.5."""
        ctx = ctx or default_context()
        img = _vol(img)
        if min(img.shape) < 4:
            raise MvsimError(_lib.MVSIM_EINVAL, "downSample2x: dims must be >= 4")
        out = np.empty(tuple(s // 2 - 1 for s in img.shape), dtype=np.float32)
        check(ctx._lib.mvsim_downsample2x(ctx.h, fptr(img), dims3(img.shape), fptr(out)), ctx.h)
        return out

    @staticmethod
    def simulateViews(gt, psfs, degrees, axis=0, delta=0.01, inc=3, poissonSNR=25.0, rnd=None, ctx=None, outs=None,
                      first_stream=0, strict_reference=True):
        """The view loop of main() (:567-613) for the acquisition stages: one ground truth, one PSF and
        one angle per view.  Ground truth is uploaded once, downloads overlap the next view.  `psfs`
        are normalised in place.  Returns the list of acquired volumes (written into `outs` if given)."""
        ctx = ctx or default_context()
        resident = isinstance(gt, DeviceVolume)       # ground truth already in HBM (uploaded once, generated there, or broadcast)
        if not resident:
            gt = _vol(gt, "gt")
        n = len(degrees)
        if len(psfs) != n:
            raise ValueError("one PSF per view")
        z, y, x = gt.shape
        oshape = ((z - 1) // inc + 1, y, x)
        if outs is None:
            outs = [np.empty(oshape, dtype=np.float32) for _ in range(n)]
        seed = _seed_from(rnd) if poissonSNR >= 0 else 0
        params = (ViewParams * n)()
        for v in range(n):
            _inplace(psfs[v], "psf")
            _inplace(outs[v], "out")
            if outs[v].shape != oshape:
                raise ValueError("out shape must be ((Z-1)//inc+1, Y, X)")
            params[v] = make_view_params(gt.shape, psfs[v].shape, axis, int(degrees[v]), delta,
                                         SimulateMultiViewDataset.minValue, SimulateMultiViewDataset.avgIntensity, inc,
                                         poissonSNR, seed, first_stream + v, strict_reference)
        fpp = C.POINTER(C.c_float)
        parr = (fpp * n)(*[fptr(p) for p in psfs])
        oarr = (fpp * n)(*[fptr(o) for o in outs])
        if resident:
            check(ctx._lib.mvsim_dev_simulate_views(ctx.h, n, params, gt.h, parr, oarr), ctx.h)
        else:
            check(ctx._lib.mvsim_simulate_views(ctx.h, n, params, fptr(gt), parr, oarr), ctx.h)
        return outs

    @staticmethod
    def simulateDataset(gt, psfs, angles, angleOffset=15, delta=0.01, inc=3, poissonSNR=25.0, osem=3.0, rnd=None, views=None, ctx=None,
                        outputs=("acq", "aligned", "aligned_psf", "weights"), sum_weights=True, strict_reference=True):
        """main()'s view loop with its post-acquisition chain (:567-663) in one device call (mvsim_simulate_dataset).

        `angles` are ALL the dataset's angles (main(): 0, angleIncrement, ... < 360); view v is acquired at angles[v] + angleOffset
        and rotated back by -angles[v].  `views` (default: all) selects the views simulated here, `psfs` holds one PSF per selected
        view (normalised in place, :255).  `gt` is a (Z, Y, X) array or a DeviceVolume.  Noise seeds are drawn like run_main: one
        nextLong() per view of `rnd` (default JavaRandom(464232194)) in view order for ALL views, stream = view index, so a view's
        counts do not depend on which subset is simulated.  Returns {"views", "acq", "aligned", "aligned_psf", "weights",
        "sum_weights"}: lists in the order of `views` (None for outputs not in `outputs`) and the sum image (or None)."""
        ctx = ctx or default_context()
        resident = isinstance(gt, DeviceVolume)
        if not resident:
            gt = _vol(gt, "gt")
        n_all = len(angles)
        views = list(range(n_all)) if views is None else [int(v) for v in views]
        n = len(views)
        if len(psfs) != n:
            raise ValueError("one PSF per simulated view")
        rnd = JavaRandom(SimulateMultiViewDataset.seed) if rnd is None else (JavaRandom(rnd) if isinstance(rnd, (int, np.integer)) else rnd)
        seeds = [_seed_from(rnd) for _ in range(n_all)]
        z, y, x = gt.shape
        za = (z - 1) // inc + 1
        params = (ViewParams * n_all)()
        for v in range(n_all):
            params[v] = make_view_params(gt.shape, psfs[views.index(v)].shape if v in views else (1, 1, 1), 0, int(angles[v]) + int(angleOffset),
                                         delta, SimulateMultiViewDataset.minValue, SimulateMultiViewDataset.avgIntensity, inc,
                                         poissonSNR, seeds[v] if poissonSNR >= 0 else 0, v, strict_reference)
        res = {"views": views, "acq": [None] * n, "aligned": [None] * n, "aligned_psf": [None] * n, "weights": [None] * n,
               "sum_weights": np.empty(gt.shape, dtype=np.float32) if sum_weights else None}
        outs = (DatasetOutputs * max(n, 1))()
        for i in range(n):
            _inplace(psfs[i], "psf")
            shapes = {"acq": (za, y, x), "aligned": ((za - 1) * inc + 1, y, x), "aligned_psf": psfs[i].shape, "weights": (z, y, x)}
            for key in outputs:
                res[key][i] = np.empty(shapes[key], dtype=np.float32)
                setattr(outs[i], key, fptr(res[key][i]))
        i32 = C.c_int32
        fpp = C.POINTER(C.c_float)
        args = (ctx.h, n_all, params, (i32 * n_all)(*[-int(a) for a in angles]), float(osem), n, (i32 * max(n, 1))(*views))
        tail = ((fpp * max(n, 1))(*[fptr(p) for p in psfs]), outs, fptr(res["sum_weights"]) if sum_weights else None)
        if resident:
            check(ctx._lib.mvsim_dev_simulate_dataset(*args, gt.h, *tail), ctx.h)
        else:
            check(ctx._lib.mvsim_simulate_dataset(*args, fptr(gt), *tail), ctx.h)
        return res


class SimulateBeads:
    """Mirror of S/SimulateBeads.java: random points (java.util.Random(535), :69), one rotated copy per angle
    (axisRotation about `axis`), each rendered as analytic Gaussians x 1000 (:168-205).  Intervals are (min_xyz, max_xyz)
    pairs like ImgLib2's FinalInterval; `FinalInterval(dims)` is ((0,0,0), dims-1)."""

    seed = 535

    def __init__(self, angles, axis, numPoints, rangeSimulation, intervalRender, sigma, ctx=None):
        self.angles = [int(a) for a in angles]
        self.axis = axis
        self.numPoints = numPoints
        self.rangeSimulation = rangeSimulation
        self.intervalRender = intervalRender
        self.sigma = [float(v) for v in sigma]
        self.ctx = ctx
        self.imgs = None

    @staticmethod
    def interval(dims_xyz):
        """new FinalInterval(dims): min 0, max dims - 1."""
        return (0, 0, 0), tuple(int(d) - 1 for d in dims_xyz)

    @staticmethod
    def randomPoints(numPoints, rangeInterval, rnd=535):
        """(:150-166) -> (numPoints, 3) float64 array of (x, y, z)."""
        mn, mx = rangeInterval
        pts = np.empty((numPoints, 3), dtype=np.float64)
        i3 = C.c_int64 * 3
        check(_lib.load().mvsim_random_points(numPoints, i3(*mn), i3(*mx), int(rnd), pts.ctypes.data_as(C.POINTER(C.c_double))))
        return pts

    @staticmethod
    def transformPoints(points, angles, axis, rangeInterval):
        """(:131-148) -> one transformed (n, 3) array per angle."""
        mn, mx = rangeInterval
        points = np.ascontiguousarray(points, dtype=np.float64)
        dp = C.POINTER(C.c_double)
        i3 = C.c_int64 * 3
        res = []
        for a in angles:
            out = np.empty_like(points)
            check(_lib.load().mvsim_transform_points(points.ctypes.data_as(dp), len(points), i3(*mn), i3(*mx), axis, int(a),
                                                     out.ctypes.data_as(dp)))
            res.append(out)
        return res

    @staticmethod
    def renderPoints(lists, interval, sigma, ctx=None):
        """(:97-121) -> one (z, y, x) float32 image per point list; like the reference the image has max - min voxels per axis."""
        ctx = ctx or default_context()
        mn, mx = interval
        shape = tuple(int(mx[d] - mn[d]) for d in (2, 1, 0))
        dp = C.POINTER(C.c_double)
        i3 = C.c_int64 * 3
        imgs = []
        for pts in lists:
            pts = np.ascontiguousarray(pts, dtype=np.float64)
            out = np.empty(shape, dtype=np.float32)
            check(ctx._lib.mvsim_render_beads(ctx.h, pts.ctypes.data_as(dp), len(pts), (C.c_double * 3)(*sigma), i3(*mn), i3(*mx),
                                              fptr(out)), ctx.h)
            imgs.append(out)
        return imgs

    def getImgs(self):
        if self.imgs is None:
            points = self.randomPoints(self.numPoints, self.rangeSimulation, self.seed)
            lists = self.transformPoints(points, self.angles, self.axis, self.rangeSimulation)
            self.imgs = self.renderPoints(lists, self.intervalRender, self.sigma, ctx=self.ctx)
        return self.imgs
