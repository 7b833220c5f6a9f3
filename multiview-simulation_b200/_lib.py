"""ctypes binding of libmvsim.so -- the same C ABI (include/mvsim.h) a JNI / Panama stub binds.

The CUDA library is the only implementation: if libmvsim.so is missing the import of this module
fails, and without a CUDA device every compute call raises MvsimError (MVSIM_ECUDA).
"""
import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MVSIM_LIB") or os.path.join(_PKG, "libmvsim.so")

MVSIM_OK, MVSIM_EINVAL, MVSIM_ENOMEM, MVSIM_ECUDA, MVSIM_ENCCL, MVSIM_EUNSUPPORTED = range(6)
STAGE_NAMES = ["h2d", "rotate", "attenuate", "psf", "fft_xfwd", "fft_yfwd", "fft_zfused", "fft_yinv", "fft_xinv",
               "adjust", "sample", "d2h", "widen"]
OPT_COUNT_TRANSPORT, OPT_HOST_THREADS, OPT_Z_KERNEL = 1, 2, 3
NSTAGES = len(STAGE_NAMES)


class MvsimError(RuntimeError):
    def __init__(self, status, message):
        super().__init__(f"mvsim status {status}: {message}")
        self.status = status


class ViewParams(C.Structure):
    _fields_ = [("dims", C.c_int64 * 3), ("kdims", C.c_int64 * 3), ("axis", C.c_int32), ("degrees", C.c_int32),
                ("delta", C.c_double), ("min_value", C.c_float), ("target_avg", C.c_float), ("inc", C.c_int32),
                ("snr", C.c_float), ("seed", C.c_uint64), ("stream", C.c_uint64), ("strict_reference", C.c_int32),
                ("reserved", C.c_int32)]


class DatasetOutputs(C.Structure):
    _fields_ = [("acq", C.POINTER(C.c_float)), ("aligned", C.POINTER(C.c_float)), ("aligned_psf", C.POINTER(C.c_float)),
                ("weights", C.POINTER(C.c_float))]


# every symbol include/mvsim.h declares: (name, restype, argtypes)
_vp = C.c_void_p
_i64p = C.POINTER(C.c_int64)
_fp = C.POINTER(C.c_float)
_dp = C.POINTER(C.c_double)
_i32p = C.POINTER(C.c_int32)
SYMBOLS = [
    ("mvsim_version", C.c_int, []),
    ("mvsim_device_count", C.c_int, [C.POINTER(C.c_int)]),
    ("mvsim_ctx_create", C.c_int, [C.c_int, C.POINTER(_vp)]),
    ("mvsim_ctx_create_on_stream", C.c_int, [C.c_int, _vp, C.POINTER(_vp)]),
    ("mvsim_ctx_destroy", C.c_int, [_vp]),
    ("mvsim_ctx_synchronize", C.c_int, [_vp]),
    ("mvsim_last_error", C.c_char_p, [_vp]),
    ("mvsim_profile_enable", C.c_int, [_vp, C.c_int]),
    ("mvsim_profile_reset", C.c_int, [_vp]),
    ("mvsim_stage_times", C.c_int, [_vp, _dp, _i64p]),
    ("mvsim_kernel_launches", C.c_int64, [_vp]),
    ("mvsim_ctx_set_option", C.c_int, [_vp, C.c_int, C.c_int64]),
    ("mvsim_psf_cache_configure", C.c_int, [_vp, C.c_size_t]),
    ("mvsim_psf_cache_stats", C.c_int, [_vp, _i64p]),
    ("mvsim_alloc_pinned", C.c_int, [C.c_size_t, C.POINTER(_vp)]),
    ("mvsim_free_pinned", C.c_int, [_vp]),
    ("mvsim_conv_padded_dims", C.c_int, [_i64p, _i64p, _i64p]),
    ("mvsim_axis_rotation", C.c_int, [_i64p, C.c_int, C.c_int, _dp, _dp]),
    ("mvsim_rotate_axis", C.c_int, [_vp, _fp, _fp, _i64p, C.c_int, C.c_int]),
    ("mvsim_attenuate", C.c_int, [_vp, _fp, _fp, _i64p, C.c_double, C.c_int]),
    ("mvsim_psf_normalize", C.c_int, [_vp, _fp, _i64p, _dp]),
    ("mvsim_convolve", C.c_int, [_vp, _fp, _i64p, _fp, _i64p, _fp]),
    ("mvsim_adjust", C.c_int, [_vp, _fp, _i64p, C.c_float, C.c_float, _dp]),
    ("mvsim_extract_slices", C.c_int, [_vp, _fp, _i64p, C.c_int, C.c_float, C.c_uint64, C.c_uint64, _fp]),
    ("mvsim_poisson", C.c_int, [_vp, _fp, C.c_size_t, C.c_double, C.c_uint64, C.c_uint64]),
    ("mvsim_simulate_view", C.c_int, [_vp, C.POINTER(ViewParams), _fp, _fp, _fp]),
    ("mvsim_simulate_views", C.c_int, [_vp, C.c_int, C.POINTER(ViewParams), _fp, C.POINTER(_fp), C.POINTER(_fp)]),
    ("mvsim_make_isotropic", C.c_int, [_vp, _fp, _i64p, C.c_int, _fp]),
    ("mvsim_weight_image", C.c_int, [_vp, _i64p, _fp]),
    ("mvsim_normalize_weights", C.c_int, [_vp, C.POINTER(_fp), C.c_int, _i64p, C.c_float, _fp]),
    ("mvsim_simulate_dataset", C.c_int, [_vp, C.c_int, C.POINTER(ViewParams), _i32p, C.c_float, C.c_int, _i32p, _fp, C.POINTER(_fp),
                                         C.POINTER(DatasetOutputs), _fp]),
    ("mvsim_dev_simulate_dataset", C.c_int, [_vp, C.c_int, C.POINTER(ViewParams), _i32p, C.c_float, C.c_int, _i32p, _vp,
                                             C.POINTER(_fp), C.POINTER(DatasetOutputs), _fp]),
    ("mvsim_dev_align_view", C.c_int, [_vp, _vp, C.c_int, C.c_int, _vp]),
    ("mvsim_dev_aligned_weights", C.c_int, [_vp, _i64p, C.c_int, _i32p, C.c_float, C.c_int, _i32p, C.POINTER(_vp), _vp]),
    ("mvsim_random_points", C.c_int, [C.c_int, _i64p, _i64p, C.c_int64, _dp]),
    ("mvsim_transform_points", C.c_int, [_dp, C.c_int, _i64p, _i64p, C.c_int, C.c_int, _dp]),
    ("mvsim_render_beads", C.c_int, [_vp, _dp, C.c_int, _dp, _i64p, _i64p, _fp]),
    ("mvsim_draw_spheres", C.c_int, [_vp, _i64p, C.c_double, C.c_double, C.c_int, C.c_int, C.c_int64, _fp, _i64p]),
    ("mvsim_downsample2x", C.c_int, [_vp, _fp, _i64p, _fp]),
    ("mvsim_simulate_phantom", C.c_int, [_vp, C.c_int, C.c_int, C.c_int64, _fp, _i64p]),
    ("mvsim_make_square", C.c_int, [_vp, _fp, _i64p, _fp]),
    ("mvsim_dev_render_beads", C.c_int, [_vp, _dp, C.c_int, _dp, _i64p, _i64p, _vp]),
    ("mvsim_dev_simulate_phantom", C.c_int, [_vp, C.c_int, C.c_int, C.c_int64, _vp, _i64p]),
    ("mvsim_volume_create", C.c_int, [_vp, _i64p, C.POINTER(_vp)]),
    ("mvsim_volume_wrap", C.c_int, [_vp, _i64p, _vp, C.POINTER(_vp)]),
    ("mvsim_volume_free", C.c_int, [_vp, _vp]),
    ("mvsim_volume_dims", C.c_int, [_vp, _i64p]),
    ("mvsim_volume_device_ptr", _vp, [_vp]),
    ("mvsim_volume_upload", C.c_int, [_vp, _vp, _fp]),
    ("mvsim_volume_download", C.c_int, [_vp, _vp, _fp]),
    ("mvsim_dev_rotate_axis", C.c_int, [_vp, _vp, _vp, C.c_int, C.c_int]),
    ("mvsim_dev_attenuate", C.c_int, [_vp, _vp, _vp, C.c_double, C.c_int]),
    ("mvsim_dev_psf_normalize", C.c_int, [_vp, _vp, _dp]),
    ("mvsim_dev_convolve", C.c_int, [_vp, _vp, _vp, _vp]),
    ("mvsim_dev_adjust", C.c_int, [_vp, _vp, C.c_float, C.c_float, _dp]),
    ("mvsim_dev_extract_slices", C.c_int, [_vp, _vp, C.c_int, C.c_float, C.c_uint64, C.c_uint64, _vp]),
    ("mvsim_dev_extract_interval", C.c_int, [_vp, _vp, _i64p, _i64p, C.c_int, C.c_float, C.c_uint64, C.c_uint64, _vp]),
    ("mvsim_dev_simulate_view", C.c_int, [_vp, C.POINTER(ViewParams), _vp, _vp, _vp]),
    ("mvsim_dev_simulate_views", C.c_int, [_vp, C.c_int, C.POINTER(ViewParams), _vp, C.POINTER(_fp), C.POINTER(_fp)]),
    ("mvsim_slabconv_create", C.c_int, [_vp, _i64p, _i64p, C.c_int, C.c_int, C.POINTER(_vp)]),
    ("mvsim_slabconv_destroy", C.c_int, [_vp, _vp]),
    ("mvsim_slabconv_info", C.c_int, [_vp, _i64p]),
    ("mvsim_slabconv_bind", C.c_int, [_vp, _vp, _vp]),
    ("mvsim_slabconv_prepare", C.c_int, [_vp, _vp, _vp, _vp]),
    ("mvsim_slabconv_forward_y", C.c_int, [_vp, _vp, C.c_int]),
    ("mvsim_slabconv_middle_z", C.c_int, [_vp, _vp]),
    ("mvsim_slabconv_inverse_y", C.c_int, [_vp, _vp, C.c_int]),
    ("mvsim_slabconv_finish", C.c_int, [_vp, _vp, _vp]),
    ("mvsim_slabconv_p2p_alloc", C.c_int, [_vp, _vp, C.c_int, _vp]),
    ("mvsim_slabconv_p2p_open", C.c_int, [_vp, _vp, _vp]),
    ("mvsim_slabconv_p2p_select", C.c_int, [_vp, C.c_int]),
    ("mvsim_slab_rotate_attenuate", C.c_int, [_vp, _vp, _i64p, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int64, C.c_int64, _vp]),
    ("mvsim_slab_sum", C.c_int, [_vp, _vp, C.c_size_t, _vp]),
    ("mvsim_slab_adjust", C.c_int, [_vp, _vp, C.c_size_t, _vp, C.c_int, C.c_double, C.c_float, C.c_float]),
    ("mvsim_slab_extract", C.c_int, [_vp, _vp, _i64p, C.c_int64, C.c_int64, C.c_int, C.c_float, C.c_uint64, C.c_uint64, _vp, _i64p]),
]

_lib = None


def load():
    """Loads libmvsim.so; raises (no fallback) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: run `python multiview-simulation_b200/build.py` "
                              "(nvcc, sm_100a). There is no CPU implementation to fall back to.")
        lib = C.CDLL(LIB_PATH)
        for name, res, args in SYMBOLS:
            fn = getattr(lib, name)        # AttributeError if the ABI lost a symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(status, ctx=None):
    if status != MVSIM_OK:
        msg = load().mvsim_last_error(ctx)
        raise MvsimError(status, msg.decode() if msg else "")


def dims3(shape_zyx):
    z, y, x = shape_zyx
    return (C.c_int64 * 3)(x, y, z)


def fptr(a):
    return a.ctypes.data_as(_fp)
