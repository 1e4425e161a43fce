"""ctypes binding of libmvtb.so (the C ABI declared in include/mvtb.h).

There is no CPU implementation behind this module: if the nvcc-built library is missing
or no CUDA device is visible, calls raise.  (tests/cuemu builds the same sources with a
host compiler for debugging index arithmetic; that build is never loaded from here.)
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmvtb.so")

MVTB_OK, MVTB_EINVAL, MVTB_EUNSUPPORTED, MVTB_ENOMEM, MVTB_ENODEVICE, MVTB_ETIMEOUT = 0, -1, -2, -3, -4, -5
MASK_NONE, MASK_DISK, MASK_CENTRED, MASK_UNIFORM = 0, 1, 2, 3
MAX_FFT_DIMS, MAX_SPIKES = 4, 8


class Spike(C.Structure):
    _fields_ = [("idx", C.c_int32 * MAX_FFT_DIMS), ("amplitude", C.c_float), ("reserved", C.c_int32)]


class ChainDesc(C.Structure):
    _fields_ = [
        ("mask_kind", C.c_int32),
        ("mask_ndim", C.c_int32),
        ("mask_thresh", C.c_int64),
        ("inside_off", C.c_int32),
        ("n_spikes", C.c_int32),
        ("wrap_alpha", C.c_float),
        ("wrap_naxes", C.c_int32),
        ("spikes", Spike * MAX_SPIKES),
        ("mask_u", C.c_void_p),
        ("mask_p", C.c_float),
        ("reserved", C.c_int32),
    ]


class SpParams(C.Structure):
    _fields_ = [("p", C.c_float), ("seed", C.c_uint64), ("offset", C.c_uint64)]


RESAMPLE_BILINEAR, RESAMPLE_NEAREST = 0, 1


class ResampleTap(C.Structure):
    _fields_ = [("i0", C.c_int32), ("i1", C.c_int32), ("w0", C.c_float), ("w1", C.c_float)]


class ResampleGeom(C.Structure):
    _fields_ = [
        ("in_shape", C.c_int32 * 3),
        ("grid_shape", C.c_int32 * 3),
        ("out_shape", C.c_int32 * 3),
        ("axis", C.c_int32 * 3),
        ("base", C.c_int32 * 3),
        ("step", C.c_int32 * 3),
        ("mode", C.c_int32),
        ("n_taps", C.c_int32),
        ("tap_grid", C.c_int32 * 3),
        ("tap_off", C.c_int32 * 3),
        ("taps", C.c_void_p),
        ("matrix", C.c_double * 12),
    ]


class MvtbError(RuntimeError):
    def __init__(self, code, text):
        super().__init__(f"libmvtb error {code}: {text}")
        self.code = code


_SYMBOLS = {
    "mvtb_version": (C.c_int, []),
    "mvtb_last_error": (C.c_int, [C.c_char_p, C.c_int]),
    "mvtb_plan_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.POINTER(C.c_int), C.c_int, C.c_int]),
    "mvtb_plan_destroy": (C.c_int, [C.c_void_p]),
    "mvtb_plan_workspace_bytes": (C.c_size_t, [C.c_void_p]),
    "mvtb_kspace_chain_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(ChainDesc), C.c_int,
                                        C.c_void_p, C.c_int, C.c_void_p]),
    "mvtb_kspace_chain_sp_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(ChainDesc), C.c_int,
                                           C.c_void_p, C.c_int, C.c_float, C.c_uint64, C.c_uint64, C.c_void_p]),
    "mvtb_kspace_chain_ex_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(ChainDesc), C.c_int, C.c_void_p,
                                           C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "mvtb_kspace_chain_ex_strided_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(ChainDesc), C.c_int,
                                                   C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p]),
    "mvtb_kspace_logabs_sum_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "mvtb_minmax_f32": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_void_p]),
    "mvtb_salt_pepper_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_uint64, C.c_uint64,
                                       C.c_float, C.c_void_p, C.c_void_p]),
    "mvtb_salt_pepper_sparse_f32": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int, C.c_uint64, C.c_uint64, C.c_float,
                                              C.c_void_p, C.c_void_p, C.c_void_p]),
    "mvtb_sparse_table": (C.c_int, [C.c_float, C.POINTER(C.c_uint32)]),
    "mvtb_philox_uniform_f32": (C.c_int, [C.c_void_p, C.c_size_t, C.c_uint64, C.c_uint64, C.c_void_p]),
    "mvtb_mt19937_jump_poly": (C.c_int, [C.c_uint64, C.c_void_p]),
    "mvtb_mt19937_advance": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "mvtb_mt19937_chunk_table": (C.c_int, [C.c_uint64, C.c_int, C.c_void_p]),
    "mvtb_mt19937_workspace_bytes": (C.c_size_t, [C.c_int]),
    "mvtb_mt19937_uniform_f32": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int,
                                           C.c_void_p, C.c_void_p]),
    "mvtb_intensity_scratch_bytes": (C.c_size_t, [C.c_int]),
    "mvtb_intensity_prologue_coeffs_f32": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                     C.c_void_p, C.c_void_p]),
    "mvtb_intensity_affine_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_void_p]),
    "mvtb_dice_scratch_bytes": (C.c_size_t, [C.c_int]),
    "mvtb_dice_sums_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mvtb_dice_grad_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mvtb_sqdiff_sum_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mvtb_crop_flip_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                     C.POINTER(C.c_int32), C.c_int, C.c_void_p]),
    "mvtb_crop_flip_batch_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                           C.c_void_p, C.c_void_p, C.c_void_p]),
    "mvtb_crop_flip_gather_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                            C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_void_p]),
    "mvtb_resample_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(ResampleGeom), C.c_void_p]),
    "mvtb_nifti_decode_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_int64), C.c_double, C.c_double,
                                        C.c_int32, C.c_void_p]),
    "mvtb_wrap_fold_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p]),
    "mvtb_wrap_odd_last_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_void_p]),
    "mvtb_plan_profile": (C.c_int, [C.c_void_p, C.c_int]),
    "mvtb_plan_profile_read": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int)]),
    "mvtb_kernel_name": (C.c_char_p, [C.c_int]),
    "mvtb_launch_count": (C.c_ulonglong, []),
    "mvtb_plan_set_path": (C.c_int, [C.c_void_p, C.c_int]),
    "mvtb_plan_tc_status": (C.c_int, [C.c_void_p]),
}
K_KINDS = 18
SP_BLOCK = 256
MT_STATE_WORDS = 640


def bind(cdll):
    """Attach prototypes for every symbol of include/mvtb.h; raises AttributeError if one is missing."""
    for name, (res, args) in _SYMBOLS.items():
        fn = getattr(cdll, name)
        fn.restype = res
        fn.argtypes = args
    return cdll


def exported_symbols():
    return sorted(_SYMBOLS)


def last_error(cdll):
    buf = C.create_string_buffer(512)
    cdll.mvtb_last_error(buf, 512)
    return buf.value.decode("utf-8", "replace")


def check(cdll, rc):
    if rc != MVTB_OK:
        raise MvtbError(rc, last_error(cdll))


_lib = None


def lib():
    """The nvcc-built library; built by __graft_entry__.build() / mvtb/build.py."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build the CUDA extension first (python __graft_entry__.py build). "
                "mvtb has no CPU fallback.")
        _lib = bind(C.CDLL(LIB_PATH))
    return _lib
