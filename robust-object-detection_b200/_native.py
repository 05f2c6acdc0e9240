"""ctypes binding of librod_b200.so -- one Python function per entry point of include/rod_b200.h.

There is NO CPU fallback: if the shared library has not been built (python -c
"import __graft_entry__ as g; g.build()") or no CUDA device is visible, calls raise.
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "librod_b200.so")

ROD_OK, ROD_ERR_INVALID_ARG, ROD_ERR_UNSUPPORTED, ROD_ERR_CUDA, ROD_ERR_NO_DEVICE, ROD_ERR_OOM = range(6)
OP_NONE, OP_NOISE, OP_BLUR, OP_LOWRES = 0, 1, 2, 3
LAUNCHES_CORRUPT_BATCH, LAUNCHES_CORRUPT_LETTERBOX, LAUNCHES_CORRUPT_CHW = 100, 101, 102
JPEGDEC_BASELINE, JPEGDEC_PROGRESSIVE = 1, 2


class ImageDesc(ctypes.Structure):
    """struct rod_image_desc"""
    _fields_ = [("src_offset", ctypes.c_uint64), ("dst_offset", ctypes.c_uint64),
                ("height", ctypes.c_int32), ("width", ctypes.c_int32),
                ("src_pitch", ctypes.c_int64), ("dst_pitch", ctypes.c_int64)]


# every symbol include/rod_b200.h declares: name -> (restype, argtypes)
_vp, _u64, _u32, _i, _f, _d = ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_int, ctypes.c_float, ctypes.c_double
SYMBOLS = {
    "rod_version": (ctypes.c_char_p, []),
    "rod_device_count": (_i, []),
    "rod_last_cuda_error": (_i, []),
    "rod_status_string": (ctypes.c_char_p, [_i]),
    "rod_plan_create": (_i, [ctypes.POINTER(ImageDesc), _i, ctypes.POINTER(_vp)]),
    "rod_plan_destroy": (None, [_vp]),
    "rod_plan_num_images": (_i, [_vp]),
    "rod_plan_payload_bytes": (_u64, [_vp]),
    "rod_plan_launches": (_i, [_vp, _i]),
    "rod_noise_u8": (_i, [_vp, _vp, _vp, _vp, _f, _u64, _u64, _u32, _vp, _vp]),
    "rod_noise_field_f32": (_i, [_vp, _vp, _f, _u64, _u64, _u32, _vp]),
    "rod_blur_h_u8": (_i, [_vp, _vp, _vp, _i, _d, _vp, _vp]),
    "rod_set_blur_kernel": (_i, [_vp, _vp, _i]),
    "rod_plan_set_gaussian_generator": (_i, [_vp, _i]),
    "rod_noise_prewarm": (_i, [_i, ctypes.c_float]),
    "rod_gauss_table_i32": (_i, [ctypes.c_float, ctypes.POINTER(ctypes.c_int32)]),
    "rod_numpy_legacy_normal_f32": (_i, [_vp, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32),
                                         ctypes.POINTER(ctypes.c_double), _d, _u64, _vp, _i]),
    "rod_numpy_legacy_normal_f32_device": (_i, [_vp, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32),
                                                ctypes.POINTER(ctypes.c_double), _d, _vp, _vp, _i, _vp,
                                                ctypes.POINTER(_i), _vp]),
    "rod_lowres_u8": (_i, [_vp, _vp, _vp, _d, _vp, _vp]),
    "rod_corrupt_batch_u8": (_i, [_vp, _vp, _vp, _vp, _vp, _f, _i, _d, _u64, _u64, _u32, _vp]),
    "rod_corrupt_letterbox_f16": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp, _f, _i, _d, _u64, _u64, _u32, _vp]),
    "rod_corrupt_chw_f32": (_i, [_vp, _vp, _vp, _vp, _vp, _f, _i, _d, _u64, _u64, _u32, _vp]),
    "rod_plan_chw_offset": (_u64, [_vp, _i]),
    "rod_restoration_pairs_f32": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _f, _i, _d, _u64, _u64, _u32, _vp]),
    "rod_resize_linear_u8": (_i, [_vp, _i, _i, ctypes.c_int64, _vp, _i, _i, ctypes.c_int64, _vp]),
    "rod_jpeg_create": (_i, [ctypes.POINTER(ImageDesc), _i, _vp, _u64, ctypes.POINTER(_vp)]),
    "rod_jpeg_destroy": (None, [_vp]),
    "rod_jpeg_trim": (None, []),
    "rod_jpeg_encode": (_i, [_vp, _vp, _vp]),
    "rod_jpeg_stream_offset": (_u64, [_vp, _i]),
    "rod_jpeg_stream_base": (_vp, [_vp]),
    "rod_jpeg_stream_lengths": (_vp, [_vp]),
    "rod_jpeg_download": (_i, [_vp, _vp, _vp, _vp]),
    "rod_jpegdec_probe": (_i, [_vp, _u64, ctypes.POINTER(_i), ctypes.POINTER(_i)]),
    "rod_jpegdec_probe_ex": (_i, [_vp, _u64, _i, ctypes.POINTER(_i), ctypes.POINTER(_i)]),
    "rod_jpegdec_create": (_i, [_vp, _vp, _i, _vp, _vp, _i, ctypes.POINTER(_vp)]),
    "rod_jpegdec_create_ex": (_i, [_vp, _vp, _i, _vp, _vp, _i, _i, ctypes.POINTER(_vp)]),
    "rod_jpegdec_destroy": (None, [_vp]),
    "rod_jpegdec_trim": (None, []),
    "rod_jpegdec_host_status": (_i, [_vp, _vp, _vp, _vp]),
    "rod_jpegdec_decode": (_i, [_vp, _vp, _vp]),
    "rod_jpegdec_status": (_i, [_vp, _vp, _vp]),
    "rod_apply_host": (_i, [_vp, _i, _vp, _vp, _vp, _f, _i, _d, _u64, _u64, _u32]),
}

_lib = None


class RodError(RuntimeError):
    pass


def lib() -> ctypes.CDLL:
    """Load (once) and return the shared library; raise if it is missing -- never fall back."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RodError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  This package has no CPU fallback.")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(handle, name)  # AttributeError if the ABI drifted
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(status: int, what: str) -> None:
    """Map a rod_status to the exceptions SURVEY 8b names."""
    if status == ROD_OK:
        return
    msg = lib().rod_status_string(status).decode()
    if status == ROD_ERR_INVALID_ARG:
        raise ValueError(f"{what}: {msg}")
    if status == ROD_ERR_UNSUPPORTED:
        raise NotImplementedError(f"{what}: {msg}")
    if status == ROD_ERR_CUDA:
        raise RodError(f"{what}: {msg} (cudaError {lib().rod_last_cuda_error()})")
    raise RodError(f"{what}: {msg}")


def require_device() -> None:
    if lib().rod_device_count() < 1:
        raise RodError("no CUDA device visible: the B200 corruption path has no CPU fallback")
