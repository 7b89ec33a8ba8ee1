"""ctypes binding of libxrseg.so (include/xrseg.h) and of libxrseg_debug.so (the same sources + the parity hooks of
include/xrseg_debug.h, used by tests/ and tools/ only).  No compute happens in Python."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIBS = {}
ABI_VERSION = 2


class XrsegError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"xrseg error {code}: {msg}")
        self.code = code


OK, ERR_INVALID, ERR_CUDA, ERR_NO_DEVICE, ERR_WEIGHTS, ERR_STATE, ERR_NO_DETECTIONS, ERR_CAPACITY = 0, -1, -2, -3, -4, -5, -6, -7
FMT_RGB8, FMT_RGBA8, FMT_BOTTOM_UP = 0, 1, 0x100
OVERFLOW_CANDIDATES, OVERFLOW_DETECTIONS = 1, 2
RESIZE_STRETCH, RESIZE_LETTERBOX = 0, 1
CONV_UMMA, CONV_DIRECT = 0, 1
BOX_PARSEBOXES, BOX_DRAWBOXES, BOX_RAW = 0, 1, 2
MASK_REFERENCE_160, MASK_CROP_160, MASK_UPSAMPLE_640, MASK_BITS_160 = 0, 1, 2, 3


class Config(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("device", C.c_int32), ("max_batch", C.c_int32), ("model_scale", C.c_int32),
        ("weights", C.c_void_p), ("weights_bytes", C.c_size_t),
        ("iou_threshold", C.c_float), ("score_threshold", C.c_float), ("mask_threshold", C.c_float),
        ("max_det", C.c_int32), ("max_candidates", C.c_int32), ("resize_mode", C.c_int32), ("conv_impl", C.c_int32),
        ("use_cuda_graph", C.c_int32), ("micro_batch", C.c_int32), ("num_classes", C.c_int32),
        ("reserved", C.c_int32 * 7),
    ]


class TensorView(C.Structure):
    _fields_ = [("device_ptr", C.c_void_p), ("dtype", C.c_int32), ("rank", C.c_int32), ("shape", C.c_int64 * 4)]


class Box(C.Structure):
    _fields_ = [("center_x", C.c_float), ("center_y", C.c_float), ("width", C.c_float), ("height", C.c_float),
                ("label_id", C.c_int32), ("frame", C.c_int32)]


class MaskParams(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("mode", C.c_int32), ("box_convention", C.c_int32),
                ("screen_w", C.c_float), ("screen_h", C.c_float), ("image_w", C.c_int32), ("image_h", C.c_int32),
                ("first", C.c_int32), ("count", C.c_int32), ("threshold", C.c_float)]


class DepthParams(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("detection", C.c_int32), ("depth_w", C.c_int32), ("depth_h", C.c_int32),
                ("sampling_step", C.c_int32), ("max_points", C.c_int32), ("confidence_threshold", C.c_float),
                ("screen_w", C.c_float), ("screen_h", C.c_float), ("camera_position", C.c_float * 3),
                ("camera_rotation", C.c_float * 4), ("focal_length", C.c_float * 2), ("principal_point", C.c_float * 2),
                ("sensor_resolution", C.c_float * 2)]


class LayerInfo(C.Structure):
    _fields_ = [("name", C.c_char * 32), ("cin", C.c_int32), ("cout", C.c_int32), ("k", C.c_int32),
                ("stride", C.c_int32), ("groups", C.c_int32), ("act", C.c_int32), ("transposed", C.c_int32),
                ("h_in", C.c_int32), ("w_in", C.c_int32)]


# every symbol include/xrseg.h declares, with its signature
_P = C.POINTER
PRODUCT_SIGNATURES = {
    "xrseg_create": (C.c_int, [_P(Config), _P(C.c_void_p)]),
    "xrseg_destroy": (None, [C.c_void_p]),
    "xrseg_last_error": (C.c_char_p, [C.c_void_p]),
    "xrseg_abi_version": (C.c_int, []),
    "xrseg_schedule": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "xrseg_schedule_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "xrseg_poll": (C.c_int, [C.c_void_p]),
    "xrseg_wait": (C.c_int, [C.c_void_p]),
    "xrseg_counts": (C.c_int, [C.c_void_p, _P(C.c_int32), C.c_int]),
    "xrseg_overflow": (C.c_int, [C.c_void_p]),
    "xrseg_peek_output": (C.c_int, [C.c_void_p, C.c_int, _P(TensorView)]),
    "xrseg_readback": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, _P(C.c_int64), _P(C.c_int)]),
    "xrseg_decode": (C.c_int, [C.c_void_p, C.c_float, C.c_float, C.c_int, _P(Box), C.c_int, _P(C.c_int)]),
    "xrseg_masks": (C.c_int, [C.c_void_p, _P(MaskParams), C.c_void_p, C.c_size_t]),
    "xrseg_collect": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, _P(MaskParams), C.c_void_p, C.c_size_t]),
    "xrseg_keep_indices": (C.c_int, [C.c_void_p, _P(C.c_int32), _P(C.c_float), C.c_int]),
    "xrseg_layer_count": (C.c_int, [C.c_int]),
    "xrseg_layer_info_get": (C.c_int, [C.c_int, C.c_int, _P(LayerInfo)]),
    "xrseg_layer_count_nc": (C.c_int, [C.c_int, C.c_int]),
    "xrseg_layer_info_get_nc": (C.c_int, [C.c_int, C.c_int, C.c_int, _P(LayerInfo)]),
    "xrseg_weights_info": (C.c_int, [C.c_void_p, C.c_size_t, _P(C.c_int32), _P(C.c_int32)]),
    "xrseg_num_classes": (C.c_int, [C.c_void_p]),
    "xrseg_last_timings": (C.c_int, [C.c_void_p, _P(C.c_float), C.c_int]),
    "xrseg_launch_count": (C.c_int, [C.c_void_p]),
    "xrseg_event_record": (C.c_int, [C.c_void_p, C.c_int]),
    "xrseg_event_elapsed_ms": (C.c_int, [C.c_void_p, C.c_int, C.c_int, _P(C.c_float)]),
    "xrseg_sync": (C.c_int, [C.c_void_p]),
    "xrseg_profile_ops": (C.c_int, [C.c_void_p, C.c_int, _P(C.c_float), C.c_char_p, _P(C.c_double), _P(C.c_double), C.c_int]),
    "xrseg_extract_points": (C.c_int, [C.c_void_p, _P(DepthParams), C.c_void_p, C.c_void_p, C.c_int, _P(C.c_int)]),
    "xrseg_associate": (C.c_int, [C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_int, C.c_float, C.c_float, C.c_float,
                                  _P(C.c_int), _P(C.c_float)]),
    "xrseg_sentis_info": (C.c_int, [C.c_void_p, C.c_size_t, _P(C.c_int32), _P(C.c_float), _P(C.c_float)]),
    "xrseg_sentis_layer": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
                                     _P(C.c_int32), _P(C.c_int32)]),
    "xrseg_host_alloc": (C.c_void_p, [C.c_size_t]),
    "xrseg_host_free": (None, [C.c_void_p]),
    "xrseg_device_count": (C.c_int, []),
}

# include/xrseg_debug.h: exported by libxrseg_debug.so only
DEBUG_SIGNATURES = {
    "xrseg_debug_fetch": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_size_t, _P(C.c_int64)]),
    "xrseg_debug_fetch_frames": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int, C.c_int, C.c_void_p, C.c_size_t, _P(C.c_int64)]),
    "xrseg_debug_launches": (C.c_int, [C.c_void_p, _P(C.c_int), _P(C.c_int), _P(C.c_int), C.c_char_p, C.c_int]),
    "xrseg_debug_post": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "xrseg_debug_post_f16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "xrseg_debug_nms": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
    "xrseg_debug_mask_threshold": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p]),
    "xrseg_debug_conv": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                   C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]),
    "xrseg_debug_bottleneck": (C.c_int, [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                         C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "xrseg_debug_pack_bneck": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t]),
    "xrseg_debug_emulate_conv": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                           C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]),
    "xrseg_debug_post_timings": (C.c_int, [C.c_void_p, _P(C.c_float), _P(C.c_double), C.c_char_p, C.c_int]),
    "xrseg_debug_attention": (C.c_int, [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
}
SIGNATURES = {**PRODUCT_SIGNATURES, **DEBUG_SIGNATURES}   # what libxrseg_debug.so exports


def library_path(debug: bool = False) -> str:
    return os.path.join(_HERE, ("libxrseg_debug" if debug else "libxrseg") + ".so")


def build_library(verbose: bool = False) -> str:
    """Compile libxrseg.so and libxrseg_debug.so in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    r = subprocess.run(["make", "-j2", "-C", os.path.join(_HERE, "csrc")], capture_output=True, text=True)
    if verbose or r.returncode != 0:
        print(r.stdout)
        print(r.stderr)
    if r.returncode != 0:
        raise RuntimeError("building libxrseg.so failed")
    return library_path()


def load_library(debug: bool = False):
    """Load libxrseg.so (debug=True: libxrseg_debug.so, the product entry points + the parity hooks); raises if it is
    missing (there is no fallback implementation)."""
    if debug in _LIBS:
        return _LIBS[debug]
    path = library_path(debug)
    if not os.path.exists(path):
        raise XrsegError(ERR_INVALID, f"{path} not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                                      f"or `make -C xr_image_segmentation_b200/csrc` (there is no CPU fallback)")
    lib = C.CDLL(path)
    for name, (res, args) in (SIGNATURES if debug else PRODUCT_SIGNATURES).items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.xrseg_abi_version() != ABI_VERSION:
        raise XrsegError(ERR_INVALID, f"{path}: ABI version mismatch")
    _LIBS[debug] = lib
    return lib


def check(rc: int, runner=None, lib=None):
    if rc < 0:
        lib = lib or load_library()
        msg = lib.xrseg_last_error(runner)
        raise XrsegError(rc, msg.decode() if msg else "")
    return rc
