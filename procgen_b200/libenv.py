"""ctypes binding of include/procgen_b200.h (the libenv C ABI + the device-resident extension).

This is the binding gym3's CEnv would make with cffi (gym3/libenv.py); it is kept dependency-free
because gym3 is not installable in this image.
"""
from __future__ import annotations

import ctypes as C
import os

from .build import LIB_PATH

MAX_NAME = 128
MAX_NDIM = 16
DTYPE_UINT8, DTYPE_INT32, DTYPE_FLOAT32 = 1, 2, 3
SPACE_OBSERVATION, SPACE_ACTION, SPACE_INFO = 1, 2, 3


class Value(C.Union):
    _fields_ = [("uint8", C.c_uint8), ("int32", C.c_int32), ("float32", C.c_float)]


class TensorType(C.Structure):
    _fields_ = [("name", C.c_char * MAX_NAME), ("scalar_type", C.c_int), ("dtype", C.c_int),
                ("shape", C.c_int * MAX_NDIM), ("ndim", C.c_int), ("low", Value), ("high", Value)]


class Option(C.Structure):
    _fields_ = [("name", C.c_char * MAX_NAME), ("dtype", C.c_int), ("count", C.c_int), ("data", C.c_void_p)]


class Options(C.Structure):
    _fields_ = [("items", C.POINTER(Option)), ("count", C.c_int)]


class Buffers(C.Structure):
    _fields_ = [("ob", C.POINTER(C.c_void_p)), ("rew", C.POINTER(C.c_float)), ("first", C.POINTER(C.c_uint8)),
                ("info", C.POINTER(C.c_void_p)), ("ac", C.POINTER(C.c_void_p))]


class DeviceBuffers(C.Structure):
    _fields_ = [("rgb", C.c_void_p), ("rew", C.c_void_p), ("first", C.c_void_p), ("prev_level_seed", C.c_void_p),
                ("prev_level_complete", C.c_void_p), ("level_seed", C.c_void_p), ("action", C.c_void_p),
                ("num_envs", C.c_int32), ("device", C.c_int32), ("stream", C.c_void_p)]


EXPORTS = ["libenv_version", "libenv_make", "libenv_get_tensortypes", "libenv_set_buffers", "libenv_observe",
           "libenv_act", "libenv_close", "pgb200_get_device_buffers", "pgb200_set_stream", "pgb200_act_device",
           "pgb200_sync", "pgb200_get_errors", "pgb200_debug_cycles", "pgb200_debug_read_env", "pgb200_kernel_launches", "pgb200_is_device_build",
           "pgb200_kernel_timing_begin", "pgb200_kernel_timing_end", "get_state", "set_state", "pgb200_set_launch_shape",
           "pgb200_frame_info", "pgb200_set_rgb_mirror", "pgb200_mirror_parity",
           "pgb200_set_consumer_output", "pgb200_consumer_slot", "pgb200_debug_phase_offset",
           "pgb200_debug_pixel_classes"]

_lib = None


def bind(lib):
    lib.libenv_version.restype = C.c_int
    lib.libenv_make.restype = C.c_void_p
    lib.libenv_make.argtypes = [C.c_int, Options]
    lib.libenv_get_tensortypes.restype = C.c_int
    lib.libenv_get_tensortypes.argtypes = [C.c_void_p, C.c_int, C.POINTER(TensorType)]
    lib.libenv_set_buffers.argtypes = [C.c_void_p, C.POINTER(Buffers)]
    lib.libenv_set_buffers.restype = None
    for f in (lib.libenv_observe, lib.libenv_act, lib.libenv_close, lib.pgb200_act_device, lib.pgb200_sync):
        f.argtypes = [C.c_void_p]
        f.restype = None
    lib.pgb200_get_device_buffers.argtypes = [C.c_void_p, C.POINTER(DeviceBuffers)]
    lib.pgb200_get_device_buffers.restype = C.c_int
    lib.pgb200_set_stream.argtypes = [C.c_void_p, C.c_void_p]
    lib.pgb200_set_stream.restype = None
    lib.pgb200_get_errors.argtypes = [C.c_void_p, C.POINTER(C.c_uint32)]
    lib.pgb200_get_errors.restype = C.c_uint32
    lib.pgb200_debug_cycles.argtypes = [C.c_void_p, C.c_void_p]
    lib.pgb200_debug_cycles.restype = C.c_int
    lib.pgb200_debug_read_env.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
    lib.pgb200_debug_read_env.restype = C.c_int
    lib.pgb200_frame_info.argtypes = [C.c_char_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.pgb200_frame_info.restype = C.c_int
    lib.pgb200_set_rgb_mirror.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.pgb200_set_rgb_mirror.restype = C.c_int
    lib.pgb200_set_consumer_output.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    lib.pgb200_set_consumer_output.restype = C.c_int
    lib.pgb200_consumer_slot.argtypes = [C.c_void_p]
    lib.pgb200_consumer_slot.restype = C.c_int
    lib.pgb200_mirror_parity.argtypes = [C.c_void_p]
    lib.pgb200_mirror_parity.restype = C.c_int
    lib.pgb200_kernel_launches.argtypes = [C.c_void_p]
    lib.pgb200_kernel_launches.restype = C.c_int64
    lib.get_state.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.c_int]
    lib.get_state.restype = C.c_int
    lib.set_state.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.c_int]
    lib.set_state.restype = None
    lib.pgb200_set_launch_shape.argtypes = [C.c_void_p, C.c_int, C.c_int]
    lib.pgb200_set_launch_shape.restype = None
    lib.pgb200_kernel_timing_begin.argtypes = [C.c_void_p, C.c_int]
    lib.pgb200_kernel_timing_begin.restype = C.c_int
    lib.pgb200_kernel_timing_end.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
    lib.pgb200_kernel_timing_end.restype = C.c_int
    lib.pgb200_is_device_build.restype = C.c_int
    return lib


def load(path: str | None = None):
    """Load the product library. There is no CPU fallback: a missing or non-GPU build is an error."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    # PROCGEN_B200_LIB: another build of the same CUDA library (kernel tuning experiments, tools/)
    p = path or os.environ.get("PROCGEN_B200_LIB") or LIB_PATH
    if not os.path.exists(p):
        raise RuntimeError(
            f"procgen_b200: CUDA library {p} is missing. Build it with "
            "`python -c 'import __graft_entry__ as g; g.build()'` (nvcc, sm_100a). There is no CPU fallback.")
    lib = bind(C.CDLL(p))
    if path is None:
        if lib.pgb200_is_device_build() != 1:
            raise RuntimeError("procgen_b200: refusing to run on a non-CUDA build of the library")
        _lib = lib
    return lib


def make_options(keep, opts: dict) -> Options:
    """dict -> libenv_options the way gym3's CEnv marshals them: str -> uint8[count], bool -> uint8,
    int -> int32 (env.py:110-124 builds the dict)."""
    items = (Option * len(opts))()
    for i, (k, v) in enumerate(opts.items()):
        items[i].name = k.encode()
        if isinstance(v, str):
            raw = v.encode()
            buf = C.create_string_buffer(raw, max(len(raw), 1))
            items[i].dtype, items[i].count = DTYPE_UINT8, len(raw)
        elif isinstance(v, bool):
            buf = (C.c_uint8 * 1)(int(v))
            items[i].dtype, items[i].count = DTYPE_UINT8, 1
        elif isinstance(v, int):
            buf = (C.c_int32 * 1)(v)
            items[i].dtype, items[i].count = DTYPE_INT32, 1
        else:
            raise TypeError(f"option {k}: unsupported type {type(v)}")
        keep.append(buf)
        items[i].data = C.cast(buf, C.c_void_p)
    keep.append(items)
    return Options(items, len(opts))
