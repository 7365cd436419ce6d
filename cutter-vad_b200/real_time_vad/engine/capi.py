"""ctypes binding of the C ABI in include/cutter_vad_b200.h (libcvad_b200.so).

The library is built in-tree by `__graft_entry__.build()` (nvcc, sm_100a).  There
is NO fallback: a missing library raises at import of this module's `lib()`, and
`cvad_create` fails with CVAD_E_NOGPU when no sm_100 device is visible.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import numpy as np

PKG_ROOT = Path(__file__).resolve().parents[2]          # .../cutter-vad_b200
LIB_PATH = PKG_ROOT / "libcvad_b200.so"
DEV_LIB_PATH = PKG_ROOT / "libcvad_b200_dev.so"     # development probes (csrc/cvad_dev.cu): tests and tools only

OK, E_INVALID, E_CUDA, E_NOGPU, E_WEIGHTS, E_CAPACITY = 0, -1, -2, -3, -4, -5
MODEL_V5, MODEL_V4, MODEL_V4_8K = 5, 4, 48
PCM_F32, PCM_S16_32767, PCM_S16_32768 = 0, 1, 2
FLAG_STARTED, FLAG_ENDED, FLAG_CONTINUING = 1, 2, 4
STATUS_NONFINITE = 1
MATH_FP32, MATH_TC, MATH_TC16, MATH_FFT = 0, 1, 2, 3
RESAMPLE_FFT, RESAMPLE_GEMM = 0, 1
PAYLOAD_NONE, PAYLOAD_EVENTS, PAYLOAD_SEGMENTS, PAYLOAD_FRAMES = 0, 1, 2, 3

EXPORTS = (
    "cvad_abi_version", "cvad_device_count", "cvad_last_error", "cvad_create", "cvad_destroy",
    "cvad_set_stream", "cvad_reset", "cvad_configure", "cvad_get_state", "cvad_set_state",
    "cvad_step", "cvad_step_submit", "cvad_step_collect", "cvad_step_device", "cvad_sync", "cvad_launch_count", "cvad_debug_dump",
    "cvad_debug_input",
    "cvad_alloc_pinned", "cvad_free_pinned", "cvad_set_timing", "cvad_read_timing", "cvad_resample_matrix",
    "cvad_set_math", "cvad_get_math", "cvad_set_resampler", "cvad_get_resampler", "cvad_set_profile", "cvad_read_profile", "cvad_read_profile_chain",
    "cvad_feeder_create", "cvad_feeder_destroy", "cvad_feeder_last_error", "cvad_feeder_open", "cvad_feeder_close",
    "cvad_feeder_clear", "cvad_feeder_is_active", "cvad_feeder_pending", "cvad_feeder_push", "cvad_feeder_push_many",
    "cvad_feeder_step", "cvad_feeder_gather_only", "cvad_feeder_deliver_only",
    "cvad_model_fingerprint", "cvad_export_states", "cvad_import_states", "cvad_feeder_export", "cvad_feeder_import",
)

# cvad_stream_state: one slot's engine state, 1,072 bytes without padding (cvad_export_states / cvad_import_states)
STATE_DTYPE = np.dtype([("h", "<f4", (128,)), ("c", "<f4", (128,)), ("frames_done", "<i8"),
                        ("vad_start_probability", "<f8"), ("vad_end_probability", "<f8"),
                        ("is_voice_active", "<i4"), ("voice_start_frame_count", "<i4"), ("voice_end_frame_count", "<i4"),
                        ("n_start", "<i4"), ("n_end", "<i4"), ("enable_denoising", "<i4")])
assert STATE_DTYPE.itemsize == 1072
FEEDER_SNAPSHOT_MAGIC, FEEDER_SNAPSHOT_VERSION = 0x53465643, 1


class Event(C.Structure):
    _fields_ = [("stream", C.c_int32), ("slot", C.c_int32), ("frame", C.c_int32), ("kind", C.c_int32),
                ("stream_frame", C.c_int64)]


class StepArgs(C.Structure):
    _fields_ = [
        ("n_streams", C.c_int32),
        ("slots", C.c_void_p),
        ("audio", C.c_void_p),
        ("pcm_format", C.c_int32),
        ("stream_stride", C.c_int64),
        ("n_frames", C.c_void_p),
        ("max_frames", C.c_int32),
        ("frame_len", C.c_int32),
        ("hop", C.c_int32),
        ("src_rate", C.c_int32),
        ("probs_out", C.c_void_p),
        ("flags_out", C.c_void_p),
        ("status_out", C.c_void_p),
        ("events_out", C.c_void_p),
        ("max_events", C.c_int32),
        ("n_events_out", C.c_void_p),
        ("src_rates", C.c_void_p),
        ("channels", C.c_int32),
    ]


class Delivery(C.Structure):
    _fields_ = [("slot", C.c_int32), ("stream", C.c_int32), ("step_frame", C.c_int32), ("flags", C.c_int32),
                ("frame", C.c_void_p), ("segment", C.c_void_p), ("segment_len", C.c_int64),
                ("frame_len", C.c_int32), ("prob", C.c_float), ("raw", C.c_void_p), ("raw_len", C.c_int64)]


class FeederResult(C.Structure):
    _fields_ = [("n_streams", C.c_int32), ("max_frames", C.c_int32), ("n_frames_total", C.c_int64),
                ("slots", C.c_void_p), ("counts", C.c_void_p), ("probs", C.c_void_p), ("flags", C.c_void_p),
                ("n_events", C.c_int32), ("n_deliveries", C.c_int32), ("events", C.c_void_p),
                ("deliveries", C.c_void_p), ("raw", C.c_void_p), ("raw_stride", C.c_int64),
                ("gather_ms", C.c_double), ("gpu_ms", C.c_double), ("deliver_ms", C.c_double)]


_lib = None
_dev_lib = None
DEV_EXPORTS = ("cvad_dev_last_error", "cvad_tc_probe", "cvad_tc_probe_mn", "cvad_tc_rate", "cvad_tc_rate_mn", "cvad_bulk_rate")


def dev_lib() -> C.CDLL:
    """libcvad_b200_dev.so: hardware probes of the tcgen05 building blocks (include/cutter_vad_b200_dev.h).  The product
    never calls this."""
    global _dev_lib
    if _dev_lib is None:
        if not DEV_LIB_PATH.exists():
            raise EngineLibraryMissing(f"{DEV_LIB_PATH} not found: build it with `python cutter-vad_b200/build.py`")
        L = C.CDLL(str(DEV_LIB_PATH))
        vp, i32 = C.c_void_p, C.c_int
        L.cvad_dev_last_error.restype = C.c_char_p
        L.cvad_tc_probe.argtypes = [i32, vp, vp, vp]
        L.cvad_tc_probe_mn.argtypes = [i32, vp, vp, vp]
        L.cvad_tc_rate.argtypes = [i32, i32, i32, i32, i32, i32, i32, vp]
        L.cvad_tc_rate_mn.argtypes = [i32, i32, i32, i32, i32, i32, i32, i32, vp]
        L.cvad_bulk_rate.argtypes = [i32, i32, i32, i32, i32, C.c_size_t, vp]
        _dev_lib = L
    return _dev_lib



class EngineLibraryMissing(RuntimeError):
    pass


def lib() -> C.CDLL:
    """Load libcvad_b200.so (once).  Raises EngineLibraryMissing if it was not built."""
    global _lib
    if _lib is not None:
        return _lib
    path = Path(os.environ.get("CVAD_B200_LIB", LIB_PATH))
    if not path.exists():
        raise EngineLibraryMissing(
            f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). This engine has no CPU or PyTorch fallback.")
    L = C.CDLL(str(path))
    vp, i32, i64, dbl = C.c_void_p, C.c_int, C.c_int64, C.c_double
    L.cvad_abi_version.restype = i32
    L.cvad_device_count.restype = i32
    L.cvad_last_error.restype = C.c_char_p
    L.cvad_last_error.argtypes = [vp]
    L.cvad_create.argtypes = [vp, C.c_size_t, i32, i32, i32, C.POINTER(vp)]
    L.cvad_destroy.argtypes = [vp]
    L.cvad_set_stream.argtypes = [vp, vp]
    L.cvad_set_math.argtypes = [vp, i32]
    L.cvad_get_math.argtypes = [vp]
    L.cvad_set_resampler.argtypes = [vp, i32]
    L.cvad_get_resampler.argtypes = [vp]
    L.cvad_set_profile.argtypes = [vp, i32]
    L.cvad_read_profile.argtypes = [vp, vp]
    L.cvad_read_profile_chain.argtypes = [vp, vp]
    L.cvad_reset.argtypes = [vp, i32, vp]
    L.cvad_configure.argtypes = [vp, i32, vp, dbl, dbl, i32, i32, i32]
    L.cvad_get_state.argtypes = [vp, i32, vp, vp, vp, vp]
    L.cvad_set_state.argtypes = [vp, i32, vp, vp, vp]
    L.cvad_step.argtypes = [vp, C.POINTER(StepArgs)]
    L.cvad_step_device.argtypes = [vp, C.POINTER(StepArgs)]
    L.cvad_resample_matrix.argtypes = [i32, vp, C.c_size_t]
    L.cvad_step_submit.argtypes = [vp, C.POINTER(StepArgs), C.POINTER(C.c_int)]
    L.cvad_step_collect.argtypes = [vp, i32]
    L.cvad_sync.argtypes = [vp]
    L.cvad_launch_count.restype = i64
    L.cvad_launch_count.argtypes = [vp]
    L.cvad_debug_dump.argtypes = [vp, C.POINTER(StepArgs), vp, C.c_size_t]
    L.cvad_debug_input.argtypes = [vp, C.POINTER(StepArgs), vp, C.c_size_t]
    L.cvad_alloc_pinned.restype = vp
    L.cvad_alloc_pinned.argtypes = [C.c_size_t]
    L.cvad_free_pinned.argtypes = [vp]
    L.cvad_set_timing.argtypes = [vp, i32]
    L.cvad_read_timing.argtypes = [vp, vp, vp, vp]
    L.cvad_feeder_create.argtypes = [vp, i32, i32, i32, i32, i32, i32, C.POINTER(vp)]
    L.cvad_feeder_destroy.argtypes = [vp]
    L.cvad_feeder_last_error.restype = C.c_char_p
    L.cvad_feeder_last_error.argtypes = [vp]
    L.cvad_feeder_open.argtypes = [vp, i32, i32, i32, dbl, i32]
    L.cvad_feeder_close.argtypes = [vp, i32]
    L.cvad_feeder_clear.argtypes = [vp, i32]
    L.cvad_feeder_is_active.argtypes = [vp, i32]
    L.cvad_feeder_pending.restype = i64
    L.cvad_feeder_pending.argtypes = [vp, i32]
    L.cvad_feeder_push.argtypes = [vp, i32, vp, i64]
    L.cvad_feeder_push_many.argtypes = [vp, i32, vp, vp, i64, i64]
    L.cvad_feeder_step.argtypes = [vp, C.POINTER(FeederResult)]
    L.cvad_feeder_gather_only.argtypes = [vp, C.POINTER(FeederResult)]
    L.cvad_feeder_deliver_only.argtypes = [vp, vp, vp, C.POINTER(FeederResult)]
    L.cvad_model_fingerprint.argtypes = [vp, C.POINTER(C.c_uint64)]
    L.cvad_export_states.argtypes = [vp, i32, vp, vp]
    L.cvad_import_states.argtypes = [vp, i32, vp, vp]
    L.cvad_feeder_export.argtypes = [vp, i32, vp, vp, C.c_size_t, C.POINTER(C.c_size_t)]
    L.cvad_feeder_import.argtypes = [vp, i32, vp, vp, C.c_size_t]
    _lib = L
    return L
