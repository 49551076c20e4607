"""ctypes binding of include/vrg_b200.h.  There is no CPU fallback: if the CUDA
library cannot be loaded, the compute entry points raise."""
from __future__ import annotations

import ctypes
import os

from . import _build

i64 = ctypes.c_int64
vp = ctypes.c_void_p

OK = 0
ERR_CUDA, ERR_ARG, ERR_LEVELS, ERR_LABEL, ERR_EMPTY_SEED, ERR_NO_BAND, ERR_NOMEM, ERR_NONFINITE = range(-1, -9, -1)
EXIT_RUNNING, EXIT_CONVERGED, EXIT_MAX_TIME, EXIT_MAX_SEGMENT, EXIT_MAX_ITER = -1, 0, 1, 2, 3
INTENSITY_F64_DENSE, INTENSITY_F64_BAND, INTENSITY_INDEX = 0, 1, 2
INTENSITY_MODES = {"f64_dense": 0, "f64_band": 1, "index": 2, "continuous": 3}
HALO = 2
MAX_LEVELS = 65536
P2P_HANDLE_BYTES = 192
DTYPE_U8, DTYPE_I8, DTYPE_I16, DTYPE_I32, DTYPE_I64, DTYPE_F32, DTYPE_F64 = range(7)  # vrg_dtype
BUF_SEG, BUF_EXCL, BUF_FLIPS, BUF_CANCELLED, BUF_LOCAL_STATS, BUF_GLOBAL_STATS, BUF_CTRL = range(7)
ST_N_IN, ST_N_OUT, ST_N_EXCL, ST_N_FLIPS, ST_N_BAND, ST_BAD_LABEL, ST_NONFINITE, ST_TIME_UP = range(8)
ST_Q_CANCELLED, ST_Q_ADD_INSIDE, ST_Q_REM_OUTSIDE, ST_Q_REPROMOTED = 8, 9, 10, 11
ST_EXTRA = 16
C_STATUS, C_ITER, C_ITER_MAX, C_MAX_SEG, C_APPLY, C_APPLIED, C_TRACE_N, C_SWEEPS = range(8)


class Config(ctypes.Structure):
    _fields_ = [("shape", i64 * 3), ("z_begin", i64), ("z_end", i64), ("device", ctypes.c_int32),
                ("intensity_mode", ctypes.c_int32), ("H", ctypes.c_double), ("iter_max", i64),
                ("max_segment_size", i64), ("max_seconds", ctypes.c_double)]


class Result(ctypes.Structure):
    _fields_ = [("iterations", i64), ("exit_reason", i64), ("n_in", i64), ("n_out", i64), ("n_excluded", i64),
                ("n_levels", i64), ("sweeps", i64), ("kernel_launches", i64), ("q_cancelled", i64),
                ("q_add_to_inside", i64), ("q_remove_to_outside", i64), ("q_cancel_repromoted", i64), ("redone_sweeps", i64)]


class StrictResult(ctypes.Structure):
    _fields_ = [("iterations", i64), ("exit_reason", i64), ("n_in", i64), ("n_out", i64), ("n_excluded", i64),
                ("n_levels", i64), ("kernel_launches", i64), ("skipped", i64), ("dropped", i64), ("rounds", i64)]


_SIGS = {
    "vrg_strict_create": [ctypes.c_int, vp, ctypes.c_double, i64, i64, ctypes.c_double, ctypes.POINTER(vp)],
    "vrg_strict_destroy": [vp],
    "vrg_strict_init": [vp, vp, vp],
    "vrg_strict_step": [vp, ctypes.POINTER(StrictResult)],
    "vrg_strict_run": [vp, ctypes.POINTER(StrictResult)],
    "vrg_strict_download": [vp, vp, vp],
    "vrg_strict_list": [vp, ctypes.c_int, vp, vp, vp, i64, ctypes.POINTER(i64)],
    "vrg_strict_get_trace": [vp, vp, i64, ctypes.POINTER(i64)],
    "vrg_strict_get_sums": [vp, vp, vp],
    "vrg_create": [ctypes.POINTER(Config), ctypes.POINTER(vp)],
    "vrg_destroy": [vp],
    "vrg_set_stream": [vp, vp],
    "vrg_upload": [vp, vp, vp],
    "vrg_upload_device": [vp, vp, vp],
    "vrg_upload_value_map": [vp, vp],
    "vrg_attach_device": [vp, vp, vp],
    "vrg_attach_device_typed": [vp, vp, vp, ctypes.c_int32],
    "vrg_attach_state_typed": [vp, vp, vp, ctypes.c_int32, vp, ctypes.c_int32],
    "vrg_scan_levels": [vp, ctypes.POINTER(i64)],
    "vrg_get_levels": [vp, vp, i64],
    "vrg_set_levels": [vp, vp, i64],
    "vrg_init": [vp],
    "vrg_run": [vp, ctypes.POINTER(Result)],
    "vrg_enqueue_decide": [vp],
    "vrg_enqueue_cancel": [vp],
    "vrg_enqueue_flip": [vp],
    "vrg_enqueue_absorb": [vp],
    "vrg_enqueue_advance": [vp],
    "vrg_poll": [vp, ctypes.POINTER(Result)],
    "vrg_dense_refresh_sweeps": [vp, ctypes.POINTER(i64)],
    "vrg_apply_flips": [vp, vp, i64, ctypes.POINTER(Result)],
    "vrg_apply_flips_device": [vp, vp, i64, ctypes.POINTER(Result)],
    "vrg_enqueue_table": [vp],
    "vrg_p2p_connect_local": [ctypes.POINTER(vp), ctypes.c_int],
    "vrg_labels_hash": [vp, ctypes.POINTER(ctypes.c_uint64)],
    "vrg_count_nonzero": [vp, ctypes.POINTER(i64)],
    "vrg_download_segmented_map_i64": [vp, vp],
    "vrg_profile": [vp, ctypes.c_int],
    "vrg_get_profile": [vp, vp, vp],
    "vrg_get_tail_profile": [vp, vp, ctypes.POINTER(i64)],
    "vrg_get_exp_evals": [vp, ctypes.POINTER(i64)],
    "vrg_exp_peak": [ctypes.c_int, ctypes.POINTER(ctypes.c_double)],
    "vrg_buffer_info": [vp, ctypes.c_int, ctypes.POINTER(vp), ctypes.POINTER(i64)],
    "vrg_plane_geometry": [vp, ctypes.POINTER(i64), ctypes.POINTER(i64), ctypes.POINTER(i64)],
    "vrg_use_separate_global_stats": [vp],
    "vrg_params_signature": [vp, ctypes.POINTER(ctypes.c_uint64)],
    "vrg_p2p_export": [vp, ctypes.c_int, vp],
    "vrg_p2p_connect": [vp, ctypes.c_int, ctypes.c_int, vp],
    "vrg_enqueue_p2p_halo": [vp, ctypes.c_int],
    "vrg_enqueue_p2p_stats": [vp],
    "vrg_download_labels": [vp, vp],
    "vrg_download_segmented_map": [vp, vp],
    "vrg_labels_device": [vp, vp],
    "vrg_labels_device_typed": [vp, vp, ctypes.c_int32, ctypes.c_int32],
    "vrg_segmented_device": [vp, vp, i64, ctypes.POINTER(i64)],
    "vrg_band_rows_device": [vp, ctypes.c_int32, vp, i64, ctypes.POINTER(i64)],
    "vrg_band_sums_device": [vp, vp, vp],
    "vrg_download_segmented": [vp, vp, i64, ctypes.POINTER(i64)],
    "vrg_get_trace": [vp, vp, i64, ctypes.POINTER(i64)],
    "vrg_get_table": [vp, vp, vp, i64],
    "vrg_get_table_levels": [vp, vp, i64],
    "vrg_get_band_sums": [vp, vp, vp, vp, i64, ctypes.POINTER(i64)],
    "vrg_edt": [ctypes.c_int, vp, vp, vp],
    "vrg_edt_device": [ctypes.c_int, vp, vp, vp, vp],
    "vrg_edt_ft": [ctypes.c_int, vp, vp, vp, vp, vp],
    "vrg_edt_ft_device": [ctypes.c_int, vp, vp, vp, vp, vp, vp],
    "vrg_release_scratch": [ctypes.c_int],
    "vrg_label_components": [ctypes.c_int, vp, vp, vp, ctypes.POINTER(i64), vp, i64],
    "vrg_label_components_device": [ctypes.c_int, vp, vp, vp, ctypes.POINTER(i64), vp, i64, vp],
    "vrg_vessel_mask": [ctypes.c_int, vp, vp, vp, ctypes.c_double, ctypes.c_double, ctypes.c_double, i64, vp, vp, vp],
    "vrg_vessel_mask_device": [ctypes.c_int, vp, vp, vp, ctypes.c_double, ctypes.c_double, ctypes.c_double, i64, vp, vp, vp, vp],
    "vrg_phantom_device": [ctypes.c_int, vp, i64, i64, vp, i64, vp, i64, i64, i64, i64, i64, ctypes.c_int, vp, vp],
}
EXPORTS = sorted(list(_SIGS) + ["vrg_last_error", "vrg_version"])

_lib = None


def library_path() -> str:
    return _build.LIB


def load(build_if_missing: bool = True):
    """Load libvrg_b200.so (building it first when nvcc is around).  Raises if that is impossible."""
    global _lib
    if _lib is not None:
        return _lib
    if build_if_missing and _build.find_nvcc() is not None:
        _build.build()  # serialised across processes by a file lock, written through a temporary file
    if not os.path.exists(_build.LIB):
        raise RuntimeError("vrg_b200: CUDA library %s is missing and cannot be built here (no nvcc); "
                           "there is no CPU fallback" % _build.LIB)
    lib = ctypes.CDLL(os.environ.get("VRG_B200_LIB") or _build.LIB)  # VRG_B200_LIB: an alternative build for A/B measurements
    for name, args in _SIGS.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = ctypes.c_int
    lib.vrg_last_error.restype = ctypes.c_char_p
    lib.vrg_version.restype = ctypes.c_int
    _lib = lib
    return lib


class LevelsError(ValueError):
    """More than 65536 distinct intensities: the level-table modes cannot run (VRG_ERR_LEVELS)."""


class VRGError(RuntimeError):
    def __init__(self, code, text):
        super().__init__("vrg_b200 error %d: %s" % (code, text))
        self.code = code


def check(rc: int):
    if rc != OK:
        text = load().vrg_last_error().decode("utf-8", "replace")
        if rc == ERR_LEVELS:
            raise LevelsError("vrg_b200: " + text)
        if rc in (ERR_ARG, ERR_LABEL, ERR_EMPTY_SEED, ERR_NO_BAND, ERR_NONFINITE):
            raise ValueError("vrg_b200: " + text)
        if rc == ERR_NOMEM:
            raise MemoryError("vrg_b200: " + text)
        raise VRGError(rc, text)
