"""TEST INFRASTRUCTURE ONLY -- CPU restatement of ``scipy.ndimage.distance_transform_edt(mask, sampling=...,
return_indices=True)``.  Only ``tests/``, ``scripts/`` and ``__graft_entry__`` may import this; the product path
(``arterynetwork_b200``) never does.

* ``ft_oracle``        the feature transform: int32 (3, Z, Y, X), for every voxel the coordinates of its nearest zero
                       voxel, with SciPy's pass order, tie rule and fp64 order of evaluation (``oracle/ft_oracle.c``)
* ``distances_from_ft`` the float64 distances SciPy derives from it, in NumPy exactly as SciPy does

Parity status: PINNED to SciPy 1.18 by ``tests/test_edt_ft_oracle.py``.
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "ft_oracle.c")
LIB = os.path.join(HERE, "_build", "libft_oracle.so")

_lib = None


def build(force: bool = False) -> str:
    if force or not os.path.exists(LIB) or os.path.getmtime(LIB) < os.path.getmtime(SRC):
        os.makedirs(os.path.dirname(LIB), exist_ok=True)
        tmp = LIB + ".tmp.%d" % os.getpid()
        subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-o", tmp, SRC])
        os.replace(tmp, LIB)
    return LIB


def _load():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build())
        i64, p = ctypes.c_int64, ctypes.c_void_p
        _lib.ft_oracle.restype = ctypes.c_int
        _lib.ft_oracle.argtypes = [p, i64, i64, i64, p, p]
    return _lib


def _spacing(sampling):
    if sampling is None:
        return None
    s = np.broadcast_to(np.asarray(sampling, dtype=np.float64), (3,))
    return np.ascontiguousarray(s)


def ft_oracle(mask, sampling=None) -> np.ndarray:
    """int32 (3, Z, Y, X): the coordinates of each voxel's nearest zero voxel as SciPy picks it (-1 where the mask has no
    zero voxel at all)."""
    m = np.ascontiguousarray(np.asarray(mask) != 0, dtype=np.uint8)
    if m.ndim != 3:
        raise ValueError("3-D volumes only")
    s = _spacing(sampling)
    ft = np.empty((3,) + m.shape, dtype=np.int32)
    rc = _load().ft_oracle(m.ctypes.data, *m.shape, None if s is None else s.ctypes.data, ft.ctypes.data)
    if rc != 0:
        raise MemoryError("feature transform oracle")
    return ft


def distances_from_ft(ft, sampling=None) -> np.ndarray:
    """float64 distances from a feature transform, in SciPy's order: per axis (feature - index) as float64, times the
    spacing, squared, summed over the axes one after the other, square root."""
    dt = (ft - np.indices(ft.shape[1:], dtype=ft.dtype)).astype(np.float64)
    s = _spacing(sampling)
    if s is not None:
        for i in range(3):
            dt[i] *= s[i]
    np.multiply(dt, dt, dt)
    return np.sqrt(np.add.reduce(dt, axis=0))
