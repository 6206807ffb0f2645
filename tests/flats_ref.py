"""ctypes binding of flats_ref.cpp: the reference for exact depression filling and flat resolution.

The library is compiled on first use into a temporary directory (keyed by the source's hash), so the tests never write
into the repository tree."""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "flats_ref.cpp")
_LIB = None
_i64 = ctypes.c_int64


def _lib():
    global _LIB
    if _LIB is None:
        tag = hashlib.sha256(open(_SRC, "rb").read()).hexdigest()[:16]
        path = os.path.join(tempfile.gettempdir(), f"dtb_flats_ref_{os.getuid()}_{tag}.so")
        if not os.path.exists(path):
            tmp = f"{path}.{os.getpid()}"
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", _SRC, "-o", tmp])
            os.replace(tmp, path)
        _LIB = ctypes.CDLL(path)
        _LIB.ref_resolve_flats_f32.restype = _i64
        _LIB.ref_resolve_flats_i16.restype = _i64
    return _LIB


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def priority_flood(dem: np.ndarray) -> np.ndarray:
    """F1: priority flood without epsilon (float32 out; int16 elevations are exact in float32)"""
    out = np.array(dem, dtype=np.float32, order="C", copy=True)
    _lib().ref_priority_flood_f32(_p(out), _i64(out.shape[0]), _i64(out.shape[1]))
    return out


def resolve_flats(dem: np.ndarray, d8: np.ndarray, with_mask: bool = False):
    """F2: (resolved d8, unresolved cells, flat cells[, mask int64: -1 off the flats, INT64_MAX in undrained flats])"""
    lib = _lib()
    if dem.dtype == np.int16:
        d, fn = np.ascontiguousarray(dem), lib.ref_resolve_flats_i16
    else:
        d, fn = np.ascontiguousarray(dem, dtype=np.float32), lib.ref_resolve_flats_f32
    out = np.array(d8, dtype=np.uint8, order="C", copy=True)
    n_flat = _i64(0)
    mask = np.empty(d.shape, np.int64) if with_mask else None
    left = fn(_p(d), _p(out), _i64(d.shape[0]), _i64(d.shape[1]), ctypes.byref(n_flat), _p(mask) if with_mask else None)
    return (out, int(left), int(n_flat.value)) + ((mask,) if with_mask else ())
