"""ctypes binding of the CPU oracle of harris and unsharp (oracle/liboracle_apps.so, built by oracle/apps.mk) — TEST
INFRASTRUCTURE ONLY.  Same conventions as oracle/pyoracle.py: numpy arrays indexed outermost-first ([c, y, x] / [y, x]),
optional Halide mins per dimension (x first)."""
import ctypes
import os
import subprocess

import numpy as np

from .pyoracle import image

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "liboracle_apps.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB):
            subprocess.check_call(["make", "-C", _HERE, "-s", "-f", "apps.mk", "liboracle_apps.so"])
        _lib = ctypes.CDLL(_LIB)
    return _lib


def unsharp_weights():
    """kernel(0..3) of unsharp as float32 (folded in double and rounded, see oracle_unsharp.cpp)."""
    w = np.zeros(4, np.float32)
    lib().oracle_unsharp_weights(w.ctypes.data_as(ctypes.c_void_p))
    return w


def harris(inp, out_shape=None, in_mins=None, out_mins=None):
    """inp: float32 [c, h, w]; returns float32 [h-6, w-6] at mins (3, 3) unless out_shape / mins say otherwise (the
    harness geometry, apps/harris/filter.cpp:25-26)."""
    if out_shape is None:
        out_shape = (inp.shape[1] - 6, inp.shape[2] - 6)
        if out_mins is None:
            base = (0, 0) if in_mins is None else in_mins[:2]
            out_mins = (base[0] + 3, base[1] + 3)
    out = np.zeros(out_shape, np.float32)
    r = lib().oracle_harris(ctypes.byref(image(inp, in_mins)), ctypes.byref(image(out, out_mins)))
    if r != 0:
        raise RuntimeError(f"oracle_harris returned {r}")
    return out


def unsharp(inp, out_shape=None, in_mins=None, out_mins=None):
    """inp: float32 [c, h, w]; returns float32 of out_shape (default: inp's shape)."""
    out = np.zeros(inp.shape if out_shape is None else out_shape, np.float32)
    r = lib().oracle_unsharp(ctypes.byref(image(inp, in_mins)), ctypes.byref(image(out, out_mins)))
    if r != 0:
        raise RuntimeError(f"oracle_unsharp returned {r}")
    return out
