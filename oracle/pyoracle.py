"""ctypes binding of the CPU oracle (oracle/liboracle.so) — TEST INFRASTRUCTURE ONLY.

Importable from tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs; never from halide_b200/ (the product has no CPU path).
Arrays are numpy, indexed outermost-first ([c, y, x] / [y, x]) like halide_b200.buffer.
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "liboracle.so")
_REF_BLUR = os.path.join(_HERE, "_ref", "libref_blur.so")


class oracle_image_t(ctypes.Structure):
    _fields_ = [("base", ctypes.c_void_p), ("min", ctypes.c_int32 * 4), ("extent", ctypes.c_int32 * 4),
                ("stride", ctypes.c_int32 * 4)]


def build():
    subprocess.check_call(["make", "-C", _HERE, "-s"])


def _load():
    if not os.path.exists(_LIB):
        build()
    l = ctypes.CDLL(_LIB)
    for name in ("oracle_halide_exp", "oracle_halide_log", "oracle_fast_exp"):
        getattr(l, name).restype = ctypes.c_float
        getattr(l, name).argtypes = [ctypes.c_float]
    l.oracle_halide_pow.restype = ctypes.c_float
    l.oracle_halide_pow.argtypes = [ctypes.c_float, ctypes.c_float]
    l.oracle_ll_remap.restype = ctypes.c_float
    l.oracle_ll_remap.argtypes = [ctypes.c_int, ctypes.c_float]
    return l


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = _load()
    return _lib


def strict_float_lib():
    """The same oracle built with -DORACLE_STRICT_FLOAT (constant divisions stay IEEE divides, as in a Halide
    `strict_float` build; halide_math.h: div_const).  Not the parity target: kept for diffing against a future
    contraction-free Halide build (SURVEY.md §8c)."""
    path = os.path.join(_HERE, "liboracle_strict.so")
    if not os.path.exists(path):
        build()
    return ctypes.CDLL(path)


def image(arr, mins=None):
    """Describe a numpy array (outermost-first indexing) as an oracle_image_t."""
    img = oracle_image_t()
    img.base = arr.ctypes.data
    nd = arr.ndim
    for d in range(nd):
        img.extent[d] = arr.shape[nd - 1 - d]
        img.stride[d] = arr.strides[nd - 1 - d] // arr.itemsize
        img.min[d] = 0 if mins is None else mins[d]
    for d in range(nd, 4):
        img.extent[d] = 1
    img._keep = arr
    return img


def blur(inp, out_shape=None, in_mins=None, out_mins=None):
    """inp: uint16 [h, w]; returns uint16 [h-2, w-2] unless out_shape/mins say otherwise."""
    h, w = inp.shape
    if out_shape is None:
        out_shape = (h - 2, w - 2)
    out = np.zeros(out_shape, np.uint16)
    r = lib().oracle_blur(ctypes.byref(image(inp, in_mins)), ctypes.byref(image(out, out_mins)))
    if r != 0:
        raise RuntimeError(f"oracle_blur returned {r}")
    return out


def local_laplacian(inp, levels, alpha, beta, out_shape=None, in_mins=None, out_mins=None, pyramid_levels=8):
    """inp: uint16 [c, h, w]; alpha is the value the filter receives (already / (levels-1))."""
    if out_shape is None:
        out_shape = inp.shape
    out = np.zeros(out_shape, np.uint16)
    r = lib().oracle_local_laplacian(ctypes.byref(image(inp, in_mins)), ctypes.c_int(levels), ctypes.c_float(alpha),
                                     ctypes.c_float(beta), ctypes.byref(image(out, out_mins)),
                                     ctypes.c_int(pyramid_levels))
    if r != 0:
        raise RuntimeError(f"oracle_local_laplacian returned {r}")
    return out


def num_threads():
    return lib().oracle_num_threads()


def use_all_cores():
    """Undo torchrun's OMP_NUM_THREADS=1 for the CPU baseline: one OpenMP thread per available core."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    lib().oracle_set_num_threads(n)
    return n


def set_threads(n):
    lib().oracle_set_num_threads(int(n))


def ref_blur(inp, fast=False):
    """The REFERENCE's own C blur (apps/blur/test.cpp:18-33 / :35-132) via oracle/_ref.
    inp: uint16 [h, w] -> uint16 [h-2, w-8] (the shapes test.cpp uses)."""
    l = ctypes.CDLL(_REF_BLUR)
    h, w = inp.shape
    inp = np.ascontiguousarray(inp)
    out = np.zeros((h - 2, w - 8), np.uint16)
    l.ref_blur(inp.ctypes.data_as(ctypes.c_void_p), w, h, out.ctypes.data_as(ctypes.c_void_p), 1 if fast else 0)
    return out


def bilateral_grid(inp, r_sigma, out_shape=None, in_mins=None, out_mins=None, s_sigma=8):
    """inp: float32 [h, w]."""
    out = np.zeros(inp.shape if out_shape is None else out_shape, np.float32)
    r = lib().oracle_bilateral_grid(ctypes.byref(image(inp, in_mins)), ctypes.c_float(r_sigma),
                                    ctypes.byref(image(out, out_mins)), ctypes.c_int(s_sigma))
    if r != 0:
        raise RuntimeError(f"oracle_bilateral_grid returned {r}")
    return out


def nl_means(inp, patch_size, search_area, sigma, out_shape=None, in_mins=None, out_mins=None):
    """inp: float32 [3, h, w]."""
    out = np.zeros(inp.shape if out_shape is None else out_shape, np.float32)
    r = lib().oracle_nl_means(ctypes.byref(image(inp, in_mins)), ctypes.c_int(patch_size), ctypes.c_int(search_area),
                              ctypes.c_float(sigma), ctypes.byref(image(out, out_mins)))
    if r != 0:
        raise RuntimeError(f"oracle_nl_means returned {r}")
    return out


def stencil_chain(inp, out_shape=None, in_mins=None, out_mins=None, stencils=32):
    """inp: uint16 [h, w]."""
    out = np.zeros(inp.shape if out_shape is None else out_shape, np.uint16)
    r = lib().oracle_stencil_chain(ctypes.byref(image(inp, in_mins)), ctypes.byref(image(out, out_mins)),
                                   ctypes.c_int(stencils))
    if r != 0:
        raise RuntimeError(f"oracle_stencil_chain returned {r}")
    return out


def camera_pipe(raw, m3200, m7000, color_temp, gamma, contrast, sharpen_strength, black, white, out_shape, in_mins=None,
                out_mins=None):
    """raw: uint16 [h, w]; m3200/m7000: float32 [3, 4]; returns uint8 [3, H, W]."""
    out = np.zeros(out_shape, np.uint8)
    r = lib().oracle_camera_pipe(ctypes.byref(image(raw, in_mins)), ctypes.byref(image(m3200)), ctypes.byref(image(m7000)),
                                 ctypes.c_float(color_temp), ctypes.c_float(gamma), ctypes.c_float(contrast),
                                 ctypes.c_float(sharpen_strength), ctypes.c_int(black), ctypes.c_int(white),
                                 ctypes.byref(image(out, out_mins)))
    if r != 0:
        raise RuntimeError(f"oracle_camera_pipe returned {r}")
    return out


def conv_layer(inp, filt, bias):
    """inp: float32 [N, H+2, W+2, CI]; filt: [CI, 3, 3, CO]; bias: [CO] -> float32 [N, H, W, CO]."""
    n, hp, wp, ci = inp.shape
    co = bias.shape[0]
    out = np.zeros((n, hp - 2, wp - 2, co), np.float32)
    inp, filt, bias = (np.ascontiguousarray(a, np.float32) for a in (inp, filt, bias))
    f = ctypes.c_void_p
    lib().oracle_conv_layer(inp.ctypes.data_as(f), filt.ctypes.data_as(f), bias.ctypes.data_as(f), out.ctypes.data_as(f), n, ci, co,
                            wp - 2, hp - 2)
    return out
