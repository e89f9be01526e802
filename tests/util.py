"""Shared helpers for the parity tests: seeded synthetic frames, C-ABI call wrappers, and the digests of what the
reference computed on the tests' inputs (tests/golden/reference_digests.json, tests/golden/make_reference_golden.py)."""
import functools
import hashlib
import json
import os

import numpy as np


@functools.lru_cache(maxsize=None)
def reference():
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_digests.json")) as f:
        return json.load(f)


def sha(data):
    """SHA-256 of a byte string, or of an array's elements in C order."""
    return hashlib.sha256(data if isinstance(data, bytes) else np.ascontiguousarray(data).tobytes()).hexdigest()


def u16_frame(shape, seed, bits=16):
    rng = np.random.default_rng(seed)
    a = rng.integers(0, 1 << 16, shape, dtype=np.uint16)
    if bits < 16:
        a &= np.uint16((1 << bits) - 1)
    return a


def smooth_u16_frame(shape, seed):
    """Low-frequency content + mild noise: exercises coherent LUT / plane selection paths."""
    rng = np.random.default_rng(seed)
    c, h, w = shape
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    out = np.empty(shape, np.uint16)
    for ch in range(c):
        base = 0.5 + 0.45 * np.sin(xx / (7.0 + ch) + seed) * np.cos(yy / (11.0 - ch))
        base += rng.normal(0, 0.02, (h, w))
        out[ch] = np.clip(base * 65535.0, 0, 65535).astype(np.uint16)
    return out


def f32_frame(shape, seed):
    rng = np.random.default_rng(seed)
    return rng.random(shape, dtype=np.float32)


def run_blur(hb, inp, out_shape, in_mins=None, out_mins=None):
    out = np.zeros(out_shape, np.uint16)
    bi = hb.HalideBuffer.from_numpy(inp, in_mins)
    bo = hb.HalideBuffer.from_numpy(out, out_mins, host_dirty=False)
    hb.filters.halide_blur(bi, bo)
    assert bo.device_dirty
    bo.copy_to_host()
    return out


def run_local_laplacian(hb, inp, levels, alpha, beta, out_shape=None, in_mins=None, out_mins=None):
    out = np.zeros(inp.shape if out_shape is None else out_shape, np.uint16)
    bi = hb.HalideBuffer.from_numpy(inp, in_mins)
    bo = hb.HalideBuffer.from_numpy(out, out_mins, host_dirty=False)
    hb.filters.local_laplacian(bi, levels, alpha, beta, bo)
    bo.copy_to_host()
    return out


# ---- conv_layer (fixed shapes of the generator) -------------------------------------------------------------------------
CONV_N, CONV_CI, CONV_CO, CONV_W, CONV_H = 5, 128, 128, 100, 80

# Per-output bound |got - ref| <= CONV_BOUND_C * (sum_k |filter_k * input_k| + |bias|) against the float64 contraction.
# Measured on a B200 (1000 W power limit) over the eight seeded data sets of tests/test_conv_layer_gpu.py, max ratio:
# 7.3e-6 for the 3xTF32 tensor-core path, 2.9e-6 for the FP32 SIMT path, 2.8e-6 for the float32 oracle (all on positive
# data, where the float32 accumulation of 1152 same-sign terms dominates; signed data: 5.6e-7, 3.6e-7, 3.9e-7).  c is 3x
# the largest.  A kernel missing a TF32 product gives at least 5.2e-5 (single round-to-nearest product), 7.1e-5 (the
# lo x hi product dropped) and 1.3e-4 (single truncating product) in a CPU emulation (tests/test_conv_layer_bound.py), so
# it fails the bound by a factor of 2 or more.
CONV_BOUND_C = 2.5e-5


def conv_make(seed, scale, signed=False, n=CONV_N):
    """Seeded conv_layer operands: input (n, H+2, W+2, CI), filter (CI, 3, 3, CO), bias (CO), uniform in [0, scale)
    (or [-scale/2, scale/2) for input and filter when `signed`; the bias stays positive)."""
    rng = np.random.default_rng(seed)
    inp = (rng.random((n, CONV_H + 2, CONV_W + 2, CONV_CI), dtype=np.float32) * scale).astype(np.float32)
    filt = (rng.random((CONV_CI, 3, 3, CONV_CO), dtype=np.float32) * scale).astype(np.float32)
    bias = (rng.random((CONV_CO,), dtype=np.float32) * scale).astype(np.float32)
    if signed:
        inp -= np.float32(0.5 * scale)
        filt -= np.float32(0.5 * scale)
    return inp, filt, bias


def conv_columns(inp, f=None):
    """The (n*H*W, 9*CI) matrix of taps of `inp` (ky, kx, ci order), each element mapped through `f`, in float64."""
    n = inp.shape[0]
    cols = np.empty((n, CONV_H, CONV_W, 3, 3, CONV_CI), np.float64)
    for ky in range(3):
        for kx in range(3):
            v = inp[:, ky:ky + CONV_H, kx:kx + CONV_W, :]
            cols[:, :, :, ky, kx, :] = v if f is None else f(v)
    return cols.reshape(-1, 9 * CONV_CI)


def conv_weights(filt, f=None):
    """The (9*CI, CO) matrix of filter taps matching conv_columns, in float64."""
    v = filt if f is None else f(filt)
    return np.asarray(v, np.float64).transpose(1, 2, 0, 3).reshape(9 * CONV_CI, CONV_CO)


def conv_reference_f64(inp, filt, bias):
    """(relu(bias + sum of taps) in float64, sum of |terms| + |bias|), both shaped like the output (n, H, W, CO)."""
    a, b = conv_columns(inp), conv_weights(filt)
    shape = (inp.shape[0], CONV_H, CONV_W, CONV_CO)
    ref = np.maximum(a @ b + bias.astype(np.float64), 0.0).reshape(shape)
    mag = (np.abs(a) @ np.abs(b) + np.abs(bias.astype(np.float64))).reshape(shape)
    return ref, mag


def conv_bound_ratio(got, ref, mag):
    """Largest |got - ref| / (sum |terms| + |bias|) over all outputs."""
    return float(np.max(np.abs(got.astype(np.float64) - ref) / mag))
