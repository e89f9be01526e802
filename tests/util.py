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
