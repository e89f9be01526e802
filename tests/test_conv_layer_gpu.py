"""GPU parity tests for conv_layer through the C ABI (fixed shapes of the generator).  Float pipeline: 1e-4 relative
against the oracle, and a per-output bound against the float64 contraction (tests/util.py CONV_BOUND_C)."""
import numpy as np
import pytest

from util import CONV_BOUND_C, conv_bound_ratio, conv_make, conv_reference_f64

pytestmark = pytest.mark.gpu
N, CI, CO, W, H = 5, 128, 128, 100, 80


def make(seed, scale):
    rng = np.random.default_rng(seed)
    inp = (rng.random((N, H + 2, W + 2, CI), dtype=np.float32) * scale).astype(np.float32)
    filt = (rng.random((CI, 3, 3, CO), dtype=np.float32) * scale).astype(np.float32)
    bias = (rng.random((CO,), dtype=np.float32) * scale).astype(np.float32)
    return inp, filt, bias


def run(hb, inp, filt, bias):
    out = np.zeros((N, H, W, CO), np.float32)
    bi, bf, bb = hb.HalideBuffer.from_numpy(inp), hb.HalideBuffer.from_numpy(filt), hb.HalideBuffer.from_numpy(bias)
    bo = hb.HalideBuffer.from_numpy(out, host_dirty=False)
    hb.filters.conv_layer(bi, bf, bb, bo)
    bo.copy_to_host()
    return out


@pytest.mark.parametrize("seed,scale", [(0, 1.0), (1, 2147483648.0)])  # the harness fills with raw rand() up to 2^31
def test_matches_oracle(hb, oracle, seed, scale):
    inp, filt, bias = make(seed, scale)
    got = run(hb, inp, filt, bias)
    want = oracle.conv_layer(inp, filt, bias)
    err = np.abs(got - want) / np.maximum(np.abs(want), 1e-30)
    assert np.isfinite(got).all() and err.max() <= 1e-4, err.max()


def test_signed_data_and_relu(hb, oracle):
    """Mixed signs cancel, so the error is bounded against the magnitude of the accumulated terms, not of the result,
    and against the float64 contraction rather than the float32 oracle."""
    inp, filt, bias = conv_make(2, 1.0, signed=True)
    got = run(hb, inp, filt, bias)
    assert (got >= 0).all() and (got == 0).any() and (got > 0).any()
    ref, mag = conv_reference_f64(inp, filt, bias)
    assert conv_bound_ratio(got, ref, mag) <= CONV_BOUND_C


@pytest.mark.parametrize("data", ["positive", "signed", "2^31"])
@pytest.mark.parametrize("tc", [1, 0])
def test_error_bound_against_float64(hb, oracle, tc, data):
    """|got - ref| <= c * (sum |terms| + |bias|) per output against the float64 contraction, for the 3xTF32 tensor-core
    path and the FP32 SIMT path, with c = CONV_BOUND_C (tests/util.py: 3x the largest ratio measured for either path and
    for the float32 oracle, and at least 2x below what a kernel with a TF32 product missing gives).  The oracle must meet
    it too, and the 1e-4 relative bar against the oracle still holds on positive data."""
    seed, scale, signed = {"positive": (6, 1.0, False), "signed": (7, 1.0, True), "2^31": (8, 2147483648.0, False)}[data]
    inp, filt, bias = conv_make(seed, scale, signed)
    l = hb.load_library()
    try:
        l.halide_b200_conv_use_tensor_cores(tc)
        got = run(hb, inp, filt, bias)
    finally:
        l.halide_b200_conv_use_tensor_cores(1)
    ref, mag = conv_reference_f64(inp, filt, bias)
    want = oracle.conv_layer(inp, filt, bias)
    assert np.isfinite(got).all()
    assert conv_bound_ratio(want, ref, mag) <= CONV_BOUND_C
    assert conv_bound_ratio(got, ref, mag) <= CONV_BOUND_C, conv_bound_ratio(got, ref, mag)
    if not signed:
        assert (np.abs(got - want) / np.abs(want)).max() <= 1e-4


def test_wrong_shape_is_a_constraint_violation(hb):
    from halide_b200 import HalideBuffer, HalideError, filters
    inp, filt, bias = make(0, 1.0)
    bi = HalideBuffer.from_numpy(inp[:, :, :-1, :].copy())
    bf, bb = HalideBuffer.from_numpy(filt), HalideBuffer.from_numpy(bias)
    bo = HalideBuffer.from_numpy(np.zeros((N, H, W, CO), np.float32))
    with pytest.raises(HalideError) as e:
        filters.conv_layer(bi, bf, bb, bo)
    assert e.value.code == -8


@pytest.mark.parametrize("seed,scale", [(3, 1.0), (4, 2147483648.0)])
def test_simt_path_matches_oracle(hb, oracle, seed, scale):
    """The default path is the tcgen05 implicit GEMM (TMA + TMEM, 3xTF32 split); the FP32 SIMT kernel it replaced stays
    selectable (HALIDE_B200_CONV=simt) and must meet the same 1e-4 bar."""
    l = hb.load_library()
    inp, filt, bias = make(seed, scale)
    want = oracle.conv_layer(inp, filt, bias)
    try:
        l.halide_b200_conv_use_tensor_cores(0)
        got = run(hb, inp, filt, bias)
    finally:
        l.halide_b200_conv_use_tensor_cores(1)
    err = np.abs(got - want) / np.maximum(np.abs(want), 1e-30)
    assert np.isfinite(got).all() and err.max() <= 1e-4, err.max()
