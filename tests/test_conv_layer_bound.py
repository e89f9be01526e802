"""CPU test of the power of conv_layer's float64 error bound (tests/util.py CONV_BOUND_C): on one image, a numpy emulation
of the tensor-core kernel's 3xTF32 split and the float32 oracle meet it, and the degraded kernels it is meant to catch
(the lo x hi product dropped, a single TF32 product truncating or rounding) violate it."""
import numpy as np
import pytest

from util import CONV_BOUND_C, conv_bound_ratio, conv_columns, conv_make, conv_reference_f64, conv_weights, CONV_H, CONV_W, CONV_CO


def tf32(x, rounding):
    """float32 -> TF32 (10 mantissa bits) by truncation (the kernel's split) or round-to-nearest-even."""
    b = np.asarray(x, np.float32).view(np.uint32).astype(np.uint64)
    if rounding:
        b = b + 0xFFF + ((b >> 13) & 1)
    return (b & ~np.uint64(0x1FFF)).astype(np.uint32).view(np.float32)


def split(x):
    """hi = tf32(x) truncated, lo = x - hi in float32, truncated again by the MMA's TF32 read."""
    hi = tf32(x, False)
    return hi, tf32(np.asarray(x, np.float32) - hi, False)


def emulate(inp, filt, bias, variant):
    ah, al = split(inp)
    bh, bl = split(filt)
    if variant == "3xtf32":
        acc = conv_columns(ah) @ conv_weights(bh) + conv_columns(ah) @ conv_weights(bl) + conv_columns(al) @ conv_weights(bh)
    elif variant == "lo_x_hi_dropped":
        acc = conv_columns(ah) @ conv_weights(bh) + conv_columns(ah) @ conv_weights(bl)
    else:
        rounding = variant == "1xtf32_rn"
        acc = conv_columns(inp, lambda v: tf32(v, rounding)) @ conv_weights(filt, lambda v: tf32(v, rounding))
    out = np.maximum(acc + bias.astype(np.float64), 0.0)
    return out.reshape(inp.shape[0], CONV_H, CONV_W, CONV_CO)


@pytest.fixture(scope="module", params=["positive", "signed"])
def one_image(request):
    inp, filt, bias = conv_make(0 if request.param == "positive" else 2, 1.0, signed=request.param == "signed")
    inp = inp[:1].copy()
    return inp, filt, bias, conv_reference_f64(inp, filt, bias)


def test_three_product_split_meets_the_bound(one_image):
    inp, filt, bias, (ref, mag) = one_image
    assert conv_bound_ratio(emulate(inp, filt, bias, "3xtf32"), ref, mag) <= CONV_BOUND_C


@pytest.mark.parametrize("variant", ["lo_x_hi_dropped", "1xtf32_rz", "1xtf32_rn"])
def test_degraded_kernels_violate_the_bound(one_image, variant):
    inp, filt, bias, (ref, mag) = one_image
    assert conv_bound_ratio(emulate(inp, filt, bias, variant), ref, mag) > CONV_BOUND_C


def test_float32_oracle_meets_the_bound(oracle, one_image):
    inp, filt, bias, (ref, mag) = one_image
    full_inp = np.concatenate([inp] + [np.zeros_like(inp)] * 4)  # the oracle takes the generator's fixed shapes
    got = oracle.conv_layer(full_inp, filt, bias)[:1]
    assert conv_bound_ratio(got, ref, mag) <= CONV_BOUND_C
