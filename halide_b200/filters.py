"""Python call sites of the C-ABI filters, one function per exported symbol.

Same names, argument order and error behaviour as the generated AOT functions the reference's
harnesses call (apps/*/process.cpp, apps/blur/test.cpp): a negative halide_error_code_t becomes a
:class:`HalideError`.  Outputs are left device-dirty, exactly like a Halide GPU filter; call
``out.copy_to_host()`` to read them on the host.
"""
import ctypes

from .lib import lib, check


def halide_blur(input, blur_y):
    """apps/blur/halide_blur_generator.cpp: 3x3 box filter, uint16."""
    return check(lib.halide_blur(input.ptr, blur_y.ptr))


def local_laplacian(input, levels, alpha, beta, output):
    """apps/local_laplacian/local_laplacian_generator.cpp.  NOTE: like the harness
    (process.cpp:31) callers pass alpha already divided by (levels - 1)."""
    return check(lib.local_laplacian(input.ptr, ctypes.c_int32(levels), ctypes.c_float(alpha),
                                     ctypes.c_float(beta), output.ptr))


def stencil_chain(input, output):
    """apps/stencil_chain/stencil_chain_generator.cpp: 32 chained 5x5 uint16 stencils."""
    return check(lib.stencil_chain(input.ptr, output.ptr))


def bilateral_grid(input, r_sigma, output):
    """apps/bilateral_grid/bilateral_grid_generator.cpp (s_sigma = 8), float32."""
    return check(lib.bilateral_grid(input.ptr, ctypes.c_float(r_sigma), output.ptr))


def nl_means(input, patch_size, search_area, sigma, output):
    """apps/nl_means/nl_means_generator.cpp, float32, output has exactly 3 channels."""
    return check(lib.nl_means(input.ptr, ctypes.c_int32(patch_size), ctypes.c_int32(search_area),
                              ctypes.c_float(sigma), output.ptr))


def camera_pipe(input, matrix_3200, matrix_7000, color_temp, gamma, contrast, sharpen_strength, blackLevel, whiteLevel,
                processed):
    """apps/camera_pipe/camera_pipe_generator.cpp: uint16 Bayer raw -> uint8 RGB."""
    return check(lib.camera_pipe(input.ptr, matrix_3200.ptr, matrix_7000.ptr, ctypes.c_float(color_temp),
                                 ctypes.c_float(gamma), ctypes.c_float(contrast), ctypes.c_float(sharpen_strength),
                                 ctypes.c_int32(blackLevel), ctypes.c_int32(whiteLevel), processed.ptr))


def conv_layer(input, filter, bias, relu):
    """apps/conv_layer/conv_layer_generator.cpp: 3x3 conv + bias + relu, fixed shapes (N5 CI128 CO128 100x80), f32."""
    return check(lib.conv_layer(input.ptr, filter.ptr, bias.ptr, relu.ptr))


def harris(input, output):
    """apps/harris/harris_generator.cpp: Harris corner response, float32 (x, y, c) -> (x, y).  No boundary condition:
    the input must cover the output box grown by 2 in x and y, and channels 0..2."""
    return check(lib.harris(input.ptr, output.ptr))


def unsharp(input, output):
    """apps/unsharp/unsharp_generator.cpp (sigma 1.5): unsharp mask, float32 (x, y, c) -> (x, y, c).  The input is
    edge-clamped for the luma blur and must cover the output's (x, y, c) box."""
    return check(lib.unsharp(input.ptr, output.ptr))
