"""CPU tests of the drop-in boundary: the library loads and exports every symbol include/*.h
declares; struct layouts match the LP64 facts of src/runtime/HalideRuntime.h:1657-1737; every F_metadata() record
matches the committed snapshot; every F_argv unpacks its arguments as F declares them."""
import ctypes
import glob
import importlib.util
import json
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def _load_metadata_dumper():
    spec = importlib.util.spec_from_file_location("make_abi_metadata", os.path.join(GOLDEN, "make_abi_metadata.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


META = _load_metadata_dumper()
with open(os.path.join(GOLDEN, "abi_metadata.json")) as _f:
    SNAPSHOT = json.load(_f)
FILTERS = sorted(SNAPSHOT)


def _declared_symbols():
    syms = set()
    for h in glob.glob(os.path.join(ROOT, "include", "*.h")):
        text = open(h).read()
        text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
        text = re.sub(r"//[^\n]*", "", text)
        for m in re.finditer(r"^(?!typedef\b)[A-Za-z_][\w \*]*?\b(\w+)\s*\([^;{]*\)\s*;", text, flags=re.M):
            syms.add(m.group(1))
    return sorted(syms)


def test_library_exports_every_declared_symbol(hb):
    l = hb.load_library()
    declared = _declared_symbols()
    assert "local_laplacian" in declared and "halide_blur" in declared and "halide_copy_to_host" in declared
    missing = [s for s in declared if not hasattr(l, s)]
    assert not missing, f"declared in include/*.h but not exported: {missing}"


def test_struct_layout(hb):
    from halide_b200.buffer import halide_buffer_t, halide_dimension_t
    assert ctypes.sizeof(halide_buffer_t) == 56
    offs = {f: getattr(halide_buffer_t, f).offset for f, _ in halide_buffer_t._fields_}
    assert offs == {"device": 0, "device_interface": 8, "host": 16, "flags": 24, "type": 32, "dimensions": 36,
                    "dim": 40, "padding": 48}
    assert ctypes.sizeof(halide_dimension_t) == 16


def test_metadata_and_target(hb):
    """tests/golden/abi_metadata.json holds one record per filter header, and every filter reports the library's own
    target string."""
    l = hb.load_library()
    assert FILTERS == META.filter_functions()
    target = hb.capi.halide_b200_target().decode()
    assert target.endswith("b200_native")
    assert [META.dump(l, fn)["target"] for fn in FILTERS] == [target] * len(FILTERS)


@pytest.mark.parametrize("fn", FILTERS)
def test_metadata_matches_snapshot(hb, fn):
    """The library reports each F_metadata() record of the snapshot field for field: names, kinds, types, scalar and
    buffer estimates, target and name."""
    assert META.dump(hb.load_library(), fn) == SNAPSHOT[fn]


_DTYPES = {(0, 32): np.int32, (1, 8): np.uint8, (1, 16): np.uint16, (2, 32): np.float32}


@pytest.mark.parametrize("fn", FILTERS)
def test_argv_matches_direct_call(hb, fn):
    """F_argv(args) is F called with *args[i] for scalars and args[i] for buffers (src/CodeGen_C.cpp:675-705).  Every
    buffer is a bounds query, which F answers before any CUDA call: both calls must return 0 and propose the same
    shapes.  Each buffer starts from its metadata estimates shifted by its position, so a swapped pair shows."""
    from halide_b200 import HalideBuffer
    from halide_b200.buffer import halide_buffer_t
    l = hb.load_library()
    args = SNAPSHOT[fn]["arguments"]

    def call(via_argv):
        bufs, values = [], []
        for i, a in enumerate(args):
            if a["kind"] == 0:
                values.append((ctypes.c_int32 if a["type"][0] == 0 else ctypes.c_float)(a["scalar_estimate"]))
            else:
                est = a["buffer_estimates"] or [0, 64] * a["dimensions"]
                b = HalideBuffer(_DTYPES[tuple(a["type"][:2])], est[1::2], mins=[m + i for m in est[0::2]])
                bufs.append(b)
                values.append(b.buf)
        if via_argv:
            argv = (ctypes.c_void_p * len(values))(*[ctypes.addressof(v) for v in values])
            rc = getattr(l, fn + "_argv")(argv)
        else:
            rc = getattr(l, fn)(*[ctypes.byref(v) if isinstance(v, halide_buffer_t) else v for v in values])
        return rc, [b.shape() for b in bufs]

    direct, via_argv = call(False), call(True)
    assert direct[0] == 0 and via_argv == direct


def test_validation_errors_without_gpu(hb):
    """Argument checks run before any CUDA call, so they are testable on a CPU-only box
    (codes pinned by test/generator/error_codes_aottest.cpp:38-135)."""
    import numpy as np
    from halide_b200 import HalideBuffer, HalideError, filters
    img = np.zeros((3, 16, 16), np.uint16)
    out = np.zeros((3, 16, 16), np.uint16)
    bi, bo = HalideBuffer.from_numpy(img), HalideBuffer.from_numpy(out)
    # wrong element type -> -3
    bad = HalideBuffer.from_numpy(np.zeros((3, 16, 16), np.float32))
    with pytest.raises(HalideError) as e:
        filters.local_laplacian(bad, 8, 1 / 7, 1.0, bo)
    assert e.value.code == -3
    # wrong dimensionality -> -43
    bad2 = HalideBuffer.from_numpy(np.zeros((16, 16), np.uint16))
    with pytest.raises(HalideError) as e:
        filters.local_laplacian(bad2, 8, 1 / 7, 1.0, bo)
    assert e.value.code == -43
    # null buffer -> -12
    l = hb.load_library()
    assert l.local_laplacian(None, 8, ctypes.c_float(0.1), ctypes.c_float(1.0), bo.ptr) == -12
    # input smaller than the output region -> -4
    small = HalideBuffer.from_numpy(np.zeros((1, 16, 16), np.uint16))
    with pytest.raises(HalideError) as e:
        filters.local_laplacian(small, 8, 1 / 7, 1.0, bo)
    assert e.value.code == -4
    # stride[0] != 1 -> -8
    bi.dims[0].stride = 2
    with pytest.raises(HalideError) as e:
        filters.local_laplacian(bi, 8, 1 / 7, 1.0, bo)
    assert e.value.code == -8
    # blur: input must cover output + 2 -> -4
    b_in = HalideBuffer.from_numpy(np.zeros((10, 10), np.uint16))
    b_out = HalideBuffer.from_numpy(np.zeros((10, 10), np.uint16))
    with pytest.raises(HalideError) as e:
        filters.halide_blur(b_in, b_out)
    assert e.value.code == -4


def test_bounds_query_mode(hb):
    """A buffer with null host and device turns the call into a bounds query
    (HalideRuntime.h:1851-1853, src/AddImageChecks.cpp:477-496): shapes are written, nothing runs."""
    import numpy as np
    from halide_b200 import HalideBuffer, filters
    out = HalideBuffer.from_numpy(np.zeros((20, 30), np.uint16), mins=(5, 7))
    q = HalideBuffer.bounds_query(np.uint16, 2)
    assert filters.halide_blur(q, out) == 0
    assert q.shape() == [(5, 32, 1), (7, 22, 32)]
    out3 = HalideBuffer.from_numpy(np.zeros((3, 20, 30), np.uint16))
    q3 = HalideBuffer.bounds_query(np.uint16, 3)
    assert filters.local_laplacian(q3, 8, 1 / 7, 1.0, out3) == 0
    assert q3.shape() == [(0, 30, 1), (0, 20, 30), (0, 3, 600)]


def _expect(code, fn, *args):
    from halide_b200 import HalideError
    with pytest.raises(HalideError) as e:
        fn(*args)
    assert e.value.code == code, (e.value.code, e.value.message)


def test_per_filter_validation_without_gpu(hb):
    """Every filter validates before touching CUDA: wrong types / shapes / regions return the generated-code error codes."""
    import numpy as np
    from halide_b200 import HalideBuffer as B, filters as F
    f32, u16, u8 = np.float32, np.uint16, np.uint8
    # bilateral_grid: float 2-D in/out, input must cover the output
    _expect(-3, F.bilateral_grid, B.from_numpy(np.zeros((8, 8), u16)), 0.1, B.from_numpy(np.zeros((8, 8), f32)))
    _expect(-4, F.bilateral_grid, B.from_numpy(np.zeros((8, 8), f32)), 0.1, B.from_numpy(np.zeros((9, 8), f32)))
    _expect(-9, F.bilateral_grid, B.from_numpy(np.zeros((8, 8), f32)), 0.0, B.from_numpy(np.zeros((8, 8), f32)))
    # nl_means: 3-D float, output channels fixed to [0,3)
    _expect(-43, F.nl_means, B.from_numpy(np.zeros((8, 8), f32)), 3, 7, 0.12, B.from_numpy(np.zeros((3, 8, 8), f32)))
    _expect(-8, F.nl_means, B.from_numpy(np.zeros((3, 8, 8), f32)), 3, 7, 0.12, B.from_numpy(np.zeros((4, 8, 8), f32)))
    _expect(-9, F.nl_means, B.from_numpy(np.zeros((3, 8, 8), f32)), 0, 7, 0.12, B.from_numpy(np.zeros((3, 8, 8), f32)))
    # stencil_chain: u16 2-D; stride[0] must be 1
    _expect(-3, F.stencil_chain, B.from_numpy(np.zeros((8, 8), f32)), B.from_numpy(np.zeros((8, 8), u16)))
    bad = B.from_numpy(np.zeros((8, 8), u16))
    bad.dims[0].stride = 2
    _expect(-8, F.stencil_chain, bad, B.from_numpy(np.zeros((8, 8), u16)))
    # conv_layer: fixed shapes and strides (generator constraints)
    ok_in, ok_f, ok_b = np.zeros((5, 82, 102, 128), f32), np.zeros((128, 3, 3, 128), f32), np.zeros((128,), f32)
    _expect(-8, F.conv_layer, B.from_numpy(ok_in), B.from_numpy(ok_f), B.from_numpy(ok_b), B.from_numpy(np.zeros((5, 80, 100, 64), f32)))
    _expect(-43, F.conv_layer, B.from_numpy(ok_in), B.from_numpy(ok_f), B.from_numpy(np.zeros((1, 128), f32)),
            B.from_numpy(np.zeros((5, 80, 100, 128), f32)))
    # camera_pipe: raw must cover the stencil footprint after the (16,12) shift; output is u8 with at most channels 0..2
    m = np.zeros((3, 4), f32)
    _expect(-4, F.camera_pipe, B.from_numpy(np.zeros((64, 64), u16)), B.from_numpy(m), B.from_numpy(m), 3700.0, 2.0, 50.0, 1.0, 25, 1023,
            B.from_numpy(np.zeros((3, 64, 64), u8)))
    _expect(-3, F.camera_pipe, B.from_numpy(np.zeros((120, 160), u16)), B.from_numpy(m), B.from_numpy(m), 3700.0, 2.0, 50.0, 1.0, 25, 1023,
            B.from_numpy(np.zeros((3, 64, 96), u16)))
    # local_laplacian: levels range
    _expect(-9, F.local_laplacian, B.from_numpy(np.zeros((3, 8, 8), u16)), 1, 1.0, 1.0, B.from_numpy(np.zeros((3, 8, 8), u16)))


def test_per_filter_bounds_queries(hb):
    import numpy as np
    from halide_b200 import HalideBuffer as B, filters as F
    # camera_pipe asks for the shifted footprint of the output region (harness: 2560x1920 out of a 2592x1968 raw)
    q = B.bounds_query(np.uint16, 2)
    m = np.zeros((3, 4), np.float32)
    out = B.from_numpy(np.zeros((3, 1920, 2560), np.uint8))
    assert F.camera_pipe(q, B.from_numpy(m), B.from_numpy(m), 3700.0, 2.0, 50.0, 1.0, 25, 1023, out) == 0
    (x0, w, _), (y0, h, _) = q.shape()
    assert x0 >= 0 and y0 >= 0 and x0 + w <= 2592 and y0 + h <= 1968  # fits the harness's raw frame
    # conv_layer proposes its fixed shapes
    qi, qf, qb = B.bounds_query(np.float32, 4), B.bounds_query(np.float32, 4), B.bounds_query(np.float32, 1)
    qo = B.bounds_query(np.float32, 4)
    assert F.conv_layer(qi, qf, qb, qo) == 0
    assert [e for (_, e, _) in qi.shape()] == [128, 102, 82, 5] and [e for (_, e, _) in qo.shape()] == [128, 100, 80, 5]
    # nl_means: every access is clamped -> input region == output region, 3 channels
    q3 = B.bounds_query(np.float32, 3)
    assert F.nl_means(q3, 3, 7, 0.12, B.from_numpy(np.zeros((3, 20, 30), np.float32))) == 0
    assert [e for (_, e, _) in q3.shape()] == [30, 20, 3]


def test_sharded_entry_point_requires_the_communicator(hb):
    """halide_b200_local_laplacian_sharded validates like the plain filter and then refuses to run without
    halide_b200_dist_init (host-only checks: no CUDA call before them)."""
    import ctypes
    import numpy as np
    from halide_b200 import HalideBuffer as B
    img = np.zeros((3, 64, 64), np.uint16)
    bi, bo = B.from_numpy(img), B.from_numpy(np.zeros_like(img), host_dirty=False)
    with pytest.raises(hb.HalideError) as e:
        hb.lib.check(hb.capi.halide_b200_local_laplacian_sharded(bi.ptr, ctypes.c_int32(8), ctypes.c_float(1 / 7), ctypes.c_float(1.0),
                                                                  bo.ptr, ctypes.c_int32(0), ctypes.c_int32(64)))
    assert "halide_b200_dist_init" in str(e.value)
    assert hb.capi.halide_b200_dist_rank() == 0 and hb.capi.halide_b200_dist_size() == 1
    # type errors are reported before anything else, with the reference's code
    bad = B.from_numpy(np.zeros((3, 64, 64), np.float32))
    rc = hb.capi.halide_b200_local_laplacian_sharded(bad.ptr, ctypes.c_int32(8), ctypes.c_float(1 / 7), ctypes.c_float(1.0), bo.ptr,
                                                    ctypes.c_int32(0), ctypes.c_int32(64))
    assert rc == -3
