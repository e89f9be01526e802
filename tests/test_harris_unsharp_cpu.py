"""CPU tests of harris and unsharp: the oracle against the committed golden vectors and against the independent numpy
restatement (oracle/np_restatement_apps.py), the folded unsharp weights, and the C-ABI entry points up to the first
CUDA call (export, metadata, validation error codes, bounds queries, a C caller that links)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from util import f32_frame

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
INC = os.path.join(ROOT, "include")
LIBDIR = os.path.join(ROOT, "halide_b200")
ENTRY_POINTS = [f + s for f in ("harris", "unsharp") for s in ("", "_argv", "_metadata", "_auto_schedule", "_auto_schedule_argv",
                                                              "_auto_schedule_metadata")]


@pytest.fixture(scope="module")
def apps():
    from oracle import pyoracle_apps
    return pyoracle_apps


@pytest.fixture(scope="module")
def npr():
    from oracle import np_restatement_apps
    return np_restatement_apps


def smooth_f32(shape, seed):
    """Low-frequency colour content with mild noise, in [0, 1]."""
    rng = np.random.default_rng(seed)
    c, h, w = shape
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    out = np.empty(shape, np.float32)
    for ch in range(c):
        base = 0.5 + 0.45 * np.sin(xx / (6.0 + ch) + seed) * np.cos(yy / (9.0 - ch))
        out[ch] = np.clip(base + rng.normal(0, 0.01, (h, w)), 0, 1)
    return out


def black_patches(a):
    """Zero every channel in a few boxes (gray == 0 there: ratio is +-inf or NaN); a 4th channel, when present, stays
    non-zero, so ratio * input is +-inf rather than NaN at the patch edges."""
    a = a.copy()
    h, w = a.shape[1:]
    for (y, x, hh, ww) in ((2, 3, 5, 7), (h // 2, w // 3, 6, 4), (h - 4, w - 6, 4, 6), (0, 0, 2, 2)):
        a[:3, y:y + hh, x:x + ww] = 0.0
    return a


def same(got, want, what=""):
    assert got.shape == want.shape, (what, got.shape, want.shape)
    bad = np.argwhere(~((got == want) | (np.isnan(got) & np.isnan(want))))
    assert bad.size == 0, f"{what}: {len(bad)} mismatches, first at {tuple(bad[0])}: {got[tuple(bad[0])]} vs {want[tuple(bad[0])]}"


# ---- oracle vs golden vectors and vs the numpy restatement ---------------------------------------------------------------

def test_goldens_bit_exact(apps):
    z = np.load(os.path.join(GOLDEN, "harris_small.npz"))
    same(apps.harris(z["input"]), z["output"], "harris golden")
    z = np.load(os.path.join(GOLDEN, "unsharp_small.npz"))
    assert np.isnan(z["output"]).any()  # the golden frame has a black patch
    same(apps.unsharp(z["input"]), z["output"], "unsharp golden")


def test_unsharp_weights_are_the_folded_constants(apps, npr):
    want = np.array([0x3e882c1b, 0x3e5a1395, 0x3ddfedac, 0x3d136e6b], np.uint32)
    assert (apps.unsharp_weights().view(np.uint32) == want).all()
    assert (npr.unsharp_weights().view(np.uint32) == want).all()
    # the run-time realisation would give w2 one ulp lower; the folded value is the one the reference uses
    assert np.float32(0.10934004).view(np.uint32) == 0x3ddfedac


@pytest.mark.parametrize("frame", ["random", "smooth"])
@pytest.mark.parametrize("h,w", [(7, 7), (20, 33), (61, 90)])
def test_harris_oracle_vs_numpy(apps, npr, frame, h, w):
    inp = (f32_frame if frame == "random" else smooth_f32)((3, h, w), h * 7 + w)
    want = npr.harris(inp, (h - 4, w - 4), out_mins=(2, 2))
    same(apps.harris(inp, (h - 4, w - 4), out_mins=(2, 2)), want, f"{frame} {h}x{w}")


def test_harris_harness_geometry_and_crops(apps, npr):
    inp = smooth_f32((3, 64, 96), 3) + f32_frame((3, 64, 96), 4) * np.float32(0.1)
    same(apps.harris(inp), npr.harris(inp, (58, 90), out_mins=(3, 3)), "harness geometry (W-6)x(H-6) at (3, 3)")
    # negative and odd mins; extra channels beyond 0..2 are not read
    inp5 = f32_frame((5, 50, 70), 5)
    kw = dict(in_mins=(-9, -4, 0), out_mins=(-5, -1))
    same(apps.harris(inp5, (31, 47), **kw), npr.harris(inp5, (31, 47), **kw), "negative mins")
    kw = dict(in_mins=(3, 7, -1), out_mins=(6, 10))
    same(apps.harris(inp5, (41, 63), **kw), npr.harris(inp5, (41, 63), **kw), "odd mins, channel min -1")
    same(apps.harris(inp5, (1, 1), in_mins=(0, 0, 0), out_mins=(2, 2)), npr.harris(inp5, (1, 1), out_mins=(2, 2)), "1x1")


def test_harris_oracle_rejects_non_covering_inputs(apps):
    inp = f32_frame((3, 20, 20), 0)
    with pytest.raises(RuntimeError):
        apps.harris(inp, (17, 16), out_mins=(2, 2))
    with pytest.raises(RuntimeError):
        apps.harris(np.ascontiguousarray(inp[:2]), (16, 16), out_mins=(2, 2))


@pytest.mark.parametrize("frame", ["random", "smooth", "black"])
@pytest.mark.parametrize("h,w", [(1, 1), (5, 9), (33, 47)])
def test_unsharp_oracle_vs_numpy(apps, npr, frame, h, w):
    inp = (smooth_f32 if frame == "smooth" else f32_frame)((3, h, w), h + 3 * w)
    if frame == "black":
        inp = black_patches(inp)
    with np.errstate(all="ignore"):
        same(apps.unsharp(inp), npr.unsharp(inp, inp.shape), f"{frame} {h}x{w}")


def test_unsharp_geometries(apps, npr):
    with np.errstate(all="ignore"):
        # output inside a larger input at negative / odd mins: the clamp follows the input's box
        inp = f32_frame((3, 40, 60), 11)
        for kw in (dict(in_mins=(-7, -3, 0), out_mins=(-5, 1, 0)), dict(in_mins=(5, 9, 0), out_mins=(8, 12, 1))):
            shape = (3 - kw["out_mins"][2], 23, 37)
            same(apps.unsharp(inp, shape, **kw), npr.unsharp(inp, shape, **kw), str(kw))
        # output flush with the input's corner: clamped rows and columns are the input's own edges
        kw = dict(in_mins=(4, 4, 0), out_mins=(4, 4, 0))
        same(apps.unsharp(inp, (3, 10, 12), **kw), npr.unsharp(inp, (3, 10, 12), **kw), "corner")
        # a 1-channel input at c-min 1: gray reads that channel three times
        one = f32_frame((1, 30, 44), 12)
        kw = dict(in_mins=(0, 0, 1), out_mins=(0, 0, 1))
        same(apps.unsharp(one, (1, 30, 44), **kw), npr.unsharp(one, (1, 30, 44), **kw), "1 channel")
        # a 4-channel output (the 4th channel only scaled by ratio), with black patches: +-inf and NaN
        four = black_patches(f32_frame((4, 26, 35), 13) + np.float32(0.5))
        got = apps.unsharp(four)
        assert np.isinf(got).any() and np.isnan(got).any()
        same(got, npr.unsharp(four, four.shape), "4 channels")


def test_unsharp_oracle_rejects_non_covering_inputs(apps):
    inp = f32_frame((3, 20, 20), 0)
    with pytest.raises(RuntimeError):
        apps.unsharp(inp, (4, 20, 20))
    with pytest.raises(RuntimeError):
        apps.unsharp(inp, (3, 20, 20), out_mins=(1, 0, 0))


# ---- the C ABI without a GPU ---------------------------------------------------------------------------------------------

class Arg(ctypes.Structure):
    _fields_ = [("name", ctypes.c_char_p), ("kind", ctypes.c_int32), ("dimensions", ctypes.c_int32), ("type", ctypes.c_uint32),
                ("scalar", ctypes.c_void_p * 4), ("buffer_estimates", ctypes.POINTER(ctypes.POINTER(ctypes.c_int64)))]


class Meta(ctypes.Structure):
    _fields_ = [("version", ctypes.c_int32), ("num_arguments", ctypes.c_int32), ("arguments", ctypes.POINTER(Arg)),
                ("target", ctypes.c_char_p), ("name", ctypes.c_char_p)]


def test_entry_points_exported(hb):
    l = hb.load_library()
    assert [s for s in ENTRY_POINTS if not hasattr(l, s)] == []


@pytest.mark.parametrize("name,estimates", [
    ("harris", [[0, 1536, 0, 2560, 0, 3], [3, 1530, 3, 2554]]),
    ("unsharp", [[0, 1536, 0, 2560, 0, 3], [0, 1536, 0, 2560, 0, 3]]),
])
def test_metadata(hb, name, estimates):
    l = hb.load_library()
    for suffix in ("", "_auto_schedule"):
        fn = getattr(l, name + suffix + "_metadata")
        fn.restype = ctypes.POINTER(Meta)
        md = fn().contents
        assert md.version == 1 and md.num_arguments == 2 and md.name == (name + suffix).encode()
        assert b"cuda" in md.target
        for i, (want_name, kind, est) in enumerate(zip((b"input", b"output"), (1, 2), estimates)):
            a = md.arguments[i]
            assert a.name == want_name and a.kind == kind and a.dimensions == len(est) // 2
            assert a.type & 0xFFFF == (32 << 8) | 2  # float32
            assert [a.buffer_estimates[k][0] for k in range(len(est))] == est


def _expect(code, fn, *args):
    from halide_b200 import HalideError
    with pytest.raises(HalideError) as e:
        fn(*args)
    assert e.value.code == code, (e.value.code, e.value.message)


def test_harris_validation_errors(hb):
    from halide_b200 import HalideBuffer as B, filters as F
    f32 = np.float32
    out = lambda: B.from_numpy(np.zeros((10, 10), f32), mins=(2, 2), host_dirty=False)  # noqa: E731
    l = hb.load_library()
    assert l.harris(None, out().ptr) == -12
    assert l.harris_auto_schedule(B.from_numpy(np.zeros((3, 14, 14), f32)).ptr, None) == -12
    _expect(-3, F.harris, B.from_numpy(np.zeros((3, 14, 14), np.uint16)), out())
    _expect(-3, F.harris, B.from_numpy(np.zeros((3, 14, 14), f32)), B.from_numpy(np.zeros((10, 10), np.uint16), mins=(2, 2)))
    _expect(-43, F.harris, B.from_numpy(np.zeros((14, 14), f32)), out())
    _expect(-43, F.harris, B.from_numpy(np.zeros((3, 14, 14), f32)), B.from_numpy(np.zeros((1, 10, 10), f32)))
    _expect(-4, F.harris, B.from_numpy(np.zeros((3, 14, 13), f32)), out())          # one column short
    _expect(-4, F.harris, B.from_numpy(np.zeros((3, 14, 14), f32), mins=(1, 0, 0)), out())
    _expect(-4, F.harris, B.from_numpy(np.zeros((2, 14, 14), f32)), out())          # too few channels
    _expect(-4, F.harris, B.from_numpy(np.zeros((3, 14, 14), f32), mins=(0, 0, 1)), out())
    bad = B.from_numpy(np.zeros((3, 14, 14), f32))
    bad.dims[0].stride = 2
    _expect(-8, F.harris, bad, out())
    # an empty output is not an error and needs no input at all
    empty = B.from_numpy(np.zeros((1, 5), f32))
    empty.dims[1].extent = 0
    assert F.harris(B.from_numpy(np.zeros((3, 1, 1), f32)), empty) == 0


def test_unsharp_validation_errors(hb):
    from halide_b200 import HalideBuffer as B, filters as F
    f32 = np.float32
    inp = lambda shape=(3, 12, 16), mins=None: B.from_numpy(np.zeros(shape, f32), mins=mins)  # noqa: E731
    out = lambda shape=(3, 12, 16), mins=None: B.from_numpy(np.zeros(shape, f32), mins=mins, host_dirty=False)  # noqa: E731
    l = hb.load_library()
    assert l.unsharp(None, out().ptr) == -12
    assert l.unsharp_auto_schedule(inp().ptr, None) == -12
    _expect(-3, F.unsharp, B.from_numpy(np.zeros((3, 12, 16), np.uint8)), out())
    _expect(-43, F.unsharp, inp((12, 16)), out())
    _expect(-43, F.unsharp, inp(), B.from_numpy(np.zeros((12, 16), f32)))
    _expect(-4, F.unsharp, inp(), out((4, 12, 16)))                  # channel 3 is read unclamped
    _expect(-4, F.unsharp, inp((1, 12, 16), (0, 0, 1)), out((1, 12, 16)))
    _expect(-4, F.unsharp, inp(), out((3, 12, 16), (1, 0, 0)))
    _expect(-4, F.unsharp, inp(), out((3, 13, 16)))
    bad = out()
    bad.dims[0].stride = 3
    _expect(-8, F.unsharp, inp(), bad)
    empty = out((1, 12, 16))
    empty.dims[2].extent = 0
    assert F.unsharp(inp(), empty) == 0


def test_bounds_queries(hb):
    from halide_b200 import HalideBuffer as B, filters as F
    # harris: the output box grown by 2 in x and y, channels 0..2 (the harness: (W-6)x(H-6) at (3, 3) of a WxH frame)
    q = B.bounds_query(np.float32, 3)
    assert F.harris(q, B.from_numpy(np.zeros((2554, 1530), np.float32), mins=(3, 3))) == 0
    assert q.shape() == [(1, 1534, 1), (1, 2558, 1534), (0, 3, 1534 * 2558)]
    q = B.bounds_query(np.float32, 3)
    assert F.harris(q, B.from_numpy(np.zeros((5, 7), np.float32), mins=(-4, 9))) == 0
    assert [(m, e) for (m, e, _) in q.shape()] == [(-6, 11), (7, 9), (0, 3)]
    # unsharp: exactly the output's (x, y, c) box
    q = B.bounds_query(np.float32, 3)
    assert F.unsharp(q, B.from_numpy(np.zeros((4, 20, 30), np.float32), mins=(-3, 5, 1))) == 0
    assert q.shape() == [(-3, 30, 1), (5, 20, 30), (1, 4, 600)]


def test_c_caller_links_the_new_entry_points(tmp_path):
    if not os.path.exists(os.path.join(LIBDIR, "libhalide_b200.so")):
        pytest.skip("library not built")
    body = '#include "halide_b200_runtime.h"\n'
    body += "".join(f'#include "{n}{s}.h"\n' for n in ("harris", "unsharp") for s in ("", "_auto_schedule"))
    body += "#include <stdio.h>\nint main(void) {\n  const struct halide_filter_metadata_t *m;\n"
    for n in ("harris", "unsharp", "harris_auto_schedule", "unsharp_auto_schedule"):
        body += f'  m = {n}_metadata();\n  if (!m || !m->name) return 1;\n  printf("%s %d\\n", m->name, m->num_arguments);\n'
        body += f"  {{ int (*fp)(void **) = {n}_argv; if (!fp) return 2; }}\n"
        body += f"  {{ int (*fp)(struct halide_buffer_t *, struct halide_buffer_t *) = {n}; if (!fp) return 3; }}\n"
    body += "  return 0;\n}\n"
    src, exe = tmp_path / "caller.c", tmp_path / "caller"
    src.write_text(body)
    out = subprocess.run(["/usr/bin/gcc", "-std=c99", "-Wall", "-Werror", f"-I{INC}", str(src), "-o", str(exe), f"-L{LIBDIR}",
                          "-lhalide_b200", f"-Wl,-rpath,{LIBDIR}", "-lpthread", "-ldl"], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr[-2000:]
    run = subprocess.run([str(exe)], capture_output=True, text=True, timeout=60)  # metadata only: no CUDA call
    assert run.returncode == 0, run.stdout + run.stderr
    assert run.stdout.split("\n")[:4] == ["harris 2", "unsharp 2", "harris_auto_schedule 2", "unsharp_auto_schedule 2"]
