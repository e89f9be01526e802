"""GPU parity tests for harris through the C ABI: bit-exact against oracle/oracle_harris.cpp (every operation is +, -, *
in source nesting; the library builds with --fmad=false).  Every host-path case runs under the allocation fills 0xFF,
0x41 and 0x00 (tests/test_poisoned_memory_gpu.py) and must give identical results under each."""
import numpy as np
import pytest

from test_poisoned_memory_gpu import (LAYOUTS_2D, LAYOUTS_3D, Filter, _device_input, device_resident, fill, poisoned,
                                      under_fills)
from test_reference_harness_gpu import _bin, _load_halide_npy, _run, _save_halide_npy
from util import f32_frame

pytestmark = pytest.mark.gpu


class Exact(Filter):
    """Bit-exact comparison in which a NaN matches a NaN at the same position."""

    def compare(self, got, want, what=""):
        assert got.shape == want.shape, (what, got.shape, want.shape)
        bad = np.argwhere(~((got == want) | (np.isnan(got) & np.isnan(want))))
        assert bad.size == 0, f"{what}: {len(bad)} mismatches, first at {tuple(bad[0])}: {got[tuple(bad[0])]} vs {want[tuple(bad[0])]}"


def _oracle(o, inp, out_shape, in_mins, out_mins):
    from oracle import pyoracle_apps
    return pyoracle_apps.harris(inp, out_shape, in_mins, out_mins if out_mins is not None else (0, 0))


def harris_f():
    return Exact("harris", np.float32, (), _oracle, True)


class Shifted(Exact):
    """harris with the input's x / y mins moved to -2 just before the call, so that an output at (0, 0) — all the
    device-resident helper can build — is covered by an input of the output's size + 4."""

    def call(self, hb, bi, bo):
        bi.dims[0].min, bi.dims[1].min = -2, -2
        super().call(hb, bi, bo)


@pytest.mark.parametrize("h,w", [(1, 1), (5, 9), (33, 47), (70, 101)])
def test_ragged_sizes(hb, oracle, h, w):
    poisoned(hb, oracle, harris_f(), f32_frame((3, h + 4, w + 4), h * 5 + w), (h, w), out_mins=(2, 2))


def test_harness_geometry(hb, oracle):
    """apps/harris/filter.cpp:25-26 on the generator's estimate frame: (W-6) x (H-6) at (3, 3) of 1536 x 2560."""
    poisoned(hb, oracle, harris_f(), f32_frame((3, 2560, 1536), 1), (2554, 1530), out_mins=(3, 3))


def test_full_4k(hb, oracle):
    poisoned(hb, oracle, harris_f(), f32_frame((3, 2164, 3844), 2), (2160, 3840), out_mins=(2, 2))


def test_negative_and_odd_mins(hb, oracle):
    inp = f32_frame((3, 60, 90), 3)
    poisoned(hb, oracle, harris_f(), inp, (37, 51), in_mins=(-11, -6, 0), out_mins=(-7, -3), what="negative mins")
    poisoned(hb, oracle, harris_f(), inp, (21, 33), in_mins=(5, 3, 0), out_mins=(9, 8), what="odd mins")
    # extra channels on both sides of 0..2: only 0..2 are read
    poisoned(hb, oracle, harris_f(), f32_frame((5, 40, 50), 4), (29, 41), in_mins=(0, 0, -1), out_mins=(3, 5),
             what="channels -1..3")


@pytest.mark.parametrize("layout", sorted(LAYOUTS_3D))
def test_host_layouts(hb, oracle, layout):
    """The layout on the input, on the output (2-D layouts only), and on both."""
    f, inp, out_shape = harris_f(), f32_frame((3, 37, 53), 5), (33, 49)
    want = f.want(oracle, inp, out_shape, None, (2, 2))
    out_layout = LAYOUTS_2D.get(layout)
    for lay_in, lay_out in ((True, False), (False, True), (True, True)):
        if lay_out and out_layout is None:
            continue
        src = LAYOUTS_3D[layout](inp) if lay_in else inp
        mk = (lambda: out_layout(np.zeros(out_shape, np.float32))) if lay_out else None
        poisoned(hb, oracle, f, src, out_shape, out_mins=(2, 2), make_out=mk, want=want,
                 what=f"{layout} in={lay_in} out={lay_out}")


@pytest.mark.parametrize("odd_input", [False, True])
@pytest.mark.parametrize("h,w", [(33, 47), (64, 128)])
def test_device_resident_padded_outputs(hb, oracle, h, w, odd_input):
    """Output = a view into a wider sentinel-filled tensor; the input optionally one float into its storage (no 16-byte
    loads possible).  64 x 128 has rows a multiple of 4 wide, so the aligned input takes the 16-byte path."""
    inp = f32_frame((3, h + 4, w + 4), h + w)
    want = _oracle(oracle, inp, (h, w), (-2, -2, 0), (0, 0))
    device_resident(hb, oracle, Shifted("harris", np.float32, (), _oracle, True), inp, (h, w), want=want, odd_input=odd_input,
                    what=f"{h}x{w} odd_input={odd_input}")


def test_device_resident_vector_paths(hb, oracle):
    """Device input and output both 16-byte aligned with strides a multiple of 4 (16-byte loads and stores), and the
    same data at an odd element offset (element-wise path): both must equal the oracle."""
    import torch
    from halide_b200 import HalideBuffer
    h, w = 40, 64
    inp = f32_frame((3, h + 4, w + 4), 9)
    want = _oracle(oracle, inp, (h, w), (-2, -2, 0), (0, 0))
    for odd in (False, True):
        def run(byte):
            out = torch.zeros((h, w), dtype=torch.float32, device="cuda")
            bi = HalideBuffer.from_torch(_device_input(inp, odd), mins=(-2, -2, 0))
            bo = HalideBuffer.from_torch(out)
            with fill(hb, byte):
                hb.filters.harris(bi, bo)
                bo.device_sync()
            return out.cpu().numpy()
        harris_f().compare(under_fills(run), want, f"odd={odd}")


def test_launch_counts(hb):
    from halide_b200 import HalideBuffer as B, filters as F
    count = hb.capi.halide_b200_kernel_launch_count
    inp = f32_frame((3, 24, 30), 6)
    out = np.zeros((20, 26), np.float32)
    bo = B.from_numpy(out, mins=(2, 2), host_dirty=False)
    n0 = count()
    F.harris(B.from_numpy(inp), bo)
    bo.copy_to_host()
    assert count() - n0 == 1
    empty = B.from_numpy(np.zeros((1, 26), np.float32), mins=(2, 2))
    empty.dims[1].extent = 0
    n0 = count()
    assert F.harris(B.from_numpy(inp), empty) == 0
    q = B.bounds_query(np.float32, 3)
    assert F.harris(q, B.from_numpy(out, mins=(2, 2), host_dirty=False)) == 0
    assert count() - n0 == 0


def test_8k_regions(hb, oracle):
    """7680 x 4320 output: regions of the full-size result against the oracle on the input crop that determines them
    (footprint 2 px)."""
    h, w = 4320, 7680
    inp = f32_frame((3, h + 4, w + 4), 7)

    def run(byte):
        out = np.zeros((h, w), np.float32)
        bi = hb.HalideBuffer.from_numpy(inp)
        bo = hb.HalideBuffer.from_numpy(out, (2, 2), host_dirty=False)
        with fill(hb, byte):
            hb.filters.harris(bi, bo)
        bo.copy_to_host()
        return out
    got = under_fills(run)
    for (y0, x0) in [(0, 0), (h - 64, w - 64), (2001, 3999), (h - 64, 0)]:
        n = 64
        crop = np.ascontiguousarray(inp[:, y0:y0 + n + 4, x0:x0 + n + 4])  # input rows / columns y0 .. y0+n+3
        want = _oracle(oracle, crop, (n, n), (x0, y0, 0), (x0 + 2, y0 + 2))
        harris_f().compare(got[y0:y0 + n, x0:x0 + n], want, f"region ({x0}, {y0})")


def test_harris_filter_cpp(tmp_path, oracle):
    """The reference's unmodified apps/harris/filter.cpp linked against the library: it must print Success! and the
    (W-6) x (H-6) result it saves at (3, 3) must equal the oracle."""
    img = f32_frame((3, 70, 96), 8)
    _save_halide_npy(tmp_path / "in.npy", img)
    out = _run([_bin("harris_filter"), str(tmp_path / "in.npy"), str(tmp_path / "out.npy")])
    assert "Manually-tuned time" in out and "Auto-scheduled time" in out
    got = _load_halide_npy(tmp_path / "out.npy")
    harris_f().compare(np.asarray(got, np.float32), _oracle(oracle, img, (64, 90), None, (3, 3)), "harness")


def test_harris_rungen_benchmark_mode():
    import subprocess
    r = subprocess.run([_bin("harris_rungen"), "--benchmarks=all", "--estimate_all", "--parsable_output"], capture_output=True,
                       text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "BEST_TIME_MSEC_PER_ITER" in r.stdout, r.stdout + r.stderr
