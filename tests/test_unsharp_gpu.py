"""GPU parity tests for unsharp through the C ABI: bit-exact against oracle/oracle_unsharp.cpp (+, -, * and one IEEE
divide in source nesting; the library builds with --fmad=false -prec-div=true), NaN positions included.  Every host-path
case runs under the allocation fills 0xFF, 0x41 and 0x00 (tests/test_poisoned_memory_gpu.py) and must give identical
results under each."""
import numpy as np
import pytest

from test_harris_gpu import Exact
from test_poisoned_memory_gpu import LAYOUTS_3D, _device_input, device_resident, fill, poisoned, under_fills
from test_reference_harness_gpu import _bin, _load_halide_npy, _run, _save_halide_npy
from util import f32_frame

pytestmark = pytest.mark.gpu


def _oracle(o, inp, out_shape, in_mins, out_mins):
    from oracle import pyoracle_apps
    with np.errstate(all="ignore"):
        return pyoracle_apps.unsharp(inp, out_shape, in_mins, out_mins)


def unsharp_f():
    return Exact("unsharp", np.float32, (), _oracle, True)


def black_patches(a):
    """Zero channels 0..2 in a few boxes: gray == 0 there, so ratio is +-inf or NaN, as in the reference."""
    a = a.copy()
    h, w = a.shape[1:]
    for (y, x, hh, ww) in ((0, 0, 3, 3), (h // 3, w // 2, 5, 6), (h - 3, w - 4, 3, 4)):
        a[:3, y:y + hh, x:x + ww] = 0.0
    return a


@pytest.mark.parametrize("black", [False, True])
@pytest.mark.parametrize("h,w", [(1, 1), (5, 9), (33, 47), (70, 101)])
def test_ragged_sizes(hb, oracle, h, w, black):
    inp = f32_frame((3, h, w), h * 3 + w)
    if black:
        inp = black_patches(inp)
    got = poisoned(hb, oracle, unsharp_f(), inp, inp.shape)
    if black and h > 1:
        assert np.isnan(got).any()


def test_harness_geometry(hb, oracle):
    """apps/unsharp/filter.cpp on the generator's estimate frame, 1536 x 2560 x 3."""
    poisoned(hb, oracle, unsharp_f(), f32_frame((3, 2560, 1536), 1), (3, 2560, 1536))


def test_full_4k(hb, oracle):
    poisoned(hb, oracle, unsharp_f(), f32_frame((3, 2160, 3840), 2), (3, 2160, 3840))


def test_crops_clamp_to_the_input_box(hb, oracle):
    """Outputs inside a larger input at negative and odd mins: the 3-pixel apron reads real input pixels beyond the
    output's box and is clamped only at the input's own edges."""
    inp = f32_frame((3, 50, 80), 3)
    poisoned(hb, oracle, unsharp_f(), inp, (3, 29, 41), in_mins=(-9, -4, 0), out_mins=(-6, -1, 0), what="negative mins")
    poisoned(hb, oracle, unsharp_f(), inp, (2, 31, 45), in_mins=(2, 6, 0), out_mins=(7, 9, 1), what="odd mins, channels 1..2")
    poisoned(hb, oracle, unsharp_f(), inp, (3, 20, 30), in_mins=(3, 3, 0), out_mins=(3, 3, 0), what="flush with the input's corner")
    poisoned(hb, oracle, unsharp_f(), inp, (3, 21, 35), in_mins=(3, 3, 0), out_mins=(48, 32, 0), what="flush with the far corner")


def test_one_channel_input(hb, oracle):
    """A 1-channel input at c-min 1: gray reads that channel three times; the output is channel 1 only."""
    inp = f32_frame((1, 33, 47), 4)
    poisoned(hb, oracle, unsharp_f(), inp, (1, 33, 47), in_mins=(0, 0, 1), out_mins=(0, 0, 1))


def test_four_channel_output(hb, oracle):
    """Channel 3 is not staged for gray: the final multiply reads it from the input directly.  Black patches in
    channels 0..2 with a non-zero channel 3 give +-inf as well as NaN."""
    inp = black_patches(f32_frame((4, 40, 57), 5) + np.float32(0.5))
    got = poisoned(hb, oracle, unsharp_f(), inp, inp.shape)
    assert np.isinf(got).any() and np.isnan(got).any()


@pytest.mark.parametrize("layout", sorted(LAYOUTS_3D))
def test_host_layouts(hb, oracle, layout):
    f, inp = unsharp_f(), f32_frame((3, 37, 53), 6)
    want = f.want(oracle, inp, inp.shape)
    make = LAYOUTS_3D[layout]
    for lay_in, lay_out in ((True, False), (False, True), (True, True)):
        src = make(inp) if lay_in else inp
        mk = (lambda: make(np.zeros(inp.shape, np.float32))) if lay_out else None
        poisoned(hb, oracle, f, src, inp.shape, make_out=mk, want=want, what=f"{layout} in={lay_in} out={lay_out}")


@pytest.mark.parametrize("odd_input", [False, True])
@pytest.mark.parametrize("h,w", [(33, 47), (64, 128)])
def test_device_resident_padded_outputs(hb, oracle, h, w, odd_input):
    """Output = a view into a wider sentinel-filled tensor; the input optionally one float into its storage (no 16-byte
    loads possible).  64 x 128 rows are a multiple of 4 wide, so the aligned input takes the 16-byte path."""
    inp = f32_frame((3, h, w), h + w)
    device_resident(hb, oracle, unsharp_f(), inp, inp.shape, odd_input=odd_input, what=f"{h}x{w} odd_input={odd_input}")


def test_device_resident_vector_paths(hb, oracle):
    """Device input and output both 16-byte aligned with strides a multiple of 4 (16-byte loads and stores), and the
    same input at an odd element offset (element-wise loads): both must equal the oracle."""
    import torch
    from halide_b200 import HalideBuffer
    inp = black_patches(f32_frame((3, 40, 64), 9))
    want = _oracle(oracle, inp, inp.shape, None, None)
    for odd in (False, True):
        def run(byte):
            out = torch.zeros(inp.shape, dtype=torch.float32, device="cuda")
            bi = HalideBuffer.from_torch(_device_input(inp, odd))
            bo = HalideBuffer.from_torch(out)
            with fill(hb, byte):
                hb.filters.unsharp(bi, bo)
                bo.device_sync()
            return out.cpu().numpy()
        unsharp_f().compare(under_fills(run), want, f"odd={odd}")


def test_launch_counts(hb):
    from halide_b200 import HalideBuffer as B, filters as F
    count = hb.capi.halide_b200_kernel_launch_count
    inp = f32_frame((3, 24, 30), 6)
    out = np.zeros_like(inp)
    bo = B.from_numpy(out, host_dirty=False)
    n0 = count()
    F.unsharp(B.from_numpy(inp), bo)
    bo.copy_to_host()
    assert count() - n0 == 1
    empty = B.from_numpy(np.zeros((1, 24, 30), np.float32))
    empty.dims[2].extent = 0
    n0 = count()
    assert F.unsharp(B.from_numpy(inp), empty) == 0
    q = B.bounds_query(np.float32, 3)
    assert F.unsharp(q, B.from_numpy(out, host_dirty=False)) == 0
    assert count() - n0 == 0


def test_8k_regions(hb, oracle):
    """7680 x 4320 x 3: regions of the full-size result against the oracle on the crop that determines them (footprint
    3 px, margin 8; crops at the frame's edges start or end there, so their clamps are the frame's)."""
    h, w = 4320, 7680
    inp = f32_frame((3, h, w), 7)

    def run(byte):
        out = np.zeros_like(inp)
        bi, bo = hb.HalideBuffer.from_numpy(inp), hb.HalideBuffer.from_numpy(out, host_dirty=False)
        with fill(hb, byte):
            hb.filters.unsharp(bi, bo)
        bo.copy_to_host()
        return out
    got = under_fills(run)
    for (y0, x0) in [(0, 0), (h - 64, w - 64), (2001, 3999), (h - 64, 0)]:
        n, m = 64, 8
        ya, yb, xa, xb = max(0, y0 - m), min(h, y0 + n + m), max(0, x0 - m), min(w, x0 + n + m)
        crop = np.ascontiguousarray(inp[:, ya:yb, xa:xb])
        want = _oracle(oracle, crop, (3, n, n), (xa, ya, 0), (x0, y0, 0))
        unsharp_f().compare(got[:, y0:y0 + n, x0:x0 + n], want, f"region ({x0}, {y0})")


def test_unsharp_filter_cpp(tmp_path, oracle):
    """The reference's unmodified apps/unsharp/filter.cpp linked against the library: it must print Success! and the
    result it saves must equal the oracle."""
    img = f32_frame((3, 70, 96), 8)
    _save_halide_npy(tmp_path / "in.npy", img)
    out = _run([_bin("unsharp_filter"), str(tmp_path / "in.npy"), str(tmp_path / "out.npy")])
    assert "Manually-tuned time" in out and "Auto-scheduled time" in out
    got = _load_halide_npy(tmp_path / "out.npy")
    unsharp_f().compare(np.asarray(got, np.float32), _oracle(oracle, img, img.shape, None, None), "harness")


def test_unsharp_rungen_benchmark_mode():
    import subprocess
    r = subprocess.run([_bin("unsharp_rungen"), "--benchmarks=all", "--estimate_all", "--parsable_output"], capture_output=True,
                       text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "BEST_TIME_MSEC_PER_ITER" in r.stdout, r.stdout + r.stderr
