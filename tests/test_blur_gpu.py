"""GPU parity tests for halide_blur through the C ABI (bit-exact, uint16)."""
import numpy as np
import pytest

from util import reference, run_blur, sha, u16_frame

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("h,w", [(3, 3), (9, 10), (34, 70), (66, 264), (130, 515), (257, 1031)])
@pytest.mark.parametrize("seed", [0, 42])
def test_blur_matches_oracle(hb, oracle, h, w, seed):
    inp = u16_frame((h, w), seed)  # full 16-bit range: exercises the mod-2^16 wrap
    got = run_blur(hb, inp, (h - 2, w - 2))
    assert np.array_equal(got, oracle.blur(inp))


def test_blur_matches_reference_c_on_harness_shape(hb):
    """apps/blur/test.cpp:162-191: 2568x1922 input, rand() & 0xfff, compared on the interior
    against the reference's own C implementations (its naive and its SSE blur)."""
    inp = u16_frame((1922, 2568), 7, bits=12)
    got = run_blur(hb, inp, (1920, 2560))
    want = reference()["blur"]["1922x2568"]
    assert sha(got) == want["slow"]
    assert sha(got) == want["fast"]


def test_blur_config1_1080p(hb, oracle):
    inp = u16_frame((1082, 1922), 1)
    got = run_blur(hb, inp, (1080, 1920))
    assert np.array_equal(got, oracle.blur(inp))


def test_blur_offsets_and_padded_strides(hb, oracle):
    """Non-zero mins, an input larger than required, and row strides that break 16-byte alignment."""
    big = u16_frame((60, 91), 5)
    inp = big[:, :83]  # row stride 91 elements: odd -> every row differently aligned
    out_store = np.zeros((40, 77), np.uint16)
    out = out_store[:, :61]
    from halide_b200 import HalideBuffer, filters
    bi = HalideBuffer.from_numpy(inp, mins=(-3, 10))
    bo = HalideBuffer.from_numpy(out, mins=(4, 15), host_dirty=False)
    filters.halide_blur(bi, bo)
    bo.copy_to_host()
    want = oracle.blur(inp, out_shape=(40, 61), in_mins=(-3, 10), out_mins=(4, 15))
    assert np.array_equal(out, want)
    assert not out_store[:, 61:].any()  # padding columns untouched


def test_blur_large_frame_checksum_property(hb):
    """8K-wide frame: too slow for the scalar oracle to be worth it; use the pipeline's linearity
    on small values: blur(c) == c for constant frames, and row/column sums of an impulse response."""
    h, w = 4322, 7682
    inp = np.full((h, w), 1234, np.uint16)
    got = run_blur(hb, inp, (h - 2, w - 2))
    assert (got == 1234).all()
    inp = np.zeros((h, w), np.uint16)
    inp[2000, 4000] = 9 * 7
    got = run_blur(hb, inp, (h - 2, w - 2))
    assert got.sum() == 9 * 7 and (got[1998:2001, 3998:4001] == 7).all()


def test_blur_device_resident_buffers(hb, oracle):
    """Inputs already in HBM (wrapped torch tensors): no host pointers at all."""
    import torch
    from halide_b200 import HalideBuffer, filters
    inp = u16_frame((130, 258), 3)
    t_in = torch.from_numpy(inp.view(np.int16)).cuda().view(torch.uint16)
    t_out = torch.zeros((128, 256), dtype=torch.uint16, device="cuda")
    bi, bo = HalideBuffer.from_torch(t_in), HalideBuffer.from_torch(t_out)
    filters.halide_blur(bi, bo)
    bo.device_sync()
    got = t_out.view(torch.int16).cpu().numpy().view(np.uint16)
    assert np.array_equal(got, oracle.blur(inp))


def test_blur_8k_full_frame_matches_oracle(hb, oracle):
    """The bench_all frame (7680x4320 output): full compare against the oracle (tens of ms on the CPU).  At this size the
    aligned kernel runs tall strips (its unclamped main loop) on unguarded 128-column strips."""
    inp = u16_frame((4322, 7682), 77)
    got = run_blur(hb, inp, (4320, 7680))
    assert np.array_equal(got, oracle.blur(inp))


@pytest.mark.parametrize("rows", [8, 13, 19, 25, 64])
def test_blur_aligned_kernel_strip_heights(hb, oracle, rows):
    """Strip heights around the prefetch depth: the row loop has an unclamped main part and a clamped tail; every split
    of a strip between them must give the same frame (widths: whole strips, a ragged last strip, an odd width)."""
    l = hb.load_library()
    try:
        l.halide_b200_blur_force_general(rows)
        for h, w in ((100, 256), (67, 300), (90, 131)):
            inp = u16_frame((h + 2, w + 2 + (w & 1)), rows + w)
            assert np.array_equal(run_blur(hb, inp, (h, w)), oracle.blur(inp, out_shape=(h, w))), (rows, h, w)
    finally:
        l.halide_b200_blur_force_general(0)


@pytest.mark.parametrize("h,w", [(64, 128), (37, 190), (130, 257), (200, 1000)])
def test_blur_pair_and_general_kernels(hb, oracle, h, w):
    """Frames whose rows keep pixel pairs 4-byte aligned (even row strides) take the aligned kernel (a lane = two pixel
    pairs); the hook routes the same frame through the general (any alignment) kernel.  Both must equal the oracle; odd
    output widths and odd column offsets (which fall back to the general kernel by themselves) included."""
    inp = u16_frame((h + 2, w + 2 + (w & 1)), 100 + w)   # even row stride
    want = oracle.blur(inp, out_shape=(h, w))
    l = hb.load_library()
    got_pair = run_blur(hb, inp, (h, w))
    try:
        l.halide_b200_blur_force_general(1)
        got_general = run_blur(hb, inp, (h, w))
    finally:
        l.halide_b200_blur_force_general(0)
    assert np.array_equal(got_pair, want) and np.array_equal(got_general, want)
    # output region starting at an odd input column: general kernel by itself
    want_off = oracle.blur(inp, out_shape=(h - 3, w - 5), in_mins=(0, 0), out_mins=(3, 2))
    got_off = run_blur(hb, inp, (h - 3, w - 5), in_mins=(0, 0), out_mins=(3, 2))
    assert np.array_equal(got_off, want_off)
