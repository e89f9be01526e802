"""GPU parity tests on poisoned device memory, unusual layouts and rarely taken launch paths.

The allocation pool recycles blocks without clearing them, so an output element a kernel forgot to store, or scratch it
read without writing, goes unnoticed whenever the stale block happens to hold the right value (often: the previous call's
answer on the same shape).  Here every call runs three times under halide_b200_debug_fill_allocations with fills 0xFF
(NaN / 65535), 0x41 (finite, plausible values that a clamp or saturating conversion would not turn into an error) and
0x00; the three results must be bit-identical (every pipeline is deterministic) and equal to the oracle.  Device-resident
cases wrap caller-owned torch tensors filled with a sentinel around the output view: only they can see a store into row
or plane padding, since copy_to_host never copies padding back.

Fixed alongside these tests:
- conv_layer moved every operand and its output in float4s, so a wrapped device buffer that was not 16-byte aligned
  (test_device_resident_conv_layer) was read and written misaligned; such buffers are now staged through aligned scratch.
"""
import ctypes
import contextlib

import numpy as np
import pytest

from util import f32_frame, u16_frame, conv_make

pytestmark = pytest.mark.gpu
FILLS = (0xFF, 0x41, 0x00)

M3200 = np.array([[1.6697, -0.2693, -0.4004, -42.4346], [-0.3576, 1.0615, 1.5949, -37.1158],
                  [-0.2175, -1.8751, 6.9640, -26.6970]], np.float32)
M7000 = np.array([[2.2997, -0.4478, 0.1706, -39.0923], [-0.3826, 1.5906, -0.2080, -25.4311],
                  [-0.0888, -0.7344, 2.2832, -20.0826]], np.float32)
CAMERA = (3700.0, 2.0, 50.0, 1.0, 25, 1023)


@contextlib.contextmanager
def fill(hb, byte):
    l = hb.load_library()
    l.halide_b200_debug_fill_allocations(byte)
    try:
        yield
    finally:
        l.halide_b200_debug_fill_allocations(-1)


@contextlib.contextmanager
def hook(hb, setter, value):
    """One of the library's variant hooks (0 restores the default selection)."""
    l = hb.load_library()
    getattr(l, setter)(value)
    try:
        yield
    finally:
        getattr(l, setter)(0)


def raw_frame(h, w, seed):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    base = 400 + 300 * np.sin(xx / 23.0) * np.cos(yy / 17.0)
    return np.clip(0.5 * base + 0.5 * rng.integers(0, 1024, (h, w)), 0, 1023).astype(np.uint16)


# ---- the filters: how to call each one and how to compare with the oracle ----------------------------------------------

def _camera_params(hb):
    return (hb.HalideBuffer.from_numpy(M3200.copy()), hb.HalideBuffer.from_numpy(M7000.copy())) + CAMERA


def _conv_params(hb, filt, bias):
    return (hb.HalideBuffer.from_numpy(filt), hb.HalideBuffer.from_numpy(bias))


class Filter:
    def __init__(self, name, out_dtype, params, oracle, exact, rel_floor=None):
        self.name, self.out_dtype, self.params, self.oracle, self.exact, self.rel_floor = (name, out_dtype, params, oracle,
                                                                                           exact, rel_floor)

    def call(self, hb, bi, bo):
        params = self.params(hb) if callable(self.params) else self.params
        getattr(hb.filters, self.name)(bi, *params, bo)

    def want(self, oracle, inp, out_shape, in_mins=None, out_mins=None):
        return self.oracle(oracle, np.ascontiguousarray(inp), out_shape, in_mins, out_mins)

    def compare(self, got, want, what=""):
        if self.exact:
            bad = np.argwhere(got != want)
            assert bad.size == 0, f"{what}: {len(bad)} mismatches, first at {tuple(bad[0])}: {got[tuple(bad[0])]} vs {want[tuple(bad[0])]}"
        else:
            assert np.isfinite(got).all(), f"{what}: non-finite output"
            err = np.abs(got.astype(np.float64) - want) / np.maximum(np.abs(want), self.rel_floor)
            assert err.max() <= 1e-4, f"{what}: max rel err {err.max()} at {np.unravel_index(err.argmax(), err.shape)}"


def blur_f():
    return Filter("halide_blur", np.uint16, (), lambda o, i, s, im, om: o.blur(i, s, im, om), True)


def ll_f(levels=8, alpha=1.0 / 7.0, beta=1.0):
    return Filter("local_laplacian", np.uint16, (levels, alpha, beta),
                  lambda o, i, s, im, om: o.local_laplacian(i, levels, alpha, beta, s, im, om), True)


def bg_f(r_sigma=0.1):
    return Filter("bilateral_grid", np.float32, (r_sigma,), lambda o, i, s, im, om: o.bilateral_grid(i, r_sigma, s, im, om),
                  False, 1e-6)


def nl_f(patch=3, search=7, sigma=0.12):
    return Filter("nl_means", np.float32, (patch, search, sigma),
                  lambda o, i, s, im, om: o.nl_means(i, patch, search, sigma, s, im, om), False, 1e-3)


def sc_f():
    return Filter("stencil_chain", np.uint16, (), lambda o, i, s, im, om: o.stencil_chain(i, s, im, om), True)


def cp_f():
    return Filter("camera_pipe", np.uint8, _camera_params,
                  lambda o, i, s, im, om: o.camera_pipe(i, M3200, M7000, *CAMERA, s, im, om), True)


# ---- the host-path runner -----------------------------------------------------------------------------------------------

def _host_call(hb, f, inp, out, in_mins, out_mins):
    bi = hb.HalideBuffer.from_numpy(inp, in_mins)
    bo = hb.HalideBuffer.from_numpy(out, out_mins, host_dirty=False)
    f.call(hb, bi, bo)
    assert bo.device_dirty
    bo.copy_to_host()


def under_fills(run):
    """run() -> output array; the same call under each fill must give bit-identical results."""
    outs = []
    for byte in FILLS:
        outs.append(run(byte))
    for byte, o in zip(FILLS[1:], outs[1:]):
        assert o.tobytes() == outs[0].tobytes(), f"result depends on what fill 0x{byte:02X} left in device memory"
    return outs[0]


def poisoned(hb, oracle, f, inp, out_shape, in_mins=None, out_mins=None, make_out=None, want=None, what=""):
    """Run `f` under every fill with a host output (`make_out()` -> a view to write into; default dense zeros); compare
    with the oracle."""
    def run(byte):
        out = np.zeros(out_shape, f.out_dtype) if make_out is None else make_out()
        with fill(hb, byte):
            _host_call(hb, f, inp, out, in_mins, out_mins)
        return np.array(out)
    got = under_fills(run)
    if want is None:
        want = f.want(oracle, inp, out_shape, in_mins, out_mins)
    f.compare(got, want, what or f.name)
    return got


# ---- the hook itself ----------------------------------------------------------------------------------------------------

def test_fill_hook_poisons_fresh_and_recycled_blocks(hb):
    """If the hook did nothing, every other test in this file would pass vacuously."""
    from halide_b200 import HalideBuffer
    iface = ctypes.c_void_p(hb.capi.halide_cuda_device_interface())
    for n in (1000, 4096 * 3 + 17):
        for byte in FILLS + (0x5A,):
            host = np.full(n, 0x33, np.uint8)
            for _ in range(2):  # a fresh block (or one from an earlier size), then the same block back from the pool
                b = HalideBuffer.from_numpy(host, host_dirty=False)
                with fill(hb, byte):
                    hb.lib.check(hb.capi.halide_device_malloc(None, b.ptr, iface))
                b.buf.flags |= 2  # device_dirty: copy_to_host brings the device bytes back
                b.copy_to_host()
                assert (host == byte).all(), (n, byte, np.unique(host))
                b.device_free()
                host[:] = 0x33


# ---- every kernel variant the hooks reach, at ragged sizes and crops ----------------------------------------------------

LL_MASKS = (0, 1, 2, 4, 7, 8, 16, 64, 128, 256)


@pytest.mark.parametrize("mask", LL_MASKS)
def test_local_laplacian_variants(hb, oracle, mask):
    img = u16_frame((3, 131, 203), 31)
    with hook(hb, "halide_b200_ll_force_generic", mask):
        poisoned(hb, oracle, ll_f(), img, img.shape, what=f"mask {mask}")
        poisoned(hb, oracle, ll_f(), u16_frame((3, 90, 120), 4), (3, 50, 61), in_mins=(-7, 3, 0), out_mins=(10, 21, 0),
                 what=f"mask {mask} crop")
        poisoned(hb, oracle, ll_f(), u16_frame((3, 140, 264), 5), (3, 120, 240), in_mins=(0, 0, 0), out_mins=(8, 5, 0),
                 what=f"mask {mask} crop at 8 columns")


@pytest.mark.parametrize("levels,alpha,beta", [(2, 1.0, 1.0), (5, 0.25, 0.7), (16, 1.0 / 15.0, 1.0)])
def test_local_laplacian_levels(hb, oracle, levels, alpha, beta):
    poisoned(hb, oracle, ll_f(levels, alpha, beta), u16_frame((3, 33, 47), levels), (3, 33, 47))
    poisoned(hb, oracle, ll_f(levels, alpha, beta), u16_frame((3, 72, 104), levels + 1), (3, 72, 104))


@pytest.mark.parametrize("mode", [0, 1, 8, 13])
def test_blur_variants(hb, oracle, mode):
    """0: default selection, 1: general kernel, 8 / 13: aligned kernel with strips of that many rows."""
    with hook(hb, "halide_b200_blur_force_general", mode):
        for h, w in ((37, 190), (130, 257), (67, 300), (1, 1)):
            inp = u16_frame((h + 2, w + 2 + (w & 1)), 100 + w)
            poisoned(hb, oracle, blur_f(), inp, (h, w), what=f"mode {mode} {h}x{w}")
        inp = u16_frame((132, 260), 7)
        poisoned(hb, oracle, blur_f(), inp, (127, 250), in_mins=(0, 0), out_mins=(3, 2), what=f"mode {mode} crop")


@pytest.mark.parametrize("variant", [0, 1, 2])
def test_nl_means_variants(hb, oracle, variant):
    with hook(hb, "halide_b200_nl_means_variant", variant):
        for h, w in ((1, 1), (33, 47), (70, 101)):
            poisoned(hb, oracle, nl_f(), f32_frame((3, h, w), h + w), (3, h, w), what=f"variant {variant} {h}x{w}")
        poisoned(hb, oracle, nl_f(7, 7, 0.12), f32_frame((3, 40, 52), 77), (3, 40, 52))
        poisoned(hb, oracle, nl_f(), f32_frame((3, 50, 70), 5), (3, 30, 41), in_mins=(-4, 2, 0), out_mins=(1, 6, 0),
                 what=f"variant {variant} crop")


@pytest.mark.parametrize("variant", [0, 1, 2])
def test_stencil_chain_variants(hb, oracle, variant):
    with hook(hb, "halide_b200_stencil_chain_variant", variant):
        for h, w in ((1, 1), (17, 40), (65, 129), (130, 256)):
            poisoned(hb, oracle, sc_f(), u16_frame((h, w), variant * 100 + h + w), (h, w), what=f"variant {variant} {h}x{w}")
        inp = u16_frame((40, 50), 3)
        poisoned(hb, oracle, sc_f(), inp, (60, 80), in_mins=(3, -2), out_mins=(-10, -9), what="output larger than input")
        poisoned(hb, oracle, sc_f(), inp, (21, 33), in_mins=(0, 0), out_mins=(7, 5), what="crop at odd offsets")


def test_camera_pipe(hb, oracle):
    for h, w in ((56, 64), (120, 200)):
        shape = (3, ((h - 24) // 32) * 32, ((w - 32) // 32) * 32)
        poisoned(hb, oracle, cp_f(), raw_frame(h, w, h), shape)
    poisoned(hb, oracle, cp_f(), raw_frame(140, 180, 9), (3, 70, 90), out_mins=(3, 5, 0), what="odd output offsets")
    poisoned(hb, oracle, cp_f(), raw_frame(140, 180, 9), (3, 69, 87), out_mins=(4, 6, 0), what="ragged output")


@pytest.mark.parametrize("tc", [1, 0])
def test_conv_layer(hb, oracle, tc):
    inp, filt, bias = conv_make(0, 1.0)
    f = Filter("conv_layer", np.float32, lambda h: _conv_params(h, filt, bias), None, False, 1e-30)
    want = oracle.conv_layer(inp, filt, bias)
    l = hb.load_library()
    try:
        l.halide_b200_conv_use_tensor_cores(tc)
        poisoned(hb, oracle, f, inp, want.shape, want=want)
    finally:
        l.halide_b200_conv_use_tensor_cores(1)


# ---- launch regimes no other test reaches -------------------------------------------------------------------------------

@pytest.mark.parametrize("r_sigma", [0.1, 0.02, 0.006])
def test_bilateral_grid_bin_counts(hb, oracle, r_sigma):
    """0.02: the histogram needs more than 48 KB of shared memory; 0.006: the slice does as well."""
    poisoned(hb, oracle, bg_f(r_sigma), f32_frame((100, 257), 3), (100, 257))
    poisoned(hb, oracle, bg_f(r_sigma), f32_frame((120, 150), 8), (70, 90), in_mins=(-13, 5), out_mins=(3, 22), what="crop")


def test_bilateral_grid_too_many_bins_is_rejected_before_any_launch(hb):
    from halide_b200 import HalideBuffer, HalideError, filters
    inp = f32_frame((40, 50), 1)
    out = np.zeros_like(inp)
    n0 = hb.capi.halide_b200_kernel_launch_count()
    with pytest.raises(HalideError) as e:
        filters.bilateral_grid(HalideBuffer.from_numpy(inp), 0.0045, HalideBuffer.from_numpy(out, host_dirty=False))
    assert e.value.code == -9
    assert hb.capi.halide_b200_kernel_launch_count() == n0


@pytest.mark.parametrize("patch,search,h,w", [(9, 21, 23, 37), (15, 31, 19, 26), (31, 63, 9, 13)])
@pytest.mark.parametrize("variant", [0, 1])
def test_nl_means_search_rows_in_chunks(hb, oracle, patch, search, h, w, variant):
    """Pairs whose search row does not fit shared memory in one piece: the kernel walks it in ragged chunks of offsets
    ((9,21) and (15,31)) or one offset at a time ((31,63))."""
    with hook(hb, "halide_b200_nl_means_variant", variant):
        poisoned(hb, oracle, nl_f(patch, search, 0.2), f32_frame((3, h, w), patch), (3, h, w))


# ---- host-side layouts --------------------------------------------------------------------------------------------------

def _padded_rows(a, pad=3):
    """The same values in an array whose rows are `pad` elements longer."""
    store = np.zeros(a.shape[:-1] + (a.shape[-1] + pad,), a.dtype)
    v = store[..., :a.shape[-1]]
    v[...] = a
    return v


def _padded_planes(a, pad=5):
    store = np.zeros((a.shape[0], a.shape[1] + pad) + a.shape[2:], a.dtype)
    v = store[:, :a.shape[1]]
    v[...] = a
    return v


def _interleaved_rows(a):
    """(c, h, w) values with strides (x 1, y 3w, c w): a row of every channel, then the next row."""
    c, h, w = a.shape
    v = np.empty((h, c, w), a.dtype).transpose(1, 0, 2)
    v[...] = a
    return v


def _flipped_rows(a):
    v = np.empty_like(a)[..., ::-1, :]
    v[...] = a
    return v


LAYOUTS_2D = {"padded_rows": _padded_rows, "flipped_rows": _flipped_rows}
LAYOUTS_3D = dict(LAYOUTS_2D, padded_planes=_padded_planes, interleaved_rows=_interleaved_rows)


def _layout_cases():
    cases = []
    for name in LAYOUTS_2D:
        cases += [("halide_blur", name), ("stencil_chain", name), ("bilateral_grid", name), ("camera_pipe", name)]
    for name in LAYOUTS_3D:
        cases += [("local_laplacian", name), ("nl_means", name)]
    return cases


def _layout_setup(name):
    """(filter, input, output shape, output mins) per filter at a ragged size."""
    if name == "halide_blur":
        return blur_f(), u16_frame((68, 132), 1), (66, 130), None
    if name == "stencil_chain":
        return sc_f(), u16_frame((65, 98), 2), (65, 98), None
    if name == "bilateral_grid":
        return bg_f(), f32_frame((70, 104), 3), (70, 104), None
    if name == "camera_pipe":
        return cp_f(), raw_frame(120, 200, 4), (3, 96, 160), None
    if name == "local_laplacian":
        return ll_f(), u16_frame((3, 66, 104), 5), (3, 66, 104), None
    if name == "nl_means":
        return nl_f(), f32_frame((3, 33, 48), 6), (3, 33, 48), None
    raise KeyError(name)


@pytest.mark.parametrize("filt,layout", _layout_cases())
def test_host_layouts(hb, oracle, filt, layout):
    """The layout on the input, on the output, and on both (camera_pipe's raw input is 2-D: 3-D layouts go on its
    output only)."""
    f, inp, out_shape, out_mins = _layout_setup(filt)
    make = (LAYOUTS_3D if inp.ndim == 3 else LAYOUTS_2D)[layout]
    want = f.want(oracle, inp, out_shape, None, out_mins)
    out_layout = (LAYOUTS_3D if len(out_shape) == 3 else LAYOUTS_2D)[layout]
    for lay_in, lay_out in ((True, False), (False, True), (True, True)):
        src = make(inp) if lay_in else inp
        mk = (lambda: out_layout(np.zeros(out_shape, f.out_dtype))) if lay_out else None
        poisoned(hb, oracle, f, src, out_shape, out_mins=out_mins, make_out=mk, want=want,
                 what=f"{filt} {layout} in={lay_in} out={lay_out}")


# ---- device-resident buffers: stores into padding ----------------------------------------------------------------------

SENTINEL = {np.uint16: 0x5A5A, np.uint8: 0x5A, np.float32: -1234.5}
_TORCH_VIEW = {np.uint16: "uint16", np.uint8: "uint8", np.float32: "float32"}


def _torch_store(shape, dtype, value):
    """A CUDA tensor of `shape` holding `value`; uint16 travels as int16 bits (torch's uint16 support is thin)."""
    import torch
    if dtype == np.uint16:
        return torch.full(shape, np.array(value, np.uint16).view(np.int16).item(), dtype=torch.int16, device="cuda")
    return torch.full(shape, value, dtype=getattr(torch, _TORCH_VIEW[dtype]), device="cuda")


def _as_halide_dtype(t, dtype):
    import torch
    return t.view(torch.uint16) if dtype == np.uint16 else t


def _to_numpy(t, dtype):
    a = t.cpu().numpy()
    return a.view(np.uint16) if dtype == np.uint16 else a


def _device_input(a, odd_offset):
    """`a` on the device, optionally as a view starting one element into its storage."""
    import torch
    dtype = a.dtype.type
    bits = a.view(np.int16) if dtype == np.uint16 else a
    flat = torch.empty(a.size + 1, dtype={np.uint16: torch.int16, np.uint8: torch.uint8, np.float32: torch.float32}[dtype],
                       device="cuda")
    k = 1 if odd_offset else 0
    flat[k:k + a.size].copy_(torch.from_numpy(np.ascontiguousarray(bits).reshape(-1)))
    return _as_halide_dtype(flat[k:k + a.size].view(a.shape), dtype)


def device_resident(hb, oracle, f, inp, out_shape, want=None, odd_input=False, what=""):
    """Output = a view into a wider sentinel-filled CUDA tensor (odd column count; 3-D outputs also padded planes).
    Every output element must equal the oracle and every sentinel outside the view must survive."""
    from halide_b200 import HalideBuffer
    dtype = f.out_dtype
    n, lead = int(np.prod(out_shape)), 3
    if len(out_shape) == 4:  # conv_layer: fixed dense strides; the view sits inside a larger flat tensor instead
        store_shape = (n + 7,)
    elif len(out_shape) == 3:
        c, h, w = out_shape
        store_shape = (c, h + 3, w + (4 if w % 2 else 3))
    else:
        h, w = out_shape
        store_shape = (h + 1, w + (4 if w % 2 else 3))
    if want is None:
        want = f.want(oracle, inp, out_shape)

    def run(byte):
        store = _torch_store(store_shape, dtype, SENTINEL[dtype])
        view = store[lead:lead + n].view(out_shape) if len(out_shape) == 4 else store[tuple(slice(0, s) for s in out_shape)]
        bi = HalideBuffer.from_torch(_device_input(inp, odd_input))
        bo = HalideBuffer.from_torch(_as_halide_dtype(view, dtype))
        with fill(hb, byte):
            f.call(hb, bi, bo)
            bo.device_sync()
        got = _to_numpy(store, dtype)
        mask = np.ones(store_shape, bool)
        if len(out_shape) == 4:
            mask[lead:lead + n] = False
            out = got[lead:lead + n].reshape(out_shape)
        else:
            mask[tuple(slice(0, s) for s in out_shape)] = False
            out = got[tuple(slice(0, s) for s in out_shape)]
        outside = got[mask]
        assert (outside == SENTINEL[dtype]).all(), \
            f"{what or f.name}: {int((outside != SENTINEL[dtype]).sum())} stores outside the output view"
        return np.ascontiguousarray(out)
    got = under_fills(run)
    f.compare(got, want, what or f.name)


def _device_cases():
    return ["halide_blur", "stencil_chain", "bilateral_grid", "camera_pipe", "local_laplacian", "nl_means"]


@pytest.mark.parametrize("odd_input", [False, True])
@pytest.mark.parametrize("filt", _device_cases())
def test_device_resident_padded_outputs(hb, oracle, filt, odd_input):
    f, inp, out_shape, _ = _layout_setup(filt)
    device_resident(hb, oracle, f, inp, out_shape, odd_input=odd_input, what=f"{filt} odd_input={odd_input}")


@pytest.mark.parametrize("odd_input", [False, True])
@pytest.mark.parametrize("tc", [1, 0])
def test_device_resident_conv_layer(hb, oracle, tc, odd_input):
    """The output sits 3 floats into a larger tensor (not 16-byte aligned), the input optionally 1 float in."""
    inp, filt, bias = conv_make(5, 1.0)
    f = Filter("conv_layer", np.float32, lambda h: _conv_params(h, filt, bias), None, False, 1e-30)
    want = oracle.conv_layer(inp, filt, bias)
    l = hb.load_library()
    try:
        l.halide_b200_conv_use_tensor_cores(tc)
        device_resident(hb, oracle, f, inp, want.shape, want=want, odd_input=odd_input, what=f"conv tc={tc}")
    finally:
        l.halide_b200_conv_use_tensor_cores(1)
