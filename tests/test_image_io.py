"""halide_b200/image_io.py against the reference's own image I/O header (tools/halide_image_io.h): element conversions
for every type pair, every format both ways, and the type / dimensionality choice of convert_and_save_image.  What the
reference computed on these inputs is committed under tests/golden/: the vectors of image_io_golden.npz
(tests/golden/make_image_io_golden.py), and digests of its whole outputs plus its sample images, cut short
(reference_digests.json and images/, tests/golden/make_reference_golden.py).  Both scripts ran the header compiled in
place (oracle/ref_image_io_tool.cpp)."""
import os

import numpy as np
import pytest

from halide_b200 import image_io
from util import reference, sha

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "image_io_golden.npz")
IMAGES = os.path.join(ROOT, "tests", "golden", "images")
NAMES = {"u8": np.uint8, "u16": np.uint16, "u32": np.uint32, "u64": np.uint64, "i8": np.int8, "i16": np.int16,
         "i32": np.int32, "i64": np.int64, "f32": np.float32, "f64": np.float64}
TNAME = {np.dtype(v): k for k, v in NAMES.items()}


def file_sha(path):
    with open(path, "rb") as f:
        return sha(f.read())


def case_id(fmt, dtype, shape):
    return f"{fmt}-{TNAME[np.dtype(dtype)]}-{'x'.join(map(str, shape))}"


def samples(dtype, n=2048, seed=0):
    """Inputs with defined behaviour in the reference: every integer pattern; floats mostly in [0, 1] plus exact halves,
    negatives and values up to a few thousand (float -> integer conversions go through lround and a modular cast)."""
    rng = np.random.default_rng(seed)
    dt = np.dtype(dtype)
    if dt.kind in "ui":
        info = np.iinfo(dt)
        edge = np.array([info.min, info.max, 0, 1, info.max // 2, info.max // 2 + 1, info.min // 2, 127, 128, 255, 256 % (info.max + 1)],
                        dtype=np.int64 if dt.kind == "i" else np.uint64).astype(dt)
        body = rng.integers(info.min, info.max, n, dtype=dt, endpoint=True)
        return np.concatenate([edge, body])
    edge = np.array([0.0, 1.0, 0.5, 0.25, 0.75, 1.0 / 255, 0.5 / 255, 1.5 / 255, 2.5 / 255, 0.5 / 65535, 1.5 / 65535, -0.25, -1.0, 1.5,
                     2.0, 100.25, 1000.5, -3.75], dtype=dt)
    return np.concatenate([edge, rng.random(n).astype(dt), (rng.random(64) * 8 - 4).astype(dt)])


@pytest.mark.parametrize("src", list(NAMES))
def test_convert_matches_reference_for_every_target(src):
    a = samples(NAMES[src], seed=len(src))
    for dst in NAMES:
        got = image_io.convert(a, NAMES[dst])
        assert got.dtype == np.dtype(NAMES[dst]) and got.shape == a.shape
        assert sha(got) == reference()["convert"][src][dst], (src, dst)


def test_convert_matches_golden_vectors():
    g = np.load(GOLDEN)
    for key in g.files:
        if not key.startswith("conv_in_"):
            continue
        src = key[len("conv_in_"):]
        for dst in NAMES:
            want = g[f"conv_{src}_{dst}"]
            got = image_io.convert(g[key], NAMES[dst])
            assert np.array_equal(got.view(np.uint8), want.view(np.uint8)), (src, dst)


def test_conversion_rules_spelled_out():
    """The rules the natural-image runs of the seven pipelines actually meet (tools/halide_image_io.h:130-240,606-616)."""
    u8 = np.arange(256, dtype=np.uint8)
    assert np.array_equal(image_io.convert(u8, np.uint16), u8.astype(np.uint16) * 257)
    assert np.array_equal(image_io.convert(image_io.convert(u8, np.uint16), np.uint8), u8)
    u16 = np.arange(65536, dtype=np.uint32).astype(np.uint16)
    assert np.array_equal(image_io.convert(u16, np.uint8), np.floor((u16.astype(np.float64) + 128.5) / 257).astype(np.uint8))
    assert image_io.convert(u8, np.float32)[255] == np.float32(1.0) and image_io.convert(u16, np.float32)[65535] == np.float32(1.0)
    f = np.array([0.0, 0.5 / 255, 1.5 / 255 + 1e-7, 1.0, 2.0, -1.0 / 255], np.float32)
    assert list(image_io.convert(f, np.uint8)) == [0, 1, 2, 255, 254, 255]   # lround, then a modular cast


FORMAT_CASES = [("pgm", np.uint8, (37, 50)), ("pgm", np.uint16, (9, 13)), ("ppm", np.uint8, (3, 21, 34)), ("ppm", np.uint16, (3, 5, 7)),
                ("npy", np.float32, (3, 6, 5)), ("npy", np.uint16, (4, 9)), ("npy", np.int64, (2, 3, 4, 5)), ("npy", np.uint8, (11,)),
                ("tmp", np.float32, (1, 3, 8, 6)), ("tmp", np.int16, (2, 2, 3, 4)), ("mat", np.float32, (3, 4)),
                ("mat", np.float64, (2, 3, 5)), ("mat", np.uint16, (4, 6))]


def random_image(dtype, shape, seed):
    rng = np.random.default_rng(seed)
    dt = np.dtype(dtype)
    if dt.kind == "f":
        return rng.random(shape).astype(dt)
    info = np.iinfo(dt)
    return rng.integers(info.min, info.max, shape, dtype=dt, endpoint=True)


@pytest.mark.parametrize("fmt,dtype,shape", FORMAT_CASES)
def test_formats_round_trip_through_the_reference(fmt, dtype, shape, tmp_path):
    """Our writer produces the reference's bytes (a .mat file carries its own file name as the variable name, hence the
    reference's name img.<fmt>), and our reader decodes them to the array written (the reference read its own file back
    to the same array when the digest was made)."""
    a = random_image(dtype, shape, len(shape) * 7 + np.dtype(dtype).itemsize)
    our_file = str(tmp_path / ("img." + fmt))
    image_io.save(a, our_file)
    assert file_sha(our_file) == reference()["formats"][case_id(fmt, dtype, shape)]
    got = image_io.load(our_file)
    assert got.dtype == a.dtype and np.array_equal(got, a)


AUTOSAVE_SHAPES = {"pgm": [(6, 7)], "ppm": [(3, 6, 7)], "npy": [(5,), (6, 7), (3, 6, 7)], "tmp": [(6, 7), (3, 6, 7), (2, 3, 6, 7)],
                   "mat": [(6, 7), (3, 6, 7)]}


@pytest.mark.parametrize("fmt", list(AUTOSAVE_SHAPES))
def test_convert_and_save_picks_the_reference_type(fmt, tmp_path):
    """convert_and_save_image writes the reference's file byte for byte: the same element type and dimensionality
    chosen for the format, the same converted values."""
    for shape in AUTOSAVE_SHAPES[fmt]:
        for src in NAMES.values():
            our_file = str(tmp_path / ("img." + fmt))
            image_io.convert_and_save_image(random_image(src, shape, 3), our_file)
            assert file_sha(our_file) == reference()["autosave"][case_id(fmt, src, shape)], (fmt, shape, src)


def test_load_and_convert_of_the_reference_images():
    """apps/images/gray_small.pgm (its first rows) and the camera_pipe colour matrices, loaded into every type the
    harnesses ask for."""
    for name, types in (("gray_small.pgm", ("u8", "u16", "f32")), ("matrix_3200.mat", ("f32",)), ("matrix_7000.mat", ("f32", "f64"))):
        for t in types:
            got = image_io.load_and_convert_image(os.path.join(IMAGES, name), NAMES[t])
            want = reference()["load_and_convert"][f"{name}:{t}"]
            assert TNAME[got.dtype] == want["dtype"] and list(got.shape) == want["shape"], (name, t)
            assert sha(got) == want["sha256"], (name, t)


def test_golden_files_decode_identically():
    """Files written by the reference (committed bytes) decode to the committed arrays, and our writers reproduce the
    reference's bytes for the formats whose encoding is fully determined."""
    g = np.load(GOLDEN)
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        for key in g.files:
            if not key.startswith("file_"):
                continue
            _, fmt, tag = key.split("_", 2)
            path = os.path.join(d, f"{tag}.{fmt}")
            open(path, "wb").write(g[key].tobytes())
            want = g[f"array_{fmt}_{tag}"]
            got = image_io.load(path)
            assert got.dtype == want.dtype and np.array_equal(got, want), key
            if fmt in ("pgm", "ppm", "npy", "tmp"):
                ours = os.path.join(d, f"ours_{tag}.{fmt}")
                image_io.save(want, ours)
                assert open(ours, "rb").read() == g[key].tobytes(), key


def test_png_codec_round_trip_and_cross_check(tmp_path):
    """PNG (the reference reads it through libpng, which is not available to its header build here): our writer / reader
    round trip for 8- and 16-bit gray, gray+alpha, RGB and RGBA, the pure-Python decoder against OpenCV's on files with
    Sub / Up / Average / Paeth rows when OpenCV is importable."""
    for dtype, shape in ((np.uint8, (20, 31)), (np.uint16, (7, 9)), (np.uint8, (3, 12, 17)), (np.uint16, (3, 6, 5)),
                         (np.uint8, (4, 5, 6)), (np.uint16, (2, 5, 6))):
        a = random_image(dtype, shape, 5)
        p = str(tmp_path / "a.png")
        image_io.save(a, p) if (np.dtype(dtype), len(shape)) in image_io.save_query(p) and (len(shape) == 2 or shape[0] == 3) \
            else image_io._save_png(a, p)
        os.environ["HALIDE_B200_PNG_PURE"] = "1"
        try:
            got = image_io.load(p)
        finally:
            del os.environ["HALIDE_B200_PNG_PURE"]
        assert got.dtype == a.dtype and np.array_equal(got, a), (dtype, shape)
    try:
        import cv2
    except Exception:
        return
    yy, xx = np.mgrid[0:40, 0:56]
    smooth = ((np.sin(xx / 5.0) * np.cos(yy / 7.0) * 0.4 + 0.5) * 65535).astype(np.uint16)   # adaptive filters pick Paeth / Average here
    for arr in (smooth, (smooth >> 8).astype(np.uint8), np.stack([smooth, smooth[::-1], smooth.T[:40, :40].repeat(2, 1)[:, :56]])):
        p = str(tmp_path / "cv.png")
        cv2.imwrite(p, arr if arr.ndim == 2 else np.ascontiguousarray(arr.transpose(1, 2, 0)[:, :, ::-1]))
        os.environ["HALIDE_B200_PNG_PURE"] = "1"
        try:
            pure = image_io.load(p)
        finally:
            del os.environ["HALIDE_B200_PNG_PURE"]
        assert np.array_equal(pure, arr) and np.array_equal(image_io.load(p), arr)


def test_reference_png_images_decode_the_same_both_ways():
    """The reference's small sample images (apps/images/*_small*.png: 8-bit gray and RGB, 16-bit RGB, 16-bit Bayer raw;
    their first rows, as filtered in the reference's files) through the pure-Python decoder and through OpenCV;
    gray_small.png must equal gray_small.pgm, which the reference's own reader decodes
    (test_load_and_convert_of_the_reference_images)."""
    images = IMAGES
    try:
        import cv2  # noqa: F401
    except Exception:
        pytest.skip("OpenCV not importable: nothing to cross-check against")
    for name in ("gray_small.png", "rgb_small.png", "rgb_small16.png", "bayer_small.png"):
        p = os.path.join(images, name)
        fast = image_io.load(p)
        os.environ["HALIDE_B200_PNG_PURE"] = "1"
        try:
            pure = image_io.load(p)
        finally:
            del os.environ["HALIDE_B200_PNG_PURE"]
        assert fast.dtype == pure.dtype and np.array_equal(fast, pure), name
    assert np.array_equal(image_io.load(os.path.join(images, "gray_small.png")), image_io.load(os.path.join(images, "gray_small.pgm")))


TIFF_CASES = [(np.uint8, (9, 14)), (np.uint16, (3, 9, 14)), (np.float32, (4, 5, 6)), (np.int32, (7,)), (np.float64, (2, 3, 4, 5)),
              (np.uint8, (6, 3, 4)), (np.int16, (1, 2, 8, 9))]


@pytest.mark.parametrize("dtype,shape", TIFF_CASES)
def test_tiff_writer_is_byte_identical(dtype, shape, tmp_path):
    """The reference writes (uncompressed, planar) TIFF and cannot read it back; ours must produce the same bytes —
    including the rule that folds a third dimension below 5 into the channel count."""
    a = random_image(dtype, shape, 11)
    our_file = str(tmp_path / "ours.tiff")
    image_io.save(a, our_file)
    assert file_sha(our_file) == reference()["tiff"][case_id("tiff", dtype, shape)]
    with pytest.raises(ValueError):
        image_io.load(our_file)


def test_natural_image_flow_like_process_cpp(tmp_path):
    """apps/local_laplacian/process.cpp end to end on the host side: load_and_convert_image(png) into uint16 planes, the
    filter (the CPU oracle stands in for it here — the GPU parity tests cover the filter itself), convert_and_save_image
    to a 16-bit PNG, reload: the file holds exactly the filter's output, and an 8-bit source enters as x * 257."""
    from oracle import pyoracle
    src = os.path.join(IMAGES, "rgb_small.png")
    native = image_io.load(src)
    assert native.dtype == np.uint8 and native.ndim == 3 and native.shape[0] == 3
    frame = image_io.load_and_convert_image(src, np.uint16)
    assert np.array_equal(frame, native.astype(np.uint16) * 257)
    frame = np.ascontiguousarray(frame[:, :96, :128])   # a crop keeps the oracle quick
    out = pyoracle.local_laplacian(frame, 8, 1.0 / 7.0, 1.0)
    dst = str(tmp_path / "out.png")
    image_io.convert_and_save_image(out, dst)
    back = image_io.load(dst)
    assert back.dtype == np.uint16 and np.array_equal(back, out)
    image_io.convert_and_save_image(out, str(tmp_path / "out8.ppm"))   # (.ppm holds uint16 too: saved as is)
    assert np.array_equal(image_io.load(str(tmp_path / "out8.ppm")), out)
