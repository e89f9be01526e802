"""Writes what the reference-parity tests compare against, so that they run without the reference:

  tests/golden/reference_digests.json   SHA-256 digests of the reference's outputs on the tests' own seeded inputs:
                                        its C blur (apps/blur/test.cpp), and its image I/O header
                                        (tools/halide_image_io.h): element conversions, the files it writes, the
                                        arrays it loads
  tests/golden/images/                  the reference's small sample images (apps/images), cut to their first
                                        IMAGE_ROWS rows: PGM rows as they are, PNG by keeping the first filtered
                                        scanlines of the image data stream (each row keeps the reference's filter
                                        type; only the zlib wrapping is redone), the colour matrices whole

The digests cover whole outputs; a test recomputes its side on the same inputs and compares digests.  Needs
oracle/_ref (built by oracle/Makefile where the reference is present).  Run from the repository root:
    python tests/golden/make_reference_golden.py REFERENCE_DIR
"""
import json
import os
import re
import struct
import subprocess
import sys
import tempfile
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from test_image_io import (AUTOSAVE_SHAPES, FORMAT_CASES, IMAGES, NAMES, TIFF_CASES, TNAME, case_id, random_image,  # noqa: E402
                           samples)
from util import sha, u16_frame  # noqa: E402

REF_IO = os.path.join(ROOT, "oracle", "_ref", "ref_image_io")
IMAGE_ROWS = 32


def write_dump(a, path):
    """The exchange format of oracle/ref_image_io_tool.cpp: a text line (type, rank, Halide extents x first) + raw data."""
    with open(path, "wb") as f:
        f.write((" ".join([TNAME[a.dtype], str(a.ndim)] + [str(e) for e in reversed(a.shape)]) + "\n").encode())
        f.write(np.ascontiguousarray(a).tobytes())


def read_dump(path):
    b = open(path, "rb").read()
    nl = b.index(b"\n")
    parts = b[:nl].decode().split()
    ext = [int(e) for e in parts[2:2 + int(parts[1])]]
    return np.frombuffer(b[nl + 1:], dtype=NAMES[parts[0]]).reshape(tuple(reversed(ext))).copy()


def ref(*args):
    subprocess.run([REF_IO] + [str(a) for a in args], check=True)


def first_rows_pgm(src, dst, rows):
    data = open(src, "rb").read()
    m = re.match(rb"P5\s+(\d+)\s+(\d+)\s+(\d+)\s", data)   # one whitespace byte ends the header; pixels may look like one
    w, h, maxval = (int(g) for g in m.groups())
    assert maxval < 256 and h >= rows
    open(dst, "wb").write(b"P5\n%d %d\n%d\n" % (w, rows, maxval) + data[m.end():m.end() + w * rows])


def first_rows_png(src, dst, rows):
    data = open(src, "rb").read()
    chunks, i = [], 8
    while i < len(data):
        (n,) = struct.unpack(">I", data[i:i + 4])
        chunks.append((data[i + 4:i + 8], data[i + 8:i + 8 + n]))
        i += 12 + n
    w, h, depth, ctype, _, _, interlace = struct.unpack(">IIBBBBB", chunks[0][1])
    assert interlace == 0 and h >= rows
    channels = {0: 1, 2: 3, 3: 1, 4: 2, 6: 4}[ctype]
    row_bytes = 1 + (w * channels * depth + 7) // 8   # filter-type byte + the row
    idat = zlib.decompress(b"".join(d for t, d in chunks if t == b"IDAT"))[:rows * row_bytes]

    def chunk(t, d):
        return struct.pack(">I", len(d)) + t + d + struct.pack(">I", zlib.crc32(t + d))
    out = data[:8] + chunk(b"IHDR", struct.pack(">IIBBBBB", w, rows, depth, ctype, 0, 0, 0))
    out += b"".join(chunk(t, d) for t, d in chunks[1:] if t not in (b"IDAT", b"IEND"))
    open(dst, "wb").write(out + chunk(b"IDAT", zlib.compress(idat, 9)) + chunk(b"IEND", b""))


def main(reference):
    from oracle import pyoracle
    os.makedirs(IMAGES, exist_ok=True)
    src_images = os.path.join(reference, "apps", "images")
    for name in ("gray_small.png", "rgb_small.png", "rgb_small16.png", "bayer_small.png"):
        first_rows_png(os.path.join(src_images, name), os.path.join(IMAGES, name), IMAGE_ROWS)
    first_rows_pgm(os.path.join(src_images, "gray_small.pgm"), os.path.join(IMAGES, "gray_small.pgm"), IMAGE_ROWS)
    for name in ("matrix_3200.mat", "matrix_7000.mat"):
        open(os.path.join(IMAGES, name), "wb").write(open(os.path.join(src_images, name), "rb").read())

    out = {"blur": {}, "convert": {}, "formats": {}, "autosave": {}, "tiff": {}, "load_and_convert": {}}
    # tests/test_oracle_prims.py and tests/test_blur_gpu.py: the reference's naive (slow) and SSE (fast) C blur
    small = (np.random.default_rng(11).integers(0, 65536, (98, 264), dtype=np.uint16) & 0xFFF).astype(np.uint16)
    for key, a in (("98x264", small), ("1922x2568", u16_frame((1922, 2568), 7, bits=12))):
        out["blur"][key] = {k: sha(pyoracle.ref_blur(a, fast=f)) for k, f in (("slow", False), ("fast", True))}

    with tempfile.TemporaryDirectory() as d:
        p = lambda *n: os.path.join(d, *n)  # noqa: E731
        for src in NAMES:
            a = samples(NAMES[src], seed=len(src))
            a.tofile(p("in.bin"))
            out["convert"][src] = {}
            for dst in NAMES:
                ref("convert", src, dst, p("in.bin"), p("out.bin"))
                out["convert"][src][dst] = sha(open(p("out.bin"), "rb").read())
        os.makedirs(p("r"))
        for fmt, dtype, shape in FORMAT_CASES:
            a = random_image(dtype, shape, len(shape) * 7 + np.dtype(dtype).itemsize)
            write_dump(a, p("a.dump"))
            ref("save", p("a.dump"), p("r", "img." + fmt))
            ref("load", p("r", "img." + fmt), p("b.dump"))   # the reference reads back what it wrote
            assert np.array_equal(read_dump(p("b.dump")), a)
            out["formats"][case_id(fmt, dtype, shape)] = sha(open(p("r", "img." + fmt), "rb").read())
        for fmt, shapes in AUTOSAVE_SHAPES.items():
            for shape in shapes:
                for src in NAMES.values():
                    write_dump(random_image(src, shape, 3), p("a.dump"))
                    ref("autosave", p("a.dump"), p("img." + fmt))
                    out["autosave"][case_id(fmt, src, shape)] = sha(open(p("img." + fmt), "rb").read())
        for dtype, shape in TIFF_CASES:
            write_dump(random_image(dtype, shape, 11), p("a.dump"))
            ref("save", p("a.dump"), p("img.tiff"))
            out["tiff"][case_id("tiff", dtype, shape)] = sha(open(p("img.tiff"), "rb").read())
        for name, types in (("gray_small.pgm", ("u8", "u16", "f32")), ("matrix_3200.mat", ("f32",)), ("matrix_7000.mat", ("f32", "f64"))):
            for t in types:
                ref("loadconv", os.path.join(IMAGES, name), t, p("x.dump"))
                a = read_dump(p("x.dump"))
                out["load_and_convert"][f"{name}:{t}"] = {"dtype": TNAME[a.dtype], "shape": list(a.shape), "sha256": sha(a)}

    with open(os.path.join(ROOT, "tests", "golden", "reference_digests.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote tests/golden/reference_digests.json and", len(os.listdir(IMAGES)), "images")


if __name__ == "__main__":
    main(sys.argv[1])
