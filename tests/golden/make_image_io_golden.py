"""Writes tests/golden/image_io_golden.npz with the reference's own image I/O header as the source of truth
(oracle/_ref/ref_image_io = tools/halide_image_io.h compiled in place, oracle/ref_image_io_tool.cpp):
  conv_in_<src>, conv_<src>_<dst>   element conversion vectors for every type pair
  file_<fmt>_<tag>, array_<fmt>_<tag>   files as the reference writes them (raw bytes) and the arrays they hold
Run from the repo root in the container that has /root/reference:  python tests/golden/make_image_io_golden.py"""
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
from make_reference_golden import REF_IO as REF, write_dump  # noqa: E402
from test_image_io import FORMAT_CASES, NAMES, TNAME, random_image, samples  # noqa: E402


def main():
    out = {}
    with tempfile.TemporaryDirectory() as d:
        for src, st in NAMES.items():
            a = samples(st, n=256, seed=100 + len(src))
            out[f"conv_in_{src}"] = a
            a.tofile(os.path.join(d, "in.bin"))
            for dst, dt in NAMES.items():
                subprocess.run([REF, "convert", src, dst, os.path.join(d, "in.bin"), os.path.join(d, "out.bin")], check=True)
                out[f"conv_{src}_{dst}"] = np.fromfile(os.path.join(d, "out.bin"), dtype=dt)
        for i, (fmt, dtype, shape) in enumerate(FORMAT_CASES):
            a = random_image(dtype, shape, 1000 + i)
            tag = f"{TNAME[np.dtype(dtype)]}_{len(shape)}d"
            write_dump(a, os.path.join(d, "a.dump"))
            path = os.path.join(d, f"x.{fmt}")
            subprocess.run([REF, "save", os.path.join(d, "a.dump"), path], check=True)
            out[f"file_{fmt}_{tag}"] = np.frombuffer(open(path, "rb").read(), dtype=np.uint8)
            out[f"array_{fmt}_{tag}"] = a
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "image_io_golden.npz"), **out)
    print("wrote", len(out), "entries")


if __name__ == "__main__":
    main()
