"""Generates tests/golden/harris_small.npz and unsharp_small.npz by running the CPU oracle of harris and unsharp
(oracle/pyoracle_apps.py) once on seeded inputs, from a generator of their own so that the other vectors
(tests/golden/make_golden.py) stay as they are.

Like those, the vectors pin our restatement and detect the oracle and the kernels drifting together
(tests/test_harris_unsharp_cpu.py checks the oracle).  Re-run only when the oracle's definition is deliberately changed:
    python tests/golden/make_golden_apps.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import pyoracle_apps  # noqa: E402


def save(name, **kw):
    np.savez_compressed(os.path.join(HERE, name), **kw)


def main():
    rng = np.random.default_rng(20261017)
    h_in = rng.random((3, 40, 56), dtype=np.float32)
    save("harris_small.npz", input=h_in, output=pyoracle_apps.harris(h_in), out_min=np.array([3, 3], np.int32))
    u_in = rng.random((3, 36, 52), dtype=np.float32)
    u_in[:, 10:16, 20:28] = 0.0  # a black patch: gray == 0, so the output holds NaN there, as the reference's does
    with np.errstate(all="ignore"):
        save("unsharp_small.npz", input=u_in, output=pyoracle_apps.unsharp(u_in))
    print("wrote harris / unsharp golden vectors")


if __name__ == "__main__":
    main()
