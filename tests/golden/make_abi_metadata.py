"""Writes tests/golden/abi_metadata.json: every F_metadata() record libhalide_b200.so exports, one per filter header in
include/ (F and, where the filter has one, F_auto_schedule).  Reading the records needs no GPU.

The snapshot pins the exported metadata (argument names, kinds, types, scalar defaults and estimates, buffer
estimates, target string) so that a change to how the records are declared cannot change what a RunGen driver or a
harness reads (tests/test_abi.py compares the library against it).  Re-run only when a filter's signature or its
estimates are deliberately changed, after building the library:
    python tests/golden/make_abi_metadata.py
"""
import ctypes
import glob
import json
import os

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
OUT = os.path.join(HERE, "abi_metadata.json")


class Arg(ctypes.Structure):  # halide_filter_argument_t
    _fields_ = [("name", ctypes.c_char_p), ("kind", ctypes.c_int32), ("dimensions", ctypes.c_int32),
                ("code", ctypes.c_uint8), ("bits", ctypes.c_uint8), ("lanes", ctypes.c_uint16),
                ("scalar_def", ctypes.c_void_p), ("scalar_min", ctypes.c_void_p), ("scalar_max", ctypes.c_void_p),
                ("scalar_estimate", ctypes.c_void_p), ("buffer_estimates", ctypes.POINTER(ctypes.POINTER(ctypes.c_int64)))]


class Meta(ctypes.Structure):  # halide_filter_metadata_t
    _fields_ = [("version", ctypes.c_int32), ("num_arguments", ctypes.c_int32), ("arguments", ctypes.POINTER(Arg)),
                ("target", ctypes.c_char_p), ("name", ctypes.c_char_p)]


def filter_functions():
    """The filter functions, one per include/F.h (the runtime header declares no filter)."""
    return sorted(os.path.basename(h)[:-2] for h in glob.glob(os.path.join(ROOT, "include", "*.h"))
                  if not h.endswith("halide_b200_runtime.h"))


def _scalar(p, code, bits):
    if not p:
        return None
    ctype = {(0, 32): ctypes.c_int32, (2, 32): ctypes.c_float}[(code, bits)]  # the filters' scalars: int32 and float
    return ctypes.cast(p, ctypes.POINTER(ctype))[0]


def dump(lib, fn):
    f = getattr(lib, fn + "_metadata")
    f.restype = ctypes.POINTER(Meta)
    md = f().contents
    args = []
    for i in range(md.num_arguments):
        a = md.arguments[i]
        est = None
        if a.buffer_estimates:
            est = [a.buffer_estimates[k][0] if a.buffer_estimates[k] else None for k in range(2 * a.dimensions)]
        args.append({"name": a.name.decode(), "kind": a.kind, "dimensions": a.dimensions,
                     "type": [a.code, a.bits, a.lanes],
                     **{s: _scalar(getattr(a, s), a.code, a.bits) for s in ("scalar_def", "scalar_min", "scalar_max", "scalar_estimate")},
                     "buffer_estimates": est})
    return {"version": md.version, "num_arguments": md.num_arguments, "target": md.target.decode(),
            "name": md.name.decode(), "arguments": args}


def dump_all(lib):
    return {fn: dump(lib, fn) for fn in filter_functions()}


def main():
    lib = ctypes.CDLL(os.path.join(ROOT, "halide_b200", "libhalide_b200.so"))
    with open(OUT, "w") as f:
        json.dump(dump_all(lib), f, indent=1, sort_keys=True)
        f.write("\n")
    print(f"wrote {OUT}")


if __name__ == "__main__":
    main()
