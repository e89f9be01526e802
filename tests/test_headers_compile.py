"""The public headers must be usable by a C caller (the boundary is a C ABI): every include/*.h compiles as C99 and as
C++17 on its own, and a small C program that takes the address of every filter entry point links against the library."""
import glob
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INC = os.path.join(ROOT, "include")
LIBDIR = os.path.join(ROOT, "halide_b200")
HEADERS = sorted(os.path.basename(h) for h in glob.glob(os.path.join(INC, "*.h")))


@pytest.mark.parametrize("header", HEADERS)
@pytest.mark.parametrize("lang", ["c", "c++"])
def test_header_compiles_standalone(tmp_path, header, lang):
    src = tmp_path / ("t.c" if lang == "c" else "t.cpp")
    src.write_text(f'#include "{header}"\nint main(void) {{ return 0; }}\n')
    cc = ["/usr/bin/gcc", "-std=c99"] if lang == "c" else ["/usr/bin/g++", "-std=c++17"]
    out = subprocess.run(cc + ["-Wall", "-Werror", "-pedantic", "-fsyntax-only", f"-I{INC}", str(src)],
                         capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr[-2000:]


def test_c_caller_links_every_entry_point(tmp_path):
    if not os.path.exists(os.path.join(LIBDIR, "libhalide_b200.so")):
        pytest.skip("library not built")
    # every filter header: F with the parameter list the header declares, F_argv and F_metadata
    names = [h[:-2] for h in HEADERS if h != "halide_b200_runtime.h"]
    params = {}
    for n in names:
        with open(os.path.join(INC, n + ".h")) as f:
            params[n] = re.search(rf"^int {n}\((.*)\);$", f.read(), flags=re.M).group(1)
    # the filter headers only forward-declare the runtime structs (like Halide's generated headers); a caller that looks
    # inside them includes the runtime header, as the reference's harnesses include HalideRuntime.h
    body = '#include "halide_b200_runtime.h"\n' + "".join(f'#include "{n}.h"\n' for n in names)
    body += "#include <stdio.h>\nint main(void) {\n  const struct halide_filter_metadata_t *m;\n"
    for n in names:
        body += f'  m = {n}_metadata();\n  if (!m || !m->name) return 1;\n  printf("%s %d\\n", m->name, m->num_arguments);\n'
        body += f"  {{ int (*fp)(void **) = {n}_argv; if (!fp) return 2; }}\n"
        body += f"  {{ int (*fp)({params[n]}) = {n}; if (!fp) return 3; }}\n"
    body += "  return 0;\n}\n"
    src, exe = tmp_path / "caller.c", tmp_path / "caller"
    src.write_text(body)
    out = subprocess.run(["/usr/bin/gcc", "-std=c99", "-Wall", "-Werror", f"-I{INC}", str(src), "-o", str(exe), f"-L{LIBDIR}",
                          "-lhalide_b200", f"-Wl,-rpath,{LIBDIR}", "-lpthread", "-ldl"], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr[-2000:]
    run = subprocess.run([str(exe)], capture_output=True, text=True, timeout=60)  # metadata only: no CUDA call
    assert run.returncode == 0, run.stdout + run.stderr
    lines = run.stdout.split("\n")
    assert [l.split()[0] for l in lines if l] == names
    assert "halide_blur 2" in lines and "camera_pipe 10" in lines and "harris_auto_schedule 2" in lines
