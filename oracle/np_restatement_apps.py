"""Second, independently structured restatement of harris and unsharp in numpy — TEST INFRASTRUCTURE ONLY.

The companion of oracle/np_restatement.py for the apps of oracle/oracle_apps.h: every Func is a whole-array float32
expression over the index range Halide's bounds inference gives it, every operation in the generator's nesting (numpy
evaluates float32 binary operations with IEEE rounding and never contracts them).  tests/test_harris_unsharp_cpu.py
compares it with oracle/oracle_harris.cpp and oracle/oracle_unsharp.cpp bit for bit.

Follows apps/harris/harris_generator.cpp:7-11,22-61 and apps/unsharp/unsharp_generator.cpp:15-51,
src/BoundaryConditions.h (repeat_edge clamps every dimension to the buffer's own box).
"""
import numpy as np

F = np.float32


def _take(inp, in_mins, xs, ys, c):
    """inp[c, ys, xs] in Halide coordinates (in_mins = (x, y, c) mins); every index must lie inside the buffer."""
    ix, iy, ic = np.asarray(xs) - in_mins[0], np.asarray(ys) - in_mins[1], c - in_mins[2]
    assert 0 <= ic < inp.shape[0], "channel outside the input"
    assert ix.min() >= 0 and ix.max() < inp.shape[2] and iy.min() >= 0 and iy.max() < inp.shape[1], "read outside the input"
    return inp[ic][iy[:, None], ix[None, :]]


def _gray(r, g, b):
    return (F(0.299) * r + F(0.587) * g) + F(0.114) * b


def harris(inp, out_shape, in_mins=(0, 0, 0), out_mins=(0, 0)):
    """inp: float32 [c, h, w]; out_shape (H, W) at out_mins (x, y)."""
    H, W = out_shape
    ox, oy = out_mins
    xs, ys = np.arange(ox - 2, ox + W + 2), np.arange(oy - 2, oy + H + 2)  # gray's box
    gray = _gray(*(_take(inp, in_mins, xs, ys, c) for c in range(3)))

    def g(dx, dy):  # gray(x + dx, y + dy) over the products' box [ox-1, ox+W] x [oy-1, oy+H]
        return gray[1 + dy:1 + dy + H + 2, 1 + dx:1 + dx + W + 2]
    k1, k2 = F(1.0) / F(12), F(2.0) / F(12)
    Iy = g(-1, -1) * -k1 + g(-1, 1) * k1 + g(0, -1) * -k2 + g(0, 1) * k2 + g(1, -1) * -k1 + g(1, 1) * k1
    Ix = g(-1, -1) * -k1 + g(1, -1) * k1 + g(-1, 0) * -k2 + g(1, 0) * k2 + g(-1, 1) * -k1 + g(1, 1) * k1

    def sum3x3(f):
        terms = [f[1 + dy:1 + dy + H, 1 + dx:1 + dx + W] for dx in (-1, 0, 1) for dy in (-1, 0, 1)]
        s = terms[0]
        for t in terms[1:]:
            s = s + t
        return s
    Sxx, Syy, Sxy = sum3x3(Ix * Ix), sum3x3(Iy * Iy), sum3x3(Ix * Iy)
    det = Sxx * Syy - Sxy * Sxy
    trace = Sxx + Syy
    return (det - F(0.04) * trace * trace).astype(F)


def unsharp_weights():
    """kernel(k) = exp(-k^2 / 4.5f) / 3.7599425f for k = 0..3, each constant division and the exp folded in double and
    rounded to float32 (see oracle/oracle_unsharp.cpp)."""
    two_sigma_sq = F(2) * F(1.5) * F(1.5)
    norm = F(np.sqrt(F(2) * F(3.14159265358979310000), dtype=F) * F(1.5))
    w = []
    for k in range(4):
        q = F(np.float64(F(-(k * k))) / np.float64(two_sigma_sq))
        e = F(np.exp(np.float64(q)))
        w.append(F(np.float64(e) / np.float64(norm)))
    return np.array(w, F)


def unsharp(inp, out_shape, in_mins=(0, 0, 0), out_mins=(0, 0, 0)):
    """inp: float32 [c, h, w]; out_shape (C, H, W) at out_mins (x, y, c)."""
    C, H, W = out_shape
    ox, oy, oc = out_mins
    w0, w1, w2, w3 = unsharp_weights()
    n_c, n_y, n_x = inp.shape
    xs = np.clip(np.arange(ox - 3, ox + W + 3), in_mins[0], in_mins[0] + n_x - 1)  # repeat_edge
    ys = np.clip(np.arange(oy - 3, oy + H + 3), in_mins[1], in_mins[1] + n_y - 1)
    cs = [int(np.clip(c, in_mins[2], in_mins[2] + n_c - 1)) for c in range(3)]
    gray = _gray(*(_take(inp, in_mins, xs, ys, c) for c in cs))  # [oy-3, oy+H+2] x [ox-3, ox+W+2]

    def g(dy):  # gray(x, y + dy) over blur_y's box [ox-3, ox+W+2] x [oy, oy+H-1]
        return gray[3 + dy:3 + dy + H, :]
    blur_y = ((w0 * g(0) + w1 * (g(-1) + g(1))) + w2 * (g(-2) + g(2))) + w3 * (g(-3) + g(3))

    def b(dx):  # blur_y(x + dx, y) over the output box
        return blur_y[:, 3 + dx:3 + dx + W]
    blur_x = ((w0 * b(0) + w1 * (b(-1) + b(1))) + w2 * (b(-2) + b(2))) + w3 * (b(-3) + b(3))
    centre = gray[3:3 + H, 3:3 + W]
    oxs, oys = np.arange(ox, ox + W), np.arange(oy, oy + H)
    with np.errstate(divide="ignore", invalid="ignore"):  # gray == 0 gives +-inf or NaN, as in the reference
        ratio = (F(2.0) * centre - blur_x) / centre
        return np.stack([ratio * _take(inp, in_mins, oxs, oys, c) for c in range(oc, oc + C)]).astype(F)
