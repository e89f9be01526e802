// oracle/oracle_harris.cpp — TEST INFRASTRUCTURE, NOT PRODUCT CODE (see oracle.h).
//
// CPU restatement of apps/harris/harris_generator.cpp:22-61.  Each Func is realised on the box its consumer reads
// (gray on the output box grown by 2, the gradient products on it grown by 1), every f32 expression in the generator's
// nesting.  The CUDA kernel must match bit for bit.
#include <vector>

#include "oracle_apps.h"

extern "C" int oracle_harris(const oracle_image_t *in, const oracle_image_t *out) {
    const int ox = out->min[0], oy = out->min[1], W = out->extent[0], H = out->extent[1];
    if (W <= 0 || H <= 0) return 0;
    if (ox - 2 < in->min[0] || ox + W + 1 > in->min[0] + in->extent[0] - 1 || oy - 2 < in->min[1] ||
        oy + H + 1 > in->min[1] + in->extent[1] - 1 || in->min[2] > 0 || in->min[2] + in->extent[2] < 3) {
        return -4;
    }
    const float *ib = (const float *)in->base;
    auto input = [&](int x, int y, int c) -> float {
        return ib[(int64_t)(x - in->min[0]) * in->stride[0] + (int64_t)(y - in->min[1]) * in->stride[1] +
                  (int64_t)(c - in->min[2]) * in->stride[2]];
    };
    // gray on [ox-2, ox+W+1] x [oy-2, oy+H+1]
    const int gw = W + 4, gh = H + 4;
    std::vector<float> gray((size_t)gw * gh);
#pragma omp parallel for
    for (int v = 0; v < gh; v++) {
        for (int u = 0; u < gw; u++) {
            const int x = ox - 2 + u, y = oy - 2 + v;
            gray[(size_t)v * gw + u] = (0.299f * input(x, y, 0) + 0.587f * input(x, y, 1)) + 0.114f * input(x, y, 2);
        }
    }
    // Ixx, Iyy, Ixy on [ox-1, ox+W] x [oy-1, oy+H]
    const int pw = W + 2, ph = H + 2;
    std::vector<float> ixx((size_t)pw * ph), iyy((size_t)pw * ph), ixy((size_t)pw * ph);
    const float m1 = -1.0f / 12, p1 = 1.0f / 12, m2 = -2.0f / 12, p2 = 2.0f / 12;
#pragma omp parallel for
    for (int v = 0; v < ph; v++) {
        for (int u = 0; u < pw; u++) {
            // g(dx, dy): gray at (x + dx, y + dy) for the product position (x, y) = (ox - 1 + u, oy - 1 + v)
            auto g = [&](int dx, int dy) { return gray[(size_t)(v + 1 + dy) * gw + (u + 1 + dx)]; };
            const float Iy = g(-1, -1) * m1 + g(-1, 1) * p1 + g(0, -1) * m2 + g(0, 1) * p2 + g(1, -1) * m1 + g(1, 1) * p1;
            const float Ix = g(-1, -1) * m1 + g(1, -1) * p1 + g(-1, 0) * m2 + g(1, 0) * p2 + g(-1, 1) * m1 + g(1, 1) * p1;
            ixx[(size_t)v * pw + u] = Ix * Ix;
            iyy[(size_t)v * pw + u] = Iy * Iy;
            ixy[(size_t)v * pw + u] = Ix * Iy;
        }
    }
    float *ob = (float *)out->base;
#pragma omp parallel for
    for (int y = 0; y < H; y++) {
        for (int x = 0; x < W; x++) {
            // sum3x3 (generator :7-11): f(x-1, y-1) + f(x-1, y) + f(x-1, y+1) + f(x, y-1) + ... + f(x+1, y+1)
            auto sum3x3 = [&](const std::vector<float> &f) {
                float s = 0.0f;
                bool first = true;
                for (int dx = -1; dx <= 1; dx++) {
                    for (int dy = -1; dy <= 1; dy++) {
                        const float t = f[(size_t)(y + 1 + dy) * pw + (x + 1 + dx)];
                        s = first ? t : s + t;
                        first = false;
                    }
                }
                return s;
            };
            const float Sxx = sum3x3(ixx), Syy = sum3x3(iyy), Sxy = sum3x3(ixy);
            const float det = Sxx * Syy - Sxy * Sxy;
            const float trace = Sxx + Syy;
            ob[(int64_t)x * out->stride[0] + (int64_t)y * out->stride[1]] = det - 0.04f * trace * trace;
        }
    }
    return 0;
}
