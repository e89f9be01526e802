// oracle/oracle_unsharp.cpp — TEST INFRASTRUCTURE, NOT PRODUCT CODE (see oracle.h).
//
// CPU restatement of apps/unsharp/unsharp_generator.cpp:15-51 with sigma = 1.5.  gray is realised on the output box
// grown by 3 (reading repeat_edge(input): x, y and c clamped to the input buffer's own box), blur_y on the output rows
// over those columns, then blur_x, sharpen, ratio and the unclamped final multiply per output pixel.  The CUDA kernel
// must match bit for bit, including the +-inf / NaN where gray is 0.
#include <math.h>

#include <vector>

#include "halide_math.h"
#include "oracle_apps.h"

// kernel(x) = exp(-x*x / (2*sigma*sigma)) / (sqrtf(2*kPi) * sigma)   (generator :15,18)
//
// The reference's GPU schedule never schedules `kernel`, so every use kernel(k) (k = 0..3, a constant) is inlined and
// constant-folded by Halide's simplifier instead of being evaluated at run time:
//   * 2*sigma*sigma and sqrtf(2*kPi)*sigma are C++ float expressions of the generator: 4.5f and 3.7599425f;
//   * -k*k / 4.5f: a division of two constants, folded in double and rounded to float (src/Simplify_Div.cpp:80);
//   * exp of a constant: std::exp in double, rounded to float (src/Simplify_Call.cpp:757-780);
//   * the final division by 3.7599425f: folded in double again, rounded to float.
// Result: 0.2659615 (0x3e882c1b), 0.21296532 (0x3e5a1395), 0.10934004 (0x3ddfedac), 0.035993975 (0x3d136e6b).  A run-time
// evaluation (halide_exp, multiply by the folded reciprocal) would give w2 = 0.109340034, one ulp lower.
extern "C" void oracle_unsharp_weights(float *w4) {
    const float sigma = 1.5f, kPi = 3.14159265358979310000f;
    const float two_sigma_sq = 2 * sigma * sigma;
    const float norm = sqrtf(2 * kPi) * sigma;
    for (int k = 0; k < 4; k++) {
        const float num = (float)(-(k * k));
        const float q = (float)((double)num / (double)two_sigma_sq);
        const float e = (float)exp((double)q);
        w4[k] = (float)((double)e / (double)norm);
    }
}

extern "C" int oracle_unsharp(const oracle_image_t *in, const oracle_image_t *out) {
    const int ox = out->min[0], oy = out->min[1], oc = out->min[2];
    const int W = out->extent[0], H = out->extent[1], C = out->extent[2];
    if (W <= 0 || H <= 0 || C <= 0) return 0;
    for (int d = 0; d < 3; d++) {
        if (out->min[d] < in->min[d] || out->min[d] + out->extent[d] > in->min[d] + in->extent[d]) return -4;
    }
    const float *ib = (const float *)in->base;
    auto at = [&](int x, int y, int c) -> float {
        return ib[(int64_t)(x - in->min[0]) * in->stride[0] + (int64_t)(y - in->min[1]) * in->stride[1] +
                  (int64_t)(c - in->min[2]) * in->stride[2]];
    };
    auto bounded = [&](int x, int y, int c) -> float {  // repeat_edge(input)
        return at(hl::clampi(x, in->min[0], in->min[0] + in->extent[0] - 1), hl::clampi(y, in->min[1], in->min[1] + in->extent[1] - 1),
                  hl::clampi(c, in->min[2], in->min[2] + in->extent[2] - 1));
    };
    float w[4];
    oracle_unsharp_weights(w);
    // gray on [ox-3, ox+W+2] x [oy-3, oy+H+2]
    const int gw = W + 6, gh = H + 6;
    std::vector<float> gray((size_t)gw * gh);
#pragma omp parallel for
    for (int v = 0; v < gh; v++) {
        for (int u = 0; u < gw; u++) {
            const int x = ox - 3 + u, y = oy - 3 + v;
            gray[(size_t)v * gw + u] = (0.299f * bounded(x, y, 0) + 0.587f * bounded(x, y, 1)) + 0.114f * bounded(x, y, 2);
        }
    }
    auto g = [&](int x, int y) { return gray[(size_t)(y - oy + 3) * gw + (x - ox + 3)]; };
    // blur_y on [ox-3, ox+W+2] x [oy, oy+H-1]
    std::vector<float> by((size_t)gw * H);
#pragma omp parallel for
    for (int y = oy; y < oy + H; y++) {
        for (int x = ox - 3; x < ox + W + 3; x++) {
            by[(size_t)(y - oy) * gw + (x - ox + 3)] =
                ((w[0] * g(x, y) + w[1] * (g(x, y - 1) + g(x, y + 1))) + w[2] * (g(x, y - 2) + g(x, y + 2))) +
                w[3] * (g(x, y - 3) + g(x, y + 3));
        }
    }
    auto b = [&](int x, int y) { return by[(size_t)(y - oy) * gw + (x - ox + 3)]; };
    float *ob = (float *)out->base;
#pragma omp parallel for
    for (int y = oy; y < oy + H; y++) {
        for (int x = ox; x < ox + W; x++) {
            const float blur_x = ((w[0] * b(x, y) + w[1] * (b(x - 1, y) + b(x + 1, y))) + w[2] * (b(x - 2, y) + b(x + 2, y))) +
                                 w[3] * (b(x - 3, y) + b(x + 3, y));
            const float sharpen = 2.0f * g(x, y) - blur_x;
            const float ratio = sharpen / g(x, y);
            for (int c = oc; c < oc + C; c++) {
                ob[(int64_t)(x - ox) * out->stride[0] + (int64_t)(y - oy) * out->stride[1] + (int64_t)(c - oc) * out->stride[2]] =
                    ratio * at(x, y, c);
            }
        }
    }
    return 0;
}
