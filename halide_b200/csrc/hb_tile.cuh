// hb_tile.cuh — the shared-memory tile loader of the fused float32 stencil kernels (harris.cu, unsharp.cu).
//
// A block stages the three colour planes of its input tile, apron included, once.  Every coordinate is clamped to the
// input buffer's own box (x, y and c), which is exactly repeat_edge for unsharp; harris requires its input to cover
// the whole footprint, so there the clamp only keeps the columns and rows that no stored output depends on (ragged
// edge tiles, 4-column alignment slack) inside the allocation.
//
// Tile columns start at a buffer-relative x that is a multiple of 4.  When the buffer's base address is 16-byte aligned
// and its row and plane strides are multiples of 4 elements, every group of four columns that lies inside the buffer
// is one 16-byte load; groups that straddle an edge, and every group of a buffer that is not aligned that way (odd
// element offsets, odd strides), are loaded element by element.  Negative strides (flipped rows) take either path.
#pragma once

#include <stdint.h>

namespace hb {

struct F32Planes {
    const float *p;     // element at the buffer's mins
    int64_t sy, sc;     // row and plane strides in elements (any sign)
    int x0, y0, c0;     // buffer mins
    int w, h, nc;       // buffer extents (all >= 1)
    int vec;            // p is 16-byte aligned and sy, sc are multiples of 4
};

__host__ inline F32Planes f32_planes(const float *dev, const halide_buffer_t *b) {
    F32Planes s;
    s.p = dev;
    s.sy = b->dim[1].stride;
    s.sc = b->dim[2].stride;
    s.x0 = b->dim[0].min; s.y0 = b->dim[1].min; s.c0 = b->dim[2].min;
    s.w = b->dim[0].extent; s.h = b->dim[1].extent; s.nc = b->dim[2].extent;
    s.vec = ((reinterpret_cast<uintptr_t>(dev) & 15) == 0 && (s.sy & 3) == 0 && (s.sc & 3) == 0) ? 1 : 0;
    return s;
}

__device__ __forceinline__ int clamp_to(int v, int lo, int hi) {
    return v < lo ? lo : (v > hi ? hi : v);
}

// t[(k * ROWS + r) * SW + j] = input(clamp(rx4 + j), clamp(ry + r), clamp(k)) for planes k < 3, rows r < ROWS and
// columns j < SW, with rx4 / ry buffer-relative (rx4 % 4 == 0) and k an absolute channel.  t must be 16-byte aligned.
template<int ROWS, int SW, int NT>
__device__ __forceinline__ void stage_planes(float *t, const F32Planes &s, int rx4, int ry) {
    static_assert(SW % 4 == 0, "tile rows are whole 16-byte groups");
    constexpr int G = SW / 4, N = 3 * ROWS * G, PER = (N + NT - 1) / NT;
    // every load of the thread is issued before the first shared-memory store, so their latencies overlap
    float4 v[PER];
#pragma unroll
    for (int j = 0; j < PER; j++) {
        const int i = threadIdx.x + j * NT;
        if (i >= N) break;
        const int k = i / (ROWS * G), rem = i - k * (ROWS * G);
        const int r = rem / G, g = rem - r * G;
        const int y = clamp_to(ry + r, 0, s.h - 1);
        const int c = clamp_to(k, s.c0, s.c0 + s.nc - 1) - s.c0;
        const float *row = s.p + (int64_t)c * s.sc + (int64_t)y * s.sy;
        const int x = rx4 + 4 * g;
        if (s.vec && x >= 0 && x + 3 < s.w) {
            v[j] = __ldg(reinterpret_cast<const float4 *>(row + x));
        } else {
            v[j].x = __ldg(row + clamp_to(x, 0, s.w - 1));
            v[j].y = __ldg(row + clamp_to(x + 1, 0, s.w - 1));
            v[j].z = __ldg(row + clamp_to(x + 2, 0, s.w - 1));
            v[j].w = __ldg(row + clamp_to(x + 3, 0, s.w - 1));
        }
    }
#pragma unroll
    for (int j = 0; j < PER; j++) {
        const int i = threadIdx.x + j * NT;
        if (i >= N) break;
        const int k = i / (ROWS * G), rem = i - k * (ROWS * G);
        const int r = rem / G, g = rem - r * G;
        *reinterpret_cast<float4 *>(t + (k * ROWS + r) * SW + 4 * g) = v[j];
    }
}

// gray = (0.299f * c0 + 0.587f * c1) + 0.114f * c2 (apps/harris/harris_generator.cpp:23-25,
// apps/unsharp/unsharp_generator.cpp:23-25), evaluated in that order.
__device__ __forceinline__ float luma(float r, float g, float b) {
    return (0.299f * r + 0.587f * g) + 0.114f * b;
}

}  // namespace hb
