// harris.cu — harris(input, output): Harris corner response of a 3-channel float32 frame, for sm_100a.
//
// Reference algorithm: apps/harris/harris_generator.cpp:22-61.
//   gray  = (0.299 r + 0.587 g) + 0.114 b
//   Iy/Ix = six-term gradient sums, coefficients +-1/12 and +-2/12, in the generator's term order (:28-35)
//   S**   = left-associated 3x3 sums of Ix*Ix, Iy*Iy, Ix*Iy: column x-1 (rows y-1, y, y+1), then x, then x+1 (:7-11)
//   out   = (Sxx*Syy - Sxy*Sxy) - (0.04 * (Sxx + Syy)) * (Sxx + Syy)
// No boundary condition: the output box [x0, x0+W) x [y0, y0+H) needs input x in [x0-2, x0+W+1], the same in y, and
// channels 0..2.  Every operation is evaluated in source nesting with IEEE rounding (the library builds with
// --fmad=false), so the result is bit-exact against oracle/oracle_harris.cpp.
//
// One fused kernel, like the reference's GPU schedule: a block stages its 32x32 tile plus a 2-pixel apron once
// (hb_tile.cuh), then gray, the gradient products and the 3x3 sums live in shared memory and registers only.
// Algorithmic traffic is 16 B/px (12 in, 4 out) against ~70 flops/px.
#include "../../include/harris.h"
#include "../../include/harris_auto_schedule.h"
#include "hb_common.h"
#include "hb_tile.cuh"

namespace {

constexpr int TX = 32, TY = 32, NT = 256;  // output tile per block; each thread computes 4 adjacent outputs of a row
constexpr int GW = TX + 4, GH = TY + 4;     // gray: 2-pixel apron
constexpr int PW = TX + 2, PH = TY + 2;     // gradient products: 1-pixel apron
constexpr int SW = ((GW + 3) + 3) / 4 * 4;  // staged columns: up to 3 of alignment slack before the first gray column

struct HarrisParams {
    hb::F32Planes src;
    float *out;  // element at the output's mins
    int64_t out_sy;
    int out_x0, out_y0, W, H;
    int out_vec;  // out 16-byte aligned and out_sy a multiple of 4
};

__global__ void __launch_bounds__(NT) harris_kernel(HarrisParams q) {
    __shared__ __align__(16) float raw[3 * GH * SW];
    __shared__ float G[GH][GW];
    __shared__ float P[3][PH][PW + 1];  // Ixx, Iyy, Ixy
    const int tid = threadIdx.x;
    const int X0 = blockIdx.x * TX, Y0 = blockIdx.y * TY;  // tile origin, output-relative
    const int gx = q.out_x0 + X0 - 2 - q.src.x0;            // buffer-relative x of gray column 0
    const int rx4 = gx & ~3, off = gx - rx4;
    hb::stage_planes<GH, SW, NT>(raw, q.src, rx4, q.out_y0 + Y0 - 2 - q.src.y0);
    __syncthreads();
    for (int t = tid; t < GH * GW; t += NT) {
        const int v = t / GW, u = t - v * GW;
        const float *r = raw + v * SW + off + u;
        G[v][u] = hb::luma(r[0], r[GH * SW], r[2 * GH * SW]);
    }
    __syncthreads();
    constexpr float k1 = 1.0f / 12, k2 = 2.0f / 12;  // the generator's C++ float constants
    for (int t = tid; t < PH * PW; t += NT) {
        const int v = t / PW, u = t - v * PW;
        // g(dx, dy) = gray at offset (dx, dy) from the centre G[v + 1][u + 1]
#define g(dx, dy) G[v + 1 + (dy)][u + 1 + (dx)]
        const float iy = g(-1, -1) * -k1 + g(-1, 1) * k1 + g(0, -1) * -k2 + g(0, 1) * k2 + g(1, -1) * -k1 + g(1, 1) * k1;
        const float ix = g(-1, -1) * -k1 + g(1, -1) * k1 + g(-1, 0) * -k2 + g(1, 0) * k2 + g(-1, 1) * -k1 + g(1, 1) * k1;
#undef g
        P[0][v][u] = ix * ix;
        P[1][v][u] = iy * iy;
        P[2][v][u] = ix * iy;
    }
    __syncthreads();
    const int row = tid >> 3, xq = (tid & 7) * 4;
    float res[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        float s[3];
#pragma unroll
        for (int k = 0; k < 3; k++) {
            // centre P[k][row + 1][xq + i + 1]; column x-1 (y-1, y, y+1), then x, then x+1
            const float *p = &P[k][row][xq + i];
            s[k] = p[0] + p[PW + 1] + p[2 * (PW + 1)] + p[1] + p[PW + 2] + p[2 * (PW + 1) + 1] + p[2] + p[PW + 3] +
                   p[2 * (PW + 1) + 2];
        }
        const float det = s[0] * s[1] - s[2] * s[2];
        const float trace = s[0] + s[1];
        res[i] = det - 0.04f * trace * trace;
    }
    const int lx = X0 + xq, ly = Y0 + row;
    if (ly >= q.H || lx >= q.W) return;
    float *o = q.out + (int64_t)ly * q.out_sy + lx;
    if (q.out_vec && lx + 3 < q.W) {
        *reinterpret_cast<float4 *>(o) = make_float4(res[0], res[1], res[2], res[3]);
    } else {
#pragma unroll
        for (int i = 0; i < 4; i++)
            if (lx + i < q.W) o[i] = res[i];
    }
}

const hb::BufferEstimates est_in({0, 1536, 0, 2560, 0, 3});
const hb::BufferEstimates est_out({3, 1530, 3, 2554});  // output.dim(d).set_estimate(3, k - 6) (generator :70-71)
const halide_filter_argument_t kArgs[2] = {
    {"input", halide_argument_kind_input_buffer, 3, {halide_type_float, 32, 0}, nullptr, nullptr, nullptr, nullptr, est_in.p},
    {"output", halide_argument_kind_output_buffer, 2, {halide_type_float, 32, 0}, nullptr, nullptr, nullptr, nullptr, est_out.p},
};
const auto &kIn = kArgs[0], &kOut = kArgs[1];

}  // namespace

extern "C" int harris(halide_buffer_t *input, halide_buffer_t *output) {
    int r;
    if ((r = hb::check_arg(input, kIn))) return r;
    if ((r = hb::check_arg(output, kOut))) return r;
    bool query = false;
    {
        // no boundary condition: the input must hold the output box grown by 2 in x and y, and channels 0..2
        const int ox = output->dim[0].min, oy = output->dim[1].min, W = output->dim[0].extent, H = output->dim[1].extent;
        int in_mins[3] = {ox - 2, oy - 2, 0}, in_ext[3] = {W + 4, H + 4, 3};
        int out_mins[2] = {ox, oy}, out_ext[2] = {W, H};
        if (hb::is_bounds_query(input)) { hb::propose_shape(input, in_mins, in_ext); query = true; }
        if (hb::is_bounds_query(output)) { hb::propose_shape(output, out_mins, out_ext); query = true; }
    }
    if (query) return 0;
    if ((r = hb::check_shape(input, kIn))) return r;
    if ((r = hb::check_shape(output, kOut))) return r;
    const int W = output->dim[0].extent, H = output->dim[1].extent;
    if (W <= 0 || H <= 0) return 0;
    if ((r = hb::check_covers(input, kIn, 0, output->dim[0].min - 2, W + 4))) return r;
    if ((r = hb::check_covers(input, kIn, 1, output->dim[1].min - 2, H + 4))) return r;
    if ((r = hb::check_covers(input, kIn, 2, 0, 3))) return r;
    void *din = nullptr, *dout = nullptr;
    if ((r = hb::acquire_input(input, kIn, &din))) return r;
    if ((r = hb::acquire_output(output, kOut, &dout))) return r;

    HarrisParams q;
    q.src = hb::f32_planes((const float *)din, input);
    q.out = (float *)dout;
    q.out_sy = output->dim[1].stride;
    q.out_x0 = output->dim[0].min; q.out_y0 = output->dim[1].min; q.W = W; q.H = H;
    q.out_vec = ((reinterpret_cast<uintptr_t>(dout) & 15) == 0 && (q.out_sy & 3) == 0) ? 1 : 0;
    cudaStream_t s = hb::stream();
    {
        hb::CallTimer timer(s);
        dim3 grid((W + TX - 1) / TX, (H + TY - 1) / TY);
        HB_LAUNCH("harris", harris_kernel, grid, NT, 0, s, q);
    }
    if ((r = hb::check_cuda(cudaGetLastError(), "harris launch", halide_error_code_device_run_failed))) return r;
    hb::mark_output_written(output);
    return 0;
}

HB_EXPORT_FILTER(harris, kArgs)
HB_EXPORT_AUTO_SCHEDULE(harris, kArgs)
