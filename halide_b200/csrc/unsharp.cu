// unsharp.cu — unsharp(input, output): unsharp mask of a float32 frame (sigma 1.5), for sm_100a.
//
// Reference algorithm: apps/unsharp/unsharp_generator.cpp:15-51.
//   gray    = (0.299 r + 0.587 g) + 0.114 b on repeat_edge(input): x, y AND c clamped to the input buffer's own box
//   blur_y  = ((w0 g(y) + w1 (g(y-1) + g(y+1))) + w2 (g(y-2) + g(y+2))) + w3 (g(y-3) + g(y+3))
//   blur_x  = the same form over blur_y in x
//   sharpen = 2 gray - blur_x;  ratio = sharpen / gray (IEEE divide);  out(x, y, c) = ratio * input(x, y, c) (unclamped)
// The input must cover the output's (x, y, c) box.  Where gray is 0 the result is +-inf or NaN, as in the reference.
// Every operation is evaluated in source nesting with IEEE rounding (--fmad=false, -prec-div=true), so the result is
// bit-exact against oracle/oracle_unsharp.cpp.
//
// The weights w_k = kernel(k) are compile-time constants in the reference (see unsharp_weights below).
//
// One fused kernel, like the reference's GPU schedule: a block stages its 32x32 tile plus a 3-pixel apron, clamped to
// the input box, once (hb_tile.cuh); gray and blur_y live in shared memory, blur_x and ratio in registers, and the final
// multiply reads the staged centre pixels.  Algorithmic traffic is 24 B/px (12 in, 12 out) against ~60 flops/px.
#include <math.h>

#include "hb_common.h"
#include "hb_tile.cuh"

namespace {

constexpr int TX = 32, TY = 32, NT = 256;  // output tile per block; each thread computes 4 adjacent pixels of a row
constexpr int GW = TX + 6, GH = TY + 6;     // gray: 3-pixel apron
constexpr int SW = ((GW + 3) + 3) / 4 * 4;  // staged columns: up to 3 of alignment slack before the first gray column

// kernel(k) = exp(-k*k / (2 sigma^2)) / (sqrtf(2 pi) sigma), sigma = 1.5 (generator :7,15,18).  The GPU schedule never
// schedules `kernel`, so each kernel(k) is inlined with a constant argument and folded by Halide's simplifier: the
// division of two constants in double (src/Simplify_Div.cpp), exp of a constant as std::exp in double
// (src/Simplify_Call.cpp), each result rounded to float.  2 sigma^2 and sqrtf(2 pi) sigma are the generator's C++ float
// expressions, 4.5f and 3.7599425f.  (Evaluating halide_exp at run time instead would give w2 one ulp lower.)
void unsharp_weights(float w[4]) {
    const float sigma = 1.5f, kPi = 3.14159265358979310000f;
    const float two_sigma_sq = 2 * sigma * sigma;
    const float norm = sqrtf(2 * kPi) * sigma;
    for (int k = 0; k < 4; k++) {
        const float e = (float)(-(double)(k * k) / (double)two_sigma_sq);
        const float x = (float)exp((double)e);
        w[k] = (float)((double)x / (double)norm);
    }
}

struct UnsharpParams {
    hb::F32Planes src;
    float *out;  // element at the output's mins
    int64_t out_sy, out_sc;
    int out_x0, out_y0, out_c0, W, H, C;
    int out_vec;  // out 16-byte aligned and out_sy, out_sc multiples of 4
    float w0, w1, w2, w3;
};

__global__ void __launch_bounds__(NT) unsharp_kernel(UnsharpParams q) {
    __shared__ __align__(16) float raw[3 * GH * SW];
    __shared__ float G[GH][GW];
    __shared__ float BY[TY][GW];
    const int tid = threadIdx.x;
    const int X0 = blockIdx.x * TX, Y0 = blockIdx.y * TY;  // tile origin, output-relative
    const int gx = q.out_x0 + X0 - 3 - q.src.x0;            // buffer-relative x of gray column 0
    const int rx4 = gx & ~3, off = gx - rx4;
    hb::stage_planes<GH, SW, NT>(raw, q.src, rx4, q.out_y0 + Y0 - 3 - q.src.y0);
    __syncthreads();
    for (int t = tid; t < GH * GW; t += NT) {
        const int v = t / GW, u = t - v * GW;
        const float *r = raw + v * SW + off + u;
        G[v][u] = hb::luma(r[0], r[GH * SW], r[2 * GH * SW]);
    }
    __syncthreads();
    const float w0 = q.w0, w1 = q.w1, w2 = q.w2, w3 = q.w3;
    for (int t = tid; t < TY * GW; t += NT) {
        const int v = t / GW, u = t - v * GW;  // centre G[v + 3][u]
        BY[v][u] = ((w0 * G[v + 3][u] + w1 * (G[v + 2][u] + G[v + 4][u])) + w2 * (G[v + 1][u] + G[v + 5][u])) +
                   w3 * (G[v][u] + G[v + 6][u]);
    }
    __syncthreads();
    const int row = tid >> 3, xq = (tid & 7) * 4;
    const int lx = X0 + xq, ly = Y0 + row;
    if (ly >= q.H || lx >= q.W) return;
    float ratio[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const float *b = &BY[row][xq + i + 3];  // centre
        const float bx = ((w0 * b[0] + w1 * (b[-1] + b[1])) + w2 * (b[-2] + b[2])) + w3 * (b[-3] + b[3]);
        const float g = G[row + 3][xq + i + 3];
        const float sharpen = 2.0f * g - bx;
        ratio[i] = sharpen / g;
    }
    const int n = min(4, q.W - lx);
    for (int c = 0; c < q.C; c++) {
        const int ca = q.out_c0 + c;  // absolute channel
        float v[4];
        if (ca >= 0 && ca < 3 && hb::clamp_to(ca, q.src.c0, q.src.c0 + q.src.nc - 1) == ca) {
            // staged plane ca holds input channel ca itself: the centre pixels are already in shared memory
            const float *r = raw + (ca * GH + row + 3) * SW + off + 3 + xq;
#pragma unroll
            for (int i = 0; i < 4; i++) v[i] = r[i];
        } else {
            const float *r = q.src.p + (int64_t)(ca - q.src.c0) * q.src.sc + (int64_t)(q.out_y0 + ly - q.src.y0) * q.src.sy +
                             (q.out_x0 + lx - q.src.x0);
#pragma unroll
            for (int i = 0; i < 4; i++) v[i] = i < n ? __ldg(r + i) : 0.0f;
        }
        float *o = q.out + (int64_t)c * q.out_sc + (int64_t)ly * q.out_sy + lx;
        if (q.out_vec && n == 4) {
            *reinterpret_cast<float4 *>(o) = make_float4(ratio[0] * v[0], ratio[1] * v[1], ratio[2] * v[2], ratio[3] * v[3]);
        } else {
#pragma unroll
            for (int i = 0; i < 4; i++)
                if (i < n) o[i] = ratio[i] * v[i];
        }
    }
}

const hb::ArgSpec kIn = {"input", halide_type_float, 32, 3, false};
const hb::ArgSpec kOut = {"output", halide_type_float, 32, 3, true};
int64_t est_i[3][2] = {{0, 1536}, {0, 2560}, {0, 3}};
const int64_t *const est_ptrs[6] = {&est_i[0][0], &est_i[0][1], &est_i[1][0], &est_i[1][1], &est_i[2][0], &est_i[2][1]};
const halide_filter_argument_t kArgs[2] = {
    {"input", halide_argument_kind_input_buffer, 3, {halide_type_float, 32, 0}, nullptr, nullptr, nullptr, nullptr, est_ptrs},
    {"output", halide_argument_kind_output_buffer, 3, {halide_type_float, 32, 0}, nullptr, nullptr, nullptr, nullptr, est_ptrs},
};
const halide_filter_metadata_t kMeta = {1, 2, kArgs, "x86-64-linux-cuda-cuda_capability_100-b200_native", "unsharp"};
const halide_filter_metadata_t kMetaAuto = {1, 2, kArgs, "x86-64-linux-cuda-cuda_capability_100-b200_native",
                                            "unsharp_auto_schedule"};

int run_unsharp(halide_buffer_t *input, halide_buffer_t *output) {
    int r;
    if ((r = hb::check_arg(input, kIn))) return r;
    if ((r = hb::check_arg(output, kOut))) return r;
    bool query = false;
    {
        // gray reads are clamped, the final multiply is not: the input must hold the output's (x, y, c) box
        int mins[3] = {output->dim[0].min, output->dim[1].min, output->dim[2].min};
        int ext[3] = {output->dim[0].extent, output->dim[1].extent, output->dim[2].extent};
        if (hb::is_bounds_query(input)) { hb::propose_shape(input, mins, ext); query = true; }
        if (hb::is_bounds_query(output)) { hb::propose_shape(output, mins, ext); query = true; }
    }
    if (query) return 0;
    if ((r = hb::check_shape(input, kIn))) return r;
    if ((r = hb::check_shape(output, kOut))) return r;
    const int W = output->dim[0].extent, H = output->dim[1].extent, C = output->dim[2].extent;
    if (W <= 0 || H <= 0 || C <= 0) return 0;
    for (int d = 0; d < 3; d++) {
        if ((r = hb::check_covers(input, kIn, d, output->dim[d].min, output->dim[d].extent))) return r;
    }
    void *din = nullptr, *dout = nullptr;
    if ((r = hb::acquire_input(input, kIn, &din))) return r;
    if ((r = hb::acquire_output(output, kOut, &dout))) return r;

    UnsharpParams q;
    q.src = hb::f32_planes((const float *)din, input);
    q.out = (float *)dout;
    q.out_sy = output->dim[1].stride; q.out_sc = output->dim[2].stride;
    q.out_x0 = output->dim[0].min; q.out_y0 = output->dim[1].min; q.out_c0 = output->dim[2].min;
    q.W = W; q.H = H; q.C = C;
    q.out_vec = ((reinterpret_cast<uintptr_t>(dout) & 15) == 0 && (q.out_sy & 3) == 0 && (q.out_sc & 3) == 0) ? 1 : 0;
    float w[4];
    unsharp_weights(w);
    q.w0 = w[0]; q.w1 = w[1]; q.w2 = w[2]; q.w3 = w[3];
    cudaStream_t s = hb::stream();
    {
        hb::CallTimer timer(s);
        dim3 grid((W + TX - 1) / TX, (H + TY - 1) / TY);
        HB_LAUNCH("unsharp", unsharp_kernel, grid, NT, 0, s, q);
    }
    if ((r = hb::check_cuda(cudaGetLastError(), "unsharp launch", halide_error_code_device_run_failed))) return r;
    hb::mark_output_written(output);
    return 0;
}

}  // namespace

extern "C" int unsharp(halide_buffer_t *input, halide_buffer_t *output) {
    return run_unsharp(input, output);
}
extern "C" int unsharp_argv(void **args) {
    return run_unsharp((halide_buffer_t *)args[0], (halide_buffer_t *)args[1]);
}
extern "C" const halide_filter_metadata_t *unsharp_metadata(void) {
    return &kMeta;
}
extern "C" int unsharp_auto_schedule(halide_buffer_t *input, halide_buffer_t *output) {
    return run_unsharp(input, output);
}
extern "C" int unsharp_auto_schedule_argv(void **args) {
    return unsharp_argv(args);
}
extern "C" const halide_filter_metadata_t *unsharp_auto_schedule_metadata(void) {
    return &kMetaAuto;
}
