// conv_layer.cu — conv_layer(input, filter, bias, relu) for sm_100a.
//
// Reference algorithm: apps/conv_layer/conv_layer_generator.cpp:17-27 with the fixed shapes the generator pins
// by constraints (:35-50): input (CI=128, W+2=102, H+2=82, N=5) channel-innermost, filter (CO=128, 3, 3, CI)
// output-channel-innermost, bias (128), relu (CO=128, W=100, H=80, N=5).
//   relu(co,x,y,n) = max(0, bias(co) + sum_{ky,kx,ci} filter(co,kx,ky,ci) * input(ci, x+kx, y+ky, n))
// Float pipeline: parity bar 1e-4 relative against oracle/oracle_conv_layer.cpp (a tiled contraction necessarily
// changes the summation order; the harness data are all positive so there is no cancellation).
//
// This round ships the FP32 SIMT contraction (register-tiled implicit GEMM, FFMA): M = 40 000 output pixels,
// N = 128, K = 1152, 11.8 GFLOP.  It is the baseline the tcgen05 path has to beat (DESIGN.md §9): TF32 tensor
// cores need a 3-term split to hold 1e-4 on rand()-scale inputs because the conversion truncates.
// Block = 10x8 output pixels x 128 output channels, 256 threads, each thread 5 pixels x 8 channels in registers;
// per (ci-chunk of 32, ky, kx) one 16 KB filter slab is staged in shared memory; the input patch (12x10 pixels
// x 32 channels) is staged once per ci-chunk.  Operand loads are warp-broadcast or 16-byte conflict-free.
#include <stdlib.h>
#include <string.h>

#include "../../include/conv_layer.h"
#include "../../include/conv_layer_auto_schedule.h"
#include "hb_common.h"

// tcgen05 / TMEM / TMA implementation (conv_layer_tc.cu)
int conv_layer_tc_run(const float *din, const float *df, const float *db, float *dout, cudaStream_t s);

namespace {

// Which contraction runs: the tcgen05 implicit GEMM (3xTF32 split) or the FP32 SIMT kernel.  HALIDE_B200_CONV=simt|tc
// picks at start-up; halide_b200_conv_use_tensor_cores() switches at run time (tests cover both).
bool g_use_tc = [] {
    const char *e = getenv("HALIDE_B200_CONV");
    return !(e && strcmp(e, "simt") == 0);  // default: tensor cores
}();

constexpr int N = 5, CI = 128, CO = 128, W = 100, H = 80;  // generator :35-50 (process.cpp:14)
constexpr int TX = 10, TY = 8;                             // output tile
constexpr int PX = TX + 2, PY = TY + 2;                    // input patch
constexpr int KC = 32;                                     // ci per chunk
constexpr int KP = KC + 4;                                 // padded channel pitch of the input patch (bank spread)

__global__ void __launch_bounds__(256) conv_layer_kernel(const float *__restrict__ in, const float *__restrict__ filt,
                                                         const float *__restrict__ bias, float *__restrict__ out) {
    __shared__ __align__(16) float s_in[PY][PX][KP];   // 17 280 B
    __shared__ __align__(16) float s_f[KC][CO];        // 16 384 B
    const int tid = threadIdx.x;
    const int tc = tid & 15, tp = tid >> 4;            // 16 channel groups x 16 pixel groups
    const int x0 = blockIdx.x * TX, y0 = blockIdx.y * TY, n = blockIdx.z;
    const int prow = tp >> 1, pcol = (tp & 1) * 5;     // this thread's 5 pixels: row prow, cols pcol..pcol+4
    // 8 output channels per thread as two quads, co = 4*tc + {0..3} and 64 + 4*tc + {0..3}: the 16 threads of a
    // channel group then read 256 contiguous bytes of the filter slab per quad (conflict-free LDS.128)
    const int co0 = tc * 4, co1 = 64 + tc * 4;
    float acc[5][8];
#pragma unroll
    for (int j = 0; j < 5; j++)
#pragma unroll
        for (int k = 0; k < 8; k++) acc[j][k] = bias[(k < 4 ? co0 : co1 - 4) + k];

    const int64_t in_sx = CI, in_sy = (int64_t)CI * (W + 2), in_sn = in_sy * (H + 2);
    const float *in_n = in + n * in_sn;
    for (int c0 = 0; c0 < CI; c0 += KC) {
        __syncthreads();  // previous chunk's consumers are done with s_in / s_f
        // input patch: PY*PX pixels x KC channels, 8 float4 per pixel
        for (int i = tid; i < PY * PX * (KC / 4); i += 256) {
            int pix = i / (KC / 4), q = i - pix * (KC / 4);
            int py = pix / PX, px = pix - py * PX;
            int gy = min(y0 + py, H + 1), gx = min(x0 + px, W + 1);  // tiles never overhang (100 % 10 == 0, 80 % 8 == 0)
            float4 v = __ldg(reinterpret_cast<const float4 *>(in_n + gy * in_sy + gx * in_sx + c0) + q);
            *reinterpret_cast<float4 *>(&s_in[py][px][4 * q]) = v;
        }
        for (int kk = 0; kk < 9; kk++) {
            const int ky = kk / 3, kx = kk - ky * 3;
            __syncthreads();  // s_f free (and, first time round, s_in visible)
            // filter slab: KC rows of CO floats at filter(0, kx, ky, c0 + r)
            for (int i = tid; i < KC * (CO / 4); i += 256) {
                int r = i / (CO / 4), q = i - r * (CO / 4);
                float4 v = __ldg(reinterpret_cast<const float4 *>(filt + (int64_t)(c0 + r) * (CO * 9) + ky * (CO * 3) + kx * CO) + q);
                *reinterpret_cast<float4 *>(&s_f[r][4 * q]) = v;
            }
            __syncthreads();
            const float *a_base = &s_in[prow + ky][pcol + kx][0];
#pragma unroll 4
            for (int ci = 0; ci < KC; ci++) {
                float a[5];
#pragma unroll
                for (int j = 0; j < 5; j++) a[j] = a_base[j * KP + ci];
                float4 b0 = *reinterpret_cast<const float4 *>(&s_f[ci][co0]);
                float4 b1 = *reinterpret_cast<const float4 *>(&s_f[ci][co1]);
                const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                for (int j = 0; j < 5; j++)
#pragma unroll
                    for (int k = 0; k < 8; k++) acc[j][k] = __fmaf_rn(b[k], a[j], acc[j][k]);
            }
        }
    }
    // relu + store: two quads of output channels per pixel
    const int64_t o_sx = CO, o_sy = (int64_t)CO * W, o_sn = o_sy * H;
#pragma unroll
    for (int j = 0; j < 5; j++) {
        float *o = out + n * o_sn + (int64_t)(y0 + prow) * o_sy + (int64_t)(x0 + pcol + j) * o_sx;
        float4 v0 = make_float4(fmaxf(acc[j][0], 0.f), fmaxf(acc[j][1], 0.f), fmaxf(acc[j][2], 0.f), fmaxf(acc[j][3], 0.f));
        float4 v1 = make_float4(fmaxf(acc[j][4], 0.f), fmaxf(acc[j][5], 0.f), fmaxf(acc[j][6], 0.f), fmaxf(acc[j][7], 0.f));
        *reinterpret_cast<float4 *>(o + co0) = v0;
        *reinterpret_cast<float4 *>(o + co1) = v1;
    }
}

// estimates = the fixed shapes (generator :52-68)
const hb::BufferEstimates est_in({0, CI, 0, W + 2, 0, H + 2, 0, N});
const hb::BufferEstimates est_f({0, CO, 0, 3, 0, 3, 0, CI});
const hb::BufferEstimates est_b({0, CO});
const hb::BufferEstimates est_out({0, CO, 0, W, 0, H, 0, N});
const halide_filter_argument_t kArgs[4] = {
    {"input", halide_argument_kind_input_buffer, 4, {halide_type_float, 32, 0}, nullptr, nullptr, nullptr, nullptr, est_in.p},
    {"filter", halide_argument_kind_input_buffer, 4, {halide_type_float, 32, 0}, nullptr, nullptr, nullptr, nullptr, est_f.p},
    {"bias", halide_argument_kind_input_buffer, 1, {halide_type_float, 32, 0}, nullptr, nullptr, nullptr, nullptr, est_b.p},
    {"relu", halide_argument_kind_output_buffer, 4, {halide_type_float, 32, 0}, nullptr, nullptr, nullptr, nullptr, est_out.p},
};
const auto &kIn = kArgs[0], &kFilt = kArgs[1], &kBias = kArgs[2], &kOut = kArgs[3];

struct Shape {
    int ext[4];
};
// the generator's set_bounds / set_stride constraints (:35-50)
const Shape kInShape = {{CI, W + 2, H + 2, N}}, kFiltShape = {{CO, 3, 3, CI}}, kOutShape = {{CO, W, H, N}};

int check_fixed(const halide_buffer_t *b, const halide_filter_argument_t &spec, const int *ext, int nd) {
    int64_t stride = 1;
    for (int d = 0; d < nd; d++) {
        if (b->dim[d].min != 0 || b->dim[d].extent != ext[d] || b->dim[d].stride != stride) {
            return hb::fail(halide_error_code_constraint_violated,
                            "Constraint violated: %s.dim(%d) is (min %d, extent %d, stride %d) but must be (0, %d, %lld)", spec.name, d,
                            b->dim[d].min, b->dim[d].extent, b->dim[d].stride, ext[d], (long long)stride);
        }
        stride *= ext[d];
    }
    return 0;
}

}  // namespace

extern "C" int conv_layer(halide_buffer_t *input, halide_buffer_t *filter, halide_buffer_t *bias, halide_buffer_t *relu) {
    int r;
    if ((r = hb::check_arg(input, kIn)) || (r = hb::check_arg(filter, kFilt)) || (r = hb::check_arg(bias, kBias)) ||
        (r = hb::check_arg(relu, kOut)))
        return r;
    bool query = false;
    const int zero4[4] = {0, 0, 0, 0};
    const int bias_ext[1] = {CO};
    if (hb::is_bounds_query(input)) { hb::propose_shape(input, zero4, kInShape.ext); query = true; }
    if (hb::is_bounds_query(filter)) { hb::propose_shape(filter, zero4, kFiltShape.ext); query = true; }
    if (hb::is_bounds_query(bias)) { hb::propose_shape(bias, zero4, bias_ext); query = true; }
    if (hb::is_bounds_query(relu)) { hb::propose_shape(relu, zero4, kOutShape.ext); query = true; }
    if (query) return 0;
    if ((r = hb::check_shape(input, kIn)) || (r = hb::check_shape(filter, kFilt)) || (r = hb::check_shape(bias, kBias)) ||
        (r = hb::check_shape(relu, kOut)))
        return r;
    if ((r = check_fixed(relu, kOut, kOutShape.ext, 4)) || (r = check_fixed(input, kIn, kInShape.ext, 4)) ||
        (r = check_fixed(filter, kFilt, kFiltShape.ext, 4)) || (r = check_fixed(bias, kBias, bias_ext, 1)))
        return r;
    void *din = nullptr, *df = nullptr, *db = nullptr, *dout = nullptr;
    if ((r = hb::acquire_input(input, kIn, &din)) || (r = hb::acquire_input(filter, kFilt, &df)) ||
        (r = hb::acquire_input(bias, kBias, &db)) || (r = hb::acquire_output(relu, kOut, &dout)))
        return r;
    cudaStream_t s = hb::stream();
    // Both contractions move every operand and the output in float4s.  A caller's device buffer that is not 16-byte
    // aligned (a wrapped tensor view at an odd element offset) is staged through pooled scratch, which is.
    hb::Scratch staging;
    float *user_out = nullptr;
    const size_t out_bytes = (size_t)N * H * W * CO * sizeof(float);
    {
        const size_t bytes[3] = {(size_t)N * (H + 2) * (W + 2) * CI * sizeof(float), (size_t)CO * 9 * CI * sizeof(float),
                                 (size_t)CO * sizeof(float)};
        void **ptrs[3] = {&din, &df, &db};
        for (int i = 0; i < 3; i++) {
            if (((uintptr_t)*ptrs[i] & 15) == 0) continue;
            void *a = staging.get<uint8_t>(bytes[i]);
            if (!a) return hb::fail(halide_error_code_device_malloc_failed, "conv_layer: staging allocation failed");
            if ((r = hb::check_cuda(cudaMemcpyAsync(a, *ptrs[i], bytes[i], cudaMemcpyDeviceToDevice, s), "conv_layer staging copy",
                                    halide_error_code_device_run_failed)))
                return r;
            *ptrs[i] = a;
        }
        if ((uintptr_t)dout & 15) {
            user_out = (float *)dout;
            if (!(dout = staging.get<uint8_t>(out_bytes)))
                return hb::fail(halide_error_code_device_malloc_failed, "conv_layer: staging allocation failed");
        }
    }
    {
        hb::CallTimer timer(s);
        if (g_use_tc) {
            if ((r = conv_layer_tc_run((const float *)din, (const float *)df, (const float *)db, (float *)dout, s))) return r;
        } else {
            dim3 grid(W / TX, H / TY, N);
            HB_LAUNCH("conv_layer_f32", conv_layer_kernel, grid, 256, 0, s, (const float *)din, (const float *)df, (const float *)db,
                      (float *)dout);
        }
    }
    if (user_out && (r = hb::check_cuda(cudaMemcpyAsync(user_out, dout, out_bytes, cudaMemcpyDeviceToDevice, s), "conv_layer staging copy",
                                        halide_error_code_device_run_failed)))
        return r;
    if ((r = hb::check_cuda(cudaGetLastError(), "conv_layer launch", halide_error_code_device_run_failed))) return r;
    hb::mark_output_written(relu);
    return 0;
}

HB_EXPORT_FILTER(conv_layer, kArgs)
HB_EXPORT_AUTO_SCHEDULE(conv_layer, kArgs)

extern "C" void halide_b200_conv_use_tensor_cores(int enable) {
    g_use_tc = enable != 0;
}
