// bilateral_grid.cu — bilateral_grid(input, r_sigma, output) for sm_100a (s_sigma = 8).
//
// Reference algorithm: apps/bilateral_grid/bilateral_grid_generator.cpp:17-67
//   histogram(x,y,zi,c) += mux(c,{val,1}) over the 8x8 pixels of cell (x,y) (offset -4), zi = int(val/r_sigma + 0.5)
//   blurz/blurx/blury: unnormalised 1-4-6-4-1 along z, x, y
//   output = trilinear slice of blury at (x/8, y/8, val/r_sigma), channel 0 / channel 1
// Float pipeline: parity bar is 1e-4 relative against oracle/oracle_bilateral_grid.cpp, so sums
// may be re-associated (all terms are non-negative: no cancellation).
//
// HBM-bound: 8 algorithmic B/px (4 in + 4 out).  Three kernels:
//   bg_hist_blurz   reads the frame once with coalesced float4 loads; each lane scatters its 4
//                   columns x 8 rows into lane-private shared-memory bins (no atomics, no
//                   conflicts: bin-major layout), the two lanes of a cell then emit blurz.
//   bg_blur_xy      blurx then blury fused: each thread owns one (cell column, z, channel) and walks
//                   down the grid rows with a 5-row register window of blurx values.
//   bg_slice        one block per 120 x 8 pixels (one row of grid cells): the 16 x 2 x nz cells it interpolates between
//                   are staged in shared memory with a plane stride of 32 cells (bank = cell, whatever the plane);
//                   4 pixels per thread (float4 in / float4 out), 8 shared 8-byte corner loads per pixel.
// Grid layout in HBM: [cell_y][cell_x][z][2] f32 — the (z, z+1) x (value, weight) quad a pixel
// needs at one corner is 16 contiguous bytes.
#include "../../include/bilateral_grid.h"
#include "../../include/bilateral_grid_auto_schedule.h"
#include "hb_common.h"
#include "hl_math.cuh"

namespace {

constexpr int S = 8;  // s_sigma GeneratorParam of the shipped app (generator :8)

struct BGParams {
    const float *in;  // element at input mins
    int64_t in_sy;
    int in_x0, in_y0, in_w, in_h;
    float *out;  // element at output mins
    int64_t out_sy;
    int out_x0, out_y0, W, H;
    float inv_r;
    int zmax;      // largest histogram bin
    int nz;        // blurred grid planes: z in [0, zmax+1]
    int gx0, gy0;  // first grid cell stored (absolute cell coordinates)
    int gw, gh;    // stored cells
    float *grid_a, *grid_b;  // [gh][gw][nz][2]
};

// ---- K1: histogram + blurz --------------------------------------------------------------------------
// One warp handles 16 horizontally adjacent cells (128 px): lane l covers columns 4l..4l+3 of the
// strip for all 8 rows of the cell row.  Bins live in shared memory as [bin][channel][thread].
__global__ void __launch_bounds__(128) bg_hist_blurz_kernel(BGParams p) {
    extern __shared__ float s_bins[];  // (zmax+1) * 2 * 128
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nb = p.zmax + 1;
    for (int b = 0; b < nb * 2; b++) s_bins[b * 128 + tid] = 0.f;
    const int cell_row = blockIdx.y;                       // index into stored rows
    const int cell_col0 = (blockIdx.x * 4 + warp) * 16;    // first stored cell column of this warp
    const int gy = p.gy0 + cell_row;
    const int px0 = (p.gx0 + cell_col0) * S - S / 2 + 4 * lane;  // absolute x of this lane's first pixel
    const bool interior_x = (px0 >= p.in_x0) && (px0 + 3 <= p.in_x0 + p.in_w - 1);
#pragma unroll
    for (int ry = 0; ry < S; ry++) {
        int y = hl::clampi(gy * S + ry - S / 2, p.in_y0, p.in_y0 + p.in_h - 1) - p.in_y0;
        const float *row = p.in + (int64_t)y * p.in_sy;
        float v[4];
        if (interior_x && ((reinterpret_cast<uintptr_t>(row + (px0 - p.in_x0)) & 15) == 0)) {
            float4 t = __ldg(reinterpret_cast<const float4 *>(row + (px0 - p.in_x0)));
            v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
        } else {
#pragma unroll
            for (int i = 0; i < 4; i++) {
                int x = hl::clampi(px0 + i, p.in_x0, p.in_x0 + p.in_w - 1) - p.in_x0;
                v[i] = __ldg(row + x);
            }
        }
#pragma unroll
        for (int i = 0; i < 4; i++) {
            float val = hl::clampf(v[i], 0.0f, 1.0f);
            int zi = (int)__fadd_rn(__fmul_rn(val, p.inv_r), 0.5f);
            zi = min(zi, p.zmax);
            s_bins[(zi * 2) * 128 + tid] += val;
            s_bins[(zi * 2 + 1) * 128 + tid] += 1.0f;
        }
    }
    __syncwarp();
    // lanes 2c, 2c+1 hold the two halves of cell c: even lane emits channel 0, odd lane channel 1
    const int cell = cell_col0 + (lane >> 1);
    if (cell >= p.gw) return;
    const int ch = lane & 1;
    const int ta = tid & ~1, tb = ta + 1;
    auto h = [&](int z) -> float {
        if (z < 0 || z > p.zmax) return 0.f;
        return s_bins[(z * 2 + ch) * 128 + ta] + s_bins[(z * 2 + ch) * 128 + tb];
    };
    float *g = p.grid_a + ((size_t)cell_row * p.gw + cell) * p.nz * 2 + ch;
    float hm2 = 0.f, hm1 = 0.f, h0 = h(0), h1 = h(1), h2 = h(2);
    for (int z = 0; z < p.nz; z++) {
        // blurz = h(z-2) + 4 h(z-1) + 6 h(z) + 4 h(z+1) + h(z+2) (generator :33-37)
        g[z * 2] = (((hm2 + hm1 * 4.0f) + h0 * 6.0f) + h1 * 4.0f) + h2;
        hm2 = hm1; hm1 = h0; h0 = h1; h1 = h2; h2 = h(z + 3);
    }
}

// ---- K2: blurx + blury on the grid -------------------------------------------------------------------
// blury is only needed on the interior (stored region shrunk by 2 cells on every side); the result is
// written over the same extent with the border cells left untouched (never read by the slice).
__global__ void __launch_bounds__(256) bg_blur_xy_kernel(BGParams p, int rows_per_block) {
    const int V = p.nz * 2;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;  // (cell_x - 2) * V + v
    const int cx = t / V + 2;
    if (cx >= p.gw - 2) return;
    const int v = t - (cx - 2) * V;
    const int y_begin = 2 + blockIdx.y * rows_per_block;
    const int y_end = min(y_begin + rows_per_block, p.gh - 2);
    if (y_begin >= y_end) return;
    // x-blur of one grid row at this thread's (cell, value): five loads, combined in the generator's order.  The loads of
    // two rows are issued together (ten in flight per thread): with one row per iteration the kernel sat on its own load
    // latency (long-scoreboard 60 % of the stall samples, DRAM 19 %: profiles/r02_blur_bilateral_ncu_b.md).
    struct Taps {
        float t[5];
    };
    auto load_taps = [&](int cy) -> Taps {
        const float *r = p.grid_a + ((size_t)cy * p.gw + cx) * V + v;
        Taps k;
        k.t[0] = __ldg(r - 2 * V); k.t[1] = __ldg(r - V); k.t[2] = __ldg(r); k.t[3] = __ldg(r + V); k.t[4] = __ldg(r + 2 * V);
        return k;
    };
    auto blurx = [](const Taps &k) -> float {
        return (((k.t[0] + k.t[1] * 4.0f) + k.t[2] * 6.0f) + k.t[3] * 4.0f) + k.t[4];
    };
    float a, b, c, d;
    {
        const Taps k0 = load_taps(y_begin - 2), k1 = load_taps(y_begin - 1), k2 = load_taps(y_begin), k3 = load_taps(y_begin + 1);
        a = blurx(k0); b = blurx(k1); c = blurx(k2); d = blurx(k3);
    }
    for (int cy = y_begin; cy < y_end; cy += 2) {
        const bool two = cy + 1 < y_end;
        const Taps k0 = load_taps(cy + 2);
        const Taps k1 = load_taps(two ? cy + 3 : cy + 2);  // (rows up to y_end + 1 <= gh - 1 exist: the grid keeps a 2-cell border)
        float e = blurx(k0);
        p.grid_b[((size_t)cy * p.gw + cx) * V + v] = (((a + b * 4.0f) + c * 6.0f) + d * 4.0f) + e;
        a = b; b = c; c = d; d = e;
        if (two) {
            e = blurx(k1);
            p.grid_b[((size_t)(cy + 1) * p.gw + cx) * V + v] = (((a + b * 4.0f) + c * 6.0f) + d * 4.0f) + e;
            a = b; b = c; c = d; d = e;
        }
    }
}

// ---- K3: trilinear slice + normalise -----------------------------------------------------------------
// One block = 128 x 8 pixels = one row of grid cells: the 17 x 2 cells (x nz planes x 2 channels) its pixels interpolate
// between are staged once into shared memory as [z][cell row][24] float2, so that a corner fetch is one 8-byte shared
// load.  Lane l of a warp owns the 4 pixels of cell (l & 15) at offset 4 * (l >> 4): the 16 lanes of a half-warp — the
// unit an 8-byte shared load is served in — then read 16 DIFFERENT cells, and with a plane stride of 48 entries
// (= 0 mod 16 bank pairs) the bank of a fetch depends on the cell only, never on the data-dependent plane zi: no
// conflicts whatever the image.  (First version: corners gathered straight from L1, 92 % of the L1 data pipe.  Second:
// shared memory, but lanes 2c and 2c+1 shared cell c, so on a noisy image — different zi — every fetch was a two-way
// conflict: 58 % of the wavefronts, L1 data pipe 96 % busy, profiles/r02_other_pipelines_ncu.md.)
constexpr int kSliceW = 128, kSliceCells = 17, kSlicePitch = 24;

__global__ void __launch_bounds__(256) bg_slice_kernel(BGParams p) {
    extern __shared__ float2 s_grid[];  // [nz][2][kSlicePitch]
    const int lane = threadIdx.x, row = threadIdx.y, tid = row * 32 + lane;
    const int X0 = (p.out_x0 & ~(S - 1)) + blockIdx.x * kSliceW, Y0 = (p.out_y0 & ~(S - 1)) + blockIdx.y * S;
    const int cx0 = (X0 >> 3) - p.gx0, cy0 = (Y0 >> 3) - p.gy0;  // first stored cell of the tile
    {
        const float2 *g = reinterpret_cast<const float2 *>(p.grid_b);
        for (int it = tid; it < 2 * kSliceCells * p.nz; it += 256) {
            // (cell fastest: consecutive lanes store to consecutive banks; the planes of a cell are contiguous in HBM, so
            // the later planes of a cell hit the line the first one brought into L1)
            const int z = it / (2 * kSliceCells), cell = it - z * (2 * kSliceCells);
            const int cr = cell >= kSliceCells ? 1 : 0, cc = cell - cr * kSliceCells;
            const int cx = min(cx0 + cc, p.gw - 1), cy = min(cy0 + cr, p.gh - 1);
            s_grid[(z * 2 + cr) * kSlicePitch + cc] = __ldg(g + ((size_t)cy * p.gw + cx) * p.nz + z);
        }
    }
    __syncthreads();
    const int y = Y0 + row, x = X0 + 8 * (lane & 15) + 4 * (lane >> 4);
    if (y < p.out_y0 || y >= p.out_y0 + p.H || x + 3 < p.out_x0 || x >= p.out_x0 + p.W) return;
    const float *ip = p.in + (int64_t)(y - p.in_y0) * p.in_sy + (x - p.in_x0);
    float *op = p.out + (int64_t)(y - p.out_y0) * p.out_sy + (x - p.out_x0);
    const float2 *c00 = s_grid + (lane & 15);  // cell (xi, yi) of this thread's four pixels; xi + 1: +1, yi + 1: +kSlicePitch
    const float yf = __fmul_rn((float)(y & (S - 1)), 0.125f);
    auto px = [&](float raw, int xx) -> float {
        const float val = hl::clampf(raw, 0.0f, 1.0f);
        const float zv = __fmul_rn(val, p.inv_r);
        int zi = (int)zv;
        const float zf = __fsub_rn(zv, (float)zi);
        zi = min(zi, p.nz - 2);
        const float xf = __fmul_rn((float)(xx & (S - 1)), 0.125f);
        const float2 *c = c00 + zi * (2 * kSlicePitch);
        const float2 a0 = c[0], b0 = c[1], d0 = c[kSlicePitch], e0 = c[kSlicePitch + 1];
        const float2 a1 = c[2 * kSlicePitch], b1 = c[2 * kSlicePitch + 1], d1 = c[3 * kSlicePitch], e1 = c[3 * kSlicePitch + 1];
        // lerp nest x -> y -> z exactly as generator :59-64
        const float v0 = hl::lerpf(hl::lerpf(hl::lerpf(a0.x, b0.x, xf), hl::lerpf(d0.x, e0.x, xf), yf),
                                   hl::lerpf(hl::lerpf(a1.x, b1.x, xf), hl::lerpf(d1.x, e1.x, xf), yf), zf);
        const float v1 = hl::lerpf(hl::lerpf(hl::lerpf(a0.y, b0.y, xf), hl::lerpf(d0.y, e0.y, xf), yf),
                                   hl::lerpf(hl::lerpf(a1.y, b1.y, xf), hl::lerpf(d1.y, e1.y, xf), yf), zf);
        return __fdiv_rn(v0, v1);
    };
    const bool full = x >= p.out_x0 && x + 3 < p.out_x0 + p.W;
    if (full && ((reinterpret_cast<uintptr_t>(ip) | reinterpret_cast<uintptr_t>(op)) & 15) == 0) {
        const float4 v = __ldg(reinterpret_cast<const float4 *>(ip));
        float4 o;
        o.x = px(v.x, x);
        o.y = px(v.y, x + 1);
        o.z = px(v.z, x + 2);
        o.w = px(v.w, x + 3);
        *reinterpret_cast<float4 *>(op) = o;
    } else {
        for (int i = 0; i < 4; i++) {
            if (x + i >= p.out_x0 && x + i < p.out_x0 + p.W) op[i] = px(__ldg(ip + i), x + i);
        }
    }
}

const hb::BufferEstimates est({0, 1536, 0, 2560});
const halide_scalar_value_t sv_rsigma = hb::scalar(0.1f);
const halide_filter_argument_t kArgs[3] = {
    {"input", halide_argument_kind_input_buffer, 2, {halide_type_float, 32, 0}, nullptr, nullptr, nullptr, nullptr, est.p},
    {"r_sigma", halide_argument_kind_input_scalar, 0, {halide_type_float, 32, 0}, nullptr, nullptr, nullptr, &sv_rsigma, nullptr},
    {"bilateral_grid", halide_argument_kind_output_buffer, 2, {halide_type_float, 32, 0}, nullptr, nullptr, nullptr, nullptr, est.p},
};
const auto &kIn = kArgs[0], &kOut = kArgs[2];

inline int fdiv(int a, int b) {  // floor division, b > 0
    int q = a / b;
    return (a % b != 0 && a < 0) ? q - 1 : q;
}

}  // namespace

extern "C" int bilateral_grid(halide_buffer_t *input, float r_sigma, halide_buffer_t *output) {
    int r;
    if ((r = hb::check_arg(input, kIn))) return r;
    if ((r = hb::check_arg(output, kOut))) return r;
    bool query = false;
    {
        // the slice reads input(x,y) unclamped (generator :50): the input must cover the output region
        int mins[2] = {output->dim[0].min, output->dim[1].min};
        int ext[2] = {output->dim[0].extent, output->dim[1].extent};
        if (hb::is_bounds_query(input)) { hb::propose_shape(input, mins, ext); query = true; }
        if (hb::is_bounds_query(output)) { hb::propose_shape(output, mins, ext); query = true; }
    }
    if (query) return 0;
    if ((r = hb::check_shape(input, kIn))) return r;
    if ((r = hb::check_shape(output, kOut))) return r;
    for (int d = 0; d < 2; d++) {
        if ((r = hb::check_covers(input, kIn, d, output->dim[d].min, output->dim[d].extent))) return r;
    }
    const int W = output->dim[0].extent, H = output->dim[1].extent;
    if (W <= 0 || H <= 0) return 0;
    if (!(r_sigma > 0.0f)) {
        return hb::fail(halide_error_code_param_too_small, "Parameter r_sigma is %g but must be positive", (double)r_sigma);
    }
    BGParams p;
    p.inv_r = 1.0f / r_sigma;
    p.zmax = (int)(1.0f * p.inv_r + 0.5f);
    p.nz = p.zmax + 2;
    const size_t bins_bytes = (size_t)(p.zmax + 1) * 2 * 128 * sizeof(float);
    if (bins_bytes > 200 * 1024) {
        return hb::fail(halide_error_code_param_too_small,
                        "Parameter r_sigma is %g: more than %d intensity bins are not supported by this build",
                        (double)r_sigma, (int)(200 * 1024 / (2 * 128 * sizeof(float))));
    }
    void *din = nullptr, *dout = nullptr;
    if ((r = hb::acquire_input(input, kIn, &din))) return r;
    if ((r = hb::acquire_output(output, kOut, &dout))) return r;

    const int ox = output->dim[0].min, oy = output->dim[1].min;
    p.in = (const float *)din;
    p.in_sy = input->dim[1].stride;
    p.in_x0 = input->dim[0].min; p.in_y0 = input->dim[1].min;
    p.in_w = input->dim[0].extent; p.in_h = input->dim[1].extent;
    p.out = (float *)dout;
    p.out_sy = output->dim[1].stride;
    p.out_x0 = ox; p.out_y0 = oy; p.W = W; p.H = H;
    // cells the slice touches are xi..xi+1; blury/blurx add 2 cells on every side
    p.gx0 = fdiv(ox, S) - 2;
    p.gy0 = fdiv(oy, S) - 2;
    p.gw = fdiv(ox + W - 1, S) + 1 + 2 - p.gx0 + 1;
    p.gh = fdiv(oy + H - 1, S) + 1 + 2 - p.gy0 + 1;
    hb::Scratch scratch;
    const size_t gelems = (size_t)p.gw * p.gh * p.nz * 2;
    p.grid_a = scratch.get<float>(gelems);
    p.grid_b = scratch.get<float>(gelems);
    if (!p.grid_a || !p.grid_b) return hb::fail(halide_error_code_device_malloc_failed, "bilateral_grid: scratch allocation failed");

    cudaStream_t s = hb::stream();
    {
        hb::CallTimer timer(s);
        static hb::PerDeviceOnce hist_attr;
        if (bins_bytes > 48 * 1024) {
            hist_attr.run([] { cudaFuncSetAttribute(bg_hist_blurz_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); });
        }
        dim3 g1((p.gw + 63) / 64, p.gh);
        HB_LAUNCH("bg_hist_blurz", bg_hist_blurz_kernel, g1, 128, bins_bytes, s, p);
        const int V = p.nz * 2;
        const int cols = (p.gw - 4) * V;
        int rows = 16;
        while (rows > 2 && (int64_t)((cols + 255) / 256) * ((p.gh - 4 + rows - 1) / rows) < 148 * 4) rows >>= 1;
        dim3 g2((cols + 255) / 256, (p.gh - 4 + rows - 1) / rows);
        HB_LAUNCH("bg_blur_xy", bg_blur_xy_kernel, g2, 256, 0, s, p, rows);
        const int tx0 = ox & ~(S - 1), ty0 = oy & ~(S - 1);
        dim3 g3((ox + W - tx0 + kSliceW - 1) / kSliceW, (oy + H - ty0 + S - 1) / S);
        const size_t slice_smem = (size_t)p.nz * 2 * kSlicePitch * sizeof(float2);
        if (slice_smem > 48 * 1024) cudaFuncSetAttribute(bg_slice_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)slice_smem);
        HB_LAUNCH("bg_slice", bg_slice_kernel, g3, dim3(32, 8), slice_smem, s, p);
    }
    if ((r = hb::check_cuda(cudaGetLastError(), "bilateral_grid launch", halide_error_code_device_run_failed))) return r;
    hb::mark_output_written(output);
    return 0;
}

HB_EXPORT_FILTER(bilateral_grid, kArgs)
HB_EXPORT_AUTO_SCHEDULE(bilateral_grid, kArgs)
