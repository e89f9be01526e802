// nl_means.cu — nl_means(input, patch_size, search_area, sigma, output) for sm_100a.
//
// Reference algorithm: apps/nl_means/nl_means_generator.cpp:24-63
//   d(x,y,dx,dy)  = sum_c (I(x,y,c) - I(x+dx,y+dy,c))^2            (clamped coordinates, c = 0..2)
//   blur_d        = box sum of d over the patch (y then x)
//   w             = fast_exp(blur_d * (-1 / (sigma^2 * patch^2)))
//   out_c         = clamp( sum_{dy,dx} w * I_c(x+dx,y+dy) / sum_{dy,dx} w , 0, 1 )
// Float pipeline: parity bar 1e-4 relative against oracle/oracle_nl_means.cpp (the box sums are
// taken in the reference's order anyway: y then x, ascending).
//
// Compute-bound (~1.5 kflop/px at patch 3 / search 7 against 24 algorithmic B/px): the frame is
// read once into a shared-memory tile with its (search/2 + patch/2) apron, then for each search row
// dy three phases run per block with the whole dx row batched between barriers:
//   A  d for all dx over the tile grown by the patch apron          -> smem D[dx][y][x]
//   B  vertical patch sums                                          -> smem V[dx][y][x]
//   C  horizontal patch sums, fast_exp, accumulate 4 running sums in registers (2 px per thread)
#include "../../include/nl_means.h"
#include "../../include/nl_means_auto_schedule.h"
#include "hb_common.h"
#include "hl_math.cuh"

namespace {

constexpr int TX = 32, TY = 16;  // output tile per block; 256 threads, 2 rows per thread

struct NLParams {
    const float *in;  // element at input mins
    int64_t in_sy, in_sc;
    int in_x0, in_y0, in_c0, in_w, in_h, in_c;
    float *out;
    int64_t out_sy, out_sc;
    int out_x0, out_y0, W, H;
    int p, s, p_lo, s_lo;  // patch/search extents and their first offsets (-(n/2))
    float inv_sigma_sq;
    int nd;                // dx offsets batched per pass
    int iw, ih;            // input tile extent (TX + p + s - 2, TY + p + s - 2)
    int dw, dh;            // D tile extent (TX + p - 1, TY + p - 1)
};

__global__ void __launch_bounds__(256) nl_means_kernel(NLParams q) {
    extern __shared__ float smem[];
    float *sI = smem;                              // [3][ih][iw]
    float *sD = sI + 3 * q.ih * q.iw;              // [nd][dh][dw]
    float *sV = sD + q.nd * q.dh * q.dw;           // [nd][TY][dw]
    const int tid = threadIdx.x;
    const int X0 = q.out_x0 + blockIdx.x * TX, Y0 = q.out_y0 + blockIdx.y * TY;
    // tile coordinate (u,v) <-> absolute (X0 + p_lo + s_lo + u, Y0 + p_lo + s_lo + v)
    const int ax0 = X0 + q.p_lo + q.s_lo, ay0 = Y0 + q.p_lo + q.s_lo;
    for (int t = tid; t < 3 * q.ih * q.iw; t += 256) {
        int c = t / (q.ih * q.iw), rem = t - c * q.ih * q.iw;
        int v = rem / q.iw, u = rem - v * q.iw;
        int x = hl::clampi(ax0 + u, q.in_x0, q.in_x0 + q.in_w - 1) - q.in_x0;
        int y = hl::clampi(ay0 + v, q.in_y0, q.in_y0 + q.in_h - 1) - q.in_y0;
        int cc = hl::clampi(c, q.in_c0, q.in_c0 + q.in_c - 1) - q.in_c0;
        sI[t] = __ldg(q.in + (int64_t)cc * q.in_sc + (int64_t)y * q.in_sy + x);
    }
    __syncthreads();
    const int plane = q.ih * q.iw;
    const int tx = tid & 31, ty = tid >> 5;  // rows ty and ty + 8
    float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
    const int off_s = -q.s_lo;               // tile offset of search offset 0
    for (int dyi = 0; dyi < q.s; dyi++) {
        for (int dx0 = 0; dx0 < q.s; dx0 += q.nd) {
            const int nd = min(q.nd, q.s - dx0);
            // ---- phase A: D[j][v][u] = d(X0 + p_lo + u, Y0 + p_lo + v, dx, dy), dx = s_lo + dx0 + j
            for (int t = tid; t < q.dh * q.dw; t += 256) {
                int v = t / q.dw, u = t - v * q.dw;
                const float *a = sI + (v + off_s) * q.iw + (u + off_s);
                const float *b = sI + (v + dyi) * q.iw + (u + dx0);
                const float a0 = a[0], a1 = a[plane], a2 = a[2 * plane];
                for (int j = 0; j < nd; j++) {
                    float e0 = a0 - b[j], e1 = a1 - b[plane + j], e2 = a2 - b[2 * plane + j];
                    sD[j * q.dh * q.dw + t] = ((0.0f + e0 * e0) + e1 * e1) + e2 * e2;
                }
            }
            __syncthreads();
            // ---- phase B: V[j][y][u] = sum_{t<p} D[j][y + t][u]
            for (int t = tid; t < TY * q.dw; t += 256) {
                int y = t / q.dw, u = t - y * q.dw;
                for (int j = 0; j < nd; j++) {
                    const float *d = sD + (j * q.dh + y) * q.dw + u;
                    float sum = 0.f;
                    for (int k = 0; k < q.p; k++) sum += d[k * q.dw];
                    sV[j * TY * q.dw + t] = sum;
                }
            }
            __syncthreads();
            // ---- phase C: horizontal sums, weights, accumulation
            for (int j = 0; j < nd; j++) {
#pragma unroll
                for (int r = 0; r < 2; r++) {
                    int y = ty + 8 * r;
                    const float *vrow = sV + (j * TY + y) * q.dw + tx;
                    float bd = 0.f;
                    for (int k = 0; k < q.p; k++) bd += vrow[k];
                    float w = hl::fast_exp(bd * q.inv_sigma_sq);
                    const float *nb = sI + (y - q.p_lo + dyi) * q.iw + (tx - q.p_lo + dx0 + j);
                    acc[r][0] += w * nb[0];
                    acc[r][1] += w * nb[plane];
                    acc[r][2] += w * nb[2 * plane];
                    acc[r][3] += w;
                }
            }
            // phase A of the next pass overwrites sD only (phase C reads sV and sI): one barrier is
            // enough between C and the next B, and the A->B barrier above provides it.
        }
    }
#pragma unroll
    for (int r = 0; r < 2; r++) {
        int lx = blockIdx.x * TX + tx, ly = blockIdx.y * TY + ty + 8 * r;
        if (lx < q.W && ly < q.H) {
#pragma unroll
            for (int c = 0; c < 3; c++) {
                float v = hl::clampf(__fdiv_rn(acc[r][c], acc[r][3]), 0.0f, 1.0f);
                q.out[(int64_t)c * q.out_sc + (int64_t)ly * q.out_sy + lx] = v;
            }
        }
    }
}

// ---- register-window version for compile-time patch / search sizes ------------------------------------------------
// The kernel above is generic in patch and search size: every tile coordinate costs an integer division by a run-time
// extent, d goes through shared memory twice (D, then V) and the loops cannot unroll — ~165 instructions per pixel and
// search offset.  With P and S fixed at compile time:
//   phase 1: a thread owns one column u of one search offset dx and walks down the tile's TY + P - 1 rows; d of the new
//            row comes from six shared loads (three channels of the centre and of the shifted tile), the vertical patch
//            sum is the explicit ascending sum over a register window ((0 + d0) + d1) + ... — the reference's order —
//            and only V is written to shared memory;
//   phase 2: as before (horizontal patch sum, fast_exp, four running sums per pixel, two rows per thread), unrolled.
// All S offsets of a search row are batched between two barriers.  Same float operations in the same order as the
// generic kernel (results are bit-identical to it; tests/test_nl_means_gpu.py runs both against the oracle).
template<int P, int S>
__global__ void __launch_bounds__(256) nl_means_window_kernel(NLParams q) {
    constexpr int IW = TX + P + S - 2, IH = TY + P + S - 2, DW = TX + P - 1, DH = TY + P - 1, PLANE = IH * IW;
    constexpr int PLO = -(P / 2), SLO = -(S / 2), OFFS = -SLO;
    extern __shared__ float smem[];
    float *sI = smem;             // [3][IH][IW]
    float *sV = sI + 3 * PLANE;   // [S][TY][DW]
    const int tid = threadIdx.x;
    const int X0 = q.out_x0 + blockIdx.x * TX, Y0 = q.out_y0 + blockIdx.y * TY;
    const int ax0 = X0 + PLO + SLO, ay0 = Y0 + PLO + SLO;  // tile (u, v) <-> absolute (ax0 + u, ay0 + v)
    for (int t = tid; t < 3 * PLANE; t += 256) {
        const int c = t / PLANE, rem = t - c * PLANE;
        const int v = rem / IW, u = rem - v * IW;
        const int x = hl::clampi(ax0 + u, q.in_x0, q.in_x0 + q.in_w - 1) - q.in_x0;
        const int y = hl::clampi(ay0 + v, q.in_y0, q.in_y0 + q.in_h - 1) - q.in_y0;
        const int cc = hl::clampi(c, q.in_c0, q.in_c0 + q.in_c - 1) - q.in_c0;
        sI[t] = __ldg(q.in + (int64_t)cc * q.in_sc + (int64_t)y * q.in_sy + x);
    }
    __syncthreads();
    const int tx = tid & 31, ty = tid >> 5;  // rows ty and ty + 8
    float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
    for (int dyi = 0; dyi < S; dyi++) {
        // ---- phase 1: V[j][y][u] = sum_{k<P} d(u, y + k) for search offset (SLO + j, SLO + dyi)
        for (int it = tid; it < DW * S; it += 256) {
            const int j = it / DW, u = it - j * DW;
            const float *a = sI + OFFS * IW + (u + OFFS);   // centre pixel of d: tile row v + OFFS
            const float *b = sI + dyi * IW + (u + j);       // shifted pixel:     tile row v + dyi
            float *vout = sV + j * TY * DW + u;
            float win[P];
#pragma unroll
            for (int v = 0; v < DH; v++) {
                const float e0 = a[v * IW] - b[v * IW], e1 = a[PLANE + v * IW] - b[PLANE + v * IW],
                            e2 = a[2 * PLANE + v * IW] - b[2 * PLANE + v * IW];
                win[v % P] = ((0.0f + e0 * e0) + e1 * e1) + e2 * e2;
                if (v >= P - 1) {
                    float sum = 0.f;
#pragma unroll
                    for (int k = 0; k < P; k++) sum += win[(v - (P - 1) + k) % P];  // rows y .. y + P - 1, ascending
                    vout[(v - (P - 1)) * DW] = sum;
                }
            }
        }
        __syncthreads();
        // ---- phase 2: horizontal sums, weights, accumulation
#pragma unroll
        for (int j = 0; j < S; j++) {
#pragma unroll
            for (int r = 0; r < 2; r++) {
                const int y = ty + 8 * r;
                const float *vrow = sV + (j * TY + y) * DW + tx;
                float bd = 0.f;
#pragma unroll
                for (int k = 0; k < P; k++) bd += vrow[k];
                const float w = hl::fast_exp(bd * q.inv_sigma_sq);
                const float *nb = sI + (y - PLO + dyi) * IW + (tx - PLO + j);
                acc[r][0] += w * nb[0];
                acc[r][1] += w * nb[PLANE];
                acc[r][2] += w * nb[2 * PLANE];
                acc[r][3] += w;
            }
        }
        __syncthreads();  // (the next search row's phase 1 overwrites sV)
    }
#pragma unroll
    for (int r = 0; r < 2; r++) {
        const int lx = blockIdx.x * TX + tx, ly = blockIdx.y * TY + ty + 8 * r;
        if (lx < q.W && ly < q.H) {
#pragma unroll
            for (int c = 0; c < 3; c++) {
                const float v = hl::clampf(__fdiv_rn(acc[r][c], acc[r][3]), 0.0f, 1.0f);
                q.out[(int64_t)c * q.out_sc + (int64_t)ly * q.out_sy + lx] = v;
            }
        }
    }
}
template<int P, int S>
constexpr size_t nl_window_smem() {
    return (size_t)(3 * (TY + P + S - 2) * (TX + P + S - 2) + S * TY * (TX + P - 1)) * sizeof(float);
}

constexpr bool kDefaultWindow = true;  // (the register-window kernel: bit-identical to the first kernel on hardware, profiles/r02_ab_variants.log)
int g_variant = 0;  // test / A-B hook (halide_b200_nl_means_variant): 0 = default, 1 = generic kernel, 2 = register-window kernel

const hb::BufferEstimates est({0, 1536, 0, 2560, 0, 3});
const halide_scalar_value_t sv_patch = hb::scalar(7), sv_search = hb::scalar(7), sv_sigma = hb::scalar(0.12f);
const halide_filter_argument_t kArgs[5] = {
    {"input", halide_argument_kind_input_buffer, 3, {halide_type_float, 32, 0}, nullptr, nullptr, nullptr, nullptr, est.p},
    {"patch_size", halide_argument_kind_input_scalar, 0, {halide_type_int, 32, 0}, nullptr, nullptr, nullptr, &sv_patch, nullptr},
    {"search_area", halide_argument_kind_input_scalar, 0, {halide_type_int, 32, 0}, nullptr, nullptr, nullptr, &sv_search, nullptr},
    {"sigma", halide_argument_kind_input_scalar, 0, {halide_type_float, 32, 0}, nullptr, nullptr, nullptr, &sv_sigma, nullptr},
    {"non_local_means", halide_argument_kind_output_buffer, 3, {halide_type_float, 32, 0}, nullptr, nullptr, nullptr, nullptr, est.p},
};
const auto &kIn = kArgs[0], &kOut = kArgs[4];

}  // namespace

extern "C" void halide_b200_nl_means_variant(int v) {
    g_variant = v;
}

extern "C" int nl_means(halide_buffer_t *input, int32_t patch_size, int32_t search_area, float sigma, halide_buffer_t *output) {
    int r;
    if ((r = hb::check_arg(input, kIn))) return r;
    if ((r = hb::check_arg(output, kOut))) return r;
    bool query = false;
    {
        // every input access is clamped: a query is answered with the output's x/y region and 3 channels
        int mins[3] = {output->dim[0].min, output->dim[1].min, 0};
        int ext[3] = {output->dim[0].extent, output->dim[1].extent, 3};
        if (hb::is_bounds_query(input)) { hb::propose_shape(input, mins, ext); query = true; }
        if (hb::is_bounds_query(output)) { hb::propose_shape(output, mins, ext); query = true; }
    }
    if (query) return 0;
    if ((r = hb::check_shape(input, kIn))) return r;
    if ((r = hb::check_shape(output, kOut))) return r;
    // explicit constraint: non_local_means.dim(2).set_bounds(0, 3) (generator :68)
    if (output->dim[2].min != 0 || output->dim[2].extent != 3) {
        return hb::fail(halide_error_code_constraint_violated,
                        "Constraint violated: non_local_means.min.2 (%d) == 0 and non_local_means.extent.2 (%d) == 3",
                        output->dim[2].min, output->dim[2].extent);
    }
    const int W = output->dim[0].extent, H = output->dim[1].extent;
    if (W <= 0 || H <= 0) return 0;
    if (input->dim[0].extent <= 0 || input->dim[1].extent <= 0 || input->dim[2].extent <= 0) {
        return hb::fail(halide_error_code_access_out_of_bounds, "Input buffer input is empty");
    }
    if (patch_size < 1 || search_area < 1 || patch_size > 31 || search_area > 63) {
        return hb::fail(patch_size < 1 || search_area < 1 ? halide_error_code_param_too_small : halide_error_code_param_too_large,
                        "nl_means: patch_size %d / search_area %d outside the supported range [1,31] / [1,63]", patch_size,
                        search_area);
    }
    void *din = nullptr, *dout = nullptr;
    if ((r = hb::acquire_input(input, kIn, &din))) return r;
    if ((r = hb::acquire_output(output, kOut, &dout))) return r;

    NLParams q;
    q.in = (const float *)din;
    q.in_sy = input->dim[1].stride; q.in_sc = input->dim[2].stride;
    q.in_x0 = input->dim[0].min; q.in_y0 = input->dim[1].min; q.in_c0 = input->dim[2].min;
    q.in_w = input->dim[0].extent; q.in_h = input->dim[1].extent; q.in_c = input->dim[2].extent;
    q.out = (float *)dout;
    q.out_sy = output->dim[1].stride; q.out_sc = output->dim[2].stride;
    q.out_x0 = output->dim[0].min; q.out_y0 = output->dim[1].min; q.W = W; q.H = H;
    q.p = patch_size; q.s = search_area;
    q.p_lo = -(patch_size / 2); q.s_lo = -(search_area / 2);
    // inv_sigma_sq = -1.0f / (sigma * sigma * patch_size * patch_size) (generator :24)
    q.inv_sigma_sq = -1.0f / (((sigma * sigma) * (float)patch_size) * (float)patch_size);
    q.iw = TX + patch_size + search_area - 2; q.ih = TY + patch_size + search_area - 2;
    q.dw = TX + patch_size - 1; q.dh = TY + patch_size - 1;
    const size_t fixed = (size_t)3 * q.iw * q.ih * sizeof(float);
    const size_t per_dx = (size_t)(q.dh + TY) * q.dw * sizeof(float);
    const size_t budget = 100 * 1024;
    int nd = search_area;
    while (nd > 1 && fixed + nd * per_dx > budget) nd--;
    q.nd = nd;
    const size_t smem = fixed + nd * per_dx;
    if (smem > 220 * 1024) {
        return hb::fail(halide_error_code_param_too_large, "nl_means: patch/search sizes need %zu bytes of shared memory", smem);
    }
    cudaStream_t s = hb::stream();
    {
        hb::CallTimer timer(s);
        // (the limit is per device; setting it is cheap, so it is simply set for every call that needs it)
        if (smem > 48 * 1024) cudaFuncSetAttribute(nl_means_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        dim3 grid((W + TX - 1) / TX, (H + TY - 1) / TY);
        const bool window = g_variant == 2 || (g_variant == 0 && kDefaultWindow);
        if (window && patch_size == 3 && search_area == 7) {
            constexpr size_t sm = nl_window_smem<3, 7>();
            static_assert(sm <= 48 * 1024, "no opt-in needed");
            HB_LAUNCH("nl_means_window", (nl_means_window_kernel<3, 7>), grid, 256, sm, s, q);
        } else if (window && patch_size == 7 && search_area == 7) {
            constexpr size_t sm = nl_window_smem<7, 7>();
            static_assert(sm <= 48 * 1024, "no opt-in needed");
            HB_LAUNCH("nl_means_window", (nl_means_window_kernel<7, 7>), grid, 256, sm, s, q);
        } else {
            HB_LAUNCH("nl_means", nl_means_kernel, grid, 256, smem, s, q);
        }
    }
    if ((r = hb::check_cuda(cudaGetLastError(), "nl_means launch", halide_error_code_device_run_failed))) return r;
    hb::mark_output_written(output);
    return 0;
}

HB_EXPORT_FILTER(nl_means, kArgs)
HB_EXPORT_AUTO_SCHEDULE(nl_means, kArgs)
