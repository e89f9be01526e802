// camera_pipe.cu — camera_pipe(input, matrix_3200, matrix_7000, color_temp, gamma, contrast,
// sharpen_strength, blackLevel, whiteLevel, processed) for sm_100a.
//
// Reference algorithm: apps/camera_pipe/camera_pipe_generator.cpp — shift(16,12) :412, hot-pixel suppression
// :240-249, GRBG deinterleave :251-261, gradient-directed demosaic :57-146, 3x4 Q8.8 colour matrix :263-295,
// 1024-entry tone curve :297-367, 1-2-1 unsharp mask :369-404.  Integer pipeline (uint16 raw -> uint8 RGB) with
// Halide's no-promotion typing; bit-exact against oracle/oracle_camera_pipe.cpp.
//
// HBM-bound by construction: 5 algorithmic bytes per output pixel (2 raw + 3 out).  Like the reference's own GPU
// schedule (generator :471-497) every intermediate of a tile lives in shared memory, so the frame is read
// once and written once:
//   cp_tables_kernel   12-entry Q8.8 matrix, 1024-entry curve (halide_pow), sharpen strength — once per call
//   camera_pipe_kernel one 64x32 output tile per block:
//        raw (+apron) -> smem -> denoised -> g_r/g_b at half resolution -> demosaic + matrix + curve (u8, tile+1)
//        -> unsharp mask -> 4 pixels per thread stored as one 32-bit word per channel
#include "../../include/camera_pipe.h"
#include "../../include/camera_pipe_auto_schedule.h"
#include "hb_common.h"
#include "hl_math.cuh"

namespace {

typedef uint16_t u16;
typedef int16_t i16;
typedef uint8_t u8;

constexpr int TW = 64, TH = 32;              // output tile
constexpr int CW = TW + 2, CH = TH + 2;      // curved tile (unsharp apron 1)
constexpr int HW = TW / 2 + 3, HH = TH / 2 + 3;  // half-res sites needed by the curved tile (any parity of the origin)
constexpr int GW = HW + 2, GH = HH + 2;      // g_r / g_b tile (demosaic apron 1)
constexpr int DW = 2 * GW, DH = 2 * GH;      // denoised tile (full-res)
constexpr int RW = DW + 4, RH = DH + 4;      // raw tile (hot-pixel apron 2)

struct CPTables {
    i16 matrix[12];  // [y*4 + x]
    u8 s32;
    u8 curve[1024];
};

struct CPParams {
    const u16 *in;  // element at the input mins
    int64_t in_sy;
    int in_x0, in_y0, in_w, in_h;
    u8 *out;  // element at the output mins
    int64_t out_sy, out_sc;
    int out_x0, out_y0, W, H, C, out_c0;
    const CPTables *tab;
};

__device__ __forceinline__ u16 avg16(u16 a, u16 b) { return (u16)(((uint32_t)a + (uint32_t)b + 1u) >> 1); }  // generator :16-19
__device__ __forceinline__ u16 absd16(u16 a, u16 b) { return a > b ? (u16)(a - b) : (u16)(b - a); }
__device__ __forceinline__ u8 avg8(u8 a, u8 b) { return (u8)(((uint32_t)a + (uint32_t)b + 1u) >> 1); }
__device__ __forceinline__ u8 blur121_8(u8 a, u8 b, u8 c) { return avg8(avg8(a, c), b); }
__device__ __forceinline__ int fdiv2(int a) { return a >> 1; }

// ---- tables: colour matrix, tone curve, sharpen strength (generator :263-271, :297-332, :372) --------------------
__global__ void cp_tables_kernel(CPTables *t, const float *m3200, int64_t m32_sx, int64_t m32_sy, const float *m7000, int64_t m70_sx,
                                 int64_t m70_sy, float color_temp, float gamma, float contrast, float sharpen_strength,
                                 int blackLevel, int whiteLevel, float inv_c_diff) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x < 12) {
        // alpha = (1/kelvin - 1/3200) / (1/7000 - 1/3200); the constant divisor is folded to a reciprocal multiply
        const float c3200 = 1.0f / 3200;
        float alpha = __fmul_rn(__fsub_rn(__fdiv_rn(1.0f, color_temp), c3200), inv_c_diff);
        int mx = x & 3, my = x >> 2;
        float a = m3200[mx * m32_sx + my * m32_sy], b = m7000[mx * m70_sx + my * m70_sy];
        float val = __fadd_rn(__fmul_rn(a, alpha), __fmul_rn(b, __fsub_rn(1.0f, alpha)));
        t->matrix[x] = (i16)(int)__fmul_rn(val, 256.0f);
    }
    if (x == 12) {
        float s = fmaxf(__fmul_rn(sharpen_strength, 32.0f), 0.0f);  // u8_sat: clamp low, saturate high, truncate
        t->s32 = s >= 255.0f ? (u8)255 : (u8)(int)s;
    }
    if (x < 1024) {
        const int minRaw = 0 + blackLevel, maxRaw = whiteLevel;
        const float invRange = __fdiv_rn(1.0f, (float)(maxRaw - minRaw));
        const float b = __fsub_rn(2.0f, hl::halide_pow(2.0f, __fmul_rn(contrast, 0.01f)));  // contrast / 100.0f folds to * 0.01f
        const float a = __fsub_rn(2.0f, __fmul_rn(2.0f, b));
        float xf = hl::clampf(__fmul_rn((float)(x - minRaw), invRange), 0.0f, 1.0f);
        float g = hl::halide_pow(xf, __fdiv_rn(1.0f, gamma));
        float omg = __fsub_rn(1.0f, g);
        float z_hi = __fsub_rn(1.0f, __fadd_rn(__fmul_rn(__fmul_rn(a, omg), omg), __fmul_rn(b, omg)));
        float z_lo = __fadd_rn(__fmul_rn(__fmul_rn(a, g), g), __fmul_rn(b, g));
        float z = g > 0.5f ? z_hi : z_lo;
        u8 val = (u8)(int)hl::clampf(__fadd_rn(__fmul_rn(z, 255.0f), 0.5f), 0.0f, 255.0f);
        t->curve[x] = x <= minRaw ? (u8)0 : (x > maxRaw ? (u8)255 : val);
    }
}

// ---- the fused tile kernel -------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) camera_pipe_kernel(CPParams p) {
    __shared__ u16 s_raw[RH][RW];
    __shared__ u16 s_den[DH][DW];
    __shared__ u16 s_gr[GH][GW];  // g_r at half-res sites
    __shared__ u16 s_gb[GH][GW];  // g_b
    __shared__ u8 s_cv[3][CH][CW + 2];
    __shared__ u8 s_curve[1024];
    __shared__ int s_m[12];
    const int tid = threadIdx.x;
    const int X0 = p.out_x0 + blockIdx.x * TW, Y0 = p.out_y0 + blockIdx.y * TH;  // absolute output coords of the tile
    // half-res origin of the sites the curved tile [X0-1, X0+TW] needs, grown by 1 for g_r / g_b
    const int gx0 = fdiv2(X0 - 1) - 1, gy0 = fdiv2(Y0 - 1) - 1;
    const int dx0 = 2 * gx0, dy0 = 2 * gy0;  // denoised tile origin (full-res, shifted coordinates)
    const int rx0 = dx0 - 2, ry0 = dy0 - 2;  // raw tile origin

    for (int i = tid; i < 1024; i += 256) s_curve[i] = p.tab->curve[i];
    if (tid < 12) s_m[tid] = (int)p.tab->matrix[tid];
    // raw tile: shifted(x,y) = input(x+16, y+12) (generator :412).  Coordinates the output never depends on may fall
    // outside the buffer at the frame's far edges of the last tiles; they are clamped (values unused).
    for (int i = tid; i < RW * RH; i += 256) {
        int ly = i / RW, lx = i - ly * RW;
        int ax = min(max(rx0 + lx + 16 - p.in_x0, 0), p.in_w - 1);  // buffer-relative, kept inside the buffer
        int ay = min(max(ry0 + ly + 12 - p.in_y0, 0), p.in_h - 1);
        s_raw[ly][lx] = __ldg(p.in + (int64_t)ay * p.in_sy + ax);
    }
    __syncthreads();
    // denoised = clamp(in, 0, max of the 4 neighbours at distance 2) (generator :240-249)
    for (int i = tid; i < DW * DH; i += 256) {
        int ly = i / DW, lx = i - ly * DW;
        int ry = ly + 2, rx = lx + 2;
        u16 a = max(max(s_raw[ry][rx - 2], s_raw[ry][rx + 2]), max(s_raw[ry - 2][rx], s_raw[ry + 2][rx]));
        s_den[ly][lx] = min(s_raw[ry][rx], a);
    }
    __syncthreads();
    // deinterleaved channel accessors at half-res site (sx, sy) relative to (gx0, gy0) (generator :57-60, :255-259)
#define G_GR(sx, sy) s_den[2 * (sy)][2 * (sx)]
#define R_R(sx, sy) s_den[2 * (sy)][2 * (sx) + 1]
#define B_B(sx, sy) s_den[2 * (sy) + 1][2 * (sx)]
#define G_GB(sx, sy) s_den[2 * (sy) + 1][2 * (sx) + 1]
    // green at red and blue sites (generator :70-82); border sites of the tile whose taps fall outside are never consumed
    for (int i = tid; i < GW * GH; i += 256) {
        int sy = i / GW, sx = i - sy * GW;
        int ym = max(sy - 1, 0), yp = min(sy + 1, GH - 1), xm = max(sx - 1, 0), xp = min(sx + 1, GW - 1);
        u16 gv_r = avg16(G_GB(sx, ym), G_GB(sx, sy)), gvd_r = absd16(G_GB(sx, ym), G_GB(sx, sy));
        u16 gh_r = avg16(G_GR(xp, sy), G_GR(sx, sy)), ghd_r = absd16(G_GR(xp, sy), G_GR(sx, sy));
        s_gr[sy][sx] = ghd_r < gvd_r ? gh_r : gv_r;
        u16 gv_b = avg16(G_GR(sx, yp), G_GR(sx, sy)), gvd_b = absd16(G_GR(sx, yp), G_GR(sx, sy));
        u16 gh_b = avg16(G_GB(xm, sy), G_GB(sx, sy)), ghd_b = absd16(G_GB(xm, sy), G_GB(sx, sy));
        s_gb[sy][sx] = ghd_b < gvd_b ? gh_b : gv_b;
    }
    __syncthreads();
    // demosaic + colour matrix + curve on the curved tile [X0-1, X0+TW] x [Y0-1, Y0+TH]
    for (int i = tid; i < CW * CH; i += 256) {
        int ly = i / CW, lx = i - ly * CW;
        int X = X0 - 1 + lx, Y = Y0 - 1 + ly;
        int x = fdiv2(X) - gx0, y = fdiv2(Y) - gy0;  // half-res site within the tiles
        bool xe = (X & 1) == 0, ye = (Y & 1) == 0;
        u16 r, g, b;
        if (ye && xe) {  // gr site (generator :89-96)
            g = G_GR(x, y);
            u16 corr = (u16)(g - avg16(s_gr[y][x], s_gr[y][x - 1]));
            r = (u16)(corr + avg16(R_R(x - 1, y), R_R(x, y)));
            corr = (u16)(g - avg16(s_gb[y][x], s_gb[y - 1][x]));
            b = (u16)(corr + avg16(B_B(x, y), B_B(x, y - 1)));
        } else if (ye) {  // r site (generator :121-130)
            r = R_R(x, y);
            g = s_gr[y][x];
            u16 corr = (u16)(g - avg16(s_gb[y][x], s_gb[y - 1][x + 1]));
            u16 bp = (u16)(corr + avg16(B_B(x, y), B_B(x + 1, y - 1)));
            u16 bpd = absd16(B_B(x, y), B_B(x + 1, y - 1));
            corr = (u16)(g - avg16(s_gb[y][x + 1], s_gb[y - 1][x]));
            u16 bn = (u16)(corr + avg16(B_B(x + 1, y), B_B(x, y - 1)));
            u16 bnd = absd16(B_B(x + 1, y), B_B(x, y - 1));
            b = bpd < bnd ? bp : bn;
        } else if (xe) {  // b site (generator :111-119)
            b = B_B(x, y);
            g = s_gb[y][x];
            u16 corr = (u16)(g - avg16(s_gr[y][x], s_gr[y + 1][x - 1]));
            u16 rp = (u16)(corr + avg16(R_R(x, y), R_R(x - 1, y + 1)));
            u16 rpd = absd16(R_R(x, y), R_R(x - 1, y + 1));
            corr = (u16)(g - avg16(s_gr[y][x - 1], s_gr[y + 1][x]));
            u16 rn = (u16)(corr + avg16(R_R(x - 1, y), R_R(x, y + 1)));
            u16 rnd = absd16(R_R(x - 1, y), R_R(x, y + 1));
            r = rpd < rnd ? rp : rn;
        } else {  // gb site (generator :98-102)
            g = G_GB(x, y);
            u16 corr = (u16)(g - avg16(s_gr[y][x], s_gr[y + 1][x]));
            r = (u16)(corr + avg16(R_R(x, y), R_R(x, y + 1)));
            corr = (u16)(g - avg16(s_gb[y][x], s_gb[y][x + 1]));
            b = (u16)(corr + avg16(B_B(x, y), B_B(x + 1, y)));
        }
        // i16 reinterpretation (generator :146), colour matrix in i32 with floor division by 256 (generator :277-292)
        const int ir = (int)(i16)r, ig = (int)(i16)g, ib = (int)(i16)b;
#pragma unroll
        for (int c = 0; c < 3; c++) {
            int acc = ((s_m[c * 4 + 3] + s_m[c * 4 + 0] * ir) + s_m[c * 4 + 1] * ig) + s_m[c * 4 + 2] * ib;
            int cc = (int)(i16)(acc >> 8);
            s_cv[c][ly][lx] = s_curve[min(max(cc, 0), 1023)];
        }
    }
    __syncthreads();
#undef G_GR
#undef R_R
#undef B_B
#undef G_GB
    // unsharp mask (generator :384-401): 4 horizontally adjacent pixels per thread, one 32-bit store per channel
    const int s32 = (int)p.tab->s32;
    for (int i = tid; i < (TW / 4) * TH * 3; i += 256) {
        int c = i / ((TW / 4) * TH), rem = i - c * (TW / 4) * TH;
        int ly = rem / (TW / 4), q = rem - ly * (TW / 4);
        if (c >= p.C) continue;
        int oy = blockIdx.y * TH + ly;
        if (oy >= p.H) continue;
        int cch = p.out_c0 + c;  // absolute channel 0..2 -> curved plane
        if (cch < 0 || cch > 2) continue;
        uint32_t packed = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            int lx = 4 * q + k;  // tile-local output x; curved tile index = lx + 1, ly + 1
            const int cx = lx + 1, cy = ly + 1;
            u8 uy_m = blur121_8(s_cv[cch][cy - 1][cx - 1], s_cv[cch][cy][cx - 1], s_cv[cch][cy + 1][cx - 1]);
            u8 uy_0 = blur121_8(s_cv[cch][cy - 1][cx], s_cv[cch][cy][cx], s_cv[cch][cy + 1][cx]);
            u8 uy_p = blur121_8(s_cv[cch][cy - 1][cx + 1], s_cv[cch][cy][cx + 1], s_cv[cch][cy + 1][cx + 1]);
            u8 unsharp = blur121_8(uy_m, uy_0, uy_p);
            int in_v = (int)s_cv[cch][cy][cx];
            i16 mask = (i16)(in_v - (int)unsharp);
            i16 prod = (i16)((int)mask * s32);          // i16 * u8 stays i16 and wraps (src/IROperator.cpp:769-816)
            int sum = (int)(i16)(in_v + ((int)prod >> 5));  // floor division by 32
            packed |= (uint32_t)min(max(sum, 0), 255) << (8 * k);
        }
        int ox = blockIdx.x * TW + 4 * q;
        u8 *dst = p.out + (int64_t)c * p.out_sc + (int64_t)oy * p.out_sy + ox;
        if (ox + 3 < p.W && (reinterpret_cast<uintptr_t>(dst) & 3) == 0) {
            *reinterpret_cast<uint32_t *>(dst) = packed;
        } else {
            for (int k = 0; k < 4; k++)
                if (ox + k < p.W) dst[k] = (u8)(packed >> (8 * k));
        }
    }
}

const hb::BufferEstimates est_in({0, 2592, 0, 1968}), est_m({0, 4, 0, 3});
const hb::BufferEstimates est_out({0, 2592, 0, 1968, 0, 3});
const halide_scalar_value_t sv[6] = {hb::scalar(3700.0f), hb::scalar(2.0f), hb::scalar(50.0f), hb::scalar(1.0f), hb::scalar(25),
                                     hb::scalar(1023)};
const halide_filter_argument_t kArgs[10] = {
    {"input", halide_argument_kind_input_buffer, 2, {halide_type_uint, 16, 0}, nullptr, nullptr, nullptr, nullptr, est_in.p},
    {"matrix_3200", halide_argument_kind_input_buffer, 2, {halide_type_float, 32, 0}, nullptr, nullptr, nullptr, nullptr, est_m.p},
    {"matrix_7000", halide_argument_kind_input_buffer, 2, {halide_type_float, 32, 0}, nullptr, nullptr, nullptr, nullptr, est_m.p},
    {"color_temp", halide_argument_kind_input_scalar, 0, {halide_type_float, 32, 0}, nullptr, nullptr, nullptr, &sv[0], nullptr},
    {"gamma", halide_argument_kind_input_scalar, 0, {halide_type_float, 32, 0}, nullptr, nullptr, nullptr, &sv[1], nullptr},
    {"contrast", halide_argument_kind_input_scalar, 0, {halide_type_float, 32, 0}, nullptr, nullptr, nullptr, &sv[2], nullptr},
    {"sharpen_strength", halide_argument_kind_input_scalar, 0, {halide_type_float, 32, 0}, nullptr, nullptr, nullptr, &sv[3], nullptr},
    {"blackLevel", halide_argument_kind_input_scalar, 0, {halide_type_int, 32, 0}, nullptr, nullptr, nullptr, &sv[4], nullptr},
    {"whiteLevel", halide_argument_kind_input_scalar, 0, {halide_type_int, 32, 0}, nullptr, nullptr, nullptr, &sv[5], nullptr},
    {"processed", halide_argument_kind_output_buffer, 3, {halide_type_uint, 8, 0}, nullptr, nullptr, nullptr, nullptr, est_out.p},
};
const auto &kIn = kArgs[0], &kM32 = kArgs[1], &kM70 = kArgs[2], &kOut = kArgs[9];

inline int fdiv(int a, int b) {
    int q = a / b;
    return (a % b != 0 && ((a < 0) != (b < 0))) ? q - 1 : q;
}

}  // namespace

extern "C" int camera_pipe(halide_buffer_t *input, halide_buffer_t *m3200, halide_buffer_t *m7000, float color_temp, float gamma,
                           float contrast, float sharpen_strength, int32_t blackLevel, int32_t whiteLevel, halide_buffer_t *out) {
    int r;
    if ((r = hb::check_arg(input, kIn))) return r;
    if ((r = hb::check_arg(m3200, kM32))) return r;
    if ((r = hb::check_arg(m7000, kM70))) return r;
    if ((r = hb::check_arg(out, kOut))) return r;
    const int ox = out->dim[0].min, oy = out->dim[1].min, W = out->dim[0].extent, H = out->dim[1].extent;
    // Required input region by interval arithmetic over the stencil chain (no boundary condition anywhere):
    // unsharp +-1 -> half-res sites -> demosaic +-1 site -> denoise +-2 -> shift (16,12).
    const int hx0 = fdiv(ox - 1, 2), hx1 = fdiv(ox + W, 2), hy0 = fdiv(oy - 1, 2), hy1 = fdiv(oy + H, 2);
    const int need_x0 = 2 * (hx0 - 1) - 2 + 16, need_x1 = 2 * (hx1 + 1) + 1 + 2 + 16;
    const int need_y0 = 2 * (hy0 - 1) - 2 + 12, need_y1 = 2 * (hy1 + 1) + 1 + 2 + 12;
    bool query = false;
    if (hb::is_bounds_query(input)) {
        int mins[2] = {need_x0, need_y0}, ext[2] = {need_x1 - need_x0 + 1, need_y1 - need_y0 + 1};
        hb::propose_shape(input, mins, ext);
        query = true;
    }
    for (halide_buffer_t *m : {m3200, m7000}) {
        if (hb::is_bounds_query(m)) {
            int mins[2] = {0, 0}, ext[2] = {4, 3};
            hb::propose_shape(m, mins, ext);
            query = true;
        }
    }
    if (hb::is_bounds_query(out)) {
        int mins[3] = {ox, oy, out->dim[2].min}, ext[3] = {W, H, out->dim[2].extent};
        hb::propose_shape(out, mins, ext);
        query = true;
    }
    if (query) return 0;
    if ((r = hb::check_shape(input, kIn)) || (r = hb::check_shape(m3200, kM32)) || (r = hb::check_shape(m7000, kM70)) ||
        (r = hb::check_shape(out, kOut)))
        return r;
    if (W <= 0 || H <= 0 || out->dim[2].extent <= 0) return 0;
    if ((r = hb::check_covers(input, kIn, 0, need_x0, need_x1 - need_x0 + 1))) return r;
    if ((r = hb::check_covers(input, kIn, 1, need_y0, need_y1 - need_y0 + 1))) return r;
    for (halide_buffer_t *m : {m3200, m7000}) {
        const halide_filter_argument_t &sp = m == m3200 ? kM32 : kM70;
        if ((r = hb::check_covers(m, sp, 0, 0, 4)) || (r = hb::check_covers(m, sp, 1, 0, 3))) return r;
    }
    if ((r = hb::check_covers(out, kOut, 2, out->dim[2].min, out->dim[2].extent))) return r;
    if (out->dim[2].min < 0 || out->dim[2].min + out->dim[2].extent > 3) {
        return hb::fail(halide_error_code_access_out_of_bounds, "Output buffer processed channel range [%d,%d) is outside [0,3)",
                        out->dim[2].min, out->dim[2].min + out->dim[2].extent);
    }
    void *din = nullptr, *d32 = nullptr, *d70 = nullptr, *dout = nullptr;
    if ((r = hb::acquire_input(input, kIn, &din)) || (r = hb::acquire_input(m3200, kM32, &d32)) ||
        (r = hb::acquire_input(m7000, kM70, &d70)) || (r = hb::acquire_output(out, kOut, &dout)))
        return r;
    hb::Scratch scratch;
    CPTables *tab = scratch.get<CPTables>(1);
    if (!tab) return hb::fail(halide_error_code_device_malloc_failed, "camera_pipe: scratch allocation failed");

    CPParams p;
    p.in = (const u16 *)din;
    p.in_sy = input->dim[1].stride;
    p.in_x0 = input->dim[0].min; p.in_y0 = input->dim[1].min;
    p.in_w = input->dim[0].extent; p.in_h = input->dim[1].extent;
    p.out = (u8 *)dout;
    p.out_sy = out->dim[1].stride; p.out_sc = out->dim[2].stride;
    p.out_x0 = ox; p.out_y0 = oy; p.W = W; p.H = H; p.C = out->dim[2].extent; p.out_c0 = out->dim[2].min;
    p.tab = tab;
    // (1/7000 - 1/3200) in float, reciprocal folded in double then rounded (src/Simplify_Div.cpp:204)
    const float c_diff = 1.0f / 7000 - 1.0f / 3200;
    const float inv_c_diff = (float)(1.0 / (double)c_diff);
    // offsets of matrix element (0,0)
    const float *m32p = (const float *)d32 - m3200->dim[0].min * (int64_t)m3200->dim[0].stride - m3200->dim[1].min * (int64_t)m3200->dim[1].stride;
    const float *m70p = (const float *)d70 - m7000->dim[0].min * (int64_t)m7000->dim[0].stride - m7000->dim[1].min * (int64_t)m7000->dim[1].stride;
    cudaStream_t s = hb::stream();
    {
        hb::CallTimer timer(s);
        HB_LAUNCH("cp_tables", cp_tables_kernel, 4, 256, 0, s, tab, m32p, (int64_t)m3200->dim[0].stride, (int64_t)m3200->dim[1].stride,
                  m70p, (int64_t)m7000->dim[0].stride, (int64_t)m7000->dim[1].stride, color_temp, gamma, contrast, sharpen_strength,
                  blackLevel, whiteLevel, inv_c_diff);
        dim3 grid((W + TW - 1) / TW, (H + TH - 1) / TH);
        HB_LAUNCH("camera_pipe", camera_pipe_kernel, grid, 256, 0, s, p);
    }
    if ((r = hb::check_cuda(cudaGetLastError(), "camera_pipe launch", halide_error_code_device_run_failed))) return r;
    hb::mark_output_written(out);
    return 0;
}

HB_EXPORT_FILTER(camera_pipe, kArgs)
HB_EXPORT_AUTO_SCHEDULE(camera_pipe, kArgs)
