// blur.cu — halide_blur(input, blur_y): 3x3 box filter on uint16, the plumbing target (config 1).
//
// Algorithm (reference: apps/blur/halide_blur_generator.cpp:39-40):
//   blur_x(x,y) = (in(x,y) + in(x+1,y) + in(x+2,y)) / 3
//   blur_y(x,y) = (blur_x(x,y) + blur_x(x,y+1) + blur_x(x,y+2)) / 3
// All arithmetic stays uint16 (Halide's u16+u16 is u16 and wraps, src/IROperator.cpp:769-816), so
// the sums are taken mod 2^16 before the unsigned divide.  There is no boundary condition: the
// input must cover [ox, ox+W+1] x [oy, oy+H+1] or the call fails with -4
// (src/AddImageChecks.cpp:404-417).
//
// Kernel shape: HBM-bound, 4 algorithmic bytes per pixel.  Two kernels, both "one warp walks a column strip top to
// bottom with the last two blur_x rows in registers, several input rows in flight per lane":
//   * blur3x3_u16_quad_kernel — frames whose rows keep pixel pairs 4-byte aligned (even row strides: the harness and
//     RunGen frames): a lane owns 4 pixels, 32-bit loads, arithmetic in high-half form, ~10 instructions per pixel,
//     strips sized to fill the resident warps a whole number of times.  29.8 us at 8K (68 % of the measured HBM peak).
//   * blur3x3_u16_kernel — any alignment: a lane owns 8 pixels, aligned 16-byte loads realigned by funnel shifts, the
//     2-pixel horizontal apron from the neighbouring lane by shuffle.  Bound by the integer pipe (49 us at 8K).
#include "../../include/halide_blur.h"
#include "hb_common.h"

namespace {

constexpr int kPxPerLane = 8;
constexpr int kStripW = 32 * kPxPerLane;  // 256 output pixels per warp per row
constexpr int kWarpsPerBlock = 4;
int g_force_general = 0;  // test hook (halide_b200_blur_force_general): 1 = route aligned frames through the general kernel too,
                          // >= 8 = aligned kernel with this strip height (small test frames then reach its unclamped main loop)

struct BlurArgs {
    const uint16_t *in;   // element (in_x0, in_y0) of the input == the one feeding output (0,0)
    uint16_t *out;        // element at output mins
    int64_t in_stride_y, out_stride_y;
    int w, h;             // output extent
    int rows_per_warp;
    // valid element range of the input allocation relative to `in`, for guarding vector loads
    int64_t in_lo, in_hi;
};

__device__ __forceinline__ uint4 load_chunk(const uint16_t *p, int64_t off, int64_t lo, int64_t hi) {
    // p+off is 16-byte aligned.  Fast path when the whole chunk is inside the allocation span.
    if (off >= lo && off + 7 <= hi) {
        return *reinterpret_cast<const uint4 *>(p + off);
    }
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        int64_t e0 = off + 2 * i, e1 = e0 + 1;
        uint32_t a = (e0 >= lo && e0 <= hi) ? p[e0] : 0u;
        uint32_t b = (e1 >= lo && e1 <= hi) ? p[e1] : 0u;
        w[i] = a | (b << 16);
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}

// Raw 16-byte chunks of one input row for this lane (issued one row ahead of their use so the loads of row y+3
// are in flight while row y+2 is being reduced).
struct RawRow {
    uint4 v, t;
    int mis;
};
__device__ __forceinline__ RawRow load_raw_row(const BlurArgs &a, int64_t row_off, int x0, int lane) {
    RawRow r;
    // Element offset (relative to a.in) of the first pixel of this warp's strip on this row.
    int64_t e = row_off + x0;
    // Misalignment of that element against 16 bytes, uniform across the warp.
    r.mis = (int)((reinterpret_cast<uintptr_t>(a.in + e) & 15) >> 1);
    int64_t base = e - r.mis;  // 16-byte aligned
    r.v = load_chunk(a.in, base + 8 * lane, a.in_lo, a.in_hi);
    r.t = make_uint4(0, 0, 0, 0);
    if (lane < 2) r.t = load_chunk(a.in, base + 8 * (32 + lane), a.in_lo, a.in_hi);
    return r;
}

// blur_x for the 8 pixels of this lane on one input row.
__device__ __forceinline__ void blur_x_row(const RawRow &raw, int lane, uint32_t bx[8]) {
    const uint4 v = raw.v, t = raw.t;
    const int mis = raw.mis;

    // words of the 3-chunk window: own chunk, next lane's chunk, first word of the chunk after that
    uint32_t w[9];
    w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
    uint32_t n0 = __shfl_down_sync(0xffffffffu, v.x, 1), n1 = __shfl_down_sync(0xffffffffu, v.y, 1);
    uint32_t n2 = __shfl_down_sync(0xffffffffu, v.z, 1), n3 = __shfl_down_sync(0xffffffffu, v.w, 1);
    uint32_t m0 = __shfl_down_sync(0xffffffffu, v.x, 2);
    uint32_t t0x = __shfl_sync(0xffffffffu, t.x, 0), t0y = __shfl_sync(0xffffffffu, t.y, 0);
    uint32_t t0z = __shfl_sync(0xffffffffu, t.z, 0), t0w = __shfl_sync(0xffffffffu, t.w, 0);
    uint32_t t1x = __shfl_sync(0xffffffffu, t.x, 1);
    if (lane == 31) { n0 = t0x; n1 = t0y; n2 = t0z; n3 = t0w; m0 = t1x; }
    if (lane == 30) { m0 = t0x; }
    w[4] = n0; w[5] = n1; w[6] = n2; w[7] = n3; w[8] = m0;

    // 10 halfwords starting at halfword `mis` of the window → 6 words starting at word mis>>1.
    int wo = mis >> 1;
    uint32_t s[6];
#pragma unroll
    for (int i = 0; i < 6; i++) {
        // wo is warp-uniform in [0,3]; select without dynamic register indexing
        uint32_t c0 = w[i], c1 = w[i + 1], c2 = w[i + 2], c3 = (i + 3 < 9) ? w[i + 3] : 0u;
        s[i] = wo == 0 ? c0 : wo == 1 ? c1 : wo == 2 ? c2 : c3;
    }
    if (mis & 1) {
#pragma unroll
        for (int i = 0; i < 5; i++) s[i] = __funnelshift_r(s[i], s[i + 1], 16);
    }
    uint32_t px[10];
#pragma unroll
    for (int i = 0; i < 5; i++) {
        px[2 * i] = s[i] & 0xffffu;
        px[2 * i + 1] = s[i] >> 16;
    }
#pragma unroll
    for (int i = 0; i < 8; i++) {
        bx[i] = ((px[i] + px[i + 1] + px[i + 2]) & 0xffffu) / 3u;
    }
}

__global__ void __launch_bounds__(32 * kWarpsPerBlock) blur3x3_u16_kernel(BlurArgs a) {
    int lane = threadIdx.x & 31;
    int warp = threadIdx.x >> 5;
    int x0 = blockIdx.x * kStripW;
    int y0 = (blockIdx.y * kWarpsPerBlock + warp) * a.rows_per_warp;
    if (y0 >= a.h) return;
    int y1 = min(y0 + a.rows_per_warp, a.h);

    uint32_t r0[8], r1[8], r2[8];
    blur_x_row(load_raw_row(a, (int64_t)y0 * a.in_stride_y, x0, lane), lane, r0);
    blur_x_row(load_raw_row(a, (int64_t)(y0 + 1) * a.in_stride_y, x0, lane), lane, r1);
    RawRow next = load_raw_row(a, (int64_t)(y0 + 2) * a.in_stride_y, x0, lane);
    int xl = x0 + lane * kPxPerLane;
    for (int y = y0; y < y1; y++) {
        const RawRow cur = next;
        if (y + 1 < y1) next = load_raw_row(a, (int64_t)(y + 3) * a.in_stride_y, x0, lane);
        blur_x_row(cur, lane, r2);
        uint32_t o[8];
#pragma unroll
        for (int i = 0; i < 8; i++) o[i] = ((r0[i] + r1[i] + r2[i]) & 0xffffu) / 3u;
        uint16_t *dst = a.out + (int64_t)y * a.out_stride_y + xl;
        if (xl + 8 <= a.w && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
            uint4 pk = make_uint4(o[0] | (o[1] << 16), o[2] | (o[3] << 16), o[4] | (o[5] << 16), o[6] | (o[7] << 16));
            *reinterpret_cast<uint4 *>(dst) = pk;
        } else {
#pragma unroll
            for (int i = 0; i < 8; i++) {
                if (xl + i < a.w) dst[i] = (uint16_t)o[i];
            }
        }
#pragma unroll
        for (int i = 0; i < 8; i++) { r0[i] = r1[i]; r1[i] = r2[i]; }
    }
}

// ---- fast path: frames whose rows keep pixel pairs 4-byte aligned (even strides, aligned bases) ----------------------
// The kernel above pays for arbitrary row misalignment with funnel shifts and selects and is bound by the integer
// pipe, not by HBM (ALU 63 %, issue 66 %, DRAM 20 % at 8K: profiles/r02_other_pipelines_ncu.md).  When every row starts
// on an even element — the harness and RunGen frames do: dense rows of W + 2 with W even — a lane can own two aligned
// pixel PAIRS (4 pixels): two 32-bit loads per row, the pair to its right from the next lane by shuffle (lane 31 loads
// it), and all arithmetic in "high-half form" (a u16 value v held as v << 16): 32-bit adds of such values wrap mod 2^16
// by themselves, umulhi(s, 0x55555556) leaves floor(v / 3) in the upper half (the lower half is (v mod 3) * 2^16 / 3
// plus an error below 1, which never carries), and one PRMT packs two results.  ~10 integer instructions per pixel.
// One warp = a 128-pixel-wide strip walked top to bottom with the last two blur_x rows in registers and kQuadAhead
// input rows in flight per lane; the strip height is chosen on the host so that the strips fill the resident warps of
// the device a whole number of times (no tail wave).
constexpr int kQuadWarps = 4, kQuadW = 128;  // (kQuadAhead: template parameter AHEAD, a multiple of 3 so the row window rotates by renaming)
constexpr uint32_t kThird = 0x55555556u;

__device__ __forceinline__ uint32_t ld_pair(const BlurArgs &a, int64_t off) {  // off even: one aligned word, or guarded halves
    if (off >= a.in_lo && off + 1 <= a.in_hi) return __ldg(reinterpret_cast<const uint32_t *>(a.in + off));
    uint32_t lo = (off >= a.in_lo && off <= a.in_hi) ? a.in[off] : 0u;
    uint32_t hi = (off + 1 >= a.in_lo && off + 1 <= a.in_hi) ? a.in[off + 1] : 0u;
    return lo | (hi << 16);
}

struct QuadRow {
    uint32_t w0, w1, w2;  // pixels (x, x+1), (x+2, x+3), (x+4, x+5); w2 is the next lane's w0 again (an L1 hit, no shuffle)
};
template<bool GUARD>
__device__ __forceinline__ QuadRow ld_quad(const BlurArgs &a, const uint16_t *row) {  // row = &in(x, y) of this lane
    QuadRow q;
    if (!GUARD) {
        const uint32_t *p = reinterpret_cast<const uint32_t *>(row);
        q.w0 = __ldg(p);
        q.w1 = __ldg(p + 1);
        q.w2 = __ldg(p + 2);
    } else {
        const int64_t off = row - a.in;
        q.w0 = ld_pair(a, off);
        q.w1 = ld_pair(a, off + 2);
        q.w2 = ld_pair(a, off + 4);
    }
    return q;
}
// blur_x of the lane's four pixels, results in high-half form with a clean lower half
__device__ __forceinline__ void blur_x_quad(const QuadRow &q, uint32_t (&b)[4]) {
    const uint32_t a0 = q.w0 << 16, a1 = q.w0 & 0xffff0000u, a2 = q.w1 << 16, a3 = q.w1 & 0xffff0000u;
    const uint32_t a4 = q.w2 << 16, a5 = q.w2 & 0xffff0000u;
    b[0] = __umulhi(a0 + a1 + a2, kThird) & 0xffff0000u;
    b[1] = __umulhi(a1 + a2 + a3, kThird) & 0xffff0000u;
    b[2] = __umulhi(a2 + a3 + a4, kThird) & 0xffff0000u;
    b[3] = __umulhi(a3 + a4 + a5, kThird) & 0xffff0000u;
}

// Walks one strip.  `rin` is the row pointer of the next input row to request, `rout` the output row pointer.  The
// bulk of the strip runs without any test per row; only the refills of the last rows (which would run past the
// strip's last input row) use the clamped request, which re-requests a valid row.
template<bool GUARD, int kQuadAhead>
struct QuadStrip {
    const BlurArgs &a;
    const uint16_t *rin;
    uint16_t *rout;
    int next_row, last_in, x;
    QuadRow q[kQuadAhead];
    uint32_t r0[4], r1[4];

    template<bool CLAMP>
    __device__ __forceinline__ QuadRow fetch() {
        const QuadRow t = ld_quad<GUARD>(a, rin);
        if (!CLAMP) {
            rin += a.in_stride_y;
        } else if (next_row < last_in) {
            next_row++;
            rin += a.in_stride_y;
        }
        return t;
    }
    template<bool CLAMP>
    __device__ __forceinline__ void row(int k) {
        uint32_t r2[4];
        blur_x_quad(q[k], r2);
        q[k] = fetch<CLAMP>();
        uint32_t o[4];
#pragma unroll
        for (int i = 0; i < 4; i++) o[i] = __umulhi(r0[i] + r1[i] + r2[i], kThird);
        const uint32_t p0 = __byte_perm(o[0], o[1], 0x7632), p1 = __byte_perm(o[2], o[3], 0x7632);
        if (!GUARD) {
            reinterpret_cast<uint32_t *>(rout)[0] = p0;
            reinterpret_cast<uint32_t *>(rout)[1] = p1;
        } else {
            if (x + 1 < a.w) reinterpret_cast<uint32_t *>(rout)[0] = p0;
            else if (x < a.w) rout[0] = (uint16_t)(p0 & 0xffffu);
            if (x + 3 < a.w) reinterpret_cast<uint32_t *>(rout)[1] = p1;
            else if (x + 2 < a.w) rout[2] = (uint16_t)(p1 & 0xffffu);
        }
        rout += a.out_stride_y;
#pragma unroll
        for (int i = 0; i < 4; i++) { r0[i] = r1[i]; r1[i] = r2[i]; }
    }
    __device__ __forceinline__ void run(int y0, int y1) {
        last_in = y1 + 1;  // last input row read; y0 + 2 <= last_in
        rin = a.in + ((int64_t)y0 * a.in_stride_y + x);
        rout = a.out + ((int64_t)y0 * a.out_stride_y + x);
        const QuadRow t0 = fetch<false>(), t1 = fetch<false>();
        next_row = y0 + 2;
#pragma unroll
        for (int k = 0; k < kQuadAhead; k++) q[k] = fetch<true>();
        blur_x_quad(t0, r0);
        blur_x_quad(t1, r1);
        int y = y0;
        // the refill of row y asks for input row y + 2 + kQuadAhead and then steps once more: unclamped while even that
        // step stays <= last_in for a whole group
        for (; y + 2 * kQuadAhead < y1; y += kQuadAhead) {
#pragma unroll
            for (int k = 0; k < kQuadAhead; k++) row<false>(k);
        }
        next_row = min(y + 2 + kQuadAhead, last_in);  // rin points at that row already
        for (; y < y1; y += kQuadAhead) {
#pragma unroll
            for (int k = 0; k < kQuadAhead; k++) {
                if (y + k < y1) row<true>(k);  // warp-uniform
            }
        }
    }
};

// a.rows_per_warp = strip height; strips are numbered x-fastest so the warps of a block read adjacent spans of a row
template<int AHEAD>
__global__ void __launch_bounds__(32 * kQuadWarps) blur3x3_u16_quad_kernel(BlurArgs a, int strips_x, int strips) {
    const int lane = threadIdx.x & 31;
    const int t = blockIdx.x * kQuadWarps + (threadIdx.x >> 5);
    if (t >= strips) return;
    const int sx = t % strips_x, sy = t / strips_x;
    const int xw = sx * kQuadW, y0 = sy * a.rows_per_warp;
    const int y1 = min(y0 + a.rows_per_warp, a.h);
    // whole strip (and the two input columns to its right) inside the output width: nothing to guard
    if (xw + kQuadW <= a.w) {
        QuadStrip<false, AHEAD> st{a};
        st.x = xw + 4 * lane;
        st.run(y0, y1);
    } else {
        QuadStrip<true, AHEAD> st{a};
        st.x = xw + 4 * lane;
        st.run(y0, y1);
    }
}

const halide_filter_argument_t kArgs[2] = {
    {"input", halide_argument_kind_input_buffer, 2, {halide_type_uint, 16, 0}, nullptr, nullptr, nullptr, nullptr, nullptr},
    {"blur_y", halide_argument_kind_output_buffer, 2, {halide_type_uint, 16, 0}, nullptr, nullptr, nullptr, nullptr, nullptr},
};
const auto &kIn = kArgs[0], &kOut = kArgs[1];

}  // namespace

extern "C" int halide_blur(halide_buffer_t *input, halide_buffer_t *blur_y) {
    int r;
    if ((r = hb::check_arg(input, kIn))) return r;
    if ((r = hb::check_arg(blur_y, kOut))) return r;

    // Bounds query (src/AddImageChecks.cpp:477-496): the input must cover the output region
    // grown by the 3-tap footprints: [ox, ox+W+1] x [oy, oy+H+1].
    const int ox = blur_y->dim[0].min, oy = blur_y->dim[1].min;
    const int w = blur_y->dim[0].extent, h = blur_y->dim[1].extent;
    bool query = false;
    if (hb::is_bounds_query(input)) {
        int mins[2] = {ox, oy}, ext[2] = {w + 2, h + 2};
        hb::propose_shape(input, mins, ext);
        query = true;
    }
    if (hb::is_bounds_query(blur_y)) {
        int mins[2] = {ox, oy}, ext[2] = {w, h};
        hb::propose_shape(blur_y, mins, ext);
        query = true;
    }
    if (query) return 0;

    if ((r = hb::check_shape(input, kIn))) return r;
    if ((r = hb::check_shape(blur_y, kOut))) return r;
    if ((r = hb::check_covers(input, kIn, 0, ox, w + 2))) return r;
    if ((r = hb::check_covers(input, kIn, 1, oy, h + 2))) return r;
    if (w <= 0 || h <= 0) return 0;

    void *din = nullptr, *dout = nullptr;
    if ((r = hb::acquire_input(input, kIn, &din))) return r;
    if ((r = hb::acquire_output(blur_y, kOut, &dout))) return r;

    BlurArgs a;
    const int64_t isy = input->dim[1].stride;
    const int64_t origin = (int64_t)(ox - input->dim[0].min) + (int64_t)(oy - input->dim[1].min) * isy;
    a.in = (const uint16_t *)din + origin;
    a.out = (uint16_t *)dout;
    a.in_stride_y = isy;
    a.out_stride_y = blur_y->dim[1].stride;
    a.w = w;
    a.h = h;
    // allocation span of the input relative to a.in (dim0 stride is 1; dim1 stride may be negative)
    int64_t reach1 = (int64_t)(input->dim[1].extent - 1) * isy;
    int64_t lo = reach1 < 0 ? reach1 : 0, hi = (reach1 > 0 ? reach1 : 0) + input->dim[0].extent - 1;
    a.in_lo = lo - origin;
    a.in_hi = hi - origin;

    // Enough warps to cover 148 SMs a few times over, but strips tall enough to amortise the
    // two-row vertical apron.
    int strips_x = (w + kStripW - 1) / kStripW;
    int rows = 32;
    while (rows > 4 && (int64_t)strips_x * ((h + rows - 1) / rows) < 148 * 8) rows >>= 1;
    a.rows_per_warp = rows;
    int warps_y = (h + rows - 1) / rows;
    dim3 grid(strips_x, (warps_y + kWarpsPerBlock - 1) / kWarpsPerBlock);

    // pixel pairs 4-byte aligned on every row of both buffers -> the pair kernel; anything else -> the general kernel
    const bool pair_ok = ((reinterpret_cast<uintptr_t>(a.in) | reinterpret_cast<uintptr_t>(a.out)) & 3) == 0 &&
                         (a.in_stride_y & 1) == 0 && (a.out_stride_y & 1) == 0 && g_force_general != 1;
    cudaStream_t s = hb::stream();
    {
        hb::CallTimer timer(s);
        if (pair_ok) {
            // strips of 128 columns; height such that the strips fill the resident warps a whole number of times
            // (six rows in flight per lane: nine — 86 registers, five blocks per SM — measured slower, 33.5 vs 29.3 us at 8K)
            static int resident = 0;  // blocks per SM x SMs (per process: one device per process)
            if (!resident) {
                int per_sm = 0, dev = 0, sms = 0;
                cudaGetDevice(&dev);
                cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
                cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, blur3x3_u16_quad_kernel<6>, 32 * kQuadWarps, 0);
                resident = (per_sm > 0 ? per_sm : 8) * (sms > 0 ? sms : 148);
            }
            const int sxq = (w + kQuadW - 1) / kQuadW;
            const int64_t slots = (int64_t)resident * kQuadWarps;
            int qrows = 8;
            for (int m = 1; m <= 64; m++) {
                const int64_t sy = m * slots / sxq;
                if (sy < 1) continue;
                const int rr = (int)((h + sy - 1) / sy);
                if (rr <= 64 || m == 64) {
                    qrows = rr < 8 ? 8 : rr;
                    break;
                }
            }
            if (g_force_general >= 8) qrows = g_force_general;
            a.rows_per_warp = qrows;
            const int strips_q = sxq * ((h + qrows - 1) / qrows);
            const int nblk = (strips_q + kQuadWarps - 1) / kQuadWarps;
            HB_LAUNCH("blur3x3_u16_quad", blur3x3_u16_quad_kernel<6>, nblk, 32 * kQuadWarps, 0, s, a, sxq, strips_q);
        } else {
            HB_LAUNCH("blur3x3_u16", blur3x3_u16_kernel, grid, 32 * kWarpsPerBlock, 0, s, a);
        }
    }
    if ((r = hb::check_cuda(cudaGetLastError(), "halide_blur launch", halide_error_code_device_run_failed))) return r;
    hb::mark_output_written(blur_y);
    return 0;
}

// Test hook: 1 = always take the general (any alignment) kernel, so both kernels stay covered by the parity tests;
// >= 8 = the aligned kernel with strips of that many rows.
extern "C" void halide_b200_blur_force_general(int enable) {
    g_force_general = enable;
}

HB_EXPORT_FILTER(halide_blur, kArgs)
