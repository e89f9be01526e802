// stencil_chain.cu — stencil_chain(input, output): 32 successive 5x5 uint16 stencils.
//
// Reference algorithm: apps/stencil_chain/stencil_chain_generator.cpp:16-34.  Stage s+1 at (x,y) is
//   e = u16(0); for i in -2..2 (x offset) for j in -2..2 (y offset): e += u16((i+3)*(j+3)) * stage_s(x+i, y+j)
// entirely in uint16, i.e. arithmetic in the ring Z/2^16.  Only the input is edge-clamped
// (repeat_edge, generator :18); later stages are pure functions evaluated on grown regions.
//
// Because Z/2^16 is a commutative ring the result does not depend on summation order, so the
// weights' outer-product structure (i+3)*(j+3) is exploited exactly: a vertical 5-tap pass with
// weights (j+3) followed by a horizontal 5-tap pass with weights (i+3), both reduced mod 2^16
// (10 multiply-adds per pixel per stage instead of 25).  Bit-exact by construction; the parity
// tests compare with the oracle's literal 25-tap source-order loop.
//
// Kernel shape: ALU/shared-memory bound (800 MAC/px in the reference formulation, 4 B/px of
// compulsory HBM traffic).  kFuse stages run per launch on a shared-memory tile with a 2*kFuse
// apron, ping-ponging between two uint16 tiles; the frame itself (7.9 MB at the harness size)
// stays L2-resident between launches.
#include "../../include/stencil_chain.h"
#include "../../include/stencil_chain_auto_schedule.h"
#include "hb_common.h"

namespace {

constexpr int kStages = 32;  // GeneratorParam `stencils` of the shipped app (generator :9)
constexpr int kFuse = 4;     // stages per launch
constexpr int kTile = 64;    // output tile edge per block
constexpr int kTileIn = kTile + 4 * kFuse;  // 80: input tile edge (2 px apron per fused stage, both sides)

struct Plane {
    const uint16_t *src;  // element (x0,y0) of the region this launch reads
    uint16_t *dst;        // element (x0+2f, y0+2f) of the region it writes
    int64_t src_sy, dst_sy;
    int src_w, src_h;     // extent of the source region
    // when reading the pipeline input: clamp coordinates into the buffer (repeat_edge)
    int clamp_x0, clamp_y0, clamp_w, clamp_h, do_clamp;
    int dst_w, dst_h;
    int fuse;             // stages in this launch (<= kFuse)
    int src_words, dst_words;  // rows of src / dst keep pixel pairs 4-byte aligned (even stride, aligned base): 32-bit accesses
};

__global__ void __launch_bounds__(256) stencil_chain_fused_kernel(Plane p) {
    __shared__ uint16_t A[kTileIn][kTileIn + 2];
    __shared__ uint16_t B[kTileIn][kTileIn + 2];
    __shared__ uint16_t C[kTileIn][kTileIn + 2];
    const int tid = threadIdx.x;
    const int ox = blockIdx.x * kTile, oy = blockIdx.y * kTile;  // tile origin in dst coordinates
    const int in_edge = kTile + 4 * p.fuse;
    // load the source tile: dst (ox,oy) corresponds to src (ox, oy) .. (ox+in_edge, oy+in_edge)
    for (int t = tid; t < in_edge * in_edge; t += 256) {
        int ly = t / in_edge, lx = t - ly * in_edge;
        int sx = ox + lx, sy = oy + ly;
        uint16_t v = 0;
        if (p.do_clamp) {
            // src points at absolute coordinate (src_x0, src_y0) folded into clamp_x0/y0 by the host:
            int cx = min(max(sx + p.clamp_x0, 0), p.clamp_w - 1);
            int cy = min(max(sy + p.clamp_y0, 0), p.clamp_h - 1);
            v = p.src[(int64_t)cy * p.src_sy + cx];
        } else if (sx < p.src_w && sy < p.src_h) {
            v = p.src[(int64_t)sy * p.src_sy + sx];
        }
        A[ly][lx] = v;
    }
    __syncthreads();
    int edge = in_edge;
    uint16_t(*cur)[kTileIn + 2] = A;
    uint16_t(*nxt)[kTileIn + 2] = B;
    for (int s = 0; s < p.fuse; s++) {
        // vertical pass: C[y][x] = sum_j (j+3) * cur[y+2+j][x], y in [0, edge-4)
        const int vh = edge - 4;
        for (int t = tid; t < vh * edge; t += 256) {
            int ly = t / edge, lx = t - ly * edge;
            uint32_t acc = 1u * cur[ly][lx] + 2u * cur[ly + 1][lx] + 3u * cur[ly + 2][lx] + 4u * cur[ly + 3][lx] +
                           5u * cur[ly + 4][lx];
            C[ly][lx] = (uint16_t)acc;
        }
        __syncthreads();
        // horizontal pass: nxt[y][x] = sum_i (i+3) * C[y][x+2+i], x in [0, edge-4)
        for (int t = tid; t < vh * vh; t += 256) {
            int ly = t / vh, lx = t - ly * vh;
            uint32_t acc = 1u * C[ly][lx] + 2u * C[ly][lx + 1] + 3u * C[ly][lx + 2] + 4u * C[ly][lx + 3] +
                           5u * C[ly][lx + 4];
            nxt[ly][lx] = (uint16_t)acc;
        }
        __syncthreads();
        edge -= 4;
        uint16_t(*tmp)[kTileIn + 2] = cur; cur = nxt; nxt = tmp;
    }
    // edge == kTile now
    for (int t = tid; t < kTile * kTile; t += 256) {
        int ly = t / kTile, lx = t - ly * kTile;
        int dx = ox + lx, dy = oy + ly;
        if (dx < p.dst_w && dy < p.dst_h) p.dst[(int64_t)dy * p.dst_sy + dx] = cur[ly][lx];
    }
}

// ---- register-window version (kFuse stages per launch, same tiles) -----------------------------------------------
// The kernel above spends ~135 instructions per pixel and stage: one pixel per thread and pass, five 16-bit shared
// loads per output and an integer division per element for the tile coordinates.  Here the tile lives in shared memory
// as 32-bit words (two pixels), every edge length is a compile-time constant, and each pass is a sliding window held
// in registers:
//   vertical:   a thread owns a column PAIR on a segment of rows — per row one 32-bit load, eight multiply-adds (four
//               per pixel: v0 + 2 v1 + 3 v2 + 4 v3 + 5 v4 starts from v0), one PRMT to repack, one 32-bit store;
//   horizontal: a thread owns a row on a segment of output pairs — per output pair one new word, eight multiply-adds.
// Sums are taken in 32 bits and truncated by the repack (Z/2^16 arithmetic: any order, any carries above bit 15).
// Row pitch = 41 words (odd): the 32 lanes of a warp — consecutive column pairs in the vertical pass, consecutive rows
// in the horizontal one — fall into 32 different banks.
constexpr int kPW = (kTileIn + 2) / 2;  // words per shared-memory row

template<int EDGE>
__device__ __forceinline__ void stencil_stage(const uint32_t *cur, uint32_t *mid, uint32_t *nxt, int tid) {
    constexpr int VH = EDGE - 4, NP = EDGE / 2;
    {   // vertical pass: mid[y][x] = sum_j (j+1) * cur[y+j][x], y in [0, VH), all EDGE columns
        constexpr int SEG = 256 / NP, LEN = (VH + SEG - 1) / SEG;
        const int sgi = tid / NP, pc = tid - sgi * NP;
        const int r0 = sgi * LEN, r1 = min(r0 + LEN, VH);
        if (sgi < SEG && r0 < r1) {
            const uint32_t *c = cur + r0 * kPW + pc;
            uint32_t w = c[0];
            uint32_t l0 = w & 0xffffu, h0 = w >> 16;
            w = c[kPW];
            uint32_t l1 = w & 0xffffu, h1 = w >> 16;
            w = c[2 * kPW];
            uint32_t l2 = w & 0xffffu, h2 = w >> 16;
            w = c[3 * kPW];
            uint32_t l3 = w & 0xffffu, h3 = w >> 16;
            uint32_t *o = mid + r0 * kPW + pc;
#pragma unroll 4
            for (int r = r0; r < r1; r++) {
                w = c[4 * kPW];
                const uint32_t l4 = w & 0xffffu, h4 = w >> 16;
                const uint32_t al = l0 + 2u * l1 + 3u * l2 + 4u * l3 + 5u * l4;
                const uint32_t ah = h0 + 2u * h1 + 3u * h2 + 4u * h3 + 5u * h4;
                *o = __byte_perm(al, ah, 0x5410);
                l0 = l1; l1 = l2; l2 = l3; l3 = l4;
                h0 = h1; h1 = h2; h2 = h3; h3 = h4;
                c += kPW;
                o += kPW;
            }
        }
    }
    __syncthreads();
    {   // horizontal pass: nxt[y][x] = sum_i (i+1) * mid[y][x+i], x in [0, VH), VH rows
        constexpr int SEG = 256 / VH, NOP = VH / 2, LEN = (NOP + SEG - 1) / SEG;
        const int sgi = tid / VH, r = tid - sgi * VH;
        const int k0 = sgi * LEN, k1 = min(k0 + LEN, NOP);
        if (sgi < SEG && k0 < k1) {
            const uint32_t *c = mid + r * kPW + k0;
            uint32_t w = c[0];
            uint32_t v0 = w & 0xffffu, v1 = w >> 16;
            w = c[1];
            uint32_t v2 = w & 0xffffu, v3 = w >> 16;
            uint32_t *o = nxt + r * kPW + k0;
#pragma unroll 4
            for (int k = k0; k < k1; k++) {
                w = c[2];
                const uint32_t v4 = w & 0xffffu, v5 = w >> 16;
                const uint32_t a0 = v0 + 2u * v1 + 3u * v2 + 4u * v3 + 5u * v4;
                const uint32_t a1 = v1 + 2u * v2 + 3u * v3 + 4u * v4 + 5u * v5;
                *o = __byte_perm(a0, a1, 0x5410);
                v0 = v2; v1 = v3; v2 = v4; v3 = v5;
                c++;
                o++;
            }
        }
    }
    __syncthreads();
}

template<int EDGE, int LEFT>
struct StencilStages {
    static __device__ __forceinline__ const uint32_t *run(uint32_t *cur, uint32_t *mid, uint32_t *nxt, int tid) {
        stencil_stage<EDGE>(cur, mid, nxt, tid);
        return StencilStages<EDGE - 4, LEFT - 1>::run(nxt, mid, cur, tid);
    }
};
template<int EDGE>
struct StencilStages<EDGE, 0> {
    static __device__ __forceinline__ const uint32_t *run(uint32_t *cur, uint32_t *, uint32_t *, int) { return cur; }
};

template<int FUSE>
__global__ void __launch_bounds__(256) stencil_chain_window_kernel(Plane p) {
    constexpr int IN = kTile + 4 * FUSE, INW = IN / 2;
    __shared__ uint32_t A[kTileIn * kPW];
    __shared__ uint32_t B[kTileIn * kPW];
    __shared__ uint32_t C[kTileIn * kPW];
    const int tid = threadIdx.x;
    const int ox = blockIdx.x * kTile, oy = blockIdx.y * kTile;  // tile origin in dst coordinates (even)
    // source tile: dst (ox, oy) needs src (ox .. ox + IN - 1, oy .. oy + IN - 1); elements outside the source region are
    // only ever combined into outputs outside the destination region, so they may hold anything (zeros here)
    for (int t = tid; t < IN * INW; t += 256) {
        const int ly = t / INW, lw = t - ly * INW;
        const int sx = ox + 2 * lw, sy = oy + ly;
        uint32_t w = 0;
        if (p.do_clamp) {
            const int cy = min(max(sy + p.clamp_y0, 0), p.clamp_h - 1);
            const int cx0 = min(max(sx + p.clamp_x0, 0), p.clamp_w - 1), cx1 = min(max(sx + 1 + p.clamp_x0, 0), p.clamp_w - 1);
            const uint16_t *row = p.src + (int64_t)cy * p.src_sy;
            w = (uint32_t)row[cx0] | ((uint32_t)row[cx1] << 16);
        } else if (sy < p.src_h) {
            const uint16_t *e = p.src + (int64_t)sy * p.src_sy + sx;
            if (p.src_words && sx + 1 < p.src_w) {
                w = *reinterpret_cast<const uint32_t *>(e);
            } else {
                if (sx < p.src_w) w = e[0];
                if (sx + 1 < p.src_w) w |= (uint32_t)e[1] << 16;
            }
        }
        A[ly * kPW + lw] = w;
    }
    __syncthreads();
    const uint32_t *res = StencilStages<IN, FUSE>::run(A, C, B, tid);
    // res holds the kTile x kTile result (kTile / 2 words per row)
    for (int t = tid; t < kTile * (kTile / 2); t += 256) {
        const int ly = t / (kTile / 2), lw = t - ly * (kTile / 2);
        const int dx = ox + 2 * lw, dy = oy + ly;
        if (dy >= p.dst_h || dx >= p.dst_w) continue;
        const uint32_t w = res[ly * kPW + lw];
        uint16_t *e = p.dst + (int64_t)dy * p.dst_sy + dx;
        if (p.dst_words && dx + 1 < p.dst_w) {
            *reinterpret_cast<uint32_t *>(e) = w;
        } else {
            e[0] = (uint16_t)w;
            if (dx + 1 < p.dst_w) e[1] = (uint16_t)(w >> 16);
        }
    }
}

constexpr bool kDefaultWindow = true;  // (the register-window kernel: bit-identical to the first kernel on hardware, profiles/r02_ab_variants.log)
int g_variant = 0;  // test / A-B hook (halide_b200_stencil_chain_variant): 0 = default, 1 = one-pixel-per-thread kernel, 2 = register-window kernel

const hb::BufferEstimates est({0, 1536, 0, 2560});
const halide_filter_argument_t kArgs[2] = {
    {"input", halide_argument_kind_input_buffer, 2, {halide_type_uint, 16, 0}, nullptr, nullptr, nullptr, nullptr, est.p},
    {"output", halide_argument_kind_output_buffer, 2, {halide_type_uint, 16, 0}, nullptr, nullptr, nullptr, nullptr, est.p},
};
const auto &kIn = kArgs[0], &kOut = kArgs[1];

}  // namespace

extern "C" void halide_b200_stencil_chain_variant(int v) {
    g_variant = v;
}

extern "C" int stencil_chain(halide_buffer_t *input, halide_buffer_t *output) {
    int r;
    if ((r = hb::check_arg(input, kIn))) return r;
    if ((r = hb::check_arg(output, kOut))) return r;
    bool query = false;
    {
        // every access to the input goes through repeat_edge: nothing beyond a non-empty buffer is
        // required; a query is answered with the output region.
        int mins[2] = {output->dim[0].min, output->dim[1].min};
        int ext[2] = {output->dim[0].extent, output->dim[1].extent};
        if (hb::is_bounds_query(input)) { hb::propose_shape(input, mins, ext); query = true; }
        if (hb::is_bounds_query(output)) { hb::propose_shape(output, mins, ext); query = true; }
    }
    if (query) return 0;
    if ((r = hb::check_shape(input, kIn))) return r;
    if ((r = hb::check_shape(output, kOut))) return r;
    const int W = output->dim[0].extent, H = output->dim[1].extent;
    if (W <= 0 || H <= 0) return 0;
    if (input->dim[0].extent <= 0 || input->dim[1].extent <= 0) {
        return hb::fail(halide_error_code_access_out_of_bounds, "Input buffer input is empty");
    }
    void *din = nullptr, *dout = nullptr;
    if ((r = hb::acquire_input(input, kIn, &din))) return r;
    if ((r = hb::acquire_output(output, kOut, &dout))) return r;

    // ping-pong buffers for the intermediate stages on their grown regions
    const int groups = (kStages + kFuse - 1) / kFuse;
    const int maxR = 2 * (kStages - kFuse);
    hb::Scratch scratch;
    const int64_t bw = (W + 2 * maxR + 1) & ~(int64_t)1, bh = H + 2 * maxR;  // (even pitch: intermediate rows keep pixel pairs word-aligned)
    uint16_t *buf[2] = {nullptr, nullptr};
    if (groups > 1) {
        buf[0] = scratch.get<uint16_t>((size_t)bw * bh);
        buf[1] = groups > 2 ? scratch.get<uint16_t>((size_t)bw * bh) : buf[0];
        if (!buf[0] || !buf[1]) return hb::fail(halide_error_code_device_malloc_failed, "stencil_chain: scratch allocation failed");
    }
    cudaStream_t s = hb::stream();
    {
        hb::CallTimer timer(s);
        int done = 0;
        for (int g = 0; g < groups; g++) {
            const int fuse = (kStages - done) < kFuse ? (kStages - done) : kFuse;
            const int Rin = 2 * (kStages - done);           // apron of the region this launch reads
            const int Rout = Rin - 2 * fuse;                // apron of the region it writes
            Plane p;
            p.fuse = fuse;
            p.dst_w = W + 2 * Rout;
            p.dst_h = H + 2 * Rout;
            p.src_w = W + 2 * Rin;
            p.src_h = H + 2 * Rin;
            if (g == 0) {
                p.src = (const uint16_t *)din;
                p.src_sy = input->dim[1].stride;
                p.do_clamp = 1;
                // source-region local (0,0) is absolute (ox - Rin, oy - Rin); buffer-relative = minus input min
                p.clamp_x0 = output->dim[0].min - Rin - input->dim[0].min;
                p.clamp_y0 = output->dim[1].min - Rin - input->dim[1].min;
                p.clamp_w = input->dim[0].extent;
                p.clamp_h = input->dim[1].extent;
            } else {
                p.src = buf[(g - 1) & 1];
                p.src_sy = bw;
                p.do_clamp = 0;
                p.clamp_x0 = p.clamp_y0 = p.clamp_w = p.clamp_h = 0;
            }
            if (g == groups - 1) {
                p.dst = (uint16_t *)dout;
                p.dst_sy = output->dim[1].stride;
            } else {
                p.dst = buf[g & 1];
                p.dst_sy = bw;
            }
            p.src_words = ((reinterpret_cast<uintptr_t>(p.src) & 3) == 0 && (p.src_sy & 1) == 0) ? 1 : 0;
            p.dst_words = ((reinterpret_cast<uintptr_t>(p.dst) & 3) == 0 && (p.dst_sy & 1) == 0) ? 1 : 0;
            dim3 grid((p.dst_w + kTile - 1) / kTile, (p.dst_h + kTile - 1) / kTile);
            const bool window = fuse == kFuse && (g_variant == 2 || (g_variant == 0 && kDefaultWindow));
            if (window) {
                HB_LAUNCH("stencil_chain_window", stencil_chain_window_kernel<kFuse>, grid, 256, 0, s, p);
            } else {
                HB_LAUNCH("stencil_chain_fused", stencil_chain_fused_kernel, grid, 256, 0, s, p);
            }
            done += fuse;
        }
    }
    if ((r = hb::check_cuda(cudaGetLastError(), "stencil_chain launch", halide_error_code_device_run_failed))) return r;
    hb::mark_output_written(output);
    return 0;
}

HB_EXPORT_FILTER(stencil_chain, kArgs)
HB_EXPORT_AUTO_SCHEDULE(stencil_chain, kArgs)
