// local_laplacian.cu — host side of local_laplacian(input, levels, alpha, beta, output) for sm_100a:
// the C-ABI entry points (reference: apps/local_laplacian/local_laplacian_generator.cpp:12-16,287 and
// the harness apps/local_laplacian/process.cpp:31), argument validation, pyramid geometry, scratch
// allocation, the launch sequence, and the row-sharded multi-GPU variant.  Kernels: ll_kernels.cuh.
//
// Data layout in HBM (all f32, callee-owned scratch):
//   lut      [2*256*(levels-1)+1]            remap(i), i in [-256(levels-1), 256(levels-1)]
//   gp[j]    [sy_j][gpitch_j][K]  j=1..J-1   gPyramid[j], the K=levels planes interleaved per
//                                            pixel (K=8 -> one 32-byte sector per pixel, so the
//                                            data-dependent (li, li+1) plane pick costs one sector)
//   ing[j]   [sy_j][gpitch_j]     j=1..J-1   inGPyramid[j]
//   outg[j]  [oy_j][opitch_j]     j=1..J-1   outGPyramid[j]
// gray / gPyramid[0] / lPyramid / outLPyramid / outGPyramid[0] are never materialised: they are
// recomputed from the uint16 input where needed (8 f32 planes at full resolution would be
// 32 B/px of traffic against 12 B/px of compulsory I/O).
#include <stdlib.h>
#include <string.h>

#include <map>
#include <mutex>
#include <vector>

#include "hb_dist.h"
#include "ll_kernels.cuh"

namespace {

using namespace llk;

int g_shard_coarse_level = 0;  // halide_b200_ll_shard_coarse_level: 0 = choose by size, n >= 2 = gather level n
int g_force_naive = 0;  // test hook bitmask (halide_b200_ll_force_generic): 1 = generic down kernels, 2 = generic up, 4 = generic final, 8 = no fused coarse launch, 16 = general-layout final kernel, 64 = no TMA frame tile in the final kernel, 256 = 48-row tiles in the TMA final kernel (default 32; 128 = 32 rows explicitly)

const hb::ArgSpec kIn = {"input", halide_type_uint, 16, 3, false};
const hb::ArgSpec kOut = {"output", halide_type_uint, 16, 3, true};

int64_t est_i[3][2] = {{0, 1536}, {0, 2560}, {0, 3}};
const int64_t *const est_ptrs[6] = {&est_i[0][0], &est_i[0][1], &est_i[1][0], &est_i[1][1], &est_i[2][0], &est_i[2][1]};
halide_scalar_value_t sv_levels, sv_alpha, sv_beta;
struct InitScalars {
    InitScalars() {
        sv_levels.u.i64 = 0; sv_levels.u.i32 = 8;
        sv_alpha.u.i64 = 0; sv_alpha.u.f32 = 1.0f;
        sv_beta.u.i64 = 0; sv_beta.u.f32 = 1.0f;
    }
} init_scalars;
// Argument records as the generator declares them (generator :12-16, estimates :92-99).
const halide_filter_argument_t kArgs[5] = {
    {"input", halide_argument_kind_input_buffer, 3, {halide_type_uint, 16, 0}, nullptr, nullptr, nullptr, nullptr, est_ptrs},
    {"levels", halide_argument_kind_input_scalar, 0, {halide_type_int, 32, 0}, nullptr, nullptr, nullptr, &sv_levels, nullptr},
    {"alpha", halide_argument_kind_input_scalar, 0, {halide_type_float, 32, 0}, nullptr, nullptr, nullptr, &sv_alpha, nullptr},
    {"beta", halide_argument_kind_input_scalar, 0, {halide_type_float, 32, 0}, nullptr, nullptr, nullptr, &sv_beta, nullptr},
    {"output", halide_argument_kind_output_buffer, 3, {halide_type_uint, 16, 0}, nullptr, nullptr, nullptr, nullptr, est_ptrs},
};
const halide_filter_metadata_t kMeta = {1, 5, kArgs, "x86-64-linux-cuda-cuda_capability_100-b200_native", "local_laplacian"};
const halide_filter_metadata_t kMetaAuto = {1, 5, kArgs, "x86-64-linux-cuda-cuda_capability_100-b200_native",
                                            "local_laplacian_auto_schedule"};


// Everything one call needs on the device: frame description + per-level buffers.
struct Plan {
    LLFrame f;
    LevelSet ls;
    ll::Geom geom;
    int J, K;
    float alpha;
    float *lut;
};

int check_and_query(halide_buffer_t *input, int levels, halide_buffer_t *output, bool *done) {
    int r;
    *done = true;
    if ((r = hb::check_arg(input, kIn))) return r;
    if ((r = hb::check_arg(output, kOut))) return r;
    // Bounds query: the only access that bypasses repeat_edge is input(x,y,c) in `color`
    // (generator :84), so the input must cover exactly the output region.
    bool query = false;
    {
        int mins[3] = {output->dim[0].min, output->dim[1].min, output->dim[2].min};
        int ext[3] = {output->dim[0].extent, output->dim[1].extent, output->dim[2].extent};
        if (hb::is_bounds_query(input)) {
            hb::propose_shape(input, mins, ext);
            query = true;
        }
        if (hb::is_bounds_query(output)) {
            hb::propose_shape(output, mins, ext);
            query = true;
        }
    }
    if (query) return 0;
    if ((r = hb::check_shape(input, kIn))) return r;
    if ((r = hb::check_shape(output, kOut))) return r;
    for (int d = 0; d < 3; d++) {
        if ((r = hb::check_covers(input, kIn, d, output->dim[d].min, output->dim[d].extent))) return r;
    }
    if (levels < 2 || levels > 32) {
        // 1/(levels-1) (generator :41) is meaningless below 2; the reference does not check, we do.
        return hb::fail(levels < 2 ? halide_error_code_param_too_small : halide_error_code_param_too_large,
                        "Parameter levels is %d but must be in [2, 32]", levels);
    }
    if (output->dim[0].extent <= 0 || output->dim[1].extent <= 0 || output->dim[2].extent <= 0) return 0;
    *done = false;
    return 0;
}

void fill_frame(Plan &p, halide_buffer_t *input, halide_buffer_t *output, void *din, void *dout, int levels, float alpha,
                float beta) {
    LLFrame &f = p.f;
    f.in = (const uint16_t *)din;
    f.in_sy = input->dim[1].stride; f.in_sc = input->dim[2].stride;
    f.in_x0 = input->dim[0].min; f.in_y0 = input->dim[1].min; f.in_c0 = input->dim[2].min;
    f.in_w = input->dim[0].extent; f.in_h = input->dim[1].extent; f.in_c = input->dim[2].extent;
    f.clamp_y0 = f.in_y0; f.clamp_h = f.in_h;
    f.halo_top = f.halo_bot = nullptr;
    f.halo_top_rows = f.halo_bot_rows = f.halo_pitch = 0;
    f.out = (uint16_t *)dout;
    f.out_sy = output->dim[1].stride; f.out_sc = output->dim[2].stride;
    f.out_x0 = output->dim[0].min; f.out_y0 = output->dim[1].min; f.out_c0 = output->dim[2].min;
    f.W = output->dim[0].extent; f.H = output->dim[1].extent; f.C = output->dim[2].extent;
    f.row0 = f.out_y0; f.nrows = f.H;
    f.levels = levels;
    f.beta = beta;
    f.flm1 = (float)(levels - 1);
    f.inv_lm1 = 1.0f / (float)(levels - 1);
    f.lut_half = 256 * (levels - 1);
    p.K = levels;
    p.J = ll::kMaxJ;
    p.alpha = alpha;
}

// ---- remap table: recomputed only when (levels, alpha) change --------------------------------------------------
// alpha is a runtime scalar, but a caller (the harness's benchmark loop, a video stream) passes the same value call
// after call: the 2*256*(levels-1)+1 halide_exp evaluations and their launch are kept per device and reused.  The table
// is immutable once built (a change of parameters builds a new one; the old ones are kept: kernels of an earlier call
// may still be reading them on another stream), and it is built synchronously, so any stream may read it afterwards.
struct LutEntry {
    int device, levels;
    float alpha;
    float *lut;
};
std::mutex g_lut_mu;
std::vector<LutEntry> g_luts;

int get_lut(Plan &p, cudaStream_t s) {
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lock(g_lut_mu);
    for (const LutEntry &e : g_luts) {
        if (e.device == dev && e.levels == p.f.levels && memcmp(&e.alpha, &p.alpha, sizeof(float)) == 0) {
            p.lut = e.lut;
            p.f.lut = e.lut;
            return 0;
        }
    }
    if (g_luts.size() >= 64) {  // a caller sweeping alpha: drop the oldest tables once nothing can still be reading them
        cudaDeviceSynchronize();
        for (const LutEntry &e : g_luts) cudaFree(e.lut);
        g_luts.clear();
    }
    float *lut = nullptr;
    const int n = 2 * p.f.lut_half + 1;
    if (cudaMalloc((void **)&lut, ((size_t)n + 3) / 4 * 16) != cudaSuccess) {
        cudaGetLastError();
        return hb::fail(halide_error_code_device_malloc_failed, "local_laplacian: remap table allocation failed");
    }
    hb::debug_fill(lut, ((size_t)n + 3) / 4 * 16, s);
    HB_LAUNCH("ll_lut", ll_lut_kernel, (n + 255) / 256, 256, 0, s, lut, p.f.lut_half, p.alpha);
    if (cudaStreamSynchronize(s) != cudaSuccess) {
        cudaGetLastError();
        cudaFree(lut);
        return hb::fail(halide_error_code_device_run_failed, "local_laplacian: remap table kernel failed");
    }
    g_luts.push_back({dev, p.f.levels, p.alpha, lut});
    p.lut = lut;
    p.f.lut = lut;
    return 0;
}

int alloc_levels(Plan &p, hb::Scratch &scratch) {
    const int nq = (p.K + 1) / 2;
    for (int j = 1; j < p.J; j++) {
        const ll::Level &lv = p.geom.lv[j];
        LevelBuf &b = p.ls.lv[j];
        b.sx = lv.sx; b.sy = lv.sy; b.ox = lv.ox; b.oy = lv.oy;
        b.cy = lv.cy; b.coy = lv.coy; b.gy = lv.gy;
        b.xo = lv.xo; b.nq = nq;
        b.gpitch = lv.gpitch; b.opitch = lv.opitch;
        b.has_pair = 0;
        size_t gpix = (size_t)lv.sy.n() * lv.gpitch;
        b.gp = scratch.get<float>(gpix * nq * 2);
        b.ing = scratch.get<float>(gpix);
        b.pair = p.K == 8 ? scratch.get<float>(gpix * 2) : b.ing;
        b.outg = scratch.get<float>((size_t)lv.oy.n() * lv.opitch);
        if (!b.gp || !b.ing || !b.pair || !b.outg) {
            return hb::fail(halide_error_code_device_malloc_failed, "local_laplacian: scratch allocation failed");
        }
    }
    p.ls.lv[0] = p.ls.lv[1];  // level 0 is never stored; keep the slot initialised
    return 0;
}

// ---- launch helpers ------------------------------------------------------------------------------------
const dim3 kBlk(32, 8);
dim3 grid_for(int w, int h) { return dim3((w + 31) / 32, (h + 7) / 8); }

// Resident block slots of a kernel on the current device.  The driver queries behind it (function attribute,
// occupancy) cost several microseconds each — at eight ranks a whole frame is ~0.8 ms of GPU time and ~17 launches — so
// the answer is cached per (kernel, device, shared-memory size); a process may drive several devices.
struct SlotKey {
    const void *kern;
    int dev;
    size_t smem;
    bool operator<(const SlotKey &o) const {
        return kern != o.kern ? kern < o.kern : (dev != o.dev ? dev < o.dev : smem < o.smem);
    }
};
std::mutex g_slots_mu;
std::map<SlotKey, int> g_slots;

template<typename Kern>
int resident_slots(Kern kern, int threads, size_t smem) {
    int dev = 0;
    cudaGetDevice(&dev);
    const SlotKey key = {(const void *)kern, dev, smem};
    std::lock_guard<std::mutex> lock(g_slots_mu);
    auto it = g_slots.find(key);
    if (it != g_slots.end()) return it->second;
    int sms = 148, per_sm = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (smem > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem) != cudaSuccess || per_sm < 1) {
        cudaGetLastError();
        per_sm = 1;
    }
    return g_slots[key] = sms * per_sm;
}

template<bool BETA1>
void launch_level1(Plan &p, cudaStream_t s) {
    LevelBuf *lb = p.ls.lv;
    const LLFrame &f = p.f;
    const size_t smem = kPairLutN * sizeof(float2) + kDWarps * sizeof(DownStage);
    // (the attribute and the occupancy are per device and cheap to query; no process-wide caching)
    const int slots = resident_slots(ll_level1_kernel<BETA1>, kDWarps * 32, smem);
    const int ns = (lb[1].sx.n() + kDCols - 1) / kDCols, nc = (lb[1].cy.n() + kDR - 1) / kDR;
    const long long units = (long long)ns * nc;
    // one block per resident slot, but never fewer than ~2 units per warp's worth of work per block
    long long g = (units + 1) / 2;
    if (g > slots) g = slots;
    if (g < 1) g = 1;
    // aligned 32-bit loads of a column pair / 32-bit element offsets from the buffer's first element
    const int wide = ((uintptr_t)f.in & 3) == 0 && (f.in_sy & 1) == 0 && (f.in_sc & 1) == 0 && (f.in_x0 & 1) == 0 &&
                     ((uintptr_t)f.halo_top & 3) == 0 && ((uintptr_t)f.halo_bot & 3) == 0 && (f.halo_pitch & 1) == 0;
    const int idx32 = f.in_sy > 0 && f.in_sc > 0 && (int64_t)f.in_h * f.in_sy + (int64_t)f.in_c * f.in_sc < (1ll << 31);
    HB_LAUNCH("ll_level1", (ll_level1_kernel<BETA1>), (int)g, kDWarps * 32, smem, s, p.f, lb[1], ns, nc, wide, idx32);
    lb[1].has_pair = 1;
}

void launch_down(Plan &p, int j, cudaStream_t s) {  // produce level j (j >= 1) rows cy
    LevelBuf *lb = p.ls.lv;
    if (lb[j].cy.n() <= 0) return;
    const bool fast = (p.K == 8) && !(g_force_naive & 1);
    if (fast) {
        const bool beta1 = p.f.beta == 1.0f;
        if (j == 1) {
            if (beta1) launch_level1<true>(p, s);
            else launch_level1<false>(p, s);
        } else {
            // stored levels: load-bound row-group kernel; no pair plane (the up-sweep of these small levels picks its two
            // planes out of the level itself)
            const int ns = (lb[j].sx.n() + kDCols - 1) / kDCols, ng = (lb[j].cy.n() + kRG - 1) / kRG;
            const long long tasks = (long long)ns * ng * 5;
            const int slots = resident_slots(ll_down_rows_kernel, 256, 0);
            long long g = (tasks + 7) / 8;
            if (g > slots) g = slots;
            HB_LAUNCH("ll_down_rows", ll_down_rows_kernel, (int)g, 256, 0, s, lb[j - 1], lb[j], ns, ng);
        }
    } else if (j == 1) {
        HB_LAUNCH("ll_level1_generic", ll_level1_naive_kernel, grid_for(lb[1].sx.n(), lb[1].cy.n()), kBlk, 0, s, p.f, lb[1]);
    } else {
        HB_LAUNCH("ll_down", ll_down_naive_kernel, grid_for(lb[j].sx.n(), lb[j].cy.n()), kBlk, 0, s, lb[j - 1], lb[j], p.K);
    }
}

dim3 up_grid(int x_lo, int x_hi, int y_lo, int y_hi, int th = kUpTH) {  // tiles on even absolute origins
    return dim3((x_hi - (x_lo & ~1) + kUpTW) / kUpTW, (y_hi - (y_lo & ~1) + th) / th);
}

void launch_up(Plan &p, int j, cudaStream_t s) {  // produce outGPyramid[j] (1 <= j <= J-1) rows coy
    LevelBuf *lb = p.ls.lv;
    if (lb[j].coy.n() <= 0) return;
    const bool fast_up = (p.K == 8) && !(g_force_naive & 2);
    if (fast_up && j < p.J - 1) {
        static const CUtensorMap no_map = {};
        HB_LAUNCH("ll_up2", (ll_up2_kernel<false, false, true>), up_grid(lb[j].ox.lo, lb[j].ox.hi, lb[j].coy.lo, lb[j].coy.hi), 256,
                  up2_smem_bytes(false, false), s, p.f, lb[j], lb[j + 1], no_map);
    } else {
        HB_LAUNCH("ll_up", ll_up_naive_kernel, grid_for(lb[j].ox.n(), lb[j].coy.n()), kBlk, 0, s, lb[j],
                  lb[j == p.J - 1 ? j : j + 1], p.f.flm1, p.f.levels, j == p.J - 1 ? 1 : 0);
    }
}

void launch_final(Plan &p, cudaStream_t s) {
    LevelBuf *lb = p.ls.lv;
    if (p.f.nrows <= 0) return;
    if (p.J > 1 && p.K == 8 && !(g_force_naive & 4) && p.f.C <= 3) {
        const LLFrame &f = p.f;
        // 48-row tiles (hook bit 256) were measured SLOWER than 32-row tiles although they spread the per-block fixed work
        // over 6 rows per thread instead of 4 (16K: 1.63 vs 1.52 ms, 4K: 61.9 vs 57.8 us): the kernel wants the fourth block
        // per SM more than it wants fewer instructions.  Kept selectable for A/B runs (tools/ab_masks.py) and tested.
        const bool tall = (g_force_naive & 256) && !(g_force_naive & 128);
        const int th = tall ? kUpTHTall : kUpTH;
        // the common layout takes the kernel's ALIGNED path (32-bit addressing, one aligned word per thread and channel)
        const int64_t in_span = (int64_t)f.in_h * f.in_sy + 3 * f.in_sc, out_span = (int64_t)f.H * f.out_sy + 3 * f.out_sc;
        const bool aligned = f.C == 3 && f.in_c0 == 0 && f.out_c0 == 0 && f.in_c >= 3 && (f.W & 1) == 0 && (f.out_x0 & 1) == 0 &&
                             (f.in_x0 & 1) == 0 && ((uintptr_t)f.in & 3) == 0 && ((uintptr_t)f.out & 3) == 0 &&
                             (f.in_sy & 1) == 0 && (f.in_sc & 1) == 0 && (f.out_sy & 1) == 0 && (f.out_sc & 1) == 0 &&
                             f.in_sy > 0 && f.in_sc > 0 && f.out_sy > 0 && f.out_sc > 0 && in_span < (1ll << 31) &&
                             out_span < (1ll << 31) && !(g_force_naive & 16);
        const bool beta1 = f.beta == 1.0f;
        // frame tile by TMA when the buffer meets TMA's rules (16-byte aligned base and strides); the map describes the
        // input buffer itself (x, y, c), so a tile reaching past it reads zeros for pixels that are never stored
        CUtensorMap in_map = {};
        bool use_tma = false;
        if (aligned && !(g_force_naive & 64)) {
            const int64_t strides[2] = {f.in_sy * 2, f.in_sc * 2};
            // (every tile's first column must also start on a 16-byte boundary: crops at other even offsets take the load path)
            if (tma::strides_ok(f.in, strides, 2) && (((f.out_x0 & ~1) - f.in_x0) & 7) == 0) {
                const uint64_t dims[3] = {(uint64_t)f.in_w, (uint64_t)f.in_h, (uint64_t)f.in_c};
                const uint32_t box[3] = {kUpInW, (uint32_t)th, 3};
                use_tma = tma::encode(&in_map, CU_TENSOR_MAP_DATA_TYPE_UINT16, 3, (void *)f.in, dims, strides, box);
            }
        }
        auto launch = [&](auto kern, bool tma_on, int tile_h = kUpTH) {
            const int smem = up2_smem_bytes(true, tma_on, tile_h);
            const dim3 g = up_grid(f.out_x0, f.out_x0 + f.W - 1, f.row0, f.row0 + f.nrows - 1, tile_h);
            (void)resident_slots(kern, 256, smem);  // (sets the > 48 KB shared-memory attribute once per kernel and device)
            HB_LAUNCH("ll_final2", kern, g, 256, smem, s, p.f, lb[1], lb[1], in_map);
        };
        if (use_tma && beta1 && tall) launch((ll_up2_kernel<true, true, true, true, kUpTHTall>), true, kUpTHTall);
        else if (use_tma && tall) launch((ll_up2_kernel<true, true, false, true, kUpTHTall>), true, kUpTHTall);
        else if (use_tma && beta1) launch(ll_up2_kernel<true, true, true, true>, true);
        else if (use_tma) launch(ll_up2_kernel<true, true, false, true>, true);
        else if (aligned && beta1) launch(ll_up2_kernel<true, true, true, false>, false);
        else if (aligned) launch(ll_up2_kernel<true, true, false, false>, false);
        else if (beta1) launch(ll_up2_kernel<true, false, true, false>, false);
        else launch(ll_up2_kernel<true, false, false, false>, false);
    } else {
        HB_LAUNCH("ll_final", ll_final_naive_kernel, grid_for(p.f.W, p.f.nrows), kBlk, 0, s, p.f, lb[1], p.J > 1 ? 1 : 0);
    }
}

// Coarse tail in one cooperative launch: levels j0+1 .. J-1 down and up (see ll_coarse_fused_kernel).
bool launch_coarse_fused(Plan &p, int j0, cudaStream_t s) {
    int dev = 0, coop = 0;
    cudaGetDevice(&dev);
    static std::map<int, int> coop_ok;  // per device (guarded by g_slots_mu)
    {
        std::lock_guard<std::mutex> lock(g_slots_mu);
        auto it = coop_ok.find(dev);
        if (it == coop_ok.end()) {
            cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
            coop_ok[dev] = coop;
        } else {
            coop = it->second;
        }
    }
    const int slots = resident_slots(ll_coarse_fused_kernel, 256, 0);  // sms * blocks per SM
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int max_blocks = coop ? (slots > 2 * sms ? 2 * sms : slots) : 0;
    if (max_blocks <= 0) return false;
    int J = p.J, K = p.K, levels = p.f.levels;
    float flm1 = p.f.flm1;
    void *args[] = {&p.ls, &J, &j0, &K, &flm1, &levels};
    hb::count_launch("ll_coarse_fused", s);
    cudaError_t e = cudaLaunchCooperativeKernel((void *)ll_coarse_fused_kernel, dim3(max_blocks), dim3(256), args, 0, s);
    hb::after_launch(s);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return true;
}

// Levels from_level+1 .. J-1 down, then J-1 .. from_level+1 up: the part of the sweep that runs on whole levels
// (everything on one GPU; the replicated coarse levels when row-sharded).  Small levels share one cooperative launch.
// (Tried and dropped: the levels of <= 12 K pixels as one 8-CTA thread-block cluster with hardware cluster barriers
// instead of grid barriers — 41 us against 35 us for the cooperative kernel at 4K: eight SMs' worth of threads cannot
// cover the L2 latency of these phases, the barriers were not the cost.)
void run_coarse_sweep(Plan &p, int from_level, cudaStream_t s) {
    int j0 = p.J - 1;
    if (!(g_force_naive & 8)) {
        // (level 1 always has its own launch: it is built from the frame, not from a stored level)
        const int j_min = from_level < 1 ? 1 : from_level;
        while (j0 > j_min && (int64_t)p.ls.lv[j0].sx.n() * p.ls.lv[j0].sy.n() <= 40 * 1024) j0--;
    }
    // j0 = last level produced by its own launch; levels j0+1.. are fused (if any)
    bool fused = false;
    for (int j = from_level + 1; j <= j0; j++) launch_down(p, j, s);
    if (j0 < p.J - 1) fused = launch_coarse_fused(p, j0, s);
    if (!fused) {
        for (int j = j0 + 1; j < p.J; j++) launch_down(p, j, s);
        for (int j = p.J - 1; j > j0; j--) launch_up(p, j, s);
    }
    for (int j = j0; j > from_level; j--) launch_up(p, j, s);
}

int run_local_laplacian(halide_buffer_t *input, int levels, float alpha, float beta, halide_buffer_t *output) {
    int r;
    bool done;
    if ((r = check_and_query(input, levels, output, &done)) || done) return r;
    void *din = nullptr, *dout = nullptr;
    if ((r = hb::acquire_input(input, kIn, &din))) return r;
    if ((r = hb::acquire_output(output, kOut, &dout))) return r;

    Plan p;
    fill_frame(p, input, output, din, dout, levels, alpha, beta);
    const int W = p.f.W, H = p.f.H;
    Span outx = {p.f.out_x0, p.f.out_x0 + W - 1}, outy = {p.f.out_y0, p.f.out_y0 + H - 1};
    Span inx = {p.f.in_x0, p.f.in_x0 + p.f.in_w - 1}, iny = {p.f.in_y0, p.f.in_y0 + p.f.in_h - 1};
    p.geom = ll::make_geom(outx, outy, inx, iny, p.J);
    hb::Scratch scratch;
    if ((r = alloc_levels(p, scratch))) return r;

    cudaStream_t s = hb::stream();
    if ((r = get_lut(p, s))) return r;
    {
        hb::CallTimer timer(s);
        run_coarse_sweep(p, 0, s);
        launch_final(p, s);
    }
    if ((r = hb::check_cuda(cudaGetLastError(), "local_laplacian launch", halide_error_code_device_run_failed))) return r;
    hb::mark_output_written(output);
    return 0;
}

// Row-sharded path: the level gathered all-to-all (levels from it upwards are replicated on every rank).
// Depends only on the whole frame's geometry and the rank count, so every rank computes the same value.
int choose_coarse_level(const ll::Geom &whole, int nranks, int J, int K) {
    if (g_shard_coarse_level > 0) return g_shard_coarse_level < 2 ? 2 : (g_shard_coarse_level > J - 1 ? J - 1 : g_shard_coarse_level);
    // The gathered level trades the two messages of a call against each other: gathering a finer level means a bigger
    // all-to-all (a rank receives (N-1)/N of the level: gPyramid + inGPyramid, (K + 1) floats per pixel) but a smaller
    // input halo (about 3 * 2^j frame rows of three uint16 channels per rank, which also is the recomputed work).  Pick the
    // level with the fewest bytes received per rank; ties go to the finer level (less recompute).  Measured on 4 x B200,
    // 16K frame: level 6 cost 65 + 55 us of NCCL time per frame, the 18.6 MB input halo alone being bandwidth-bound.
    const double frame_row_bytes = (double)whole.lv[0].sx.n() * 3 * sizeof(uint16_t);
    int best = J - 1;
    double best_bytes = 1e300;
    for (int j = 2; j < J; j++) {
        const double halo = 3.0 * (double)(1 << j) * frame_row_bytes;
        const double level = (double)whole.lv[j].sy.n() * whole.lv[j].gpitch * (K + 1) * sizeof(float);
        const double bytes = halo + level * (nranks - 1) / (nranks > 0 ? nranks : 1);
        if (bytes < best_bytes) {
            best_bytes = bytes;
            best = j;
        }
    }
    return best;
}

// ---- row-sharded variant (one process per GPU) -----------------------------------------------------------
// `input`/`output` describe this rank's band: all columns and channels of the frame, rows
// [dim[1].min, dim[1].min + extent) in the frame's coordinates.  frame_y_min/extent give the rows of the whole
// frame; ranks must be ordered top to bottom (rank r-1 holds the rows directly above rank r's).
// Communication per call (SURVEY.md §8e, see ll_geom.h): ONE exchange of input halo rows with the two neighbours
// (the only place the stencil footprint of the sharded levels crosses the shard boundary — every pyramid row a band
// needs beyond itself is recomputed from them) and ONE all-to-all gather of the coarse level jr; both are NCCL
// point-to-point groups on the compute stream.  Everything else is the single-GPU kernels on this rank's rows.
struct ShardPlan {  // per geometry: every rank's band (gathered once), reused call after call
    int key[10];
    bool valid = false;
    std::vector<int> bands;  // [lo, hi] per rank
};
ShardPlan g_shard;

int run_local_laplacian_sharded(halide_buffer_t *input, int levels, float alpha, float beta, halide_buffer_t *output,
                                int frame_y_min, int frame_y_extent) {
    int r;
    bool done;
    if ((r = check_and_query(input, levels, output, &done)) || done) return r;
    if (!hbdist::active()) {
        return hb::fail(halide_error_code_generic_error, "local_laplacian_sharded: call halide_b200_dist_init first");
    }
    const int rank = hbdist::rank(), nranks = hbdist::size();
    Span band = {output->dim[1].min, output->dim[1].min + output->dim[1].extent - 1};
    if (input->dim[1].min != band.lo || input->dim[1].extent != band.n()) {
        return hb::fail(halide_error_code_constraint_violated,
                        "local_laplacian_sharded: input rows [%d,%d) must equal the output band [%d,%d)", input->dim[1].min,
                        input->dim[1].min + input->dim[1].extent, band.lo, band.hi + 1);
    }
    const bool first = rank == 0, last = rank == nranks - 1;
    Span frame_y = {frame_y_min, frame_y_min + frame_y_extent - 1};
    if ((first && band.lo != frame_y.lo) || (last && band.hi != frame_y.hi) || band.lo < frame_y.lo || band.hi > frame_y.hi) {
        return hb::fail(halide_error_code_constraint_violated, "local_laplacian_sharded: band [%d,%d] inconsistent with frame rows [%d,%d] on rank %d/%d",
                        band.lo, band.hi, frame_y.lo, frame_y.hi, rank, nranks);
    }
    if (input->dim[0].min != output->dim[0].min || input->dim[0].extent != output->dim[0].extent) {
        return hb::fail(halide_error_code_constraint_violated, "local_laplacian_sharded: input and output bands must span the same columns");
    }
    void *din = nullptr, *dout = nullptr;
    if ((r = hb::acquire_input(input, kIn, &din))) return r;
    if ((r = hb::acquire_output(output, kOut, &dout))) return r;

    Plan p;
    fill_frame(p, input, output, din, dout, levels, alpha, beta);
    const int W = p.f.W, C = p.f.in_c;
    Span outx = {p.f.out_x0, p.f.out_x0 + W - 1};
    Span inx = {p.f.in_x0, p.f.in_x0 + p.f.in_w - 1};
    const ll::Geom whole = ll::make_geom(outx, frame_y, inx, frame_y, p.J);
    const int jr = choose_coarse_level(whole, nranks, p.J, p.K);

    // every rank's band: gathered once per geometry (collective on first use / change)
    const int key[10] = {W, band.lo, band.hi, frame_y.lo, frame_y.hi, rank, nranks, C, jr, levels};
    if (!g_shard.valid || memcmp(g_shard.key, key, sizeof(key)) != 0) {
        int mine[2] = {band.lo, band.hi};
        g_shard.bands.assign(2 * (size_t)nranks, 0);
        if ((r = hbdist::allgather_bytes(mine, g_shard.bands.data(), sizeof(mine)))) return r;
        for (int q = 0; q + 1 < nranks; q++) {
            if (g_shard.bands[2 * q + 1] + 1 != g_shard.bands[2 * q + 2]) {
                return hb::fail(halide_error_code_constraint_violated,
                                "local_laplacian_sharded: rank %d's band ends at row %d but rank %d's starts at %d", q,
                                g_shard.bands[2 * q + 1], q + 1, g_shard.bands[2 * q + 2]);
            }
        }
        memcpy(g_shard.key, key, sizeof(key));
        g_shard.valid = true;
    }
    auto band_of = [&](int q) { return Span{g_shard.bands[2 * q], g_shard.bands[2 * q + 1]}; };
    auto rows_of = [&](int q, ll::ShardLevel *sl, Span *need) {
        ll::compute_shard_rows(whole, frame_y, band_of(q), q == 0, q == nranks - 1, jr, sl, need);
    };
    ll::ShardLevel sl[ll::kMaxJ];
    Span in_need;
    rows_of(rank, sl, &in_need);
    for (int j = 1; j <= jr && j < p.J; j++) {
        if (sl[j].own.n() < 1) {
            return hb::fail(halide_error_code_constraint_violated,
                            "local_laplacian_sharded: band of %d rows is too small for %d ranks (level %d owns no row)", band.n(), nranks, j);
        }
    }
    p.geom = ll::make_shard_geom(whole, sl, jr);
    p.f.clamp_y0 = frame_y.lo;
    p.f.clamp_h = frame_y.n();
    hb::Scratch scratch;
    if ((r = alloc_levels(p, scratch))) return r;

    // ---- input halo: rows [in_need.lo, band.lo) from the rank above, (band.hi, in_need.hi] from the rank below ----
    const int ht = band.lo - in_need.lo, hbn = in_need.hi - band.hi;
    const size_t rowb = (size_t)p.f.in_w * sizeof(uint16_t);
    uint16_t *halo_top = nullptr, *halo_bot = nullptr, *send_up = nullptr, *send_dn = nullptr;
    int up_need = 0, dn_need = 0;  // rows the rank below needs from my bottom / the rank above needs from my top
    if (!first) {
        ll::ShardLevel t[ll::kMaxJ];
        Span n;
        rows_of(rank - 1, t, &n);
        up_need = n.hi - band_of(rank - 1).hi;  // its bottom halo = my first rows
    }
    if (!last) {
        ll::ShardLevel t[ll::kMaxJ];
        Span n;
        rows_of(rank + 1, t, &n);
        dn_need = band_of(rank + 1).lo - n.lo;  // its top halo = my last rows
    }
    if (ht > (first ? 0 : band_of(rank - 1).n()) || hbn > (last ? 0 : band_of(rank + 1).n()) || up_need > band.n() || dn_need > band.n()) {
        return hb::fail(halide_error_code_constraint_violated,
                        "local_laplacian_sharded: bands of %d rows are smaller than the input halo (%d above, %d below)", band.n(), ht, hbn);
    }
    if (ht) halo_top = scratch.get<uint16_t>((size_t)C * ht * p.f.in_w);
    if (hbn) halo_bot = scratch.get<uint16_t>((size_t)C * hbn * p.f.in_w);
    if (up_need) send_up = scratch.get<uint16_t>((size_t)C * up_need * p.f.in_w);
    if (dn_need) send_dn = scratch.get<uint16_t>((size_t)C * dn_need * p.f.in_w);
    if ((ht && !halo_top) || (hbn && !halo_bot) || (up_need && !send_up) || (dn_need && !send_dn)) {
        return hb::fail(halide_error_code_device_malloc_failed, "local_laplacian_sharded: scratch allocation failed");
    }
    p.f.halo_pitch = p.f.in_w;
    p.f.halo_top = halo_top; p.f.halo_bot = halo_bot;
    p.f.halo_top_rows = ht; p.f.halo_bot_rows = hbn;

    cudaStream_t s = hb::stream();
    if ((r = get_lut(p, s))) return r;
    {
        hb::CallTimer timer(s);
        // pack my boundary rows per channel ([c][row][w], the layout of the receiver's halo arrays) and exchange — on a
        // second stream, so that the level-1 kernel's interior rows (every source row inside the band) run meanwhile;
        // only the few level-1 rows at the band's edges wait for the halo (HALIDE_B200_SHARD_OVERLAP=0: one stream)
        static const bool overlap = [] {
            const char *e = getenv("HALIDE_B200_SHARD_OVERLAP");
            return !(e && e[0] == '0');
        }();
        static thread_local cudaStream_t comm_stream = nullptr;
        static thread_local cudaEvent_t ev_in = nullptr, ev_halo = nullptr;
        if (overlap && !comm_stream) {
            cudaStreamCreateWithFlags(&comm_stream, cudaStreamNonBlocking);
            cudaEventCreateWithFlags(&ev_in, cudaEventDisableTiming);
            cudaEventCreateWithFlags(&ev_halo, cudaEventDisableTiming);
        }
        bool exchanged_async = false;
        {
            cudaStream_t xs = overlap ? comm_stream : s;
            if (overlap) {  // the input (and the previous call's use of the scratch blocks) is ordered on s
                cudaEventRecord(ev_in, s);
                cudaStreamWaitEvent(xs, ev_in, 0);
            }
            hbdist::Msg msgs[4];
            int n = 0;
            for (int c = 0; c < C; c++) {
                const uint16_t *plane = (const uint16_t *)din + (int64_t)c * p.f.in_sc;
                if (up_need) {
                    cudaMemcpy2DAsync(send_up + (size_t)c * up_need * p.f.in_w, rowb, plane, (size_t)p.f.in_sy * sizeof(uint16_t), rowb,
                                      up_need, cudaMemcpyDeviceToDevice, xs);
                }
                if (dn_need) {
                    cudaMemcpy2DAsync(send_dn + (size_t)c * dn_need * p.f.in_w, rowb, plane + (int64_t)(p.f.in_h - dn_need) * p.f.in_sy,
                                      (size_t)p.f.in_sy * sizeof(uint16_t), rowb, dn_need, cudaMemcpyDeviceToDevice, xs);
                }
            }
            if (up_need) msgs[n++] = {send_up, (size_t)C * up_need * rowb, rank - 1, true};
            if (dn_need) msgs[n++] = {send_dn, (size_t)C * dn_need * rowb, rank + 1, true};
            if (ht) msgs[n++] = {halo_top, (size_t)C * ht * rowb, rank - 1, false};
            if (hbn) msgs[n++] = {halo_bot, (size_t)C * hbn * rowb, rank + 1, false};
            if (n) {
                hb::profile_begin("nccl_input_halo", xs);  // (event-bracketed in profile mode like a kernel launch; not counted as one)
                r = hbdist::exchange(msgs, n, xs);
                hb::after_launch(xs);
                if (r) return r;
                if (overlap) {
                    cudaEventRecord(ev_halo, xs);
                    exchanged_async = true;
                }
            }
        }
        LevelBuf *lb = p.ls.lv;
        if (exchanged_async && p.K == 8 && !(g_force_naive & 1)) {
            // level 1 in up to three launches: interior rows (taps 2y-1 .. 2y+2 all inside the band) now, edge rows after the halo
            const Span cy = lb[1].cy;
            int i_lo = (p.f.in_y0 + 2) >> 1;                    // smallest y with 2y-1 >= in_y0
            int i_hi = (p.f.in_y0 + p.f.in_h - 3) >> 1;          // largest y with 2y+2 <= in_y0 + in_h - 1
            if (i_lo < cy.lo) i_lo = cy.lo;
            if (i_hi > cy.hi) i_hi = cy.hi;
            if (i_lo <= i_hi) {
                lb[1].cy = {i_lo, i_hi};
                launch_down(p, 1, s);
            }
            cudaStreamWaitEvent(s, ev_halo, 0);
            if (i_lo > i_hi) {  // (band too thin to have interior rows)
                lb[1].cy = cy;
                launch_down(p, 1, s);
            } else {
                if (cy.lo < i_lo) {
                    lb[1].cy = {cy.lo, i_lo - 1};
                    launch_down(p, 1, s);
                }
                if (i_hi < cy.hi) {
                    lb[1].cy = {i_hi + 1, cy.hi};
                    launch_down(p, 1, s);
                }
            }
            lb[1].cy = cy;
        } else {
            if (exchanged_async) cudaStreamWaitEvent(s, ev_halo, 0);
            launch_down(p, 1, s);
        }
        for (int j = 2; j <= jr; j++) launch_down(p, j, s);  // (level jr: only the rows this rank owns)
        // ---- gather level jr: my rows to every rank, every rank's rows into my whole-frame copy ----
        {
            std::vector<hbdist::Msg> msgs;
            const size_t gp_row = (size_t)lb[jr].nq * lb[jr].gpitch * 2 * sizeof(float), ing_row = (size_t)lb[jr].gpitch * sizeof(float);
            auto rows_msg = [&](Span rows, int peer, bool send) {
                if (rows.n() <= 0) return;
                const size_t off = (size_t)(rows.lo - lb[jr].sy.lo);
                msgs.push_back({(char *)lb[jr].gp + off * gp_row, (size_t)rows.n() * gp_row, peer, send});
                msgs.push_back({(char *)lb[jr].ing + off * ing_row, (size_t)rows.n() * ing_row, peer, send});
            };
            for (int q = 0; q < nranks; q++) {
                if (q == rank) continue;
                Span own_q[ll::kMaxJ];
                ll::compute_band_own(whole, band_of(q), q == 0, q == nranks - 1, own_q);
                rows_msg(sl[jr].own, q, true);
                rows_msg(own_q[jr], q, false);
            }
            if (!msgs.empty()) {
                hb::profile_begin("nccl_level_gather", s);
                r = hbdist::exchange(msgs.data(), (int)msgs.size(), s);
                hb::after_launch(s);
                if (r) return r;
            }
        }
        lb[jr].cy = lb[jr].sy;   // from here on level jr is complete (its pair plane is not: the up-sweep gathers from gp)
        lb[jr].has_pair = 0;
        run_coarse_sweep(p, jr, s);          // levels jr+1.. down, ..jr+1 up, whole frame, on every rank
        launch_up(p, jr, s);
        for (int j = jr - 1; j >= 1; j--) launch_up(p, j, s);
        launch_final(p, s);
    }
    if ((r = hb::check_cuda(cudaGetLastError(), "local_laplacian_sharded launch", halide_error_code_device_run_failed))) return r;
    hb::mark_output_written(output);
    return 0;
}

}  // namespace

extern "C" int local_laplacian(halide_buffer_t *input, int32_t levels, float alpha, float beta, halide_buffer_t *output) {
    return run_local_laplacian(input, levels, alpha, beta, output);
}
extern "C" int local_laplacian_argv(void **args) {
    return run_local_laplacian((halide_buffer_t *)args[0], *(int32_t *)args[1], *(float *)args[2], *(float *)args[3],
                               (halide_buffer_t *)args[4]);
}
extern "C" const halide_filter_metadata_t *local_laplacian_metadata(void) {
    return &kMeta;
}
// The harness's second AOT variant (apps/local_laplacian/process.cpp:44-48): same implementation.
extern "C" int local_laplacian_auto_schedule(halide_buffer_t *input, int32_t levels, float alpha, float beta,
                                             halide_buffer_t *output) {
    return run_local_laplacian(input, levels, alpha, beta, output);
}
extern "C" int local_laplacian_auto_schedule_argv(void **args) {
    return local_laplacian_argv(args);
}
extern "C" const halide_filter_metadata_t *local_laplacian_auto_schedule_metadata(void) {
    return &kMetaAuto;
}

// Test hook: route K == 8 calls through the generic (any `levels`) kernels so both paths stay covered.
extern "C" void halide_b200_ll_force_generic(int enable) {
    g_force_naive = enable;
}

// Row-sharded path: which pyramid level is gathered all-to-all (see run_local_laplacian_sharded).  Collective
// setting: every rank must use the same value.  0 = choose by size (default), n >= 2 = level n.
extern "C" void halide_b200_ll_shard_coarse_level(int level) {
    g_shard_coarse_level = level < 0 ? 0 : level;
}

// Probe for the CPU-side tests (no CUDA calls): the level halide_b200_local_laplacian_sharded gathers for a
// frame of frame_w x frame_h split over nranks ranks.
extern "C" int halide_b200_ll_shard_plan_level(int32_t frame_w, int32_t frame_h, int32_t nranks) {
    Span fx = {0, frame_w - 1}, fy = {0, frame_h - 1};
    return choose_coarse_level(ll::make_geom(fx, fy, fx, fy, ll::kMaxJ), nranks, ll::kMaxJ, 8);
}

// Row-sharded entry point (B200 extension; see run_local_laplacian_sharded).
extern "C" int halide_b200_local_laplacian_sharded(halide_buffer_t *input, int32_t levels, float alpha, float beta,
                                                   halide_buffer_t *output, int32_t frame_y_min, int32_t frame_y_extent) {
    return run_local_laplacian_sharded(input, levels, alpha, beta, output, frame_y_min, frame_y_extent);
}

// Band geometry probe for the CPU-side tests of the sharding logic (no CUDA calls): for a band [band_lo, band_hi] of a
// frame_w x frame_h frame and gathered level jr, fills out[j*8 .. j*8+7] = {own.lo, own.hi, d.lo, d.hi, u.lo, u.hi,
// S_j.lo, S_j.hi} (ll_geom.h: ShardLevel; S_j = the level's stored rows on the whole frame) for j = 0..7 and
// out[64..65] = the input rows [lo, hi] the band's level-1 rows read.
extern "C" int halide_b200_ll_band_geometry(int32_t frame_w, int32_t frame_h, int32_t band_lo, int32_t band_hi, int32_t first,
                                            int32_t last, int32_t jr, int32_t *out) {
    Span fx = {0, frame_w - 1}, fy = {0, frame_h - 1};
    ll::Geom whole = ll::make_geom(fx, fy, fx, fy, ll::kMaxJ);
    ll::ShardLevel sl[ll::kMaxJ];
    Span need;
    ll::compute_shard_rows(whole, fy, Span{band_lo, band_hi}, first != 0, last != 0, jr, sl, &need);
    for (int j = 0; j < ll::kMaxJ; j++) {
        int32_t *o = out + j * 8;
        o[0] = sl[j].own.lo; o[1] = sl[j].own.hi; o[2] = sl[j].d.lo; o[3] = sl[j].d.hi;
        o[4] = sl[j].u.lo; o[5] = sl[j].u.hi; o[6] = whole.lv[j].sy.lo; o[7] = whole.lv[j].sy.hi;
    }
    out[64] = need.lo;
    out[65] = need.hi;
    return 0;
}

// Device self-test of the arithmetic shortcuts used by the fast kernels (shared-reciprocal division, magic-number
// conversions): returns the number of mismatches against div.rn / cvt over n pseudo-random operand sets, or -1.
extern "C" long long halide_b200_selftest_arith(unsigned long long n, unsigned long long seed) {
    unsigned long long *bad = nullptr, host = 0;
    if (cudaMalloc(&bad, sizeof(*bad)) != cudaSuccess) return -1;
    cudaMemset(bad, 0, sizeof(*bad));
    cudaStream_t s = hb::stream();
    HB_LAUNCH("ll_selftest", ll_selftest_kernel, 148 * 8, 256, 0, s, n, seed, bad);
    if (cudaMemcpyAsync(&host, bad, sizeof(host), cudaMemcpyDeviceToHost, s) != cudaSuccess || cudaStreamSynchronize(s) != cudaSuccess) {
        cudaFree(bad);
        return -1;
    }
    cudaFree(bad);
    return (long long)host;
}
