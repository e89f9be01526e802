/* halide_b200_runtime.h — the C ABI boundary of the B200-native Halide apps library.
 *
 * This header re-declares (it does not copy) the binary layout a Halide AOT filter and its
 * harness agree on, so that `apps/<app>/process.cpp|filter.cpp|test.cpp` of the reference link
 * against libhalide_b200.so unchanged.  Every declaration cites the reference interface it
 * replaces; all paths are relative to /root/reference.
 *
 *   halide_buffer_t            src/runtime/HalideRuntime.h:1710-1737   (56 bytes, LP64)
 *   halide_dimension_t         src/runtime/HalideRuntime.h:1657-1685   (16 bytes)
 *   halide_type_t              src/runtime/HalideRuntime.h:521-545     (4 bytes: code, bits, reserved)
 *   halide_device_interface_t  src/runtime/HalideRuntime.h:875-899     (15 function pointers + impl)
 *   halide_error_code_t        src/runtime/HalideRuntime.h:1152-1357
 *   halide_filter_metadata_t   src/runtime/HalideRuntime.h:1937-1977
 *   halide_cuda_* entry points src/runtime/HalideRuntimeCuda.h:40-81
 *
 * If the reference's own HalideRuntime.h was included first (harness builds), the type
 * re-declarations below are skipped and only the function prototypes remain, so both headers
 * can coexist in one translation unit.
 */
#ifndef HALIDE_B200_RUNTIME_H
#define HALIDE_B200_RUNTIME_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#ifndef HALIDE_HALIDERUNTIME_H /* the reference header's include guard */
#define HALIDE_B200_OWNS_ABI_TYPES 1

/* Element type codes (HalideRuntime.h:492-503). */
enum {
    halide_type_int = 0,
    halide_type_uint = 1,
    halide_type_float = 2,
    halide_type_handle = 3,
    halide_type_bfloat = 4
};

/* 4-byte type word: code@0, bits@1, 16 reserved bits@2 (HalideRuntime.h:521-545). */
struct halide_type_t {
    uint8_t code;
    uint8_t bits;
    uint16_t reserved;
};

/* One dimension: coordinates [min, min+extent), stride in ELEMENTS (HalideRuntime.h:1657-1685). */
typedef struct halide_dimension_t {
    int32_t min, extent, stride;
    uint32_t flags;
} halide_dimension_t;

/* Dirty bits in halide_buffer_t::flags (HalideRuntime.h:1699-1702). */
enum {
    halide_buffer_flag_host_dirty = 1,
    halide_buffer_flag_device_dirty = 2
};

struct halide_device_interface_t;

/* The image handle crossing the boundary (HalideRuntime.h:1710-1737).  `host` addresses the element
 * whose coordinates are the per-dimension mins; caller owns host memory and the dim[] array. */
typedef struct halide_buffer_t {
    uint64_t device;                                          /* @0  device handle (CUdeviceptr) or 0 */
    const struct halide_device_interface_t *device_interface; /* @8  */
    uint8_t *host;                                            /* @16 */
    uint64_t flags;                                           /* @24 */
    struct halide_type_t type;                                /* @32 */
    int32_t dimensions;                                       /* @36 */
    halide_dimension_t *dim;                                  /* @40 */
    void *padding;                                            /* @48 */
} halide_buffer_t;

struct halide_device_interface_impl_t;

/* Function table every buffer with a device allocation points at (HalideRuntime.h:875-899).
 * Halide::Runtime::Buffer calls copy_to_host / device_sync / device_free through it
 * (src/runtime/HalideBuffer.h:352-358,1810-1815). */
struct halide_device_interface_t {
    int (*device_malloc)(void *user_context, struct halide_buffer_t *buf,
                         const struct halide_device_interface_t *device_interface);
    int (*device_free)(void *user_context, struct halide_buffer_t *buf);
    int (*device_sync)(void *user_context, struct halide_buffer_t *buf);
    void (*device_release)(void *user_context, const struct halide_device_interface_t *device_interface);
    int (*copy_to_host)(void *user_context, struct halide_buffer_t *buf);
    int (*copy_to_device)(void *user_context, struct halide_buffer_t *buf,
                          const struct halide_device_interface_t *device_interface);
    int (*device_and_host_malloc)(void *user_context, struct halide_buffer_t *buf,
                                  const struct halide_device_interface_t *device_interface);
    int (*device_and_host_free)(void *user_context, struct halide_buffer_t *buf);
    int (*buffer_copy)(void *user_context, struct halide_buffer_t *src,
                       const struct halide_device_interface_t *dst_device_interface, struct halide_buffer_t *dst);
    int (*device_crop)(void *user_context, const struct halide_buffer_t *src, struct halide_buffer_t *dst);
    int (*device_slice)(void *user_context, const struct halide_buffer_t *src, int slice_dim, int slice_pos,
                        struct halide_buffer_t *dst);
    int (*device_release_crop)(void *user_context, struct halide_buffer_t *buf);
    int (*wrap_native)(void *user_context, struct halide_buffer_t *buf, uint64_t handle,
                       const struct halide_device_interface_t *device_interface);
    int (*detach_native)(void *user_context, struct halide_buffer_t *buf);
    int (*compute_capability)(void *user_context, int *major, int *minor);
    const struct halide_device_interface_impl_t *impl;
};

/* Return codes (HalideRuntime.h:1152-1357); only the ones this library can produce are named. */
enum halide_error_code_t {
    halide_error_code_success = 0,
    halide_error_code_generic_error = -1,
    halide_error_code_explicit_bounds_too_small = -2,
    halide_error_code_bad_type = -3,
    halide_error_code_access_out_of_bounds = -4,
    halide_error_code_buffer_allocation_too_large = -5,
    halide_error_code_buffer_extents_too_large = -6,
    halide_error_code_constraints_make_required_region_smaller = -7,
    halide_error_code_constraint_violated = -8,
    halide_error_code_param_too_small = -9,
    halide_error_code_param_too_large = -10,
    halide_error_code_out_of_memory = -11,
    halide_error_code_buffer_argument_is_null = -12,
    halide_error_code_copy_to_host_failed = -14,
    halide_error_code_copy_to_device_failed = -15,
    halide_error_code_device_malloc_failed = -16,
    halide_error_code_device_sync_failed = -17,
    halide_error_code_device_free_failed = -18,
    halide_error_code_no_device_interface = -19,
    halide_error_code_unimplemented = -20,
    halide_error_code_internal_error = -22,
    halide_error_code_device_run_failed = -23,
    halide_error_code_buffer_extents_negative = -28,
    halide_error_code_gpu_device_error = -29,
    halide_error_code_device_wrap_native_failed = -32,
    halide_error_code_device_detach_native_failed = -33,
    halide_error_code_host_is_null = -34,
    halide_error_code_host_and_device_dirty = -37,
    halide_error_code_buffer_is_null = -38,
    halide_error_code_device_buffer_copy_failed = -39,
    halide_error_code_device_crop_unsupported = -40,
    halide_error_code_incompatible_device_interface = -42,
    halide_error_code_bad_dimensions = -43,
    halide_error_code_device_dirty_with_no_device_support = -44
};

/* Scalar value cell used by the metadata tables (HalideRuntime.h:1880-1900). */
struct halide_scalar_value_t {
    union {
        uint8_t b;
        int8_t i8;
        int16_t i16;
        int32_t i32;
        int64_t i64;
        uint8_t u8;
        uint16_t u16;
        uint32_t u32;
        uint64_t u64;
        float f32;
        double f64;
        void *handle;
    } u;
};

enum halide_argument_kind_t {
    halide_argument_kind_input_scalar = 0,
    halide_argument_kind_input_buffer = 1,
    halide_argument_kind_output_buffer = 2
};

/* Per-argument metadata record (HalideRuntime.h:1937-1951). */
struct halide_filter_argument_t {
    const char *name;
    int32_t kind;
    int32_t dimensions;
    struct halide_type_t type;
    const struct halide_scalar_value_t *scalar_def, *scalar_min, *scalar_max, *scalar_estimate;
    int64_t const *const *buffer_estimates;
};

/* What F_metadata() returns (HalideRuntime.h:1954-1977); apps/blur/test.cpp:158 reads ->target. */
struct halide_filter_metadata_t {
    int32_t version;
    int32_t num_arguments;
    const struct halide_filter_argument_t *arguments;
    const char *target;
    const char *name;
};

typedef void (*halide_error_handler_t)(void *, const char *);
typedef void *(*halide_malloc_t)(void *, size_t);
typedef void (*halide_free_t)(void *, void *);
typedef void (*halide_print_t)(void *, const char *);

#endif /* HALIDE_HALIDERUNTIME_H */

/* ---- runtime shim: the subset of the Halide runtime the filters and harnesses call ---- */

/* Error reporting (HalideRuntime.h:173-195; default handler prints "Error: ..." and aborts,
 * src/runtime/posix_error_handler.cpp:9-41).  halide_set_error_handler returns the old handler. */
void halide_error(void *user_context, const char *msg);
halide_error_handler_t halide_set_error_handler(halide_error_handler_t handler);

/* Host allocator hooks (HalideRuntime.h; installed by tools/halide_malloc_trace.h in apps/camera_pipe/process.cpp). */
halide_malloc_t halide_set_custom_malloc(halide_malloc_t user_malloc);
halide_free_t halide_set_custom_free(halide_free_t user_free);
/* The rest of the host-side hooks tools/RunGenMain.cpp links (HalideRuntime.h:170-181,434-465,2343). */
void *halide_default_malloc(void *user_context, size_t x);
void halide_default_free(void *user_context, void *ptr);
void *halide_malloc(void *user_context, size_t x);
void halide_free(void *user_context, void *ptr);
halide_print_t halide_set_custom_print(halide_print_t print);
void halide_print(void *user_context, const char *msg);
void *halide_get_symbol(const char *name);
#ifdef __cplusplus
int halide_reuse_device_allocations(void *user_context, bool enable);
#else
int halide_reuse_device_allocations(void *user_context, _Bool enable);
#endif

/* Device bookkeeping (src/runtime/device_interface.cpp:30-56,154-205). */
int halide_device_malloc(void *user_context, struct halide_buffer_t *buf,
                         const struct halide_device_interface_t *device_interface);
int halide_device_free(void *user_context, struct halide_buffer_t *buf);
int halide_device_sync(void *user_context, struct halide_buffer_t *buf);
int halide_copy_to_host(void *user_context, struct halide_buffer_t *buf);
/* Copy the region `dst` describes out of `src` (HalideRuntime.h halide_buffer_copy; src/runtime/device_interface.cpp:154-205):
 * to dst's device side when dst_device_interface is halide_cuda_device_interface(), to its host side when it is NULL. */
int halide_buffer_copy(void *user_context, struct halide_buffer_t *src,
                       const struct halide_device_interface_t *dst_device_interface, struct halide_buffer_t *dst);
int halide_copy_to_device(void *user_context, struct halide_buffer_t *buf,
                          const struct halide_device_interface_t *device_interface);
void halide_device_release(void *user_context, const struct halide_device_interface_t *device_interface);

/* CUDA device API (src/runtime/HalideRuntimeCuda.h:21,40-81). */
const struct halide_device_interface_t *halide_cuda_device_interface(void);
int halide_cuda_wrap_device_ptr(void *user_context, struct halide_buffer_t *buf, uint64_t device_ptr);
int halide_cuda_detach_device_ptr(void *user_context, struct halide_buffer_t *buf);
uintptr_t halide_cuda_get_device_ptr(void *user_context, struct halide_buffer_t *buf);
int halide_cuda_release_unused_device_allocations(void *user_context);

/* ---- B200 library extensions (no reference equivalent; plain pointers and sizes only) ---- */

/* Stream every kernel and copy of this thread's subsequent filter calls is issued on
 * (a cudaStream_t passed as void*; NULL = the legacy default stream, which is also torch's
 * default current stream).  Replaces halide_set_cuda_get_stream (HalideRuntimeCuda.h:66-81). */
void halide_b200_set_stream(void *cuda_stream);
void *halide_b200_get_stream(void);
/* A non-blocking stream for a caller thread that pipelines frames (one stream per thread: copies of
 * one thread's frame overlap kernels and copies of another's); destroy synchronises first. */
void *halide_b200_stream_create(void);
int halide_b200_stream_destroy(void *cuda_stream);
/* Select the CUDA device for this process (replaces HL_GPU_DEVICE, src/runtime/gpu_device_selection.cpp). */
int halide_b200_set_device(int ordinal);
/* Number of kernels this library has launched since process start (bench.py's gpu_launches). */
uint64_t halide_b200_kernel_launch_count(void);
/* Library/target identification string, e.g. "x86-64-linux-cuda-cuda_capability_100-b200_native". */
const char *halide_b200_target(void);
/* Bracket the kernels of one filter call with CUDA events on the library stream and report the
 * device time of the most recent call in milliseconds (negative if timing is disabled). */
void halide_b200_set_timing(int enable);
float halide_b200_last_kernel_ms(void);
/* Per-kernel profile: when enabled, every kernel launch is bracketed by CUDA events on its
 * stream.  The report is text, one "name count total_ms" line per kernel; returns bytes needed. */
void halide_b200_profile_enable(int enable);
void halide_b200_profile_reset(void);
int halide_b200_profile_report(char *out, int out_size);


/* ---- multi-GPU (one process per GPU; the reference has no counterpart, SURVEY.md §8e) ---- */

/* NCCL bootstrap: rank 0 obtains a 128-byte id, the host's control plane broadcasts it, every rank
 * joins.  Ranks are ordered top to bottom over the frame's rows. */
int halide_b200_dist_unique_id(char *out128);
int halide_b200_dist_init(int rank, int nranks, const char *id128);
int halide_b200_dist_shutdown(void);
int halide_b200_dist_rank(void);
int halide_b200_dist_size(void);

/* local_laplacian on this rank's row band of a frame whose rows are [frame_y_min, frame_y_min +
 * frame_y_extent): `input`/`output` hold the band's rows (all columns/channels) with dim[1].min in
 * frame coordinates; ranks are ordered top to bottom.  Communication per call: one exchange of input halo rows with
 * the two row neighbours (every pyramid row a band needs beyond itself is recomputed from them) and one all-to-all
 * gather of a coarse pyramid level.  Bit-identical to the single-GPU filter on the whole frame. */
int halide_b200_local_laplacian_sharded(struct halide_buffer_t *input, int32_t levels, float alpha, float beta,
                                        struct halide_buffer_t *output, int32_t frame_y_min, int32_t frame_y_extent);

/* Host-only probe of the band geometry for tests: with level jr gathered, out[j*8..j*8+7] = {own.lo, own.hi, d.lo, d.hi,
 * u.lo, u.hi, S.lo, S.hi} per pyramid level j = 0..7 (rows owned in the gather partition / Gaussian-side rows computed and
 * held / outGPyramid rows needed / the level's rows on the whole frame), out[64..65] = input rows read; out[66]. */
int halide_b200_ll_band_geometry(int32_t frame_w, int32_t frame_h, int32_t band_lo, int32_t band_hi, int32_t first,
                                 int32_t last, int32_t jr, int32_t *out);
/* Row-sharded local_laplacian: pyramid level gathered all-to-all so that the coarser levels are computed
 * redundantly on every rank without further exchange.  0 = chosen by size (default), n >= 2 = level n.
 * Collective setting: all ranks must agree. */
void halide_b200_ll_shard_coarse_level(int level);
/* The level the sharded call gathers for a frame_w x frame_h frame over nranks ranks; host-only. */
int halide_b200_ll_shard_plan_level(int32_t frame_w, int32_t frame_h, int32_t nranks);
/* Test hook: bitmask routing levels==8 calls through the generic kernels (1 down, 2 up, 4 final,
 * 8 no fused coarse launch, 16 general-layout final kernel, 64 no TMA frame tile in the final
 * kernel, 256 = the 48-row-tile variant of the TMA final kernel, 128 = its default 32-row tiles) so
 * every code path stays covered by the parity tests. */
void halide_b200_ll_force_generic(int mask);
/* halide_blur test hook: 1 = route 4-byte-aligned frames through the general (any alignment) kernel as well;
 * >= 8 = aligned kernel with strips of that many rows (0 restores the defaults). */
void halide_b200_blur_force_general(int enable);
/* nl_means test / A-B hook: 0 = default kernel, 1 = generic kernel, 2 = register-window kernel (patch 3 or 7, search 7). */
void halide_b200_nl_means_variant(int variant);
/* stencil_chain test / A-B hook: 0 = default kernel, 1 = one-pixel-per-thread tile kernel, 2 = register-window tile kernel. */
void halide_b200_stencil_chain_variant(int variant);
/* conv_layer: 1 = tcgen05/TMEM/TMA implicit GEMM (3xTF32 split), 0 = FP32 SIMT kernel (also HALIDE_B200_CONV=tc|simt). */
void halide_b200_conv_use_tensor_cores(int enable);
/* Test hook: byte in 0..255 makes every device block the library hands out (buffer device_malloc, filter scratch,
 * the local_laplacian remap table) start filled with that byte, memset on the calling thread's stream before the
 * block is returned, so an unwritten output element or unwritten scratch shows up as a wrong value instead of
 * whatever the recycled block last held; -1 (the default) turns it off. */
void halide_b200_debug_fill_allocations(int byte);
/* Device self-test of the fast kernels' arithmetic shortcuts; returns mismatches vs div.rn / cvt, or -1. */
long long halide_b200_selftest_arith(unsigned long long n, unsigned long long seed);

#ifdef __cplusplus
}
#endif

#endif /* HALIDE_B200_RUNTIME_H */
