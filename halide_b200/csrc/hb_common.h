// hb_common.h — internal helpers shared by the filter translation units of libhalide_b200.so.
//
// Host side of the drop-in boundary: argument validation in the order a Halide-generated
// filter prologue performs it (reference: src/AddImageChecks.cpp:311-347,404-476,560-686),
// bounds-query mode (src/AddImageChecks.cpp:477-496,710-716), host/device residency
// (src/InjectHostDevBufferCopies.cpp, src/runtime/device_interface.cpp:154-205) and the
// kernel-launch bookkeeping.  Nothing here computes pixels.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/halide_b200_runtime.h"

namespace hb {

// ---- error reporting -------------------------------------------------------------------------
// Formats a message, hands it to the (replaceable) halide_error handler and returns `code`,
// mirroring the halide_error_* helpers in src/runtime/errors.cpp:5-80.
int fail(int code, const char *fmt, ...) __attribute__((format(printf, 2, 3)));

// ---- stream / launch accounting --------------------------------------------------------------
cudaStream_t stream();
void count_launch(const char *name, cudaStream_t s);
void profile_begin(const char *name, cudaStream_t s);  // event bracket only (closed by after_launch), not counted as a launch
void after_launch(cudaStream_t s);
int check_cuda(cudaError_t e, const char *what, int code);

// RAII bracket around the kernels of one filter call (halide_b200_set_timing).
struct CallTimer {
    explicit CallTimer(cudaStream_t s);
    ~CallTimer();
    cudaStream_t s;
};

// ---- once-per-device set-up (function attributes are per device / context; keyed by the CURRENT device, and safe
// to race: two threads at worst both run `fn`, which must be idempotent) -----------------------------------------
struct PerDeviceOnce {
    unsigned long long done = 0;  // bit d = device d set up (devices >= 64: always run fn)
    template<typename F>
    void run(F fn) {
        int dev = 0;
        cudaGetDevice(&dev);
        const unsigned long long bit = dev < 64 ? 1ull << dev : 0ull;
        if (bit && (__atomic_load_n(&done, __ATOMIC_ACQUIRE) & bit)) return;
        fn();
        if (bit) __atomic_fetch_or(&done, bit, __ATOMIC_RELEASE);
    }
};

// ---- device scratch (callee-owned intermediates; pooled, src/runtime/cuda.cpp:760-870 analogue) ---
void *scratch_alloc(size_t bytes);  // returns nullptr on failure (caller maps to -16)
void scratch_free(void *p);         // stream-ordered: safe to call right after the last launch
// Under halide_b200_debug_fill_allocations, memset a fresh device block to the fill byte on `s` (no-op when off).
void *debug_fill(void *p, size_t bytes, cudaStream_t s);

struct Scratch {  // frees everything it handed out when the filter call returns
    static constexpr int kMax = 48;
    void *ptrs[kMax];
    int n = 0;
    ~Scratch() {
        for (int i = 0; i < n; i++) scratch_free(ptrs[i]);
    }
    template<typename T>
    T *get(size_t count) {
        if (n >= kMax) return nullptr;
        void *p = scratch_alloc(count * sizeof(T));
        if (p) ptrs[n++] = p;
        return (T *)p;
    }
};

// ---- buffer validation -----------------------------------------------------------------------
struct ArgSpec {
    const char *name;  // "Input buffer input", "Output buffer output" style prefix is added by fail()
    uint8_t code;      // halide_type_uint / halide_type_float ...
    uint8_t bits;
    int dimensions;
    bool is_output;
};

inline bool is_bounds_query(const halide_buffer_t *b) {
    return b->host == nullptr && b->device == 0;  // HalideRuntime.h:1851-1853
}

// null → -12, type → -3, dimensions → -43.  (Extent/stride checks need the required region and
// are done by check_shape after the bounds-query early-out, as in the generated prologue.)
int check_arg(const halide_buffer_t *b, const ArgSpec &spec);

// negative extent → -28, |extent*stride| and allocation size limits → -5/-6, stride[0] != 1 → -8.
int check_shape(const halide_buffer_t *b, const ArgSpec &spec);

// required [min, min+extent) per dimension must lie inside the buffer → else -4.
int check_covers(const halide_buffer_t *b, const ArgSpec &spec, int dim, int req_min, int req_extent);

// Bounds-query answer: write min/extent and dense strides (src/AddImageChecks.cpp:386-436).
void propose_shape(halide_buffer_t *b, const int *mins, const int *extents);

// ---- residency -------------------------------------------------------------------------------
// Make the buffer's contents available on the device and return the device address of the
// element at the mins.  Inputs: allocate + H2D when host_dirty or no device allocation yet.
// Outputs: allocate only.  Returns 0 or a negative halide_error_code_t.
int acquire_input(halide_buffer_t *b, const ArgSpec &spec, void **dev_ptr);
int acquire_output(halide_buffer_t *b, const ArgSpec &spec, void **dev_ptr);
void mark_output_written(halide_buffer_t *b);

inline size_t elem_bytes(const halide_buffer_t *b) {
    return (b->type.bits + 7) / 8;
}

}  // namespace hb

// Launch macro: counts the launch, optionally brackets it with events for the per-kernel
// profile (halide_b200_profile_*), and surfaces launch-configuration errors immediately.
#define HB_LAUNCH(NAME, KERNEL, GRID, BLOCK, SMEM, STREAM, ...)        \
    do {                                                               \
        hb::count_launch(NAME, STREAM);                                \
        KERNEL<<<(GRID), (BLOCK), (SMEM), (STREAM)>>>(__VA_ARGS__);    \
        hb::after_launch(STREAM);                                      \
    } while (0)

extern "C" {
// Per-kernel profile: when enabled every HB_LAUNCH is bracketed by CUDA events on its stream.
void halide_b200_profile_enable(int enable);
void halide_b200_profile_reset(void);
// Writes lines "name count total_ms\n" into out (NUL-terminated); returns bytes needed.
int halide_b200_profile_report(char *out, int out_size);
}
