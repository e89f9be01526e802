// hb_runtime.cu — the slice of the Halide runtime that the AOT filters and the reference
// harnesses call, rebuilt on the CUDA runtime API for a single B200 per process.
//
// Replaces (behaviour, not code): src/runtime/cuda.cpp (device malloc/free pool :760-870, copies
// :884-1017, sync), src/runtime/device_interface.cpp (dirty-bit protocol :30-56,154-205),
// src/runtime/posix_error_handler.cpp:9-41 (default handler prints and aborts) and
// src/runtime/errors.cpp (message + code pairs).  No driver-API module loading is needed because
// the kernels are compiled into this library.
#include "hb_common.h"

#include <dlfcn.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <map>
#include <mutex>
#include <string>
#include <vector>

namespace {

std::atomic<halide_error_handler_t> g_handler{nullptr};
std::atomic<uint64_t> g_launches{0};
std::atomic<int> g_fill_byte{-1};  // halide_b200_debug_fill_allocations: -1 = off
thread_local cudaStream_t t_stream = nullptr;

// ---- device allocation pool ------------------------------------------------------------------
// Exact-size free lists, one per stream.  Blocks returned by device_free / scratch_free become reusable
// by later work on the *same* stream without a sync (stream order makes that safe); a caller thread that
// runs on its own stream (halide_b200_set_stream is thread-local) therefore never receives a block whose
// last use is still in flight on another thread's stream.  Blocks go back to the driver only through
// halide_cuda_release_unused_device_allocations / halide_device_release.
struct Pool {
    using Key = std::pair<cudaStream_t, size_t>;
    std::mutex mu;
    std::multimap<Key, void *> free_blocks;
    std::map<void *, size_t> live;
    size_t cached_bytes = 0;

    void *alloc(size_t bytes) {
        if (bytes == 0) bytes = 256;
        bytes = (bytes + 255) & ~size_t(255);
        {
            std::lock_guard<std::mutex> lock(mu);
            auto it = free_blocks.find(Key(t_stream, bytes));
            if (it != free_blocks.end()) {
                void *p = it->second;
                free_blocks.erase(it);
                cached_bytes -= bytes;
                live[p] = bytes;
                return hb::debug_fill(p, bytes, t_stream);
            }
        }
        void *p = nullptr;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) {
            release_unused();
            e = cudaMalloc(&p, bytes);
            if (e != cudaSuccess) {
                cudaGetLastError();
                return nullptr;
            }
        }
        {
            std::lock_guard<std::mutex> lock(mu);
            live[p] = bytes;
        }
        return hb::debug_fill(p, bytes, t_stream);
    }
    void free(void *p) {
        if (!p) return;
        std::lock_guard<std::mutex> lock(mu);
        auto it = live.find(p);
        if (it == live.end()) return;  // wrapped / foreign pointer: not ours to recycle
        free_blocks.emplace(Key(t_stream, it->second), p);
        cached_bytes += it->second;
        live.erase(it);
    }
    void release_unused() {
        std::vector<void *> victims;
        {
            std::lock_guard<std::mutex> lock(mu);
            for (auto &kv : free_blocks) victims.push_back(kv.second);
            free_blocks.clear();
            cached_bytes = 0;
        }
        if (!victims.empty()) cudaDeviceSynchronize();
        for (void *p : victims) cudaFree(p);
    }
};
Pool &pool() {
    static Pool *p = new Pool;  // intentionally leaked: buffers may be freed during static destruction
    return *p;
}

// ---- per-kernel profile ----------------------------------------------------------------------
struct ProfEntry {
    const char *name;
    cudaEvent_t e0, e1;
};
std::atomic<int> g_prof_on{0};
std::mutex g_prof_mu;
std::vector<ProfEntry> g_prof_pending;
std::map<std::string, std::pair<int, double>> g_prof_totals;
thread_local cudaEvent_t t_prof_e1 = nullptr;

std::atomic<int> g_timing_on{0};
thread_local cudaEvent_t t_call_e0 = nullptr, t_call_e1 = nullptr;
thread_local bool t_call_valid = false;

void prof_drain_locked() {
    for (auto &p : g_prof_pending) {
        cudaEventSynchronize(p.e1);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, p.e0, p.e1);
        auto &t = g_prof_totals[p.name];
        t.first += 1;
        t.second += ms;
        cudaEventDestroy(p.e0);
        cudaEventDestroy(p.e1);
    }
    g_prof_pending.clear();
}

// Span of a buffer in elements relative to the element at the mins: [lo, hi].
void span_elems(const halide_buffer_t *b, int64_t *lo, int64_t *hi) {
    int64_t l = 0, h = 0;
    for (int d = 0; d < b->dimensions; d++) {
        int64_t reach = (int64_t)(b->dim[d].extent - 1) * b->dim[d].stride;
        if (b->dim[d].extent <= 0) continue;
        if (reach < 0) l += reach; else h += reach;
    }
    *lo = l;
    *hi = h;
}

bool any_empty(const halide_buffer_t *b) {
    for (int d = 0; d < b->dimensions; d++) {
        if (b->dim[d].extent <= 0) return true;
    }
    return false;
}

// -- device interface implementation -----------------------------------------------------------
extern const halide_device_interface_t g_cuda_interface;

int if_device_malloc(void *uc, halide_buffer_t *buf, const halide_device_interface_t *iface) {
    if (!buf) return hb::fail(halide_error_code_buffer_is_null, "device_malloc: buffer is null");
    if (buf->device) {
        if (buf->device_interface != &g_cuda_interface) {
            return hb::fail(halide_error_code_incompatible_device_interface,
                            "device_malloc: buffer already has a device allocation of another interface");
        }
        return 0;
    }
    int64_t lo, hi;
    span_elems(buf, &lo, &hi);
    size_t bytes = (size_t)(hi - lo + 1) * hb::elem_bytes(buf);
    void *p = pool().alloc(bytes);
    if (!p) {
        return hb::fail(halide_error_code_device_malloc_failed, "CUDA: cudaMalloc of %zu bytes failed", bytes);
    }
    // device handle addresses the element at the mins, like `host` does.
    buf->device = (uint64_t)((uint8_t *)p - lo * (int64_t)hb::elem_bytes(buf));
    buf->device_interface = &g_cuda_interface;
    return 0;
}

void *alloc_base(const halide_buffer_t *buf) {
    int64_t lo, hi;
    span_elems(buf, &lo, &hi);
    return (uint8_t *)buf->device + lo * (int64_t)hb::elem_bytes(buf);
}

int if_device_free(void *uc, halide_buffer_t *buf) {
    if (!buf || !buf->device) return 0;
    pool().free(alloc_base(buf));
    buf->device = 0;
    buf->device_interface = nullptr;
    buf->flags &= ~(uint64_t)halide_buffer_flag_device_dirty;
    return 0;
}

int if_device_sync(void *uc, halide_buffer_t *buf) {
    cudaError_t e = cudaStreamSynchronize(hb::stream());
    if (e != cudaSuccess) {
        return hb::fail(halide_error_code_device_sync_failed, "CUDA: stream synchronize failed: %s",
                        cudaGetErrorString(e));
    }
    return 0;
}

void if_device_release(void *uc, const halide_device_interface_t *iface) {
    cudaDeviceSynchronize();
    pool().release_unused();
}

// Copy exactly the elements a buffer describes (reference: src/runtime/device_buffer_utils.h make_buffer_copy /
// copy_memory_helper and cuda.cpp:884-1017): dimensions are sorted by stride, dimensions that are contiguous on both
// sides are folded into one chunk, the next dimension becomes the rows of a 2-D memcpy and the remaining ones are
// looped.  Gaps between rows / planes (padded or cropped buffers) are never touched on either side.
struct CopyDim {
    int64_t extent, sstride, dstride;  // strides in bytes
};

int copy_nd(uint8_t *dst, const uint8_t *src, CopyDim *dims, int n, size_t eb, cudaMemcpyKind kind, cudaStream_t s) {
    for (int i = 0; i < n; i++) {
        if (dims[i].extent <= 0) return 0;
    }
    // drop unit dimensions, sort by destination stride (insertion sort; n <= 4 in practice)
    int m = 0;
    for (int i = 0; i < n; i++) {
        if (dims[i].extent != 1) dims[m++] = dims[i];
    }
    for (int i = 1; i < m; i++) {
        CopyDim d = dims[i];
        int j = i;
        while (j > 0 && llabs(dims[j - 1].dstride) > llabs(d.dstride)) {
            dims[j] = dims[j - 1];
            j--;
        }
        dims[j] = d;
    }
    int64_t chunk = (int64_t)eb;
    int first = 0;
    while (first < m && dims[first].sstride == chunk && dims[first].dstride == chunk) {
        chunk *= dims[first].extent;
        first++;
    }
    auto fail_copy = [&](cudaError_t e) {
        return hb::fail(kind == cudaMemcpyDeviceToHost ? halide_error_code_copy_to_host_failed
                                                       : (kind == cudaMemcpyHostToDevice ? halide_error_code_copy_to_device_failed
                                                                                         : halide_error_code_device_buffer_copy_failed),
                        "CUDA: memcpy of %lld-byte chunks failed: %s", (long long)chunk, cudaGetErrorString(e));
    };
    if (first == m) {
        cudaError_t e = cudaMemcpyAsync(dst, src, (size_t)chunk, kind, s);
        return e == cudaSuccess ? 0 : fail_copy(e);
    }
    // rows of a 2-D copy when both pitches are positive and at least one chunk wide; otherwise chunk by chunk
    const CopyDim row = dims[first];
    const bool two_d = row.sstride >= chunk && row.dstride >= chunk;
    const int outer0 = two_d ? first + 1 : first;
    int64_t idx[8] = {0};
    for (;;) {
        int64_t so = 0, dof = 0;
        for (int i = outer0; i < m; i++) {
            so += idx[i] * dims[i].sstride;
            dof += idx[i] * dims[i].dstride;
        }
        cudaError_t e = two_d ? cudaMemcpy2DAsync(dst + dof, (size_t)row.dstride, src + so, (size_t)row.sstride, (size_t)chunk,
                                                  (size_t)row.extent, kind, s)
                              : cudaMemcpyAsync(dst + dof, src + so, (size_t)chunk, kind, s);
        if (e != cudaSuccess) return fail_copy(e);
        int i = outer0;
        for (; i < m; i++) {
            if (++idx[i] < dims[i].extent) break;
            idx[i] = 0;
        }
        if (i == m) break;
    }
    return 0;
}

int copy_span(halide_buffer_t *buf, bool to_host) {
    if (any_empty(buf)) return 0;
    if (buf->dimensions > 8) return hb::fail(halide_error_code_bad_dimensions, "copy: buffers of more than 8 dimensions are not supported");
    const size_t eb = hb::elem_bytes(buf);
    CopyDim dims[8];
    for (int d = 0; d < buf->dimensions; d++) {
        dims[d] = {buf->dim[d].extent, (int64_t)buf->dim[d].stride * (int64_t)eb, (int64_t)buf->dim[d].stride * (int64_t)eb};
    }
    uint8_t *h = buf->host, *d = (uint8_t *)buf->device;
    return to_host ? copy_nd(h, d, dims, buf->dimensions, eb, cudaMemcpyDeviceToHost, hb::stream())
                   : copy_nd(d, h, dims, buf->dimensions, eb, cudaMemcpyHostToDevice, hb::stream());
}

int if_copy_to_host(void *uc, halide_buffer_t *buf) {
    if (!buf) return hb::fail(halide_error_code_buffer_is_null, "copy_to_host: buffer is null");
    if (!(buf->flags & halide_buffer_flag_device_dirty)) return 0;
    if (buf->flags & halide_buffer_flag_host_dirty) {
        return hb::fail(halide_error_code_host_and_device_dirty, "copy_to_host: buffer is dirty on both host and device");
    }
    if (!buf->host) return hb::fail(halide_error_code_host_is_null, "copy_to_host: host pointer is null");
    if (!buf->device) return hb::fail(halide_error_code_no_device_interface, "copy_to_host: no device allocation");
    int r = copy_span(buf, true);
    if (r) return r;
    cudaError_t e = cudaStreamSynchronize(hb::stream());
    if (e != cudaSuccess) {
        return hb::fail(halide_error_code_copy_to_host_failed, "CUDA: copy_to_host failed: %s", cudaGetErrorString(e));
    }
    buf->flags &= ~(uint64_t)halide_buffer_flag_device_dirty;
    return 0;
}

int if_copy_to_device(void *uc, halide_buffer_t *buf, const halide_device_interface_t *iface) {
    if (!buf) return hb::fail(halide_error_code_buffer_is_null, "copy_to_device: buffer is null");
    bool fresh = buf->device == 0;
    int r = if_device_malloc(uc, buf, iface);
    if (r) return r;
    if (buf->flags & halide_buffer_flag_host_dirty) {
        if (buf->flags & halide_buffer_flag_device_dirty) {
            return hb::fail(halide_error_code_host_and_device_dirty, "copy_to_device: buffer is dirty on both host and device");
        }
        if (!buf->host) return hb::fail(halide_error_code_host_is_null, "copy_to_device: host pointer is null");
        r = copy_span(buf, false);
        if (r) return r;
        buf->flags &= ~(uint64_t)halide_buffer_flag_host_dirty;
    } else if (fresh && buf->host) {
        // A brand-new device allocation has no contents yet; the host copy is the truth.
        r = copy_span(buf, false);
        if (r) return r;
    }
    return 0;
}

int if_device_and_host_malloc(void *uc, halide_buffer_t *buf, const halide_device_interface_t *iface) {
    int64_t lo, hi;
    span_elems(buf, &lo, &hi);
    size_t eb = hb::elem_bytes(buf);
    size_t bytes = (size_t)(hi - lo + 1) * eb;
    void *h = nullptr;
    if (cudaMallocHost(&h, bytes) != cudaSuccess) {
        cudaGetLastError();
        return hb::fail(halide_error_code_device_malloc_failed, "CUDA: pinned host allocation of %zu bytes failed", bytes);
    }
    buf->host = (uint8_t *)h - lo * (int64_t)eb;
    int r = if_device_malloc(uc, buf, iface);
    if (r) {
        cudaFreeHost(h);
        buf->host = nullptr;
    }
    return r;
}

int if_device_and_host_free(void *uc, halide_buffer_t *buf) {
    if (buf->host) {
        int64_t lo, hi;
        span_elems(buf, &lo, &hi);
        cudaFreeHost(buf->host + lo * (int64_t)hb::elem_bytes(buf));
        buf->host = nullptr;
    }
    return if_device_free(uc, buf);
}

// halide_buffer_copy (src/runtime/device_interface.cpp:154-205, cuda.cpp:884-1017): copy the region `dst` describes out of
// `src` (which must cover it) — from the device side of src when that is the valid copy, to the device side of dst when
// dst_iface is this interface, to its host side when dst_iface is null.  Dirty bits follow the reference's rules.
int if_buffer_copy(void *uc, halide_buffer_t *src, const halide_device_interface_t *dst_iface, halide_buffer_t *dst) {
    if (!src || !dst) return hb::fail(halide_error_code_buffer_is_null, "buffer_copy: buffer is null");
    if (dst_iface && dst_iface != &g_cuda_interface) {
        return hb::fail(halide_error_code_incompatible_device_interface, "buffer_copy: destination interface is not this runtime's");
    }
    if (src->dimensions != dst->dimensions || src->type.bits != dst->type.bits || src->dimensions > 8) {
        return hb::fail(halide_error_code_device_buffer_copy_failed, "buffer_copy: source and destination differ in dimensions or element size");
    }
    const bool from_host = src->device == 0 || (src->flags & halide_buffer_flag_host_dirty) ||
                           (src->host != nullptr && !(src->flags & halide_buffer_flag_device_dirty));
    const bool to_host = dst_iface == nullptr;
    if (from_host && !src->host) return hb::fail(halide_error_code_host_is_null, "buffer_copy: source has no valid copy");
    if (to_host && !dst->host) return hb::fail(halide_error_code_host_is_null, "buffer_copy: destination host pointer is null");
    if (!to_host) {
        int r = if_device_malloc(uc, dst, dst_iface);
        if (r) return r;
    }
    const size_t eb = hb::elem_bytes(src);
    CopyDim dims[8];
    int64_t src_off = 0;
    for (int d = 0; d < src->dimensions; d++) {
        const int lo = dst->dim[d].min, ext = dst->dim[d].extent;
        if (ext > 0 && (lo < src->dim[d].min || lo + ext > src->dim[d].min + src->dim[d].extent)) {
            return hb::fail(halide_error_code_access_out_of_bounds, "buffer_copy: destination region [%d, %d] of dimension %d is outside the source [%d, %d]",
                            lo, lo + ext - 1, d, src->dim[d].min, src->dim[d].min + src->dim[d].extent - 1);
        }
        src_off += (int64_t)(lo - src->dim[d].min) * src->dim[d].stride * (int64_t)eb;
        dims[d] = {ext, (int64_t)src->dim[d].stride * (int64_t)eb, (int64_t)dst->dim[d].stride * (int64_t)eb};
    }
    const uint8_t *sp = (from_host ? src->host : (const uint8_t *)src->device) + src_off;
    uint8_t *dp = to_host ? dst->host : (uint8_t *)dst->device;
    const cudaMemcpyKind kind = from_host ? (to_host ? cudaMemcpyHostToHost : cudaMemcpyHostToDevice)
                                          : (to_host ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice);
    int r = copy_nd(dp, sp, dims, src->dimensions, eb, kind, hb::stream());
    if (r) return r;
    if (to_host || from_host) {  // host memory involved: the caller may touch it as soon as we return
        cudaError_t e = cudaStreamSynchronize(hb::stream());
        if (e != cudaSuccess) return hb::fail(halide_error_code_device_buffer_copy_failed, "CUDA: buffer_copy failed: %s", cudaGetErrorString(e));
    }
    if (to_host) {
        dst->flags |= halide_buffer_flag_host_dirty;
        dst->flags &= ~(uint64_t)halide_buffer_flag_device_dirty;
    } else {
        dst->flags |= halide_buffer_flag_device_dirty;
        dst->flags &= ~(uint64_t)halide_buffer_flag_host_dirty;
    }
    return 0;
}
int if_device_crop(void *uc, const halide_buffer_t *src, halide_buffer_t *dst) {
    // Same allocation, shifted handle: dst->dim already holds the cropped mins.
    int64_t off = 0;
    for (int d = 0; d < src->dimensions; d++) {
        off += (int64_t)(dst->dim[d].min - src->dim[d].min) * src->dim[d].stride;
    }
    dst->device = src->device + off * hb::elem_bytes(src);
    dst->device_interface = src->device_interface;
    return 0;
}
int if_device_slice(void *uc, const halide_buffer_t *src, int slice_dim, int slice_pos, halide_buffer_t *dst) {
    int64_t off = (int64_t)(slice_pos - src->dim[slice_dim].min) * src->dim[slice_dim].stride;
    dst->device = src->device + off * hb::elem_bytes(src);
    dst->device_interface = src->device_interface;
    return 0;
}
int if_device_release_crop(void *uc, halide_buffer_t *buf) {
    buf->device = 0;
    buf->device_interface = nullptr;
    return 0;
}
int if_wrap_native(void *uc, halide_buffer_t *buf, uint64_t handle, const halide_device_interface_t *iface) {
    if (buf->device) {
        return hb::fail(halide_error_code_device_wrap_native_failed, "wrap_native: buffer already has a device allocation");
    }
    buf->device = handle;
    buf->device_interface = &g_cuda_interface;
    return 0;
}
int if_detach_native(void *uc, halide_buffer_t *buf) {
    buf->device = 0;
    buf->device_interface = nullptr;
    return 0;
}
int if_compute_capability(void *uc, int *major, int *minor) {
    int dev = 0;
    cudaDeviceProp prop;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaGetDeviceProperties(&prop, dev) != cudaSuccess) {
        cudaGetLastError();
        return hb::fail(halide_error_code_gpu_device_error, "CUDA: no usable device");
    }
    *major = prop.major;
    *minor = prop.minor;
    return 0;
}

const halide_device_interface_t g_cuda_interface = {
    if_device_malloc, if_device_free, if_device_sync, if_device_release, if_copy_to_host, if_copy_to_device,
    if_device_and_host_malloc, if_device_and_host_free, if_buffer_copy, if_device_crop, if_device_slice,
    if_device_release_crop, if_wrap_native, if_detach_native, if_compute_capability, nullptr};

}  // namespace

// ------------------------------------------------------------------------------------------------
namespace hb {

int fail(int code, const char *fmt, ...) {
    char msg[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(msg, sizeof(msg), fmt, ap);
    va_end(ap);
    halide_error(nullptr, msg);
    return code;
}

cudaStream_t stream() {
    return t_stream;
}

int check_cuda(cudaError_t e, const char *what, int code) {
    if (e == cudaSuccess) return 0;
    return fail(code, "CUDA: %s failed: %s", what, cudaGetErrorString(e));
}

void count_launch(const char *name, cudaStream_t s) {
    g_launches.fetch_add(1, std::memory_order_relaxed);
    profile_begin(name, s);
}

// The event bracket alone (for stream work that is not one of this library's kernels, e.g. an NCCL group): shows up in the
// per-kernel profile, not in halide_b200_kernel_launch_count.
void profile_begin(const char *name, cudaStream_t s) {
    if (g_prof_on.load(std::memory_order_relaxed)) {
        cudaEvent_t e0, e1;
        cudaEventCreate(&e0);
        cudaEventCreate(&e1);
        cudaEventRecord(e0, s);
        t_prof_e1 = e1;
        std::lock_guard<std::mutex> lock(g_prof_mu);
        g_prof_pending.push_back({name, e0, e1});
    }
}

void after_launch(cudaStream_t s) {
    if (t_prof_e1) {
        cudaEventRecord(t_prof_e1, s);
        t_prof_e1 = nullptr;
    }
}

CallTimer::CallTimer(cudaStream_t s_) : s(s_) {
    if (g_timing_on.load(std::memory_order_relaxed)) {
        if (!t_call_e0) {
            cudaEventCreate(&t_call_e0);
            cudaEventCreate(&t_call_e1);
        }
        cudaEventRecord(t_call_e0, s);
    }
}
CallTimer::~CallTimer() {
    if (g_timing_on.load(std::memory_order_relaxed) && t_call_e0) {
        cudaEventRecord(t_call_e1, s);
        t_call_valid = true;
    }
}

void *scratch_alloc(size_t bytes) {
    return pool().alloc(bytes);
}
void scratch_free(void *p) {
    pool().free(p);
}
void *debug_fill(void *p, size_t bytes, cudaStream_t s) {
    const int b = g_fill_byte.load(std::memory_order_relaxed);
    if (p && b >= 0) cudaMemsetAsync(p, b, bytes, s);
    return p;
}

static const char *kind(const ArgSpec &s) {
    return s.is_output ? "Output" : "Input";
}

int check_arg(const halide_buffer_t *b, const ArgSpec &spec) {
    if (!b) {
        return fail(halide_error_code_buffer_argument_is_null, "Buffer argument %s is nullptr", spec.name);
    }
    // Compare code+bits only: this reference keeps the upper 16 bits reserved=0 while Halide
    // releases store lanes=1 there (SURVEY.md §8b "Type word").
    if (b->type.code != spec.code || b->type.bits != spec.bits) {
        return fail(halide_error_code_bad_type, "%s buffer %s has type code %d bits %d but expected code %d bits %d",
                    kind(spec), spec.name, b->type.code, b->type.bits, spec.code, spec.bits);
    }
    if (b->dimensions != spec.dimensions) {
        return fail(halide_error_code_bad_dimensions, "%s buffer %s requires a buffer of exactly %d dimensions, but the buffer passed in has %d dimensions",
                    kind(spec), spec.name, spec.dimensions, b->dimensions);
    }
    if (b->dimensions > 0 && !b->dim) {
        return fail(halide_error_code_buffer_is_null, "%s buffer %s has a null dim array", kind(spec), spec.name);
    }
    return 0;
}

int check_shape(const halide_buffer_t *b, const ArgSpec &spec) {
    int64_t total = 1;
    for (int d = 0; d < b->dimensions; d++) {
        const halide_dimension_t &dm = b->dim[d];
        if (dm.extent < 0) {
            return fail(halide_error_code_buffer_extents_negative, "The extents for buffer %s dimension %d is negative (%d)",
                        spec.name, d, dm.extent);
        }
        int64_t stride = dm.stride < 0 ? -(int64_t)dm.stride : dm.stride;
        int64_t sz = (int64_t)dm.extent * stride;
        if (sz > 0x7fffffffLL) {
            return fail(halide_error_code_buffer_allocation_too_large,
                        "Total allocation for buffer %s is %lld, which exceeds the maximum size of 2147483647",
                        spec.name, (long long)sz);
        }
        total *= dm.extent;
        if (total > 0x7fffffffLL) {
            return fail(halide_error_code_buffer_extents_too_large,
                        "Product of extents for buffer %s is %lld, which exceeds the maximum size of 2147483647",
                        spec.name, (long long)total);
        }
    }
    if (b->dimensions > 0 && b->dim[0].stride != 1) {
        return fail(halide_error_code_constraint_violated, "Constraint violated: %s.stride.0 (%d) == 1 (1)",
                    spec.name, b->dim[0].stride);
    }
    return 0;
}

int check_covers(const halide_buffer_t *b, const ArgSpec &spec, int d, int req_min, int req_extent) {
    if (req_extent <= 0) return 0;
    const halide_dimension_t &dm = b->dim[d];
    int req_max = req_min + req_extent - 1;
    int have_max = dm.min + dm.extent - 1;
    if (req_min < dm.min || req_max > have_max) {
        return fail(halide_error_code_access_out_of_bounds,
                    "%s buffer %s is accessed at %d, which is %s the %s (%d) in dimension %d",
                    kind(spec), spec.name, req_min < dm.min ? req_min : req_max,
                    req_min < dm.min ? "before" : "beyond", req_min < dm.min ? "min" : "max",
                    req_min < dm.min ? dm.min : have_max, d);
    }
    return 0;
}

void propose_shape(halide_buffer_t *b, const int *mins, const int *extents) {
    int64_t stride = 1;
    for (int d = 0; d < b->dimensions; d++) {
        b->dim[d].min = mins[d];
        b->dim[d].extent = extents[d];
        b->dim[d].stride = (int32_t)stride;
        stride *= extents[d];
    }
}

int acquire_input(halide_buffer_t *b, const ArgSpec &spec, void **dev_ptr) {
    if (b->device && b->device_interface != &g_cuda_interface) {
        return fail(halide_error_code_incompatible_device_interface,
                    "Input buffer %s has a device allocation of a different device interface", spec.name);
    }
    if (!b->device && !b->host) {
        return fail(halide_error_code_host_is_null, "Input buffer %s has neither host nor device memory", spec.name);
    }
    int r = if_copy_to_device(nullptr, b, &g_cuda_interface);
    if (r) return r;
    *dev_ptr = (void *)b->device;
    return 0;
}

int acquire_output(halide_buffer_t *b, const ArgSpec &spec, void **dev_ptr) {
    if (b->device && b->device_interface != &g_cuda_interface) {
        return fail(halide_error_code_incompatible_device_interface,
                    "Output buffer %s has a device allocation of a different device interface", spec.name);
    }
    int r = if_device_malloc(nullptr, b, &g_cuda_interface);
    if (r) return r;
    *dev_ptr = (void *)b->device;
    return 0;
}

void mark_output_written(halide_buffer_t *b) {
    b->flags &= ~(uint64_t)halide_buffer_flag_host_dirty;
    b->flags |= halide_buffer_flag_device_dirty;
}

}  // namespace hb

// ------------------------------------------------------------------------------------------------
extern "C" {

void halide_error(void *user_context, const char *msg) {
    halide_error_handler_t h = g_handler.load();
    if (h) {
        h(user_context, msg);
        return;
    }
    // Default behaviour of the reference runtime: print and abort (posix_error_handler.cpp:9-41).
    fprintf(stderr, "Error: %s\n", msg);
    abort();
}

halide_error_handler_t halide_set_error_handler(halide_error_handler_t handler) {
    return g_handler.exchange(handler);
}

// Host allocator hooks (HalideRuntime.h halide_set_custom_malloc/free; tools/halide_malloc_trace.h installs tracing
// versions through them).  The filters allocate no host memory, so the hooks are only recorded.
static std::atomic<halide_malloc_t> g_malloc{nullptr};
static std::atomic<halide_free_t> g_free{nullptr};
halide_malloc_t halide_set_custom_malloc(halide_malloc_t user_malloc) {
    return g_malloc.exchange(user_malloc);
}
halide_free_t halide_set_custom_free(halide_free_t user_free) {
    return g_free.exchange(user_free);
}
// Default host allocator of the reference runtime: 128-byte aligned (src/runtime/posix_allocator.cpp); tools/RunGenMain.cpp
// wraps it for its allocation statistics.
void *halide_default_malloc(void *user_context, size_t x) {
    void *p = nullptr;
    if (posix_memalign(&p, 128, x ? x : 1) != 0) return nullptr;
    return p;
}
void halide_default_free(void *user_context, void *ptr) {
    free(ptr);
}
void *halide_malloc(void *user_context, size_t x) {
    halide_malloc_t m = g_malloc.load();
    return m ? m(user_context, x) : halide_default_malloc(user_context, x);
}
void halide_free(void *user_context, void *ptr) {
    halide_free_t f = g_free.load();
    if (f) f(user_context, ptr);
    else halide_default_free(user_context, ptr);
}
// halide_print hook (HalideRuntime.h:170-181)
static std::atomic<halide_print_t> g_print{nullptr};
halide_print_t halide_set_custom_print(halide_print_t print) {
    return g_print.exchange(print);
}
void halide_print(void *user_context, const char *msg) {
    halide_print_t p = g_print.load();
    if (p) p(user_context, msg);
    else fputs(msg, stderr);
}
// Device allocations are always pooled here (src/runtime/cuda.cpp:760-870 keeps them when enabled); switching reuse off
// just returns the cached blocks to the driver.
int halide_reuse_device_allocations(void *user_context, bool enable) {
    if (!enable) pool().release_unused();
    return 0;
}
void *halide_get_symbol(const char *name) {
    return dlsym(RTLD_DEFAULT, name);
}

int halide_device_malloc(void *uc, halide_buffer_t *buf, const halide_device_interface_t *iface) {
    if (!iface) iface = &g_cuda_interface;
    return iface->device_malloc(uc, buf, iface);
}
int halide_device_free(void *uc, halide_buffer_t *buf) {
    if (!buf) return hb::fail(halide_error_code_buffer_is_null, "halide_device_free: buffer is null");
    if (!buf->device_interface) return 0;
    return buf->device_interface->device_free(uc, buf);
}
int halide_device_sync(void *uc, halide_buffer_t *buf) {
    return if_device_sync(uc, buf);
}
int halide_copy_to_host(void *uc, halide_buffer_t *buf) {
    if (!buf) return hb::fail(halide_error_code_buffer_is_null, "halide_copy_to_host: buffer is null");
    if (!buf->device_interface) {
        if (buf->flags & halide_buffer_flag_device_dirty) {
            return hb::fail(halide_error_code_no_device_interface, "halide_copy_to_host: device dirty but no device interface");
        }
        return 0;
    }
    return buf->device_interface->copy_to_host(uc, buf);
}
int halide_copy_to_device(void *uc, halide_buffer_t *buf, const halide_device_interface_t *iface) {
    if (!iface) iface = &g_cuda_interface;
    return iface->copy_to_device(uc, buf, iface);
}
// src/runtime/device_interface.cpp:154-205: a null dst_device_interface means "to the host side of dst".
int halide_buffer_copy(void *uc, halide_buffer_t *src, const halide_device_interface_t *dst_iface, halide_buffer_t *dst) {
    return if_buffer_copy(uc, src, dst_iface, dst);
}
void halide_device_release(void *uc, const halide_device_interface_t *iface) {
    if_device_release(uc, iface);
}

const halide_device_interface_t *halide_cuda_device_interface(void) {
    return &g_cuda_interface;
}
int halide_cuda_wrap_device_ptr(void *uc, halide_buffer_t *buf, uint64_t device_ptr) {
    return if_wrap_native(uc, buf, device_ptr, &g_cuda_interface);
}
int halide_cuda_detach_device_ptr(void *uc, halide_buffer_t *buf) {
    return if_detach_native(uc, buf);
}
uintptr_t halide_cuda_get_device_ptr(void *uc, halide_buffer_t *buf) {
    return (uintptr_t)buf->device;
}
int halide_cuda_release_unused_device_allocations(void *uc) {
    pool().release_unused();
    return 0;
}

void halide_b200_set_stream(void *s) {
    t_stream = (cudaStream_t)s;
}
void *halide_b200_get_stream(void) {
    return (void *)t_stream;
}
void *halide_b200_stream_create(void) {
    cudaStream_t s = nullptr;
    if (cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) != cudaSuccess) {
        hb::fail(halide_error_code_gpu_device_error, "CUDA: stream creation failed: %s", cudaGetErrorString(cudaGetLastError()));
        return nullptr;
    }
    return (void *)s;
}
int halide_b200_stream_destroy(void *stream) {
    if (!stream) return 0;
    cudaStream_t s = (cudaStream_t)stream;
    cudaStreamSynchronize(s);
    if (t_stream == s) t_stream = nullptr;
    if (cudaStreamDestroy(s) != cudaSuccess) {
        return hb::fail(halide_error_code_gpu_device_error, "CUDA: stream destroy failed: %s", cudaGetErrorString(cudaGetLastError()));
    }
    return 0;
}
int halide_b200_set_device(int ordinal) {
    cudaError_t e = cudaSetDevice(ordinal);
    if (e != cudaSuccess) {
        return hb::fail(halide_error_code_gpu_device_error, "CUDA: cudaSetDevice(%d) failed: %s", ordinal, cudaGetErrorString(e));
    }
    return 0;
}
uint64_t halide_b200_kernel_launch_count(void) {
    return g_launches.load();
}
const char *halide_b200_target(void) {
    return "x86-64-linux-cuda-cuda_capability_100-b200_native";
}

void halide_b200_debug_fill_allocations(int byte) {
    g_fill_byte.store(byte >= 0 && byte <= 255 ? byte : -1);
}

void halide_b200_set_timing(int enable) {
    g_timing_on.store(enable);
}
float halide_b200_last_kernel_ms(void) {
    if (!t_call_valid) return -1.f;
    cudaEventSynchronize(t_call_e1);
    float ms = -1.f;
    cudaEventElapsedTime(&ms, t_call_e0, t_call_e1);
    return ms;
}

void halide_b200_profile_enable(int enable) {
    g_prof_on.store(enable);
}
void halide_b200_profile_reset(void) {
    std::lock_guard<std::mutex> lock(g_prof_mu);
    prof_drain_locked();
    g_prof_totals.clear();
}
int halide_b200_profile_report(char *out, int out_size) {
    std::lock_guard<std::mutex> lock(g_prof_mu);
    prof_drain_locked();
    std::string s;
    char line[256];
    for (auto &kv : g_prof_totals) {
        snprintf(line, sizeof(line), "%s %d %.6f\n", kv.first.c_str(), kv.second.first, kv.second.second);
        s += line;
    }
    if (out && out_size > 0) {
        int n = (int)s.size() < out_size - 1 ? (int)s.size() : out_size - 1;
        memcpy(out, s.data(), n);
        out[n] = 0;
    }
    return (int)s.size() + 1;
}

}  // extern "C"
