// registration.cpp — static-init registration of one filter with a RunGen-style driver, the counterpart of the
// `registration` output of a Halide generator (reference: src/Module.cpp:151-207; consumer tools/RunGenMain.cpp, which
// defines halide_register_argv_and_metadata, HalideRuntime.h:1979-1992).  Compile with -DHB_FILTER=<F> and link with
// libhalide_b200.so into tools/RunGenMain.cpp to get F's RunGen driver.
#ifndef HB_FILTER
#error "compile with -DHB_FILTER=<filter name>"
#endif

#define HB_CAT2(a, b) a##b
#define HB_CAT(a, b) HB_CAT2(a, b)

struct halide_filter_metadata_t;

extern "C" {
int HB_CAT(HB_FILTER, _argv)(void **args);
const struct halide_filter_metadata_t *HB_CAT(HB_FILTER, _metadata)(void);
void halide_register_argv_and_metadata(int (*filter_argv_call)(void **), const struct halide_filter_metadata_t *filter_metadata,
                                       const char *const *extra_key_value_pairs);
}

namespace {
struct Registerer {
    Registerer() {
        halide_register_argv_and_metadata(HB_CAT(HB_FILTER, _argv), HB_CAT(HB_FILTER, _metadata)(), nullptr);
    }
} registerer;
}  // namespace
