// unsharp_registration.cpp — static-init registration of the filter with a RunGen-style driver, the counterpart of the
// `registration` output of a Halide generator (reference: src/Module.cpp:151-207; consumer tools/RunGenMain.cpp, which
// defines halide_register_argv_and_metadata, HalideRuntime.h:1979-1992).  Link this file + libhalide_b200.so into
// tools/RunGenMain.cpp to get `unsharp.rungen`.
#include "unsharp.h"

extern "C" void halide_register_argv_and_metadata(int (*filter_argv_call)(void **), const struct halide_filter_metadata_t *filter_metadata,
                                                  const char *const *extra_key_value_pairs);

namespace {
struct Registerer {
    Registerer() {
        halide_register_argv_and_metadata(unsharp_argv, unsharp_metadata(), nullptr);
    }
} registerer;
}  // namespace
