/* unsharp.h — stands in for the header Halide's AOT compiler emits for this filter
 * (src/CodeGen_C.cpp:1083-1108 argument order: generator inputs in declaration order, then outputs;
 *  src/CodeGen_C.cpp:675-721 for the _argv and _metadata companions).
 * Generator: /root/reference/apps/unsharp/unsharp_generator.cpp:7-10,114
 * Returns 0 or a negative halide_error_code_t (include/halide_b200_runtime.h).
 */
#ifndef HALIDE_B200_UNSHARP_H
#define HALIDE_B200_UNSHARP_H

#include <stdint.h>

struct halide_buffer_t;
struct halide_filter_metadata_t;

#ifdef __cplusplus
extern "C" {
#endif

int unsharp(struct halide_buffer_t *input, struct halide_buffer_t *output);
int unsharp_argv(void **args);
const struct halide_filter_metadata_t *unsharp_metadata(void);

#ifdef __cplusplus
}
#endif

#endif /* HALIDE_B200_UNSHARP_H */
