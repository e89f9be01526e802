/* harris.h — stands in for the header Halide's AOT compiler emits for this filter
 * (src/CodeGen_C.cpp:1083-1108 argument order: generator inputs in declaration order, then outputs;
 *  src/CodeGen_C.cpp:675-721 for the _argv and _metadata companions).
 * Generator: /root/reference/apps/harris/harris_generator.cpp:15-16,131
 * Returns 0 or a negative halide_error_code_t (include/halide_b200_runtime.h).
 */
#ifndef HALIDE_B200_HARRIS_H
#define HALIDE_B200_HARRIS_H

#include <stdint.h>

struct halide_buffer_t;
struct halide_filter_metadata_t;

#ifdef __cplusplus
extern "C" {
#endif

int harris(struct halide_buffer_t *input, struct halide_buffer_t *output);
int harris_argv(void **args);
const struct halide_filter_metadata_t *harris_metadata(void);

#ifdef __cplusplus
}
#endif

#endif /* HALIDE_B200_HARRIS_H */
