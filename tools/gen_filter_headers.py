"""Writes include/<filter>.h (+ _auto_schedule variants) — the stand-ins for the headers Halide's
AOT compiler emits.  Run with the filter names to (re)generate: python tools/gen_filter_headers.py stencil_chain"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FILTERS = {
    "halide_blur": ("apps/blur/halide_blur_generator.cpp:31-40,117",
                    "struct halide_buffer_t *input, struct halide_buffer_t *blur_y", False),
    "local_laplacian": ("apps/local_laplacian/local_laplacian_generator.cpp:12-16,287",
                        "struct halide_buffer_t *input, int32_t levels, float alpha, float beta, struct halide_buffer_t *output", True),
    "bilateral_grid": ("apps/bilateral_grid/bilateral_grid_generator.cpp:8-16,203",
                       "struct halide_buffer_t *input, float r_sigma, struct halide_buffer_t *bilateral_grid", True),
    "nl_means": ("apps/nl_means/nl_means_generator.cpp:9-18,162",
                 "struct halide_buffer_t *input, int32_t patch_size, int32_t search_area, float sigma, struct halide_buffer_t *non_local_means", True),
    "stencil_chain": ("apps/stencil_chain/stencil_chain_generator.cpp:7-14,150",
                      "struct halide_buffer_t *input, struct halide_buffer_t *output", True),
    "conv_layer": ("apps/conv_layer/conv_layer_generator.cpp:9-16,207",
                   "struct halide_buffer_t *input, struct halide_buffer_t *filter, struct halide_buffer_t *bias, struct halide_buffer_t *relu", True),
    "camera_pipe": ("apps/camera_pipe/camera_pipe_generator.cpp:218-238,622",
                    "struct halide_buffer_t *input, struct halide_buffer_t *matrix_3200, struct halide_buffer_t *matrix_7000, float color_temp, float gamma, float contrast, float sharpen_strength, int32_t blackLevel, int32_t whiteLevel, struct halide_buffer_t *processed", True),
    "harris": ("apps/harris/harris_generator.cpp:15-16,131",
               "struct halide_buffer_t *input, struct halide_buffer_t *output", True),
    "unsharp": ("apps/unsharp/unsharp_generator.cpp:7-10,114",
                "struct halide_buffer_t *input, struct halide_buffer_t *output", True),
}


def emit(name):
    cite, args, has_auto = FILTERS[name]
    for suffix in (("", "_auto_schedule") if has_auto else ("",)):
        fn = name + suffix
        guard = "HALIDE_B200_" + fn.upper() + "_H"
        note = "" if not suffix else (
            f" * `{fn}` is the second AOT variant the harness links (the app harness, when built without\n"
            f" * -DNO_AUTO_SCHEDULE calls it); here it is the same sm_100a implementation under the second name.\n")
        with open(os.path.join(ROOT, "include", fn + ".h"), "w") as f:
            f.write(f"""/* {fn}.h — stands in for the header Halide's AOT compiler emits for this filter
 * (src/CodeGen_C.cpp:1083-1108 argument order: generator inputs in declaration order, then outputs;
 *  src/CodeGen_C.cpp:675-721 for the _argv and _metadata companions).
 * Generator: /root/reference/{cite}
{note} * Returns 0 or a negative halide_error_code_t (include/halide_b200_runtime.h).
 */
#ifndef {guard}
#define {guard}

#include <stdint.h>

struct halide_buffer_t;
struct halide_filter_metadata_t;

#ifdef __cplusplus
extern "C" {{
#endif

int {fn}({args});
int {fn}_argv(void **args);
const struct halide_filter_metadata_t *{fn}_metadata(void);

#ifdef __cplusplus
}}
#endif

#endif /* {guard} */
""")


if __name__ == "__main__":
    for n in sys.argv[1:]:
        emit(n)
