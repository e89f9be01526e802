// oracle/oracle_apps.h — TEST INFRASTRUCTURE, NOT PRODUCT CODE.
//
// C entry points of the CPU oracle for the apps beyond the seven pipelines of oracle.h (the same image view, the same
// conventions: every Func is evaluated on the box its consumers touch, f32 expressions in source nesting with IEEE
// rounding and no contraction).  Built into liboracle_apps.so by oracle/apps.mk; bound by oracle/pyoracle_apps.py.
#pragma once
#include "oracle.h"

#ifdef __cplusplus
extern "C" {
#endif

// apps/harris/harris_generator.cpp:22-61.  in: f32 3-D, out: f32 2-D.  No boundary condition: returns -4 unless in
// covers x in [x0-2, x0+W+1], the same in y, and channels 0..2.
int oracle_harris(const oracle_image_t *in, const oracle_image_t *out);

// apps/unsharp/unsharp_generator.cpp:15-51 (sigma 1.5).  in, out: f32 3-D.  gray reads repeat_edge(in) (x, y and c
// clamped to in's box); the final multiply reads in unclamped, so in must cover out's (x, y, c) box, else -4.
int oracle_unsharp(const oracle_image_t *in, const oracle_image_t *out);

// The four folded weights kernel(0..3) of unsharp (oracle_unsharp.cpp explains the derivation).
void oracle_unsharp_weights(float *w4);

#ifdef __cplusplus
}
#endif
