// The row / column coefficient profiles of emotion_recognition.PDELayer, shared by every emotion kernel
// (explicit.cu, emotion_tiled.cuh, emotion_halo.cu) so that all plane sizes use identical coefficient arithmetic.
#pragma once

#include "common.cuh"

namespace pde {
namespace expl {

// a_i = 0.5 dt (w1 + w2 sin 2 pi y_i + w3 sin 4 pi y_i) / dx^2     emotion_recognition.py:76-77
// b_j =     dt (w1 + w2 cos 2 pi x_j + w3 cos 4 pi x_j) / dy^2     emotion_recognition.py:79-80
// evaluated in the reference's order with correctly rounded fp32 ops (no contraction).
__device__ __forceinline__ void emo_profile(const pde_emo_desc &d, const float *__restrict__ w6,
                                            const float *__restrict__ xs, const float *__restrict__ ys, int i,
                                            float *a, float *b) {
    const float two_pi = (float)(2.0 * 3.141592653589793), four_pi = (float)(4.0 * 3.141592653589793);
    const float y = ys[i], x = xs[i];
    const float s1 = sinf(__fmul_rn(two_pi, y)), s2 = sinf(__fmul_rn(four_pi, y));
    const float c1 = cosf(__fmul_rn(two_pi, x)), c2 = cosf(__fmul_rn(four_pi, x));
    const float sa = __fadd_rn(__fadd_rn(w6[0], __fmul_rn(w6[1], s1)), __fmul_rn(w6[2], s2));
    const float sb = __fadd_rn(__fadd_rn(w6[3], __fmul_rn(w6[4], c1)), __fmul_rn(w6[5], c2));
    *a = __fdiv_rn(__fmul_rn(d.half_dt, sa), d.dx2);
    *b = __fdiv_rn(__fmul_rn(d.dt, sb), d.dy2);
}

}  // namespace expl
}  // namespace pde
