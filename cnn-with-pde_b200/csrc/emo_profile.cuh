// The row / column coefficient profiles of emotion_recognition.PDELayer, shared by every emotion kernel
// (explicit.cu, emotion_tiled.cuh, emotion_halo.cu) so that all plane sizes use identical coefficient arithmetic,
// and the plane loads / stores of those kernels in either I/O type.
#pragma once

#include <cuda_bf16.h>

#include "common.cuh"

namespace pde {
namespace expl {

// Plane I/O of the emotion kernels: fp32 or bf16 planes in HBM, fp32 everywhere else.  A bf16 value is widened
// exactly on load; a result is rounded once, to nearest even, on its store.
__device__ __forceinline__ float io_widen(float v) { return v; }
__device__ __forceinline__ float io_widen(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T>
__device__ __forceinline__ T io_round(float v) {
    if constexpr (sizeof(T) == 4) return v;
    else return __float2bfloat16_rn(v);
}
template <typename T>
__device__ __forceinline__ float io_ldg(const T *p) { return io_widen(__ldg(p)); }
template <typename T>
__device__ __forceinline__ float io_ldcs(const T *p) { return io_widen(__ldcs(p)); }
template <typename T>
__device__ __forceinline__ void io_stcs(T *p, float v) { __stcs(p, io_round<T>(v)); }

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
