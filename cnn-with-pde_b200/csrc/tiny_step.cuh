// The per-cell arithmetic of tiny_imagenet's explicit step, shared by the whole-plane ring kernels (explicit.cu)
// and the tiled kernels (tiny_tiled.cu) so that both compute it op for op alike.
#pragma once

#include "common.cuh"

namespace pde {
namespace expl {

__device__ __forceinline__ float clamp_alpha(const pde_tiny_desc &d, float raw, bool *inside) {
    *inside = raw >= d.cmin && raw <= d.cmax;
    return raw < d.cmin ? d.cmin : (raw > d.cmax ? d.cmax : raw);
}

__device__ __forceinline__ float blend1(float u, float sc, float adt, float lap, float bl) {
    const float v = u * sc;
    const float w = fmaf(adt, lap, v);
    return fmaf(bl, w - u, u);
}

}  // namespace expl
}  // namespace pde
