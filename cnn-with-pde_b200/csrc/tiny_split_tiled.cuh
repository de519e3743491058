// Host interface of the line-streaming kernels for tiny_imagenet's dormant methods (tiny_split_tiled.cu): planes of
// any shape up to kMaxEdge x kMaxEdge, element-aligned I/O.  tiny_split.cu decides which planes come here
// (tsplit_on_chip).
#pragma once

#include <cuda_runtime.h>

#include "common.cuh"

namespace pde {
namespace tsplit_tiled {

constexpr int kMaxEdge = 4096;

// d valid, 1 <= H, W <= kMaxEdge, d->B > 0; u and out element-aligned (they may be one buffer in modes 0-2 and must
// not overlap in modes 3-4)
int tiny_split_tiled(const pde_tiny_split_desc *d, const float *u, float *out, const DeviceProps &props,
                     cudaStream_t st);

}  // namespace tsplit_tiled
}  // namespace pde
