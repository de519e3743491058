// Host interface of the tiled tiny_imagenet kernels (tiny_tiled.cu): planes of any shape up to
// kTiledMaxEdge x kTiledMaxEdge, up to kTiledMaxSteps steps, element-aligned I/O.  explicit.cu decides which
// configurations come here (tiny_route).
#pragma once

#include <cuda_runtime.h>

#include "common.cuh"

namespace pde {
namespace tiled {

constexpr int kTiledMaxEdge = 4096;
constexpr int kTiledMaxSteps = 16;
constexpr int kTiledMaxChannels = 1024;

// the tiled kernels' domain, for a descriptor tiny_validate did not call invalid
inline bool tiny_tiled_domain(const pde_tiny_desc *d) {
    return d->H <= kTiledMaxEdge && d->W <= kTiledMaxEdge && d->steps <= kTiledMaxSteps && d->C <= kTiledMaxChannels;
}

// backward workspace: one double (alpha, scaling) partial pair per block, for any grid the launcher may pick
inline size_t tiny_tiled_workspace_bytes(const pde_tiny_desc *d, int sm_count) {
    return ((size_t)sm_count * 8 + (size_t)d->C) * 2 * sizeof(double) + 256;
}

// io_bytes: 4 (fp32 planes) or 2 (bf16 planes); pointers need only be element-aligned; d->B > 0
int tiny_tiled_forward(const pde_tiny_desc *d, int io_bytes, const void *u, const float *alpha, const float *scal,
                       void *out, const DeviceProps &props, cudaStream_t st);
int tiny_tiled_backward(const pde_tiny_desc *d, int io_bytes, const void *u, const void *gout, const float *alpha,
                        const float *scal, void *gin, float *g_alpha, float *g_scal, void *workspace,
                        size_t workspace_bytes, const DeviceProps &props, cudaStream_t st);

}  // namespace tiled
}  // namespace pde
