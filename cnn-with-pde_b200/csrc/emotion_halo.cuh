// Host interface of the halo-tiled emotion kernels (emotion_halo.cu): square planes from 65 x 65 up to
// kHaloMaxN x kHaloMaxN, up to kHaloMaxSteps steps, element-aligned fp32 or bf16 I/O.  explicit.cu decides which
// descriptors come here (emo_route).
#pragma once

#include <cuda_runtime.h>

#include "common.cuh"

namespace pde {
namespace halo {

constexpr int kHaloMaxN = 4096;
constexpr int kHaloMaxSteps = 16;
constexpr size_t kHaloWorkspaceCap = (size_t)1 << 30;   // per-chunk workspace the backward aims to stay under

// the halo kernels' domain, for a descriptor emo_validate did not call invalid and whose plane is too large for
// the whole-plane kernels
inline bool emo_halo_domain(const pde_emo_desc *d) { return d->N <= kHaloMaxN && d->Nt <= kHaloMaxSteps; }

// bytes pde_emotion_backward(_bf16) uses on this path (a function of the descriptor and the I/O type's size only)
size_t emo_halo_workspace_bytes(const pde_emo_desc *d, int io_bytes);

// d->B > 0; pointers need only be element-aligned.  T: float or __nv_bfloat16 (instantiated in emotion_halo.cu)
template <typename T>
int emo_halo_forward(const pde_emo_desc *d, const T *u0, const float *w6, const float *xs, const float *ys, T *out,
                     const DeviceProps &props, cudaStream_t st);
template <typename T>
int emo_halo_backward(const pde_emo_desc *d, const T *u0, const T *gout, const float *w6, const float *xs,
                      const float *ys, T *gin, float *g_w6, void *workspace, size_t workspace_bytes,
                      const DeviceProps &props, cudaStream_t st);

}  // namespace halo
}  // namespace pde
