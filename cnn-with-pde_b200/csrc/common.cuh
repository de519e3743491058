// Shared device helpers for libpde_b200.so (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdlib>
#include <map>
#include <mutex>

#include "pde_b200.h"

#define PDE_CUDA_TRY(expr)                          \
    do {                                            \
        cudaError_t e__ = (expr);                   \
        if (e__ != cudaSuccess) return (int)e__;    \
    } while (0)

namespace pde {

constexpr unsigned kFullMask = 0xffffffffu;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFullMask, v, o);
    return v;
}

// Named barrier over `nthreads` threads (a multiple of 32); id 0 is __syncthreads().
__device__ __forceinline__ void named_barrier(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// Streaming (evict-first) 128-bit global accesses for data touched once per kernel.
__device__ __forceinline__ float4 ld_stream(const float4 *p) { return __ldcs(p); }
__device__ __forceinline__ void st_stream(float4 *p, float4 v) { __stcs(p, v); }

inline int cuda_last_error() {
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? PDE_OK : (int)e;
}

inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

struct DeviceProps {
    int sm_count;
    int max_smem_optin;
};

// ------------------------------------------------------------------------------------------
// Launch-attribute cache.  Device properties, a kernel's register count / static shared memory,
// "dynamic shared-memory limit raised" and occupancy answers never change for a (device, kernel)
// pair; asking the runtime on every call costs more host time than the small-batch kernels run.
// Read-mostly, filled on first use under a mutex; it holds nothing a caller can observe.
// ------------------------------------------------------------------------------------------
struct KernelInfo {
    int regs;
    size_t static_smem;
};

namespace detail {
struct KernelKey {
    int dev;
    const void *kern;
    int threads;     // 0 for the attribute entry
    size_t smem;     // 0 for the attribute entry
    bool operator<(const KernelKey &o) const {
        if (dev != o.dev) return dev < o.dev;
        if (kern != o.kern) return kern < o.kern;
        if (threads != o.threads) return threads < o.threads;
        return smem < o.smem;
    }
};
struct KernelEntry {
    KernelInfo info;
    size_t smem_limit;   // largest dynamic shared-memory size the kernel has been opted in to
    int occ;
};
inline std::mutex &cache_mutex() {
    static std::mutex m;
    return m;
}
inline std::map<KernelKey, KernelEntry> &kernel_cache() {
    static std::map<KernelKey, KernelEntry> c;
    return c;
}
inline std::map<int, DeviceProps> &props_cache() {
    static std::map<int, DeviceProps> c;
    return c;
}
}  // namespace detail

inline int query_props(DeviceProps *p) {
    int dev = 0;
    PDE_CUDA_TRY(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(detail::cache_mutex());
    auto &c = detail::props_cache();
    auto it = c.find(dev);
    if (it == c.end()) {
        DeviceProps q;
        PDE_CUDA_TRY(cudaDeviceGetAttribute(&q.sm_count, cudaDevAttrMultiProcessorCount, dev));
        PDE_CUDA_TRY(cudaDeviceGetAttribute(&q.max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
        it = c.emplace(dev, q).first;
    }
    *p = it->second;
    return PDE_OK;
}

// Registers and static shared memory of `kern`; makes sure it may be launched with `smem` bytes of
// dynamic shared memory.
inline int kernel_info(const void *kern, size_t smem, KernelInfo *out) {
    int dev = 0;
    PDE_CUDA_TRY(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(detail::cache_mutex());
    auto &c = detail::kernel_cache();
    const detail::KernelKey key{dev, kern, 0, 0};
    auto it = c.find(key);
    if (it == c.end()) {
        cudaFuncAttributes fa;
        PDE_CUDA_TRY(cudaFuncGetAttributes(&fa, kern));
        detail::KernelEntry e{};
        e.info.regs = fa.numRegs;
        e.info.static_smem = fa.sharedSizeBytes;
        e.smem_limit = 48 * 1024;
        it = c.emplace(key, e).first;
    }
    if (smem > it->second.smem_limit) {
        PDE_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        it->second.smem_limit = smem;
    }
    if (out) *out = it->second.info;
    return PDE_OK;
}

// cudaOccupancyMaxActiveBlocksPerMultiprocessor, remembered (also opts the kernel in to `smem`)
inline int cached_occupancy(const void *kern, int threads, size_t smem, int *per_sm) {
    int rc = kernel_info(kern, smem, nullptr);
    if (rc) return rc;
    int dev = 0;
    PDE_CUDA_TRY(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(detail::cache_mutex());
    auto &c = detail::kernel_cache();
    const detail::KernelKey key{dev, kern, threads, smem + 1};
    auto it = c.find(key);
    if (it == c.end()) {
        detail::KernelEntry e{};
        PDE_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&e.occ, kern, threads, smem));
        if (e.occ < 1) e.occ = 1;
        it = c.emplace(key, e).first;
    }
    *per_sm = it->second.occ;
    return PDE_OK;
}

// PDE_B200_DEBUG=1 prints the launch plans; read once per process (it changes no result)
inline bool debug_enabled() {
    static const bool on = [] {
        const char *v = getenv("PDE_B200_DEBUG");
        return v && *v && *v != '0';
    }();
    return on;
}

}  // namespace pde

// ------------------------------------------------------------------------------------------
// TMA 1-D bulk copy + mbarrier (PTX; SASS: UBLKCP / SYNCS).  Planes are contiguous in NCHW,
// so a whole plane is one bulk copy: size and both addresses must be multiples of 16 bytes.
// ------------------------------------------------------------------------------------------
namespace pde {

__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}

// make the barrier initialisation visible to the async proxy before any TMA refers to it
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}

__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

// global -> shared, completion signalled on `bar` as `bytes` transaction bytes
__device__ __forceinline__ void tma_load_1d(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// shared -> global, tracked in the issuing thread's bulk groups (commit, then wait_group)
__device__ __forceinline__ void tma_store_1d(void *dst_gmem, const void *src_smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// at most N of the thread's bulk groups still read shared memory (their source may then be refilled)
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
// every bulk group of the thread is complete (its global writes done)
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// order prior generic-proxy accesses to shared memory before later async-proxy (TMA) accesses
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

}  // namespace pde

// ------------------------------------------------------------------------------------------
// Tensor memory (TMEM) as lane-private scratch.  512 columns x 128 lanes x 32 bit per SM; a warp
// reaches the 32 lanes of its quadrant (warp % 4), each thread its own lane.  Used by the
// implicit backward kernel to hold the per-pixel gradient accumulators: they are private to a
// lane, too many for registers, and keeping them out of shared memory frees both capacity and
// LSU bandwidth (TMEM has its own datapath; SASS: LDTM / STTM).  Probe: tools/probes/tmem_probe.cu.
// ------------------------------------------------------------------------------------------
namespace pde {

// one warp allocates `cols` (power of two >= 32) columns for the CTA; the base address lands in smem
__device__ __forceinline__ void tmem_alloc(uint32_t *slot, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tmem_fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// 16 consecutive columns of this thread's lane <-> 16 registers (issue only; wait separately)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float *v) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float *v) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(
            taddr),
        "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
        "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
        "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
        "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
        : "memory");
}

}  // namespace pde

// ------------------------------------------------------------------------------------------
// Packed fp32 pairs (PTX .f32x2, SASS FFMA2 / FMUL2 / FADD2): one instruction advances the same
// cell of two samples.  The FMA pipe spends two cycles on a packed op, so peak flops are those
// of scalar FFMA, but the issue slot, the shared-memory instruction and the coefficient operand
// (a scalar register, broadcast by the instruction) are spent once per pair.
// Probe: tools/probes/ffma2_probe.cu.
// ------------------------------------------------------------------------------------------
namespace pde {

struct f2 {
    unsigned long long v;
};

__device__ __forceinline__ f2 f2_make(float lo, float hi) {
    f2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r.v) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ f2 f2_bc(float s) { return f2_make(s, s); }
__device__ __forceinline__ float f2_lo(f2 a) {
    float x, y;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(x), "=f"(y) : "l"(a.v));
    return x;
}
__device__ __forceinline__ float f2_hi(f2 a) {
    float x, y;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(x), "=f"(y) : "l"(a.v));
    return y;
}
__device__ __forceinline__ float f2_hsum(f2 a) { return f2_lo(a) + f2_hi(a); }
__device__ __forceinline__ f2 f2_fma(f2 a, f2 b, f2 c) {
    f2 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r.v) : "l"(a.v), "l"(b.v), "l"(c.v));
    return r;
}
__device__ __forceinline__ f2 f2_mul(f2 a, f2 b) {
    f2 r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v));
    return r;
}
__device__ __forceinline__ f2 f2_add(f2 a, f2 b) {
    f2 r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v));
    return r;
}
__device__ __forceinline__ f2 f2_sub(f2 a, f2 b) {
    f2 r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v));
    return r;
}
// scalar coefficient times / fused with a pair
__device__ __forceinline__ f2 f2_muls(float s, f2 b) { return f2_mul(f2_bc(s), b); }
__device__ __forceinline__ f2 f2_fmas(float s, f2 b, f2 c) { return f2_fma(f2_bc(s), b, c); }

}  // namespace pde
