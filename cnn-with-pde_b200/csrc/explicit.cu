// Explicit 5-point-stencil layers, forward and adjoint, for sm_100a.
//
//   tiny_*   tiny_imagenet.ImprovedDiffusionLayer live path (tiny_imagenet.py:34-72):
//            u <- u + blend * ((s u + alpha dt Lap0(s u)) - u), zero ghosts, per-channel scalars.
//            One step per call in the reference model, so the kernel is a pure HBM stream:
//            whole planes arrive by TMA bulk copy into a 3-stage shared-memory ring
//            (mbarrier completion), every thread works on float4 strips, results leave with
//            128-bit streaming stores.  All num_steps run on-chip.
//   emo_*    emotion_recognition.PDELayer (emotion_recognition.py:76-97): Nt explicit steps
//            on a reflect-padded plane whose ghost ring stays frozen at its initial values.
//            The padded plane ping-pongs between two shared-memory buffers; a thread owns a
//            column strip of 8 rows and slides a 3-row register window down it.
//
// Backward kernels recompute the forward states on-chip (nothing but the layer input is
// saved), run the hand-derived adjoint, and reduce the coefficient gradients per thread ->
// per block -> tiny finishing kernel (double accumulation, fixed order: deterministic).
#include <cstdlib>

#include <cuda_bf16.h>

#include "common.cuh"
#include "tiny_step.cuh"
#include "tiny_tiled.cuh"

namespace pde {
namespace expl {

// ==========================================================================================
// tiny_imagenet
// ==========================================================================================
constexpr int kTinyThreads = 256;
constexpr int kMaxStages = 3;

// u, gout, out, gin: fp32 or bf16 planes (the kernels are instantiated for both I/O types; arithmetic,
// parameters and parameter gradients are fp32 either way)
struct TinyArgs {
    pde_tiny_desc d;
    const void *u, *gout;
    const float *alpha, *scal;
    void *out, *gin;
    float *part;
    int nplanes, stages, need_gin;
};

// four results leave as one streaming store: 16 bytes of fp32 or 8 bytes of bf16 (round to nearest even)
template <typename T>
__device__ __forceinline__ void st_stream4(T *dst, int q, float4 v);
template <>
__device__ __forceinline__ void st_stream4<float>(float *dst, int q, float4 v) {
    st_stream(reinterpret_cast<float4 *>(dst) + q, v);
}
template <>
__device__ __forceinline__ void st_stream4<__nv_bfloat16>(__nv_bfloat16 *dst, int q, float4 v) {
    const __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
    uint2 w;
    w.x = *reinterpret_cast<const unsigned *>(&lo);
    w.y = *reinterpret_cast<const unsigned *>(&hi);
    __stcs(reinterpret_cast<uint2 *>(dst) + q, w);
}

// bf16 -> fp32 is a shift: two cells per 32-bit word, the lower address in the lower half
__device__ __forceinline__ float4 widen4(uint2 w) {
    return make_float4(__uint_as_float(w.x << 16), __uint_as_float(w.x & 0xffff0000u), __uint_as_float(w.y << 16),
                       __uint_as_float(w.y & 0xffff0000u));
}
__device__ __forceinline__ float widen1(const __nv_bfloat16 *p) {
    return __uint_as_float((unsigned)(*reinterpret_cast<const unsigned short *>(p)) << 16);
}

struct Strip {
    float4 c, up, dn;
    float lf, rt;
};

// The four cells at chunk q of a dense H x W plane with their four neighbour strips; zero ghosts.  The plane is
// fp32 (16-byte chunks) or bf16 as it arrived from HBM (8-byte chunks, widened on the way into registers).
__device__ __forceinline__ Strip load_strip(const float *src, int q, int H, int W) {
    const float4 *s4 = reinterpret_cast<const float4 *>(src);
    const int idx = 4 * q, row = idx / W, col = idx - row * W, w4 = W >> 2;
    const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
    Strip s;
    s.c = s4[q];
    s.up = row > 0 ? s4[q - w4] : zero;
    s.dn = row < H - 1 ? s4[q + w4] : zero;
    s.lf = col > 0 ? src[idx - 1] : 0.0f;
    s.rt = col + 4 < W ? src[idx + 4] : 0.0f;
    return s;
}
__device__ __forceinline__ Strip load_strip(const __nv_bfloat16 *src, int q, int H, int W) {
    const uint2 *s2 = reinterpret_cast<const uint2 *>(src);
    const int idx = 4 * q, row = idx / W, col = idx - row * W, w4 = W >> 2;
    const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
    Strip s;
    s.c = widen4(s2[q]);
    s.up = row > 0 ? widen4(s2[q - w4]) : zero;
    s.dn = row < H - 1 ? widen4(s2[q + w4]) : zero;
    s.lf = col > 0 ? widen1(src + idx - 1) : 0.0f;
    s.rt = col + 4 < W ? widen1(src + idx + 4) : 0.0f;
    return s;
}

// Lap0 of (k * plane) at the four cells of a strip: conv2d(padding=1) with [[0,1,0],[1,-4,1],[0,1,0]]
__device__ __forceinline__ float4 lap0_scaled(const Strip &s, float k) {
    const float c0 = s.c.x * k, c1 = s.c.y * k, c2 = s.c.z * k, c3 = s.c.w * k;
    const float lf = s.lf * k, rt = s.rt * k;
    float4 r;
    r.x = (((s.up.x * k + lf) + (-4.0f * c0)) + c1) + s.dn.x * k;
    r.y = (((s.up.y * k + c0) + (-4.0f * c1)) + c2) + s.dn.y * k;
    r.z = (((s.up.z * k + c1) + (-4.0f * c2)) + c3) + s.dn.z * k;
    r.w = (((s.up.w * k + c2) + (-4.0f * c3)) + rt) + s.dn.w * k;
    return r;
}

// one explicit step of a whole plane: src in shared memory, dst in shared or global memory
template <bool kStream, typename S = float, typename T = float>
__device__ __forceinline__ void tiny_step(const S *src, T *dst, int H, int W, float sc, float adt,
                                          float bl, int tid) {
    const int nq = (H * W) >> 2;
    for (int q = tid; q < nq; q += kTinyThreads) {
        const Strip s = load_strip(src, q, H, W);
        const float4 lp = lap0_scaled(s, sc);
        float4 o;
        o.x = blend1(s.c.x, sc, adt, lp.x, bl);
        o.y = blend1(s.c.y, sc, adt, lp.y, bl);
        o.z = blend1(s.c.z, sc, adt, lp.z, bl);
        o.w = blend1(s.c.w, sc, adt, lp.w, bl);
        if (kStream)
            st_stream4<T>(dst, q, o);
        else
            reinterpret_cast<float4 *>(dst)[q] = o;
    }
}

template <typename T>
__global__ void __launch_bounds__(kTinyThreads) tiny_fwd_kernel(const TinyArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const pde_tiny_desc &d = a.d;
    const int HW = d.H * d.W, tid = threadIdx.x, stages = a.stages;
    const uint32_t bytes = (uint32_t)HW * (uint32_t)sizeof(T);
    const T *gu = static_cast<const T *>(a.u);
    T *gout = static_cast<T *>(a.out);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw);
    T *ring = reinterpret_cast<T *>(smem_raw + 128);
    float *work = reinterpret_cast<float *>(smem_raw + 128 + (size_t)stages * bytes);  // two fp32 planes, only touched when steps > 1
    const int n_my = a.nplanes > (int)blockIdx.x ? (a.nplanes - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    if (tid == 0) {
        for (int s = 0; s < stages; ++s) mbar_init(&bars[s], 1);
        mbar_fence_init();
    }
    __syncthreads();
    if (tid == 0) {
        for (int k = 0; k < stages - 1 && k < n_my; ++k) {
            mbar_expect_tx(&bars[k], bytes);
            tma_load_1d(ring + (size_t)k * HW, gu + (size_t)(blockIdx.x + (size_t)k * gridDim.x) * HW, bytes, &bars[k]);
        }
    }
    for (int k = 0; k < n_my; ++k) {
        const int st = k % stages;
        const int kn = k + stages - 1;
        if (tid == 0 && kn < n_my) {
            const int sn = kn % stages;
            fence_proxy_async();
            mbar_expect_tx(&bars[sn], bytes);
            tma_load_1d(ring + (size_t)sn * HW, gu + (size_t)(blockIdx.x + (size_t)kn * gridDim.x) * HW, bytes, &bars[sn]);
        }
        mbar_wait(&bars[st], (uint32_t)((k / stages) & 1));
        const size_t plane = blockIdx.x + (size_t)k * gridDim.x;
        const int c = (int)(plane % d.C);
        bool inside;
        const float al = clamp_alpha(d, __ldg(a.alpha + c), &inside);
        const float adt = al * d.dt, sc = __ldg(a.scal + c);
        const T *in = ring + (size_t)st * HW;    // the plane as it arrived (fp32 or bf16)
        T *gdst = gout + plane * HW;
        if (d.steps == 0) {
            for (int q = tid; q < (HW >> 2); q += kTinyThreads) st_stream4<T>(gdst, q, load_strip(in, q, d.H, d.W).c);
        } else if (d.steps == 1) {
            tiny_step<true, T, T>(in, gdst, d.H, d.W, sc, adt, d.blend, tid);
        } else {
            // several steps: the intermediate states are fp32 planes in shared memory
            tiny_step<false, T, float>(in, work, d.H, d.W, sc, adt, d.blend, tid);
            __syncthreads();
            const float *src = work;
            for (int s = 1; s < d.steps; ++s) {
                if (s == d.steps - 1) {
                    tiny_step<true, float, T>(src, gdst, d.H, d.W, sc, adt, d.blend, tid);
                } else {
                    float *dst = work + (size_t)(s & 1) * HW;
                    tiny_step<false, float, float>(src, dst, d.H, d.W, sc, adt, d.blend, tid);
                    __syncthreads();
                    src = dst;
                }
            }
        }
        __syncthreads();  // everyone is done with ring[st] before it is refilled
    }
}

// Backward.  Ring stage = {u plane, gout plane}.  For steps > 1 the forward states u_1..u_{K-1}
// are rebuilt into `hist` and the adjoint ping-pongs through `gwork`.
template <typename T>
__global__ void __launch_bounds__(kTinyThreads) tiny_bwd_kernel(const TinyArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const pde_tiny_desc &d = a.d;
    const int HW = d.H * d.W, tid = threadIdx.x, stages = a.stages, K = d.steps;
    const uint32_t bytes = (uint32_t)HW * (uint32_t)sizeof(T);
    const T *gu = static_cast<const T *>(a.u), *ggout = static_cast<const T *>(a.gout);
    T *ggin = static_cast<T *>(a.gin);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw);
    T *ring = reinterpret_cast<T *>(smem_raw + 128);                                        // [stages][2][HW]
    float *hist = reinterpret_cast<float *>(smem_raw + 128 + (size_t)stages * 2 * bytes);    // [K-1][HW]
    float *gwork = hist + (size_t)(K > 1 ? K - 1 : 0) * HW;                                  // [2][HW]
    __shared__ float red[2][kTinyThreads / 32];
    const int n_my = a.nplanes > (int)blockIdx.x ? (a.nplanes - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    // gridDim.x is a multiple of C, so every plane of this block has the same channel
    const int c = blockIdx.x % d.C;
    bool inside;
    const float al = clamp_alpha(d, __ldg(a.alpha + c), &inside);
    const float adt = al * d.dt, sc = __ldg(a.scal + c), bl = d.blend;
    float accA = 0.0f, accS = 0.0f;
    if (tid == 0) {
        for (int s = 0; s < stages; ++s) mbar_init(&bars[s], 1);
        mbar_fence_init();
    }
    __syncthreads();
    auto issue = [&](int k) {
        const int sn = k % stages;
        const size_t plane = blockIdx.x + (size_t)k * gridDim.x;
        mbar_expect_tx(&bars[sn], 2 * bytes);
        tma_load_1d(ring + (size_t)sn * 2 * HW, gu + plane * HW, bytes, &bars[sn]);
        tma_load_1d(ring + (size_t)sn * 2 * HW + HW, ggout + plane * HW, bytes, &bars[sn]);
    };
    if (tid == 0)
        for (int k = 0; k < stages - 1 && k < n_my; ++k) issue(k);
    for (int k = 0; k < n_my; ++k) {
        const int st = k % stages;
        if (tid == 0 && k + stages - 1 < n_my) {
            fence_proxy_async();
            issue(k + stages - 1);
        }
        mbar_wait(&bars[st], (uint32_t)((k / stages) & 1));
        const size_t plane = blockIdx.x + (size_t)k * gridDim.x;
        const T *u0 = ring + (size_t)st * 2 * HW, *g0 = u0 + HW;   // the planes as they arrived (fp32 or bf16)
        // forward states u_1 .. u_{K-1} (fp32 planes in shared memory)
        for (int s = 0; s + 1 < K; ++s) {
            if (s == 0) tiny_step<false, T, float>(u0, hist, d.H, d.W, sc, adt, bl, tid);
            else tiny_step<false, float, float>(hist + (size_t)(s - 1) * HW, hist + (size_t)s * HW, d.H, d.W, sc, adt, bl, tid);
            __syncthreads();
        }
        T *gfinal = a.need_gin ? ggin + plane * HW : nullptr;          // step 0 writes grad_input
        // one reversed step: state `us` and adjoint `g` in, adjoint out (to gdst, or grad_input at step 0)
        auto reverse = [&](const auto *us, const auto *g, float *gdst, bool last) {
            for (int q = tid; q < (HW >> 2); q += kTinyThreads) {
                const Strip su = load_strip(us, q, d.H, d.W);
                const Strip sg = load_strip(g, q, d.H, d.W);
                const float4 lv = lap0_scaled(su, sc);   // Lap0(v), v = s u
                const float4 lg = lap0_scaled(sg, bl);   // Lap0(g_w), g_w = blend g
                const float gw0 = sg.c.x * bl, gw1 = sg.c.y * bl, gw2 = sg.c.z * bl, gw3 = sg.c.w * bl;
                const float z0 = fmaf(adt, lg.x, gw0), z1 = fmaf(adt, lg.y, gw1), z2 = fmaf(adt, lg.z, gw2),
                            z3 = fmaf(adt, lg.w, gw3);
                accA = fmaf(gw0, lv.x, accA); accA = fmaf(gw1, lv.y, accA);
                accA = fmaf(gw2, lv.z, accA); accA = fmaf(gw3, lv.w, accA);
                accS = fmaf(z0, su.c.x, accS); accS = fmaf(z1, su.c.y, accS);
                accS = fmaf(z2, su.c.z, accS); accS = fmaf(z3, su.c.w, accS);
                if (last ? gfinal != nullptr : true) {
                    float4 o;
                    o.x = fmaf(sc, z0, sg.c.x - gw0);
                    o.y = fmaf(sc, z1, sg.c.y - gw1);
                    o.z = fmaf(sc, z2, sg.c.z - gw2);
                    o.w = fmaf(sc, z3, sg.c.w - gw3);
                    if (last)
                        st_stream4<T>(gfinal, q, o);
                    else
                        reinterpret_cast<float4 *>(gdst)[q] = o;
                }
            }
        };
        if constexpr (sizeof(T) == 4) {
            // fp32 I/O: ring planes and shared-memory planes have one type, so one loop (and one copy of the body) serves every step
            const float *g = reinterpret_cast<const float *>(g0);
            for (int s = K - 1; s >= 0; --s) {
                const float *us = s == 0 ? reinterpret_cast<const float *>(u0) : hist + (size_t)(s - 1) * HW;
                float *gdst = s == 0 ? nullptr : gwork + (size_t)(s & 1) * HW;
                reverse(us, g, gdst, s == 0);
                if (s > 0) {
                    __syncthreads();
                    g = gdst;
                }
            }
        } else if (K == 1) {
            reverse(u0, g0, nullptr, true);                // the model's case: both planes straight from the ring
        } else if (K > 1) {
            // step K-1 takes the upstream gradient from the ring, the others the adjoint plane of the step after
            float *gdst = gwork + (size_t)((K - 1) & 1) * HW;
            reverse(hist + (size_t)(K - 2) * HW, g0, gdst, false);
            __syncthreads();
            const float *g = gdst;
            for (int s = K - 2; s >= 1; --s) {
                gdst = gwork + (size_t)(s & 1) * HW;
                reverse(hist + (size_t)(s - 1) * HW, g, gdst, false);
                __syncthreads();
                g = gdst;
            }
            reverse(u0, g, nullptr, true);
        }
        if (K == 0 && a.need_gin)
            for (int q = tid; q < (HW >> 2); q += kTinyThreads) st_stream4<T>(ggin + plane * HW, q, load_strip(g0, q, d.H, d.W).c);
        __syncthreads();
    }
    accA = warp_sum(accA);
    accS = warp_sum(accS);
    if ((tid & 31) == 0) { red[0][tid >> 5] = accA; red[1][tid >> 5] = accS; }
    __syncthreads();
    if (tid == 0) {
        float sa = 0.f, ss = 0.f;
        for (int w = 0; w < kTinyThreads / 32; ++w) { sa += red[0][w]; ss += red[1][w]; }
        a.part[2 * blockIdx.x] = inside ? sa * d.dt : 0.0f;
        a.part[2 * blockIdx.x + 1] = ss;
    }
}

__global__ void tiny_finish_kernel(int C, int nblocks, const float *__restrict__ part, float *g_alpha, float *g_scal) {
    const int c = threadIdx.x;
    if (c >= C) return;
    double sa = 0.0, ss = 0.0;
    for (int b = c; b < nblocks; b += C) { sa += (double)part[2 * b]; ss += (double)part[2 * b + 1]; }
    g_alpha[c] = (float)sa;
    g_scal[c] = (float)ss;
}

static int tiny_validate(const pde_tiny_desc *d, int io_bytes = 4) {
    if (!d) return PDE_ERR_INVALID;
    if (d->B < 0 || d->C < 1 || d->H < 1 || d->W < 1 || d->steps < 0) return PDE_ERR_INVALID;
    if (d->W % 4 != 0) return PDE_ERR_UNSUPPORTED;          // float4 strips, 16-byte TMA granularity
    if (io_bytes == 2 && (d->H * d->W) % 8 != 0) return PDE_ERR_UNSUPPORTED;   // bf16 planes: 16-byte granularity too
    if (d->C > 1024) return PDE_ERR_UNSUPPORTED;
    return PDE_OK;
}

// shared-memory plan: ring stages first (planes in their I/O type), then the extra fp32 planes (work / history
// for several steps); fewer stages if it does not fit
static int tiny_plan(const pde_tiny_desc *d, bool bwd, int max_smem, int *stages, size_t *smem, int io_bytes = 4) {
    const size_t plane = (size_t)d->H * d->W * sizeof(float), io_plane = (size_t)d->H * d->W * io_bytes;
    const size_t extra = bwd ? ((size_t)(d->steps > 1 ? d->steps - 1 : 0) + (d->steps > 1 ? 2 : 0)) * plane
                             : (d->steps > 1 ? 2 * plane : 0);
    for (int s = kMaxStages; s >= 1; --s) {
        const size_t need = 128 + (size_t)s * (bwd ? 2 : 1) * io_plane + extra;
        if (need <= (size_t)max_smem) {
            *stages = s;
            *smem = need;
            return PDE_OK;
        }
    }
    return PDE_ERR_UNSUPPORTED;
}

static int tiny_grid(const pde_tiny_desc *d, const DeviceProps &props, size_t smem, bool multiple_of_c) {
    const long nplanes = (long)d->B * d->C;
    int per_sm = (int)((size_t)(227 * 1024) / (smem + 1024));
    if (per_sm > 8) per_sm = 8;
    if (per_sm < 1) per_sm = 1;
    long grid = (long)props.sm_count * per_sm;
    if (grid > nplanes) grid = nplanes;
    if (multiple_of_c) {
        grid -= grid % d->C;
        if (grid < d->C) grid = d->C;
    }
    return (int)(grid < 1 ? 1 : grid);
}

// Which kernels serve one pass of a tiny configuration with B > 0: the whole-plane ring kernels keep every
// configuration they serve (tiny_validate and tiny_plan both pass), the tiled kernels (tiny_tiled.cu) take the
// rest of their domain, anything else is PDE_ERR_UNSUPPORTED.  The launches and the workspace query all ask here.
static int tiny_route(const pde_tiny_desc *d, bool bwd, int io_bytes, int max_smem, bool *tiled, int *stages,
                      size_t *smem) {
    const int rc = tiny_validate(d, io_bytes);
    if (rc == PDE_ERR_INVALID) return rc;
    *tiled = rc != PDE_OK || tiny_plan(d, bwd, max_smem, stages, smem, io_bytes) != PDE_OK;
    return *tiled && !tiled::tiny_tiled_domain(d) ? PDE_ERR_UNSUPPORTED : PDE_OK;
}

// the checks that come before the batch is looked at: B = 0 is a no-op wherever some kernel could serve B > 0
static int tiny_precheck(const pde_tiny_desc *d, int io_bytes) {
    const int rc = tiny_validate(d, io_bytes);
    if (rc == PDE_ERR_UNSUPPORTED && tiled::tiny_tiled_domain(d)) return PDE_OK;
    return rc;
}

// pointers a kernel may be handed: 16-byte aligned for the ring kernels' vector loads and bulk copies, element
// aligned for the tiled kernels
static bool tiny_aligned(const void *p, bool tiled, int io_bytes) {
    return tiled ? (reinterpret_cast<uintptr_t>(p) % (uintptr_t)io_bytes) == 0 : aligned16(p);
}

// ==========================================================================================
// emotion_recognition
// ==========================================================================================
constexpr int kEmoRows = 8;       // rows per thread strip
constexpr int kEmoMaxN = 64;

struct EmoArgs {
    pde_emo_desc d;
    const float *u0, *gout, *w6, *xs, *ys;
    float *out, *gin, *part;
    int need_gin;
};

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

// interior of the padded plane <- global plane (coalesced), then the reflected ghost ring
__device__ __forceinline__ void emo_load_padded(const float *__restrict__ g, float *buf, float *buf2, int N,
                                                int tid, int nthreads) {
    const int M = N + 2;
    for (int idx = tid; idx < N * N; idx += nthreads) {
        const int i = idx / N, j = idx - i * N;
        buf[(i + 1) * M + j + 1] = __ldcs(g + idx);
    }
    __syncthreads();
    if (tid < N) {
        const int q = tid + 1;
        const float top = buf[2 * M + q], bot = buf[(N - 1) * M + q];
        const float lf = buf[q * M + 2], rt = buf[q * M + N - 1];
        buf[q] = top; buf[(N + 1) * M + q] = bot; buf[q * M] = lf; buf[q * M + N + 1] = rt;
        buf2[q] = top; buf2[(N + 1) * M + q] = bot; buf2[q * M] = lf; buf2[q * M + N + 1] = rt;
    }
    if (tid == 0) {  // corners are never read; keep them finite
        buf[0] = buf[N + 1] = buf[(N + 1) * M] = buf[(N + 1) * M + N + 1] = 0.f;
        buf2[0] = buf2[N + 1] = buf2[(N + 1) * M] = buf2[(N + 1) * M + N + 1] = 0.f;
    }
    __syncthreads();
}

__device__ __forceinline__ void emo_step(const float *src, float *dst, const float *sa, int N, int j, int r0,
                                         int r1, float bj) {
    const int M = N + 2;
    float up = src[r0 * M + j + 1], ct = src[(r0 + 1) * M + j + 1];
    for (int i = r0; i < r1; ++i) {
        const float dn = src[(i + 2) * M + j + 1];
        const float lf = src[(i + 1) * M + j], rt = src[(i + 1) * M + j + 2];
        const float two = 2.0f * ct;
        const float dr = (dn - two) + up;
        const float dc = (rt - two) + lf;
        dst[(i + 1) * M + j + 1] = fmaf(bj, dc, fmaf(sa[i], dr, ct));
        up = ct;
        ct = dn;
    }
}

__global__ void emo_fwd_kernel(const EmoArgs a) {
    extern __shared__ __align__(16) float smem[];
    const pde_emo_desc &d = a.d;
    const int N = d.N, M = N + 2, PP = M * M, tid = threadIdx.x, nthreads = blockDim.x;
    float *sa = smem, *sb = smem + kEmoMaxN, *buf0 = smem + 2 * kEmoMaxN, *buf1 = buf0 + PP;
    if (tid < N) emo_profile(d, a.w6, a.xs, a.ys, tid, &sa[tid], &sb[tid]);
    __syncthreads();
    const int j = tid % N, rb = tid / N;
    const int r0 = rb * kEmoRows, r1 = min(r0 + kEmoRows, N);
    const bool active = r0 < N;
    const float bj = sb[j];
    for (int plane = blockIdx.x; plane < d.B; plane += gridDim.x) {
        emo_load_padded(a.u0 + (size_t)plane * N * N, buf0, buf1, N, tid, nthreads);
        float *src = buf0, *dst = buf1;
        for (int k = 0; k < d.Nt; ++k) {
            if (active) emo_step(src, dst, sa, N, j, r0, r1, bj);
            __syncthreads();
            float *tmp = src; src = dst; dst = tmp;
        }
        float *o = a.out + (size_t)plane * N * N;
        for (int idx = tid; idx < N * N; idx += nthreads) {
            const int i = idx / N, jj = idx - i * N;
            __stcs(o + idx, src[(i + 1) * M + jj + 1]);
        }
        __syncthreads();
    }
}

// Backward: rebuild u^0..u^{Nt-1} (padded planes) in shared memory, then run the adjoint
//   lam'(i,j) = lam (1 - 2 a_i - 2 b_j) + a_{i-1} lam(i-1,j) + a_{i+1} lam(i+1,j)
//                                       + b_{j-1} lam(i,j-1) + b_{j+1} lam(i,j+1)
// on a padded lam plane whose ring stays zero; what would flow into the (frozen, input-derived)
// ghost ring is summed over all steps in four edge vectors and folded back through the
// reflection at the end.  dA_i += lam * d2_row u, dB_j += lam * d2_col u per thread.
__global__ void emo_bwd_kernel(const EmoArgs a) {
    extern __shared__ __align__(16) float smem[];
    const pde_emo_desc &d = a.d;
    const int N = d.N, M = N + 2, PP = M * M, tid = threadIdx.x, nthreads = blockDim.x, Nt = d.Nt;
    float *sa = smem;                       // a padded: sa[0] = a_{-1} = 0, sa[1 + i] = a_i, sa[N + 1] = 0
    float *sb = smem + (kEmoMaxN + 2);
    float *edge = sb + (kEmoMaxN + 2);      // top, bottom, left, right: 4 x kEmoMaxN
    float *sumA = edge + 4 * kEmoMaxN, *sumB = sumA + kEmoMaxN;
    float *hist = sumB + kEmoMaxN;          // [Nt + 1][PP]  (the extra plane is ping-pong space)
    float *lam0 = hist + (size_t)(Nt + 1) * PP, *lam1 = lam0 + PP;
    if (tid < N) {
        float av, bv;
        emo_profile(d, a.w6, a.xs, a.ys, tid, &av, &bv);
        sa[tid + 1] = av; sb[tid + 1] = bv;
        sumA[tid] = 0.f; sumB[tid] = 0.f;
    }
    if (tid == 0) { sa[0] = sa[N + 1] = 0.f; sb[0] = sb[N + 1] = 0.f; }
    for (int idx = tid; idx < 2 * PP; idx += nthreads) lam0[idx] = 0.f;  // zero rings (and interiors)
    __syncthreads();
    const int j = tid % N, rb = tid / N;
    const int r0 = rb * kEmoRows, r1 = min(r0 + kEmoRows, N);
    const bool active = r0 < N;
    const float bj = sb[j + 1], bjm = sb[j], bjp = sb[j + 2];
    float dA[kEmoRows], dB = 0.f;
#pragma unroll
    for (int r = 0; r < kEmoRows; ++r) dA[r] = 0.f;

    for (int plane = blockIdx.x; plane < d.B; plane += gridDim.x) {
        // forward states: hist[k] = u^k, k = 0..Nt-1 (hist[Nt] receives u^Nt, unused)
        emo_load_padded(a.u0 + (size_t)plane * N * N, hist, hist + PP, N, tid, nthreads);
        for (int k = 0; k < Nt; ++k) {
            float *nxt = hist + (size_t)(k + 1) * PP;
            if (k > 0 && tid < N) {  // ring of the next plane (hist[1] already has it)
                const int q = tid + 1;
                nxt[q] = hist[q]; nxt[(N + 1) * M + q] = hist[(N + 1) * M + q];
                nxt[q * M] = hist[q * M]; nxt[q * M + N + 1] = hist[q * M + N + 1];
            }
            if (active) emo_step(hist + (size_t)k * PP, nxt, sa + 1, N, j, r0, r1, bj);
            __syncthreads();
        }
        const float *go = a.gout + (size_t)plane * N * N;
        for (int idx = tid; idx < N * N; idx += nthreads) {
            const int i = idx / N, jj = idx - i * N;
            lam0[(i + 1) * M + jj + 1] = __ldcs(go + idx);
        }
        if (tid < 4 * kEmoMaxN) edge[tid] = 0.f;
        for (int idx = tid + nthreads; idx < 4 * kEmoMaxN; idx += nthreads) edge[idx] = 0.f;
        __syncthreads();
        float *lsrc = lam0, *ldst = lam1;
        for (int k = Nt - 1; k >= 0; --k) {
            const float *uk = hist + (size_t)k * PP;
            if (active) {
                float lup = lsrc[r0 * M + j + 1], lct = lsrc[(r0 + 1) * M + j + 1];
                float uup = uk[r0 * M + j + 1], uct = uk[(r0 + 1) * M + j + 1];
#pragma unroll
                for (int r = 0; r < kEmoRows; ++r) {
                    const int i = r0 + r;
                    if (i < r1) {
                        const float ldn = lsrc[(i + 2) * M + j + 1], llf = lsrc[(i + 1) * M + j], lrt = lsrc[(i + 1) * M + j + 2];
                        const float udn = uk[(i + 2) * M + j + 1], ulf = uk[(i + 1) * M + j], urt = uk[(i + 1) * M + j + 2];
                        const float two = 2.0f * uct;
                        const float dr = (udn - two) + uup, dc = (urt - two) + ulf;
                        dA[r] = fmaf(lct, dr, dA[r]);
                        dB = fmaf(lct, dc, dB);
                        const float ai = sa[i + 1];
                        const float al = ai * lct, blv = bj * lct;
                        float nv = (lct - 2.0f * al) - 2.0f * blv;
                        nv = fmaf(sa[i], lup, nv);
                        nv = fmaf(sa[i + 2], ldn, nv);
                        nv = fmaf(bjm, llf, nv);
                        nv = fmaf(bjp, lrt, nv);
                        ldst[(i + 1) * M + j + 1] = nv;
                        if (i == 0) edge[j] += al;
                        if (i == N - 1) edge[kEmoMaxN + j] += al;
                        if (j == 0) edge[2 * kEmoMaxN + i] += blv;
                        if (j == N - 1) edge[3 * kEmoMaxN + i] += blv;
                        lup = lct; lct = ldn; uup = uct; uct = udn;
                    }
                }
            }
            __syncthreads();
            float *tmp = lsrc; lsrc = ldst; ldst = tmp;
        }
        if (a.need_gin) {
            float *gi = a.gin + (size_t)plane * N * N;
            for (int idx = tid; idx < N * N; idx += nthreads) {
                const int i = idx / N, jj = idx - i * N;
                float v = lsrc[(i + 1) * M + jj + 1];
                if (i == 1) v += edge[jj];
                if (i == N - 2) v += edge[kEmoMaxN + jj];
                if (jj == 1) v += edge[2 * kEmoMaxN + i];
                if (jj == N - 2) v += edge[3 * kEmoMaxN + i];
                __stcs(gi + idx, v);
            }
        }
        __syncthreads();
    }
    if (active) {
#pragma unroll
        for (int r = 0; r < kEmoRows; ++r)
            if (r0 + r < r1) atomicAdd(&sumA[r0 + r], dA[r]);
        atomicAdd(&sumB[j], dB);
    }
    __syncthreads();
    if (tid < N) {
        a.part[(size_t)blockIdx.x * 2 * kEmoMaxN + tid] = sumA[tid];
        a.part[(size_t)blockIdx.x * 2 * kEmoMaxN + kEmoMaxN + tid] = sumB[tid];
    }
}

__global__ void emo_finish_kernel(pde_emo_desc d, int nblocks, const float *__restrict__ part,
                                  const float *__restrict__ xs, const float *__restrict__ ys, float *g_w6) {
    __shared__ double sA[kEmoMaxN], sB[kEmoMaxN];
    const int i = threadIdx.x;
    if (i < d.N) {
        double a = 0.0, b = 0.0;
        for (int blk = 0; blk < nblocks; ++blk) {
            a += (double)part[(size_t)blk * 2 * kEmoMaxN + i];
            b += (double)part[(size_t)blk * 2 * kEmoMaxN + kEmoMaxN + i];
        }
        sA[i] = a; sB[i] = b;
    }
    __syncthreads();
    if (i == 0) {
        const float two_pi = (float)(2.0 * 3.141592653589793), four_pi = (float)(4.0 * 3.141592653589793);
        const double ka = (double)d.half_dt / (double)d.dx2, kb = (double)d.dt / (double)d.dy2;
        double g[6] = {0, 0, 0, 0, 0, 0};
        for (int q = 0; q < d.N; ++q) {
            const double s1 = (double)sinf(__fmul_rn(two_pi, ys[q])), s2 = (double)sinf(__fmul_rn(four_pi, ys[q]));
            const double c1 = (double)cosf(__fmul_rn(two_pi, xs[q])), c2 = (double)cosf(__fmul_rn(four_pi, xs[q]));
            g[0] += ka * sA[q]; g[1] += ka * sA[q] * s1; g[2] += ka * sA[q] * s2;
            g[3] += kb * sB[q]; g[4] += kb * sB[q] * c1; g[5] += kb * sB[q] * c2;
        }
        for (int q = 0; q < 6; ++q) g_w6[q] = (float)g[q];
    }
}

static int emo_validate(const pde_emo_desc *d) {
    if (!d) return PDE_ERR_INVALID;
    if (d->B < 0 || d->N < 3 || d->Nt < 0) return PDE_ERR_INVALID;
    if (d->N > kEmoMaxN) return PDE_ERR_UNSUPPORTED;
    return PDE_OK;
}

static int emo_threads(int N) {
    const int rb = (N + kEmoRows - 1) / kEmoRows;
    return ((N * rb + 31) / 32) * 32;
}

static size_t emo_fwd_smem(const pde_emo_desc *d) {
    return ((size_t)2 * kEmoMaxN + (size_t)2 * (d->N + 2) * (d->N + 2)) * sizeof(float);
}
static size_t emo_bwd_smem(const pde_emo_desc *d) {
    const size_t PP = (size_t)(d->N + 2) * (d->N + 2);
    return ((size_t)2 * (kEmoMaxN + 2) + 6 * kEmoMaxN + (size_t)(d->Nt + 3) * PP) * sizeof(float);
}

static int emo_bwd_grid(const pde_emo_desc *d, const DeviceProps &props, size_t smem) {
    int per_sm = (int)((size_t)(227 * 1024) / (smem + 1024));
    if (per_sm < 1) per_sm = 1;
    if (per_sm > 4) per_sm = 4;
    long grid = (long)props.sm_count * per_sm;
    if (grid > d->B) grid = d->B;
    return (int)(grid < 1 ? 1 : grid);
}

// the register-tiled kernels serve plane edges 16 / 32 / 48 unless the descriptor asks for the generic ones
static bool emo_use_tiled(const pde_emo_desc *d) {
    return (d->N == 16 || d->N == 32 || d->N == 48) && !(d->tuning & PDE_EMO_TUNE_GENERIC);
}

}  // namespace expl
}  // namespace pde

#include "emotion_tiled.cuh"

using namespace pde;
using namespace pde::expl;

// ------------------------------------------------------------------------------------------ tiny
extern "C" size_t pde_tiny_backward_workspace_bytes(const pde_tiny_desc *d) {
    if (tiny_precheck(d, 4) != PDE_OK) return 0;
    DeviceProps props;
    if (query_props(&props) != PDE_OK) return 0;
    // one query serves both I/O types: the tiled kernels' need wherever either backward pass goes there
    bool tiled32 = false, tiled16 = false;
    int stages;
    size_t smem;
    const bool ok32 = tiny_route(d, true, 4, props.max_smem_optin, &tiled32, &stages, &smem) == PDE_OK;
    const bool ok16 = tiny_route(d, true, 2, props.max_smem_optin, &tiled16, &stages, &smem) == PDE_OK;
    if ((ok32 && tiled32) || (ok16 && tiled16)) return tiled::tiny_tiled_workspace_bytes(d, props.sm_count);
    if (!ok32 && !ok16) return 0;
    // one (alpha, scaling) partial pair per block; blocks <= 8 per SM
    return ((size_t)props.sm_count * 8 + (size_t)d->C) * 2 * sizeof(float) + 256;
}

template <typename T>
static int tiny_forward_impl(const pde_tiny_desc *d, const void *u, const float *alpha_base, const float *channel_scaling,
                             void *out, void *stream) {
    constexpr int io = (int)sizeof(T);
    int rc = tiny_precheck(d, io);
    if (rc) return rc;
    if (d->B == 0) return PDE_OK;   // empty batch: a no-op, its tensor pointers may be NULL
    if (!u || !alpha_base || !channel_scaling || !out) return PDE_ERR_INVALID;
    DeviceProps props;
    rc = query_props(&props);
    if (rc) return rc;
    TinyArgs a{};
    size_t smem;
    bool tiled;
    rc = tiny_route(d, false, io, props.max_smem_optin, &tiled, &a.stages, &smem);
    if (rc) return rc;
    if (!tiny_aligned(u, tiled, io) || !tiny_aligned(out, tiled, io)) return PDE_ERR_INVALID;
    if (tiled)
        return tiled::tiny_tiled_forward(d, io, u, alpha_base, channel_scaling, out, props, static_cast<cudaStream_t>(stream));
    a.d = *d; a.u = u; a.alpha = alpha_base; a.scal = channel_scaling; a.out = out;
    a.nplanes = d->B * d->C;
    const int grid = tiny_grid(d, props, smem, false);
    rc = kernel_info(reinterpret_cast<const void *>(tiny_fwd_kernel<T>), smem, nullptr);
    if (rc) return rc;
    tiny_fwd_kernel<T><<<grid, kTinyThreads, smem, static_cast<cudaStream_t>(stream)>>>(a);
    return cuda_last_error();
}

template <typename T>
static int tiny_backward_impl(const pde_tiny_desc *d, const void *u, const void *gout, const float *alpha_base,
                              const float *channel_scaling, void *gin, float *g_alpha_base, float *g_channel_scaling,
                              void *workspace, size_t workspace_bytes, void *stream) {
    constexpr int io = (int)sizeof(T);
    int rc = tiny_precheck(d, io);
    if (rc) return rc;
    if (!g_alpha_base || !g_channel_scaling) return PDE_ERR_INVALID;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (d->B == 0) {   // empty batch: zero gradients; u / gout / gin may be NULL
        PDE_CUDA_TRY(cudaMemsetAsync(g_alpha_base, 0, d->C * sizeof(float), st));
        PDE_CUDA_TRY(cudaMemsetAsync(g_channel_scaling, 0, d->C * sizeof(float), st));
        return PDE_OK;
    }
    if (!u || !gout || !alpha_base || !channel_scaling) return PDE_ERR_INVALID;
    DeviceProps props;
    rc = query_props(&props);
    if (rc) return rc;
    TinyArgs a{};
    size_t smem;
    bool tiled;
    rc = tiny_route(d, true, io, props.max_smem_optin, &tiled, &a.stages, &smem);
    if (rc) return rc;
    if (!tiny_aligned(u, tiled, io) || !tiny_aligned(gout, tiled, io) || (gin && !tiny_aligned(gin, tiled, io)))
        return PDE_ERR_INVALID;
    if (tiled)
        return tiled::tiny_tiled_backward(d, io, u, gout, alpha_base, channel_scaling, gin, g_alpha_base, g_channel_scaling,
                                          workspace, workspace_bytes, props, st);
    a.d = *d; a.u = u; a.gout = gout; a.alpha = alpha_base; a.scal = channel_scaling; a.gin = gin;
    a.need_gin = gin != nullptr;
    a.nplanes = d->B * d->C;
    const int grid = tiny_grid(d, props, smem, true);
    const size_t need = (size_t)grid * 2 * sizeof(float) + 256;
    if (!workspace || workspace_bytes < need) return PDE_ERR_WORKSPACE;
    a.part = reinterpret_cast<float *>((reinterpret_cast<uintptr_t>(workspace) + 255u) & ~(uintptr_t)255u);
    rc = kernel_info(reinterpret_cast<const void *>(tiny_bwd_kernel<T>), smem, nullptr);
    if (rc) return rc;
    tiny_bwd_kernel<T><<<grid, kTinyThreads, smem, st>>>(a);
    rc = cuda_last_error();
    if (rc) return rc;
    tiny_finish_kernel<<<1, ((d->C + 31) / 32) * 32, 0, st>>>(d->C, grid, a.part, g_alpha_base, g_channel_scaling);
    return cuda_last_error();
}

extern "C" int pde_tiny_forward(const pde_tiny_desc *d, const float *u, const float *alpha_base,
                                const float *channel_scaling, float *out, void *stream) {
    return tiny_forward_impl<float>(d, u, alpha_base, channel_scaling, out, stream);
}

extern "C" int pde_tiny_backward(const pde_tiny_desc *d, const float *u, const float *gout,
                                 const float *alpha_base, const float *channel_scaling, float *gin,
                                 float *g_alpha_base, float *g_channel_scaling, void *workspace,
                                 size_t workspace_bytes, void *stream) {
    return tiny_backward_impl<float>(d, u, gout, alpha_base, channel_scaling, gin, g_alpha_base, g_channel_scaling, workspace,
                                     workspace_bytes, stream);
}

extern "C" int pde_tiny_forward_bf16(const pde_tiny_desc *d, const void *u, const float *alpha_base,
                                     const float *channel_scaling, void *out, void *stream) {
    return tiny_forward_impl<__nv_bfloat16>(d, u, alpha_base, channel_scaling, out, stream);
}

extern "C" int pde_tiny_backward_bf16(const pde_tiny_desc *d, const void *u, const void *gout, const float *alpha_base,
                                      const float *channel_scaling, void *gin, float *g_alpha_base,
                                      float *g_channel_scaling, void *workspace, size_t workspace_bytes, void *stream) {
    return tiny_backward_impl<__nv_bfloat16>(d, u, gout, alpha_base, channel_scaling, gin, g_alpha_base, g_channel_scaling,
                                             workspace, workspace_bytes, stream);
}

// --------------------------------------------------------------------------------------- emotion
extern "C" size_t pde_emotion_backward_workspace_bytes(const pde_emo_desc *d) {
    if (emo_validate(d) != PDE_OK) return 0;
    DeviceProps props;
    if (query_props(&props) != PDE_OK) return 0;
    const size_t generic = (size_t)props.sm_count * 4 * 2 * kEmoMaxN * sizeof(float) + 256;
    if (emo_use_tiled(d)) {
        const size_t tiled = emo_tiled_workspace_bytes(d, props.sm_count);
        return tiled > generic ? tiled : generic;
    }
    return generic;
}

extern "C" int pde_emotion_forward(const pde_emo_desc *d, const float *u0, const float *w6, const float *xs,
                                   const float *ys, float *out, void *stream) {
    int rc = emo_validate(d);
    if (rc) return rc;
    if (d->B == 0) return PDE_OK;   // empty batch: a no-op, its tensor pointers may be NULL
    if (!u0 || !w6 || !xs || !ys || !out) return PDE_ERR_INVALID;
    DeviceProps props;
    rc = query_props(&props);
    if (rc) return rc;
    EmoArgs a{};
    a.d = *d; a.u0 = u0; a.w6 = w6; a.xs = xs; a.ys = ys; a.out = out;
    if (emo_use_tiled(d))
        return emo_tiled_forward(a, props.sm_count, static_cast<cudaStream_t>(stream));
    const size_t smem = emo_fwd_smem(d);
    const int threads = emo_threads(d->N);
    long grid = (long)props.sm_count * 6;
    if (grid > d->B) grid = d->B;
    rc = kernel_info(reinterpret_cast<const void *>(emo_fwd_kernel), smem, nullptr);
    if (rc) return rc;
    emo_fwd_kernel<<<(int)grid, threads, smem, static_cast<cudaStream_t>(stream)>>>(a);
    return cuda_last_error();
}

extern "C" int pde_emotion_backward(const pde_emo_desc *d, const float *u0, const float *gout, const float *w6,
                                    const float *xs, const float *ys, float *gin, float *g_w6, void *workspace,
                                    size_t workspace_bytes, void *stream) {
    int rc = emo_validate(d);
    if (rc) return rc;
    if (!g_w6) return PDE_ERR_INVALID;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (d->B == 0) {   // empty batch: zero gradients; u0 / gout / gin may be NULL
        PDE_CUDA_TRY(cudaMemsetAsync(g_w6, 0, 6 * sizeof(float), st));
        return PDE_OK;
    }
    if (!u0 || !gout || !w6 || !xs || !ys) return PDE_ERR_INVALID;
    DeviceProps props;
    rc = query_props(&props);
    if (rc) return rc;
    if (emo_use_tiled(d)) {
        if (!workspace || workspace_bytes < emo_tiled_workspace_bytes(d, props.sm_count)) return PDE_ERR_WORKSPACE;
        EmoArgs t{};
        t.d = *d; t.u0 = u0; t.gout = gout; t.w6 = w6; t.xs = xs; t.ys = ys; t.gin = gin;
        t.need_gin = gin != nullptr;
        return emo_tiled_backward(t, props.sm_count, workspace, xs, g_w6, st);
    }
    const size_t smem = emo_bwd_smem(d);
    if (smem > (size_t)props.max_smem_optin) return PDE_ERR_UNSUPPORTED;
    const int grid = emo_bwd_grid(d, props, smem);
    const size_t need = (size_t)grid * 2 * kEmoMaxN * sizeof(float) + 256;
    if (!workspace || workspace_bytes < need) return PDE_ERR_WORKSPACE;
    EmoArgs a{};
    a.d = *d; a.u0 = u0; a.gout = gout; a.w6 = w6; a.xs = xs; a.ys = ys; a.gin = gin;
    a.need_gin = gin != nullptr;
    a.part = reinterpret_cast<float *>((reinterpret_cast<uintptr_t>(workspace) + 255u) & ~(uintptr_t)255u);
    rc = kernel_info(reinterpret_cast<const void *>(emo_bwd_kernel), smem, nullptr);
    if (rc) return rc;
    emo_bwd_kernel<<<grid, emo_threads(d->N), smem, st>>>(a);
    rc = cuda_last_error();
    if (rc) return rc;
    emo_finish_kernel<<<1, kEmoMaxN, 0, st>>>(*d, grid, a.part, xs, ys, g_w6);
    return cuda_last_error();
}
