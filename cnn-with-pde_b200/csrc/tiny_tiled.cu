// tiny_imagenet.ImprovedDiffusionLayer on planes the whole-plane ring kernels of explicit.cu cannot hold:
// any H x W up to 4096 x 4096 (odd widths and rectangles included), 0 ... 16 steps, fp32 or bf16 I/O.
//
// A block owns a kTH x kTW tile of output cells of one plane and reads the tile's window: the tile plus K
// cells of halo on every side.  Window cells outside the plane are the zero ghosts of conv2d(padding=1); they
// stay zero in every step.  Each step is computed on a window shrunk by one more cell, so after K steps
// exactly the tile is valid.  Blocks are persistent and stride over (plane, tile) items, channel fastest; the
// next item's window is loaded into registers (coalesced, element-aligned loads) while the current one
// computes out of shared memory, and results leave as streaming stores.
//
// Backward.  The step is linear in u with fixed alpha and s, so its adjoint does not depend on u:
// grad_input on the tile needs gout on the window only, and step s's parameter-gradient terms on the tile
// need u_s and lambda_{s+1} on the tile + 1 -- both inside the window.  A block loads u and gout on the
// window and counts each step's products over its own tile's cells only, so every (cell, step) is summed
// exactly once.  The forward states u_1 ... u_{K-1} are recomputed from u_0 per reversed step (K (K - 1) / 2
// window steps): nothing but two windows of shared memory, and for K = 1, the model's case, nothing at all.
//
// Arithmetic is op for op that of explicit.cu's lap0_scaled / blend1 / reverse.  Parameter gradients:
// fp32 per thread and item, folded into double per thread, summed per block in a fixed order, finished in
// double per channel: bit-reproducible run to run.
#include <cstdio>

#include <cuda_bf16.h>

#include "common.cuh"
#include "tiny_step.cuh"
#include "tiny_tiled.cuh"

namespace pde {
namespace tiled {

using expl::blend1;
using expl::clamp_alpha;

constexpr int kThreads = 256, kWarps = kThreads / 32;
constexpr int kTH = 32, kTW = 64;   // output tile: a warp per row, 64 fp32 columns = two 128-byte lines

struct TiledArgs {
    pde_tiny_desc d;
    const void *u, *gout;
    const float *alpha, *scal;
    void *out, *gin;
    double *part;
    int ntw, ntiles;
    long long nitems;
};

__device__ __forceinline__ float ld1(const float *p) { return __ldg(p); }
__device__ __forceinline__ float ld1(const __nv_bfloat16 *p) {
    return __uint_as_float((unsigned)__ldg(reinterpret_cast<const unsigned short *>(p)) << 16);
}
__device__ __forceinline__ void st1(float *p, float v) { __stcs(p, v); }
__device__ __forceinline__ void st1(__nv_bfloat16 *p, float v) {
    const __nv_bfloat16 h = __float2bfloat16_rn(v);   // round to nearest even, as the ring kernels do
    __stcs(reinterpret_cast<unsigned short *>(p), *reinterpret_cast<const unsigned short *>(&h));
}

// Lap0 of (k * plane) at one cell, in lap0_scaled's order
__device__ __forceinline__ float lap1(const float *p, int ww, float k) {
    const float lf = p[-1] * k, c = p[0] * k, rt = p[1] * k;
    return (((p[-ww] * k + lf) + (-4.0f * c)) + rt) + p[ww] * k;
}

struct Item {
    size_t plane;   // b * C + c
    int c, gr0, gc0;   // channel; plane coordinates of window cell (0, 0)
};

__device__ __forceinline__ Item decode(const TiledArgs &a, long long item) {
    const int C = a.d.C, K = a.d.steps;
    Item it;
    it.c = (int)(item % C);
    const long long rest = item / C;
    const int tile = (int)(rest % a.ntiles);
    const long long b = rest / a.ntiles;
    it.plane = (size_t)b * C + it.c;
    it.gr0 = (tile / a.ntw) * kTH - K;
    it.gc0 = (tile % a.ntw) * kTW - K;
    return it;
}

// A window in flight: warp w holds rows w, w + 8, ...; lane l holds columns l, l + 32, ...  KH is the largest
// halo the instantiation serves, so the register array covers every window it is given.
template <int KH>
struct Regs {
    static constexpr int kRows = (kTH + 2 * KH + kWarps - 1) / kWarps, kCols = (kTW + 2 * KH + 31) / 32;
    float v[kRows][kCols];
};

template <int KH, typename T>
__device__ __forceinline__ void load_window(Regs<KH> &r, const T *plane, const Item &it, int H, int W, int WH, int WW,
                                            int warp, int lane) {
#pragma unroll
    for (int y = 0; y < Regs<KH>::kRows; ++y) {
        const int i = warp + y * kWarps, gr = it.gr0 + i;
#pragma unroll
        for (int x = 0; x < Regs<KH>::kCols; ++x) {
            const int j = lane + 32 * x, gc = it.gc0 + j;
            const bool in = i < WH && j < WW && (unsigned)gr < (unsigned)H && (unsigned)gc < (unsigned)W;
            r.v[y][x] = in ? ld1(plane + (size_t)gr * W + gc) : 0.0f;
        }
    }
}

template <int KH>
__device__ __forceinline__ void store_window(const Regs<KH> &r, float *win, int WH, int WW, int warp, int lane) {
#pragma unroll
    for (int y = 0; y < Regs<KH>::kRows; ++y) {
        const int i = warp + y * kWarps;
#pragma unroll
        for (int x = 0; x < Regs<KH>::kCols; ++x) {
            const int j = lane + 32 * x;
            if (i < WH && j < WW) win[i * WW + j] = r.v[y][x];
        }
    }
}

// one forward step on window cells [lo, WH - lo) x [lo, WW - lo): into shared memory (zero outside the plane)
// or, when gdst is set, into the plane in global memory (cells inside it only)
template <typename T>
__device__ __forceinline__ void fwd_step(const float *src, float *dst, T *gdst, int lo, int WH, int WW, const Item &it,
                                         int H, int W, float sc, float adt, float bl, int warp, int lane) {
    for (int i = lo + warp; i < WH - lo; i += kWarps) {
        const int gr = it.gr0 + i;
        const bool row_in = (unsigned)gr < (unsigned)H;
        for (int j = lo + lane; j < WW - lo; j += 32) {
            const int gc = it.gc0 + j;
            const bool in = row_in && (unsigned)gc < (unsigned)W;
            const float *p = src + i * WW + j;
            if (gdst) {
                if (in) st1(gdst + (size_t)gr * W + gc, blend1(p[0], sc, adt, lap1(p, WW, sc), bl));
            } else {
                dst[i * WW + j] = in ? blend1(p[0], sc, adt, lap1(p, WW, sc), bl) : 0.0f;
            }
        }
    }
}

// the tile (window cells [K, K + kTH) x [K, K + kTW)) of a shared-memory window into the plane
template <typename T>
__device__ __forceinline__ void copy_tile(const float *src, T *gdst, int K, int WW, const Item &it, int H, int W,
                                          int warp, int lane) {
    for (int i = K + warp; i < K + kTH; i += kWarps) {
        const int gr = it.gr0 + i;
        if ((unsigned)gr >= (unsigned)H) continue;
        for (int j = K + lane; j < K + kTW; j += 32) {
            const int gc = it.gc0 + j;
            if ((unsigned)gc < (unsigned)W) st1(gdst + (size_t)gr * W + gc, src[i * WW + j]);
        }
    }
}

__device__ __forceinline__ void channel_coeffs(const TiledArgs &a, int c, float *sc, float *adt, bool *inside) {
    const float al = clamp_alpha(a.d, __ldg(a.alpha + c), inside);
    *adt = al * a.d.dt;
    *sc = __ldg(a.scal + c);
}

template <typename T, int KH>
__global__ void __launch_bounds__(kThreads) tiny_tiled_fwd_kernel(const TiledArgs a) {
    extern __shared__ __align__(16) float win[];
    const pde_tiny_desc &d = a.d;
    const int K = d.steps, H = d.H, W = d.W, WH = kTH + 2 * K, WW = kTW + 2 * K;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float *w0 = win, *w1 = win + WH * WW;   // w1: only touched when K > 1
    const T *gu = static_cast<const T *>(a.u);
    T *gout = static_cast<T *>(a.out);
    long long item = blockIdx.x;
    if (item >= a.nitems) return;
    Item nxt = decode(a, item);
    Regs<KH> r;
    load_window(r, gu + nxt.plane * H * W, nxt, H, W, WH, WW, warp, lane);
    for (; item < a.nitems; item += gridDim.x) {
        const Item it = nxt;
        __syncthreads();   // everyone is done with the previous item's windows
        store_window(r, w0, WH, WW, warp, lane);
        __syncthreads();
        if (item + gridDim.x < a.nitems) {   // the next window streams in while this one computes
            nxt = decode(a, item + gridDim.x);
            load_window(r, gu + nxt.plane * H * W, nxt, H, W, WH, WW, warp, lane);
        }
        float sc, adt;
        bool inside;
        channel_coeffs(a, it.c, &sc, &adt, &inside);
        T *dst = gout + it.plane * H * W;
        if (K == 0) {
            copy_tile(w0, dst, 0, WW, it, H, W, warp, lane);
            continue;
        }
        const float *src = w0;
        for (int s = 1; s < K; ++s) {
            float *nb = (s & 1) ? w1 : w0;
            fwd_step<T>(src, nb, nullptr, s, WH, WW, it, H, W, sc, adt, d.blend, warp, lane);
            __syncthreads();
            src = nb;
        }
        fwd_step<T>(src, nullptr, dst, K, WH, WW, it, H, W, sc, adt, d.blend, warp, lane);
    }
}

// Backward windows: U = u_0, L0 / L1 = adjoint ping-pong (L0 receives gout), A / B = recomputed forward states.
// K <= 1 touches U and L0 only.
template <typename T, int KH>
__global__ void __launch_bounds__(kThreads) tiny_tiled_bwd_kernel(const TiledArgs a) {
    extern __shared__ __align__(16) float win[];
    const pde_tiny_desc &d = a.d;
    const int K = d.steps, H = d.H, W = d.W, WH = kTH + 2 * K, WW = kTW + 2 * K, WA = WH * WW;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    float *U = win, *L0 = win + WA, *L1 = win + 2 * WA, *A = win + 3 * WA, *Bw = win + 4 * WA;
    const T *gu = static_cast<const T *>(a.u), *gg = static_cast<const T *>(a.gout);
    T *ggin = static_cast<T *>(a.gin);
    __shared__ double red[2][kWarps];
    // gridDim.x is a multiple of C and items are channel-fastest, so every item of this block has one channel
    float sc, adt;
    bool inside;
    channel_coeffs(a, blockIdx.x % d.C, &sc, &adt, &inside);
    const float bl = d.blend;
    double dA = 0.0, dS = 0.0;
    long long item = blockIdx.x;
    Regs<KH> ru, rg;
    Item nxt{};
    if (item < a.nitems) {
        nxt = decode(a, item);
        load_window(ru, gu + nxt.plane * H * W, nxt, H, W, WH, WW, warp, lane);
        load_window(rg, gg + nxt.plane * H * W, nxt, H, W, WH, WW, warp, lane);
    }
    for (; item < a.nitems; item += gridDim.x) {
        const Item it = nxt;
        __syncthreads();
        store_window(ru, U, WH, WW, warp, lane);
        store_window(rg, L0, WH, WW, warp, lane);
        __syncthreads();
        if (item + gridDim.x < a.nitems) {
            nxt = decode(a, item + gridDim.x);
            load_window(ru, gu + nxt.plane * H * W, nxt, H, W, WH, WW, warp, lane);
            load_window(rg, gg + nxt.plane * H * W, nxt, H, W, WH, WW, warp, lane);
        }
        T *gdst = a.gin ? ggin + it.plane * H * W : nullptr;
        if (K == 0) {
            if (gdst) copy_tile(L0, gdst, 0, WW, it, H, W, warp, lane);
            continue;
        }
        float accA = 0.0f, accS = 0.0f;
        const float *g = L0;
        for (int s = K - 1; s >= 0; --s) {
            // u_s, valid on window cells [s, WH - s)
            const float *us = U;
            for (int t = 1; t <= s; ++t) {
                float *nb = (t & 1) ? A : Bw;
                fwd_step<T>(us, nb, nullptr, t, WH, WW, it, H, W, sc, adt, bl, warp, lane);
                __syncthreads();
                us = nb;
            }
            // lambda_s on window cells [K - s, WH - K + s) from lambda_{s+1}; s = 0 is the tile, to grad_input
            float *ldst = s == 0 ? nullptr : (g == L0 ? L1 : L0);
            const int lo = K - s;
            for (int i = lo + warp; i < WH - lo; i += kWarps) {
                const int gr = it.gr0 + i;
                const bool row_in = (unsigned)gr < (unsigned)H, row_tile = i >= K && i < K + kTH;
                for (int j = lo + lane; j < WW - lo; j += 32) {
                    const int gc = it.gc0 + j;
                    if (!row_in || (unsigned)gc >= (unsigned)W) {
                        if (ldst) ldst[i * WW + j] = 0.0f;
                        continue;
                    }
                    const float *pg = g + i * WW + j;
                    const float gc0 = pg[0], gw = gc0 * bl;
                    const float z = fmaf(adt, lap1(pg, WW, bl), gw);   // Lap0(g_w), g_w = blend g
                    if (row_tile && j >= K && j < K + kTW) {
                        const float *pu = us + i * WW + j;
                        accA = fmaf(gw, lap1(pu, WW, sc), accA);       // Lap0(v), v = s u
                        accS = fmaf(z, pu[0], accS);
                    }
                    const float o = fmaf(sc, z, gc0 - gw);
                    if (ldst) ldst[i * WW + j] = o;
                    else if (gdst) st1(gdst + (size_t)gr * W + gc, o);
                }
            }
            if (s > 0) {
                __syncthreads();
                g = ldst;
            }
        }
        dA += (double)accA;
        dS += (double)accS;
    }
    for (int o = 16; o > 0; o >>= 1) {
        dA += __shfl_xor_sync(0xffffffffu, dA, o);
        dS += __shfl_xor_sync(0xffffffffu, dS, o);
    }
    if (lane == 0) { red[0][warp] = dA; red[1][warp] = dS; }
    __syncthreads();
    if (tid == 0) {
        double sa = 0.0, ss = 0.0;
        for (int w = 0; w < kWarps; ++w) { sa += red[0][w]; ss += red[1][w]; }
        a.part[2 * blockIdx.x] = sa;
        a.part[2 * blockIdx.x + 1] = ss;
    }
}

// per channel c: the partials of blocks c, c + C, ... in block order; the alpha gradient is 0 for a clamped channel
__global__ void tiny_tiled_finish_kernel(pde_tiny_desc d, int nblocks, const double *__restrict__ part,
                                         const float *__restrict__ alpha, float *g_alpha, float *g_scal) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= d.C) return;
    double sa = 0.0, ss = 0.0;
    for (int b = c; b < nblocks; b += d.C) { sa += part[2 * b]; ss += part[2 * b + 1]; }
    bool inside;
    clamp_alpha(d, alpha[c], &inside);
    g_alpha[c] = inside ? (float)(sa * (double)d.dt) : 0.0f;
    g_scal[c] = (float)ss;
}

// ------------------------------------------------------------------------------------------ host
struct TiledPlan {
    const void *kern;
    size_t smem;
    int per_sm;
    int grid;
    TiledArgs a;
};

template <typename T>
static const void *pick_kernel(bool bwd, int K) {
    if (bwd) return K <= 1 ? reinterpret_cast<const void *>(tiny_tiled_bwd_kernel<T, 1>)
                           : reinterpret_cast<const void *>(tiny_tiled_bwd_kernel<T, kTiledMaxSteps>);
    return K <= 1 ? reinterpret_cast<const void *>(tiny_tiled_fwd_kernel<T, 1>)
                  : reinterpret_cast<const void *>(tiny_tiled_fwd_kernel<T, kTiledMaxSteps>);
}

static int plan_tiled(const pde_tiny_desc *d, int io_bytes, bool bwd, const DeviceProps &props, TiledPlan *p) {
    const int K = d->steps;
    const size_t wa = (size_t)(kTH + 2 * K) * (kTW + 2 * K) * sizeof(float);
    p->smem = (bwd ? (K > 1 ? 5 : 2) : (K > 1 ? 2 : 1)) * wa;
    p->kern = io_bytes == 2 ? pick_kernel<__nv_bfloat16>(bwd, K) : pick_kernel<float>(bwd, K);
    int rc = cached_occupancy(p->kern, kThreads, p->smem, &p->per_sm);
    if (rc) return rc;
    TiledArgs &a = p->a;
    a = TiledArgs{};
    a.d = *d;
    a.ntw = (d->W + kTW - 1) / kTW;
    a.ntiles = a.ntw * ((d->H + kTH - 1) / kTH);
    a.nitems = (long long)d->B * d->C * a.ntiles;
    long long grid = (long long)props.sm_count * (p->per_sm < 8 ? p->per_sm : 8);
    if (grid > a.nitems) grid = a.nitems;
    if (bwd) {   // a multiple of C (one channel per block), at most sm_count * 8 + C: the workspace query's bound
        grid -= grid % d->C;
        if (grid < d->C) grid = d->C;
    }
    p->grid = (int)grid;
    return PDE_OK;
}

int tiny_tiled_forward(const pde_tiny_desc *d, int io_bytes, const void *u, const float *alpha, const float *scal,
                       void *out, const DeviceProps &props, cudaStream_t st) {
    TiledPlan p;
    int rc = plan_tiled(d, io_bytes, false, props, &p);
    if (rc) return rc;
    p.a.u = u; p.a.alpha = alpha; p.a.scal = scal; p.a.out = out;
    if (debug_enabled())
        fprintf(stderr, "[pde_b200] tiny tiled fwd plan: B=%d C=%d H=%d W=%d K=%d io=%s tile=%dx%d window=%dx%d smem=%zu "
                "occ=%d grid=%d items=%lld\n", d->B, d->C, d->H, d->W, d->steps, io_bytes == 2 ? "bf16" : "fp32", kTH, kTW,
                kTH + 2 * d->steps, kTW + 2 * d->steps, p.smem, p.per_sm, p.grid, p.a.nitems);
    void *kargs[] = {&p.a};
    PDE_CUDA_TRY(cudaLaunchKernel(p.kern, dim3((unsigned)p.grid), dim3(kThreads), kargs, p.smem, st));
    return cuda_last_error();
}

int tiny_tiled_backward(const pde_tiny_desc *d, int io_bytes, const void *u, const void *gout, const float *alpha,
                        const float *scal, void *gin, float *g_alpha, float *g_scal, void *workspace,
                        size_t workspace_bytes, const DeviceProps &props, cudaStream_t st) {
    if (!workspace || workspace_bytes < tiny_tiled_workspace_bytes(d, props.sm_count)) return PDE_ERR_WORKSPACE;
    TiledPlan p;
    int rc = plan_tiled(d, io_bytes, true, props, &p);
    if (rc) return rc;
    p.a.u = u; p.a.gout = gout; p.a.alpha = alpha; p.a.scal = scal; p.a.gin = gin;
    p.a.part = reinterpret_cast<double *>((reinterpret_cast<uintptr_t>(workspace) + 255u) & ~(uintptr_t)255u);
    if (debug_enabled())
        fprintf(stderr, "[pde_b200] tiny tiled bwd plan: B=%d C=%d H=%d W=%d K=%d io=%s tile=%dx%d window=%dx%d smem=%zu "
                "occ=%d grid=%d items=%lld gin=%d\n", d->B, d->C, d->H, d->W, d->steps, io_bytes == 2 ? "bf16" : "fp32",
                kTH, kTW, kTH + 2 * d->steps, kTW + 2 * d->steps, p.smem, p.per_sm, p.grid, p.a.nitems, gin != nullptr);
    void *kargs[] = {&p.a};
    PDE_CUDA_TRY(cudaLaunchKernel(p.kern, dim3((unsigned)p.grid), dim3(kThreads), kargs, p.smem, st));
    rc = cuda_last_error();
    if (rc) return rc;
    tiny_tiled_finish_kernel<<<(d->C + 127) / 128, 128, 0, st>>>(*d, p.grid, p.a.part, alpha, g_alpha, g_scal);
    return cuda_last_error();
}

}  // namespace tiled
}  // namespace pde
