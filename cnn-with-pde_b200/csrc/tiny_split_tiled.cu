// tiny_imagenet.ImprovedDiffusionLayer's dormant methods (tiny_split.cu) on the planes tiny_split_kernel cannot
// hold: any H x W up to 4096 x 4096 beyond 64 x 64.  Same maps, same arithmetic, lines of any length.
//
// Implicit modes.  One lane owns one line (a row for the x solve, a column for the y solve) and runs the serial
// recurrence of tiny_split.cu's solve_line op for op, so on a line both kernels compute the results are equal bit
// for bit.  A warp owns 32 adjacent lines of one plane and walks them in chunks of 32 cells: each chunk is a
// 32 x 32 tile staged through the warp's own shared-memory tile (odd pitch: a lane walking its line and a lane
// holding a tile row both hit 32 distinct banks), moved between memory one 128-byte tile row per instruction, so
// row and column solves both load and store coalesced.  The next chunk's loads are issued before the current
// chunk's recurrence.  Forward elimination parks its values in `out`, back substitution reads them back in reverse
// order; the last chunk stays in shared memory between the two.  Every cell of a line is read and written by the
// line's own lane only, so a solve may run in place: the ADI step is the x solve into `out`, then the y solve on
// `out`.  The pivots depend on the bands, eps and the line length only; every block factorises its axis into
// shared memory (c'_i and 1 / denom_i, 32 KB at n = 4096) while its warps' first loads are in flight.
//
// Explicit modes: a warp per plane row, a lane per cell, explicit_line's operation order; u and out must not overlap.
#include <cstdio>

#include "common.cuh"
#include "tiny_split_tiled.cuh"

namespace pde {
namespace tsplit_tiled {

constexpr int kWarps = 8, kThreads = 32 * kWarps;
constexpr int kPitch = 33;   // tile row pitch in floats

struct SolveArgs {
    const float *u;
    float *out;
    size_t plane;        // H * W
    long long units;     // B * groups: a unit is 32 adjacent lines of one plane
    int groups;          // units per plane
    int n, nlines, W;    // line length, lines per plane, plane width (row pitch)
    float am, bmid, bend, eps;
};

// factorise() of tiny_split.cu into cp[0, n) and inv[0, n), by the whole block.  A middle row's pivot is a function
// of the previous row's alone, denom_i = clamp(bmid - am * (am / denom_{i-1}), eps), so once two consecutive middle
// pivots are equal bit for bit, every later middle row repeats them.  Thread 0 runs the recurrence up to that row
// (through all n rows when it never settles), the block copies the repeated row, and thread 0 finishes the last row.
__device__ void factorise_block(float *cp, float *inv, int n, float am, float bmid, float bend, float eps) {
    __shared__ int s_rep;   // the first middle row that repeats its predecessor, n if none does
    if (threadIdx.x == 0) {
        float c = __fdiv_rn(am, bend);
        cp[0] = c;
        inv[0] = __fdiv_rn(1.0f, bend);
        int rep = n;
        unsigned prev = 0;
        for (int i = 1; i < n; ++i) {
            const float b = i == n - 1 ? bend : bmid;
            float denom = __fsub_rn(b, __fmul_rn(am, c));
            denom = denom < eps ? eps : denom;
            c = i < n - 1 ? __fdiv_rn(am, denom) : 0.0f;
            cp[i] = c;
            inv[i] = __fdiv_rn(1.0f, denom);
            if (i >= 2 && i < n - 1 && __float_as_uint(denom) == prev) {
                rep = i;
                break;
            }
            prev = __float_as_uint(denom);
        }
        s_rep = rep;
    }
    __syncthreads();
    const int rep = s_rep;
    if (rep < n) {
        const float c = cp[rep], iv = inv[rep];
        for (int i = rep + 1 + threadIdx.x; i < n - 1; i += blockDim.x) {
            cp[i] = c;
            inv[i] = iv;
        }
        if (threadIdx.x == 0) {
            float denom = __fsub_rn(bend, __fmul_rn(am, c));
            denom = denom < eps ? eps : denom;
            cp[n - 1] = 0.0f;
            inv[n - 1] = __fdiv_rn(1.0f, denom);
        }
        __syncthreads();
    }
}

// Offset in the plane of cell e of line a.  A tile row is 32 consecutive cells in memory: lane = cell for rows,
// lane = line for columns; r is the other index.
template <bool kRows>
__device__ __forceinline__ int cell_of(int r, int lane, int l0, int c0, int W, int *a, int *e) {
    *a = kRows ? r : lane;
    *e = kRows ? lane : r;
    return kRows ? (l0 + r) * W + c0 + lane : (c0 + r) * W + l0 + lane;
}

// chunk [c0, c0 + 32) of lines [l0, l0 + 32) into registers: streamed input, or values this lane parked earlier
template <bool kRows, bool kParked>
__device__ __forceinline__ void load_tile(float (&v)[32], const float *plane, int l0, int c0, const SolveArgs &s,
                                          int lane) {
#pragma unroll
    for (int r = 0; r < 32; ++r) {
        int a, e;
        const int off = cell_of<kRows>(r, lane, l0, c0, s.W, &a, &e);
        const bool in = l0 + a < s.nlines && c0 + e < s.n;
        v[r] = in ? (kParked ? __ldcg(plane + off) : __ldcs(plane + off)) : 0.0f;
    }
}

// registers -> tile: line a at tile[a * kPitch], cell e of the chunk at + e
template <bool kRows>
__device__ __forceinline__ void put_tile(float *tile, const float (&v)[32], int lane) {
#pragma unroll
    for (int r = 0; r < 32; ++r) tile[kRows ? r * kPitch + lane : lane * kPitch + r] = v[r];
}

// tile -> chunk [c0, c0 + 32) of lines [l0, l0 + 32): parked (kept in L2 for the read back) or final
template <bool kRows, bool kFinal>
__device__ __forceinline__ void store_tile(float *plane, const float *tile, int l0, int c0, const SolveArgs &s,
                                           int lane) {
#pragma unroll
    for (int r = 0; r < 32; ++r) {
        int a, e;
        const int off = cell_of<kRows>(r, lane, l0, c0, s.W, &a, &e);
        if (l0 + a < s.nlines && c0 + e < s.n) {
            const float x = tile[a * kPitch + e];
            if (kFinal) __stcs(plane + off, x);
            else __stcg(plane + off, x);
        }
    }
}

template <bool kRows>
__global__ void __launch_bounds__(kThreads, 3) tiny_split_solve_kernel(const SolveArgs s) {
    extern __shared__ float sm[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, n = s.n, nk = (n + 31) / 32;
    float *cp = sm, *inv = sm + n, *tile = sm + 2 * n + warp * 32 * kPitch;
    float *mine = tile + lane * kPitch;   // this lane's line in the tile
    const float am = s.am;
    long long unit = (long long)blockIdx.x * kWarps + warp;
    const long long stride = (long long)gridDim.x * kWarps;
    float v[32];
    if (unit < s.units)
        load_tile<kRows, false>(v, s.u + (size_t)(unit / s.groups) * s.plane, (int)(unit % s.groups) * 32, 0, s, lane);
    factorise_block(cp, inv, n, am, s.bmid, s.bend, s.eps);
    for (; unit < s.units; unit += stride) {
        const size_t base = (size_t)(unit / s.groups) * s.plane;
        const int l0 = (int)(unit % s.groups) * 32;
        const float *src = s.u + base;
        float *dst = s.out + base;
        // forward elimination: x_i = (x_i - am x_{i-1}) / denom_i
        float prev = 0.0f;
        for (int k = 0; k < nk; ++k) {
            const int c0 = k * 32;
            __syncwarp();
            put_tile<kRows>(tile, v, lane);
            __syncwarp();
            if (k + 1 < nk) load_tile<kRows, false>(v, src, l0, c0 + 32, s, lane);
            else if (nk > 1) load_tile<kRows, true>(v, dst, l0, c0 - 32, s, lane);   // back substitution's first
#pragma unroll
            for (int e = 0; e < 32; ++e) {
                if (c0 + e < n) {
                    float x = mine[e];
                    x = c0 + e == 0 ? __fmul_rn(x, inv[0]) : __fmul_rn(__fsub_rn(x, __fmul_rn(am, prev)), inv[c0 + e]);
                    mine[e] = x;
                    prev = x;
                }
            }
            if (k + 1 < nk) {
                __syncwarp();
                store_tile<kRows, false>(dst, tile, l0, c0, s, lane);
            }
        }
        // back substitution: x_i -= c'_i x_{i+1}; the tile holds the last chunk
        float next = 0.0f;
        for (int k = nk - 1; k >= 0; --k) {
            const int c0 = k * 32;
            if (k + 1 < nk) {
                __syncwarp();
                put_tile<kRows>(tile, v, lane);
                __syncwarp();
                if (k > 0) load_tile<kRows, true>(v, dst, l0, c0 - 32, s, lane);
            }
            if (k == 0 && unit + stride < s.units)   // the next unit's first chunk streams in under this one
                load_tile<kRows, false>(v, s.u + (size_t)((unit + stride) / s.groups) * s.plane,
                                        (int)((unit + stride) % s.groups) * 32, 0, s, lane);
#pragma unroll
            for (int e = 31; e >= 0; --e) {
                const int i = c0 + e;
                if (i < n) {
                    float x = mine[e];
                    if (i < n - 1) x = __fsub_rn(x, __fmul_rn(cp[i], next));
                    mine[e] = x;
                    next = x;
                }
            }
            __syncwarp();
            store_tile<kRows, true>(dst, tile, l0, c0, s, lane);
        }
    }
}

// u + k (Neumann second difference) along one axis, explicit_line's order; a warp per row, lanes over its cells
template <bool kRows>
__global__ void __launch_bounds__(kThreads) tiny_split_explicit_kernel(const float *__restrict__ u,
                                                                       float *__restrict__ out, long long rows, int H,
                                                                       int W, float k) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (long long row = (long long)blockIdx.x * kWarps + warp; row < rows; row += (long long)gridDim.x * kWarps) {
        const int h = (int)(row % H);
        const size_t base = (size_t)row * W;
        const int n = kRows ? W : H, st = kRows ? 1 : W;
        for (int w = lane; w < W; w += 32) {
            const int i = kRows ? w : h;
            const float *p = u + base + w;
            const float x = __ldg(p);
            float y = x;
            if (n >= 2) {
                float acc;
                if (i == 0) acc = __fsub_rn(__ldg(p + st), x);
                else if (i == n - 1) acc = __fsub_rn(__ldg(p - st), x);
                else acc = __fadd_rn(__fsub_rn(__ldg(p - st), __fmul_rn(2.0f, x)), __ldg(p + st));
                y = __fadd_rn(x, __fmul_rn(k, acc));
            }
            __stcs(out + base + w, y);
        }
    }
}

// ------------------------------------------------------------------------------------------ host
struct Launch {
    const void *kern;
    size_t smem;
    int grid, regs, occ;
};

static int plan(const void *kern, size_t smem, long long blocks, const DeviceProps &props, Launch *l) {
    KernelInfo ki;
    int rc = kernel_info(kern, smem, &ki);
    if (rc) return rc;
    rc = cached_occupancy(kern, kThreads, smem, &l->occ);
    if (rc) return rc;
    const long long cap = (long long)props.sm_count * l->occ;
    l->kern = kern;
    l->smem = smem;
    l->regs = ki.regs;
    l->grid = (int)(blocks < cap ? blocks : cap);
    return PDE_OK;
}

static int solve_plan(const pde_tiny_split_desc *d, bool rows, const float *u, float *out, const DeviceProps &props,
                      SolveArgs *s, Launch *l) {
    const float *c = rows ? d->cx : d->cy;
    *s = SolveArgs{};
    s->u = u;
    s->out = out;
    s->plane = (size_t)d->H * d->W;
    s->n = rows ? d->W : d->H;
    s->nlines = rows ? d->H : d->W;
    s->W = d->W;
    s->groups = (s->nlines + 31) / 32;
    s->units = (long long)d->B * s->groups;
    s->am = c[0];
    s->bmid = c[1];
    s->bend = c[2];
    s->eps = d->eps;
    const void *kern = rows ? reinterpret_cast<const void *>(tiny_split_solve_kernel<true>)
                            : reinterpret_cast<const void *>(tiny_split_solve_kernel<false>);
    const size_t smem = (size_t)(2 * s->n + kWarps * 32 * kPitch) * sizeof(float);
    return plan(kern, smem, (s->units + kWarps - 1) / kWarps, props, l);
}

int tiny_split_tiled(const pde_tiny_split_desc *d, const float *u, float *out, const DeviceProps &props,
                     cudaStream_t st) {
    const int mode = d->mode;
    if (mode >= 3) {
        const bool rows = mode == 3;
        const long long nrows = (long long)d->B * d->H;
        const void *kern = rows ? reinterpret_cast<const void *>(tiny_split_explicit_kernel<true>)
                                : reinterpret_cast<const void *>(tiny_split_explicit_kernel<false>);
        Launch l;
        int rc = plan(kern, 0, (nrows + kWarps - 1) / kWarps, props, &l);
        if (rc) return rc;
        if (debug_enabled())
            fprintf(stderr, "[pde_b200] tiny split tiled plan: mode=%d B=%d H=%d W=%d explicit_%c threads=%d grid=%d "
                    "smem=0 regs=%d occ=%d\n", mode, d->B, d->H, d->W, rows ? 'x' : 'y', kThreads, l.grid, l.regs, l.occ);
        const float *uu = u;
        float *oo = out;
        long long r = nrows;
        int H = d->H, W = d->W;
        float k = rows ? d->cx[0] : d->cy[0];
        void *kargs[] = {&uu, &oo, &r, &H, &W, &k};
        PDE_CUDA_TRY(cudaLaunchKernel(l.kern, dim3((unsigned)l.grid), dim3(kThreads), kargs, 0, st));
        return cuda_last_error();
    }
    // x solve (modes 0, 1) into out, then y solve (modes 0, 2): on out for the ADI step
    SolveArgs sx, sy;
    Launch lx{}, ly{};
    int rc;
    if (mode != 2 && (rc = solve_plan(d, true, u, out, props, &sx, &lx))) return rc;
    if (mode != 1 && (rc = solve_plan(d, false, mode == 0 ? out : u, out, props, &sy, &ly))) return rc;
    if (debug_enabled())
        fprintf(stderr, "[pde_b200] tiny split tiled plan: mode=%d B=%d H=%d W=%d threads=%d x: grid=%d smem=%zu regs=%d "
                "occ=%d y: grid=%d smem=%zu regs=%d occ=%d\n", mode, d->B, d->H, d->W, kThreads, lx.grid, lx.smem,
                lx.regs, lx.occ, ly.grid, ly.smem, ly.regs, ly.occ);
    if (mode != 2) {
        void *kargs[] = {&sx};
        PDE_CUDA_TRY(cudaLaunchKernel(lx.kern, dim3((unsigned)lx.grid), dim3(kThreads), kargs, lx.smem, st));
        if ((rc = cuda_last_error())) return rc;
    }
    if (mode != 1) {
        void *kargs[] = {&sy};
        PDE_CUDA_TRY(cudaLaunchKernel(ly.kern, dim3((unsigned)ly.grid), dim3(kThreads), kargs, ly.smem, st));
        if ((rc = cuda_last_error())) return rc;
    }
    return PDE_OK;
}

}  // namespace tsplit_tiled
}  // namespace pde
