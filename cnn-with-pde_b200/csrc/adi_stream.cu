// Implicit ADI layers on planes beyond one block's shared memory: every configuration with 1 <= C <= 64 and
// 2 <= N <= 4096 (include/pde_b200.h, pde_adi_stream_*; DESIGN.md section 4.13).
//
// The reference classes take any `size` and `channels`; adi_generic.cu and adi_wide.cu hold one sample's planes in
// one block's shared memory and so stop at C * N * (N | 1) * 4 bytes <= 200 KB.  Here the state lives in global
// memory and every pass is its own launch:
//
//   * tables: one sweep's (r, 1 / pivot, r / pivot, mask) float4 per cell, [c][i][line], computed by
//     generic::prepare_line (gprepare_kernel's operations, op for op) just before the sweep and shared by the batch -- a
//     ring of one sweep (16 C N^2 bytes), never the whole call's 16 S C N^2;
//   * sweeps: one lane per (sample, channel, line) runs sweep_line's recurrence op for op.  A warp owns 32 adjacent
//     lines of one plane and moves 32 x 32 tiles through its own shared-memory tile (odd pitch), so rows (x sweeps)
//     and columns (y sweeps) both load and store coalesced; forward elimination is parked in the destination and
//     the next chunk's loads are issued before the current chunk's recurrence (tiny_split_tiled.cu, DESIGN 4.8);
//   * channel ops: a thread per pixel keeps the pixel's C values in registers, mix_pixels' summation order, in
//     place; the skip blend is the generic kernels' expression.  Outputs equal adi_generic.cu / adi_wide.cu bit for
//     bit where both serve;
//   * backward: the state at the end of every step is kept (steps planes a sample) and each step is replayed from
//     its start when it is reversed, so the workspace is (steps + sweeps per step + 1) C N^2 floats a sample in
//     flight (samples in chunks that fit 1 GiB; one sample may exceed it).  The adjoint of a sweep runs
//     reverse_line's recurrences and writes each sample's lambda . (L x) over the sweep's output, which it no longer
//     needs; one launch then sums those over the chunk's samples in fixed order (double) and applies the smoothing
//     transpose, dt / h^2 and the clamp mask once per sweep, adding into the map gradients (no atomics).  Channel
//     and skip gradients are double partials over fixed pixel ranges, summed in fixed order at the end.
#include "adi_lines.cuh"

namespace pde {
namespace adi {
namespace stream {

constexpr int kMaxN = 4096;
constexpr int kPitch = 33;                               // tile row pitch in floats
constexpr int kSweepWarps = 8;                           // forward sweeps: one tile a warp
constexpr int kAdjWarps = 4;                             // adjoint sweeps: two tiles a warp
constexpr int kChanParts = 64;                           // pixel ranges of the channel-gradient partials
constexpr int kSkipParts = 256;                          // blocks of the skip-gradient partials
constexpr size_t kChunkBytes = (size_t)1 << 30;          // state planes of the samples in flight

static size_t cnn(const pde_adi_desc &d) { return (size_t)d.C * d.N * d.N; }

// ------------------------------------------------------------------------------------------ domain and sizes
static int validate(const pde_adi_desc *d) {
    if (!d) return PDE_ERR_INVALID;
    if (d->B < 0 || d->C < 1 || d->N < 1 || d->steps < 0 || d->chan_op < 0 || d->chan_op > 2) return PDE_ERR_INVALID;
    if (d->N < 2 || d->N > kMaxN || d->C > PDE_ADI_MAX_CHANNELS) return PDE_ERR_UNSUPPORTED;
    if (d->steps * sweeps_per_step(*d) > PDE_MAX_SWEEPS) return PDE_ERR_UNSUPPORTED;
    return PDE_OK;
}

static size_t per_sample_bytes(const pde_adi_desc &d) {
    return ((size_t)d.steps + sweeps_per_step(d) + 1) * cnn(d) * sizeof(float);
}

static long long chunk_of(const pde_adi_desc &d) {
    long long k = (long long)(kChunkBytes / per_sample_bytes(d));
    const long long b = d.B > 1 ? d.B : 1;
    if (k > b) k = b;
    return k < 1 ? 1 : k;
}

static size_t forward_bytes(const pde_adi_desc &d) { return 16 * cnn(d); }

struct Layout {   // backward workspace, in this order (every region starts 16-byte aligned)
    size_t chan, skip, tab, state, total;
};

static Layout backward_layout(const pde_adi_desc &d) {
    Layout l;
    l.chan = 0;
    l.skip = l.chan + (d.chan_op ? (size_t)kChanParts * d.C * d.C * sizeof(double) : 0);
    l.tab = l.skip + (d.skip ? (size_t)kSkipParts * sizeof(double) : 0);
    l.state = l.tab + 16 * cnn(d);
    l.total = l.state + (size_t)chunk_of(d) * per_sample_bytes(d);
    return l;
}

// ------------------------------------------------------------------------------------------ kernels
// tables of one sweep: a thread per (channel, line)
__global__ void __launch_bounds__(128) sprep_kernel(const __grid_constant__ pde_adi_desc d, int axis, float tt, float dts,
                                                    float h2, const float *__restrict__ ab, const float *__restrict__ bb,
                                                    const float *__restrict__ atc, const float *__restrict__ btc,
                                                    float4 *tab) {
    const int id = blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= d.C * d.N) return;
    const int l = id % d.N, c = id / d.N;
    generic::prepare_line(d, axis, c, l, tt, dts, h2, ab, bb, atc, btc, tab + (size_t)c * d.N * d.N + l);
}

// Offset in a plane of tile row r, lane `lane`, for the unit of lines [l0, l0 + 32) and the chunk of cells
// [c0, c0 + 32).  A tile row is 32 consecutive floats in memory: lane = cell for rows, lane = line for columns.
template <bool kRows>
__device__ __forceinline__ size_t cell_of(int r, int lane, int l0, int c0, int N, int *a, int *e) {
    *a = kRows ? r : lane;   // line within the unit
    *e = kRows ? lane : r;   // cell within the chunk
    return kRows ? (size_t)(l0 + r) * N + c0 + lane : (size_t)(c0 + r) * N + l0 + lane;
}

template <bool kRows>
__device__ __forceinline__ void load_tile(float (&v)[32], const float *plane, int l0, int c0, int N, int lane) {
#pragma unroll
    for (int r = 0; r < 32; ++r) {
        int a, e;
        const size_t off = cell_of<kRows>(r, lane, l0, c0, N, &a, &e);
        v[r] = (l0 + a < N && c0 + e < N) ? __ldcg(plane + off) : 0.0f;
    }
}

// registers -> tile: line a at tile[a * kPitch], cell e of the chunk at + e
template <bool kRows>
__device__ __forceinline__ void put_tile(float *tile, const float (&v)[32], int lane) {
#pragma unroll
    for (int r = 0; r < 32; ++r) tile[kRows ? r * kPitch + lane : lane * kPitch + r] = v[r];
}

template <bool kRows>
__device__ __forceinline__ void store_tile(float *plane, const float *tile, int l0, int c0, int N, int lane) {
#pragma unroll
    for (int r = 0; r < 32; ++r) {
        int a, e;
        const size_t off = cell_of<kRows>(r, lane, l0, c0, N, &a, &e);
        if (l0 + a < N && c0 + e < N) __stcg(plane + off, tile[a * kPitch + e]);
    }
}

struct SweepArgs {
    const float *src;      // [nb][C][N][N]
    float *dst;            // may be src
    const float4 *tab;     // this sweep's tables, [c][i][line]
    long long units;       // nb * C * groups: a unit is 32 adjacent lines of one plane
    int groups, N, C;
};

// One implicit sweep of every line: sweep_line's recurrences (adi_lines.cuh) op for op.
template <bool kRows>
__global__ void __launch_bounds__(32 * kSweepWarps) ssweep_kernel(const SweepArgs s) {
    __shared__ float tiles[kSweepWarps][32 * kPitch];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, N = s.N, nk = (N + 31) / 32;
    const size_t NN = (size_t)N * N;
    float *tile = tiles[warp], *mine = tile + lane * kPitch;
    const long long stride = (long long)gridDim.x * kSweepWarps;
    long long unit = (long long)blockIdx.x * kSweepWarps + warp;
    float v[32];
    if (unit < s.units) load_tile<kRows>(v, s.src + (size_t)(unit / s.groups) * NN, (int)(unit % s.groups) * 32, 0, N, lane);
    for (; unit < s.units; unit += stride) {
        const long long pl = unit / s.groups;   // (sample, channel) plane
        const int l0 = (int)(unit % s.groups) * 32, l = l0 + lane;
        const bool live = l < N;
        const float4 *tq = s.tab + (size_t)(pl % s.C) * NN + l;
        const float *src = s.src + (size_t)pl * NN;
        float *dst = s.dst + (size_t)pl * NN;
        // forward elimination: d*_i = (d_i + r_i d*_{i-1}) / pivot_i
        float ds = 0.0f;
        for (int k = 0; k < nk; ++k) {
            const int c0 = k * 32;
            __syncwarp();
            put_tile<kRows>(tile, v, lane);
            __syncwarp();
            if (k + 1 < nk) load_tile<kRows>(v, src, l0, c0 + 32, N, lane);
            else if (nk > 1) load_tile<kRows>(v, dst, l0, c0 - 32, N, lane);   // back substitution's first
            if (live) {
#pragma unroll 8
                for (int e = 0; e < 32; ++e) {
                    const int i = c0 + e;
                    if (i < N) {
                        const float4 q = __ldg(tq + (size_t)i * N);
                        ds = i == 0 ? mine[e] * q.y : fmaf(q.x, ds, mine[e]) * q.y;
                        mine[e] = ds;
                    }
                }
            }
            if (k + 1 < nk) {
                __syncwarp();
                store_tile<kRows>(dst, tile, l0, c0, N, lane);
            }
        }
        // back substitution: x_i = d*_i + (r_i / pivot_i) x_{i+1}; the tile holds the last chunk
        float x = ds;
        for (int k = nk - 1; k >= 0; --k) {
            const int c0 = k * 32;
            if (k + 1 < nk) {
                __syncwarp();
                put_tile<kRows>(tile, v, lane);
                __syncwarp();
                if (k > 0) load_tile<kRows>(v, dst, l0, c0 - 32, N, lane);
            }
            if (k == 0 && unit + stride < s.units)   // the next unit's first chunk streams in under this one
                load_tile<kRows>(v, s.src + (size_t)((unit + stride) / s.groups) * NN, (int)((unit + stride) % s.groups) * 32, 0,
                                 N, lane);
            if (live) {
#pragma unroll 8
                for (int e = 31; e >= 0; --e) {
                    const int i = c0 + e;
                    if (i < N - 1) {
                        x = fmaf(__ldg(&tq[(size_t)i * N].z), x, mine[e]);
                        mine[e] = x;
                    }
                }
            }
            __syncwarp();
            store_tile<kRows>(dst, tile, l0, c0, N, lane);
        }
    }
}

struct AdjArgs {
    float *g;              // [nb][C][N][N]: adjoint of the sweep's output in, of its input out
    float *x;              // [nb][C][N][N]: the sweep's output in, lambda . (L x) per cell out
    const float4 *tab;
    long long units;
    int groups, N, C;
};

// Adjoint of one sweep (reverse_line's recurrences): w_i = g_i + e_{i-1} w_{i-1};
// lambda_i = (w_i + r_{i+1} lambda_{i+1}) / pivot_i; gs_i = lambda_i (L x)_i.
template <bool kRows>
__global__ void __launch_bounds__(32 * kAdjWarps) sadj_kernel(const AdjArgs s) {
    __shared__ float gt[kAdjWarps][32 * kPitch], xt[kAdjWarps][32 * kPitch];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, N = s.N, nk = (N + 31) / 32;
    const size_t NN = (size_t)N * N;
    float *gtile = gt[warp], *xtile = xt[warp];
    float *gmine = gtile + lane * kPitch, *xmine = xtile + lane * kPitch;
    for (long long unit = (long long)blockIdx.x * kAdjWarps + warp; unit < s.units; unit += (long long)gridDim.x * kAdjWarps) {
        const long long pl = unit / s.groups;
        const int l0 = (int)(unit % s.groups) * 32, l = l0 + lane;
        const bool live = l < N;
        const float4 *tq = s.tab + (size_t)(pl % s.C) * NN + l;
        float *g = s.g + (size_t)pl * NN, *xs = s.x + (size_t)pl * NN;
        float v[32];
        load_tile<kRows>(v, g, l0, 0, N, lane);
        float w = 0.0f;
        for (int k = 0; k < nk; ++k) {
            const int c0 = k * 32;
            __syncwarp();
            put_tile<kRows>(gtile, v, lane);
            __syncwarp();
            if (k + 1 < nk) load_tile<kRows>(v, g, l0, c0 + 32, N, lane);
            if (live) {
#pragma unroll 8
                for (int e = 0; e < 32; ++e) {
                    const int i = c0 + e;
                    if (i < N) {
                        w = i == 0 ? gmine[e] : fmaf(__ldg(&tq[(size_t)(i - 1) * N].z), w, gmine[e]);
                        gmine[e] = w;
                    }
                }
            }
            if (k + 1 < nk) {
                __syncwarp();
                store_tile<kRows>(g, gtile, l0, c0, N, lane);
            }
        }
        float lam = 0.0f, r_up = 0.0f, xp = 0.0f;
        for (int k = nk - 1; k >= 0; --k) {
            const int c0 = k * 32;
            __syncwarp();
            if (k + 1 < nk) {
                load_tile<kRows>(v, g, l0, c0, N, lane);
                put_tile<kRows>(gtile, v, lane);
            }
            load_tile<kRows>(v, xs, l0, c0, N, lane);
            put_tile<kRows>(xtile, v, lane);
            // x_{c0 - 1}: the previous chunk's last cell, not yet overwritten
            const float xlast = (live && c0 > 0) ? __ldcg(xs + (kRows ? (size_t)l * N + c0 - 1 : (size_t)(c0 - 1) * N + l)) : 0.0f;
            __syncwarp();
            if (live) {
#pragma unroll 8
                for (int e = 31; e >= 0; --e) {
                    const int i = c0 + e;
                    if (i < N) {
                        const float4 q = __ldg(tq + (size_t)i * N);
                        lam = i == N - 1 ? gmine[e] * q.y : fmaf(r_up, lam, gmine[e]) * q.y;
                        gmine[e] = lam;
                        const float xc = xmine[e];
                        const float xm = i == 0 ? 0.0f : (e > 0 ? xmine[e - 1] : xlast);
                        const float lx = i == N - 1 ? xm - xc : (i == 0 ? xp - xc : (xm - xc) + (xp - xc));
                        xmine[e] = lam * lx;
                        xp = xc;
                        r_up = q.x;
                    }
                }
            }
            __syncwarp();
            store_tile<kRows>(g, gtile, l0, c0, N, lane);
            store_tile<kRows>(xs, xtile, l0, c0, N, lane);
        }
    }
}

// The map gradients of one sweep: gs summed over the chunk's samples (double, sample order), then smoothing^T,
// dt / h^2 and the clamp mask as reverse_line applies them, added to the gradients (cell q owned by one thread).
__global__ void __launch_bounds__(256) sred_kernel(const __grid_constant__ pde_adi_desc d, int nb, int axis, float tt,
                                                   float scale, const float *__restrict__ gs, const float *__restrict__ base,
                                                   const float *__restrict__ tc, float *g_base, float *g_tc) {
    const int N = d.N;
    const size_t NN = (size_t)N * N, CNN = (size_t)d.C * NN, st = axis ? (size_t)N : 1;
    const float wgt = d.smooth ? scale * (1.0f / 3.0f) : scale;
    for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < CNN; q += (size_t)gridDim.x * blockDim.x) {
        const int i = axis ? (int)((q / N) % N) : (int)(q % N);
        auto sum = [&](size_t p) {
            double a = 0.0;
            for (int b = 0; b < nb; ++b) a += (double)gs[(size_t)b * CNN + p];
            return (float)a;
        };
        const float s0 = sum(q);
        float g = s0;
        if (d.smooth) {   // replicate padding: an end cell's missing neighbour is the cell itself
            const float sm = i > 0 ? sum(q - st) : s0, sp = i < N - 1 ? sum(q + st) : s0;
            g = (sp + s0) + sm;
        }
        const float raw = __fadd_rn(__ldg(base + q), __fmul_rn(__ldg(tc + q), tt));
        bool m = raw >= d.cmin;
        if (d.has_max) m = m && raw <= d.cmax;
        const float gc = g * wgt * (m ? 1.0f : 0.0f);
        g_base[q] = g_base[q] + gc;
        g_tc[q] = fmaf(gc, tt, g_tc[q]);
    }
}

// dst[b][o][p] = sum_i M[o][i] src[b][i][p] (kT: M[i][o]), i ascending from 0.0f: mix_pixels' order.  In place allowed.
template <int CB, bool kT>
__global__ void __launch_bounds__(256) smix_kernel(const float *src, float *dst, const float *__restrict__ mat, int C,
                                                   size_t NN, long long pixels) {
    __shared__ float ms[PDE_ADI_MAX_CHANNELS * PDE_ADI_MAX_CHANNELS];
    for (int q = threadIdx.x; q < C * C; q += blockDim.x) ms[q] = __ldg(mat + q);
    __syncthreads();
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < pixels; p += (long long)gridDim.x * blockDim.x) {
        const long long b = p / (long long)NN;
        const size_t off = (size_t)b * C * NN + (size_t)(p - b * (long long)NN);
        float v[CB];
#pragma unroll
        for (int c = 0; c < CB; ++c) v[c] = c < C ? src[off + (size_t)c * NN] : 0.0f;
        for (int o = 0; o < C; ++o) {
            float acc = 0.0f;
#pragma unroll
            for (int i = 0; i < CB; ++i)
                if (i < C) acc = fmaf(kT ? ms[i * C + o] : ms[o * C + i], v[i], acc);
            dst[off + (size_t)o * NN] = acc;
        }
    }
}

// channel-gradient partials: part[c][d][range] += sum over the chunk's samples and the range's pixels of g[c] x[d]
__global__ void __launch_bounds__(256) sdot_kernel(const float *__restrict__ g, const float *__restrict__ x, int C, size_t NN,
                                                   int nb, double *part) {
    __shared__ double red[8];
    const int pair = blockIdx.y, c = pair / C, dd = pair - c * C;
    const size_t lo = NN * blockIdx.x / kChanParts, hi = NN * (blockIdx.x + 1) / kChanParts;
    double s = 0.0;
    for (int b = 0; b < nb; ++b) {
        const float *gp = g + ((size_t)b * C + c) * NN, *xp = x + ((size_t)b * C + dd) * NN;
        for (size_t p = lo + threadIdx.x; p < hi; p += blockDim.x) s += (double)gp[p] * (double)xp[p];
    }
    s = generic::block_sum(s, red);
    if (threadIdx.x == 0) part[(size_t)pair * kChanParts + blockIdx.x] += s;
}

// adjoint of the layer's output -> adjoint of the last step's output; skip partials (out = sig u0 + (1 - sig) uF)
__global__ void __launch_bounds__(256) sinit_kernel(const float *__restrict__ gout, const float *__restrict__ u0,
                                                    const float *uF, float *G, long long n, const float *skipw, int skip,
                                                    double *part) {
    __shared__ double red[8];
    const float sig = skip ? generic::sigmoid_of(skipw) : 0.0f;
    double s = 0.0;
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < n; q += (long long)gridDim.x * blockDim.x) {
        float gv = __ldcs(gout + q);
        if (skip) {
            s += (double)gv * ((double)__ldg(u0 + q) - (double)uF[q]);
            gv *= 1.0f - sig;
        }
        G[q] = gv;
    }
    if (skip) {
        s = generic::block_sum(s, red);
        if (threadIdx.x == 0) part[blockIdx.x] += s;
    }
}

__global__ void __launch_bounds__(256) sgin_kernel(const float *__restrict__ G, const float *__restrict__ gout, float *gin,
                                                   long long n, const float *skipw, int skip) {
    const float sig = skip ? generic::sigmoid_of(skipw) : 0.0f;
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < n; q += (long long)gridDim.x * blockDim.x) {
        float v = G[q];
        if (skip) v = fmaf(sig, __ldcs(gout + q), v);
        __stcs(gin + q, v);
    }
}

// out <- skip blend of (steps ? out : u) with u (SVHN.py:74), the generic kernels' expression
__global__ void __launch_bounds__(256) sout_kernel(const float *__restrict__ u0, float *out, long long n, int steps,
                                                   const float *skipw, int skip) {
    const float sig = skip ? generic::sigmoid_of(skipw) : 0.0f;
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < n; q += (long long)gridDim.x * blockDim.x) {
        float v = steps ? out[q] : __ldg(u0 + q);
        if (skip) v = sig * __ldg(u0 + q) + (1.0f - sig) * v;
        __stcs(out + q, v);
    }
}

__global__ void sfin_kernel(int C, const double *__restrict__ chan_part, const double *__restrict__ skip_part,
                            const float *skipw, float *g_chan, float *g_skip) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (g_chan && q < C * C) {
        double s = 0.0;
        for (int k = 0; k < kChanParts; ++k) s += chan_part[(size_t)q * kChanParts + k];
        g_chan[q] = (float)s;
    }
    if (g_skip && q == 0) {
        double s = 0.0;
        for (int k = 0; k < kSkipParts; ++k) s += skip_part[k];
        const float sg = generic::sigmoid_of(skipw);
        g_skip[0] = (float)(s * (double)sg * (1.0 - (double)sg));
    }
}

// ------------------------------------------------------------------------------------------ host
struct Ctx {
    const pde_adi_desc &d;
    const pde_adi_schedule &sch;
    const float *ab, *bb, *atc, *btc, *chan;
    float4 *tab;
    cudaStream_t st;
    int sm_count;
    int prepared;   // the sweep whose tables the ring holds, -1 for none
};

static int grid_for(const void *kern, int threads, long long blocks, int sm_count) {
    int occ = 1;
    if (cached_occupancy(kern, threads, 0, &occ)) occ = 1;
    const long long cap = (long long)sm_count * occ;
    if (blocks > cap) blocks = cap;
    return (int)(blocks < 1 ? 1 : blocks);
}

static long long flat_blocks(long long n) { return (n + 255) / 256; }

static int prep(Ctx &c, int s) {
    if (c.prepared == s) return PDE_OK;
    const int axis = sweep_axis(s % sweeps_per_step(c.d)), lines = c.d.C * c.d.N;
    sprep_kernel<<<(lines + 127) / 128, 128, 0, c.st>>>(c.d, axis, c.sch.t[s], c.sch.dts[s], c.sch.h2[s], c.ab, c.bb, c.atc,
                                                         c.btc, c.tab);
    c.prepared = s;
    return cuda_last_error();
}

template <typename A>
static void fill_units(A *a, const pde_adi_desc &d, long long nb) {
    a->N = d.N;
    a->C = d.C;
    a->groups = (d.N + 31) / 32;
    a->units = nb * d.C * a->groups;
}

static int sweep(Ctx &c, int s, const float *src, float *dst, long long nb) {
    int rc = prep(c, s);
    if (rc) return rc;
    SweepArgs a{};
    a.src = src;
    a.dst = dst;
    a.tab = c.tab;
    fill_units(&a, c.d, nb);
    const bool rows = sweep_axis(s % sweeps_per_step(c.d)) == 0;
    const void *kern = rows ? reinterpret_cast<const void *>(ssweep_kernel<true>) : reinterpret_cast<const void *>(ssweep_kernel<false>);
    const int grid = grid_for(kern, 32 * kSweepWarps, (a.units + kSweepWarps - 1) / kSweepWarps, c.sm_count);
    void *kargs[] = {&a};
    PDE_CUDA_TRY(cudaLaunchKernel(kern, dim3(grid), dim3(32 * kSweepWarps), kargs, 0, c.st));
    return cuda_last_error();
}

static const void *mix_kernel_for(int C, bool transposed) {
#define PDE_MIX(CB) (transposed ? reinterpret_cast<const void *>(smix_kernel<CB, true>) : reinterpret_cast<const void *>(smix_kernel<CB, false>))
    if (C <= 4) return PDE_MIX(4);
    if (C <= 8) return PDE_MIX(8);
    if (C <= 16) return PDE_MIX(16);
    if (C <= 32) return PDE_MIX(32);
    return PDE_MIX(64);
#undef PDE_MIX
}

static int mix(Ctx &c, const float *src, float *dst, long long nb, bool transposed) {
    const void *kern = mix_kernel_for(c.d.C, transposed);
    size_t NN = (size_t)c.d.N * c.d.N;
    long long pixels = nb * (long long)NN;
    const float *mat = c.chan;
    int C = c.d.C;
    const int grid = grid_for(kern, 256, flat_blocks(pixels), c.sm_count);
    void *kargs[] = {&src, &dst, &mat, &C, &NN, &pixels};
    PDE_CUDA_TRY(cudaLaunchKernel(kern, dim3(grid), dim3(256), kargs, 0, c.st));
    return cuda_last_error();
}

static int launch_grid(Ctx &c, const void *kern, long long n) { return grid_for(kern, 256, flat_blocks(n), c.sm_count); }

static void print_plan(const char *pass, const pde_adi_desc &d, long long chunk, size_t ws) {
    const void *kerns[] = {reinterpret_cast<const void *>(sprep_kernel), reinterpret_cast<const void *>(ssweep_kernel<true>),
                           reinterpret_cast<const void *>(ssweep_kernel<false>), reinterpret_cast<const void *>(sadj_kernel<true>),
                           reinterpret_cast<const void *>(sadj_kernel<false>), reinterpret_cast<const void *>(sred_kernel),
                           mix_kernel_for(d.C, false)};
    const char *names[] = {"sprep", "ssweep<rows>", "ssweep<cols>", "sadj<rows>", "sadj<cols>", "sred", "smix"};
    const int n = pass[0] == 'f' ? 3 : 7;
    const long long units = (long long)chunk * d.C * ((d.N + 31) / 32);
    fprintf(stderr, "[pde_b200] stream %s plan: B=%d C=%d N=%d steps=%d chunk=%lld units=%lld ws=%zu", pass, d.B, d.C, d.N,
            d.steps, chunk, units, ws);
    for (int i = 0; i < n; ++i) {
        KernelInfo ki{};
        kernel_info(kerns[i], 0, &ki);
        fprintf(stderr, " %s(regs=%d smem=%zu)", names[i], ki.regs, ki.static_smem);
    }
    fprintf(stderr, "\n");
}

static bool maps_ok(const pde_adi_desc &d, const float *ab, const float *bb, const float *atc, const float *btc) {
    return d.steps == 0 || (ab && bb && atc && btc);
}

int forward(const pde_adi_desc &d, const pde_adi_schedule &sch, const float *ab, const float *bb, const float *atc,
            const float *btc, const float *u, const float *chan, const float *skipw, float *out, void *ws, size_t ws_bytes,
            cudaStream_t st) {
    if (d.B == 0) return PDE_OK;
    if (!u || !out || (d.chan_op && !chan) || (d.skip && !skipw) || !maps_ok(d, ab, bb, atc, btc)) return PDE_ERR_INVALID;
    if (!ws || ws_bytes < forward_bytes(d) || (reinterpret_cast<uintptr_t>(ws) & 255u)) return PDE_ERR_WORKSPACE;
    DeviceProps props;
    int rc = query_props(&props);
    if (rc) return rc;
    if (debug_enabled()) print_plan("fwd", d, d.B, forward_bytes(d));
    Ctx c{d, sch, ab, bb, atc, btc, chan, static_cast<float4 *>(ws), st, props.sm_count, -1};
    const int sps = sweeps_per_step(d);
    const long long nb = d.B;
    for (int step = 0; step < d.steps; ++step) {
        const float *cur = step ? out : u;
        if (d.chan_op == 1) {
            if ((rc = mix(c, cur, out, nb, false))) return rc;
            cur = out;
        }
        for (int k = 0; k < sps; ++k) {
            if ((rc = sweep(c, step * sps + k, cur, out, nb))) return rc;
            cur = out;
        }
        if (d.chan_op == 2 && (rc = mix(c, out, out, nb, false))) return rc;
    }
    if (d.steps == 0 || d.skip) {
        const long long n = nb * (long long)cnn(d);
        sout_kernel<<<launch_grid(c, reinterpret_cast<const void *>(sout_kernel), n), 256, 0, st>>>(u, out, n, d.steps, skipw, d.skip);
        if ((rc = cuda_last_error())) return rc;
    }
    return PDE_OK;
}

static int adjoint(Ctx &c, int s, float *G, float *X, long long nb, float *const *gmaps) {
    int rc = prep(c, s);
    if (rc) return rc;
    const pde_adi_desc &d = c.d;
    AdjArgs a{};
    a.g = G;
    a.x = X;
    a.tab = c.tab;
    fill_units(&a, d, nb);
    const int axis = sweep_axis(s % sweeps_per_step(d));
    const void *kern = axis == 0 ? reinterpret_cast<const void *>(sadj_kernel<true>) : reinterpret_cast<const void *>(sadj_kernel<false>);
    const int grid = grid_for(kern, 32 * kAdjWarps, (a.units + kAdjWarps - 1) / kAdjWarps, c.sm_count);
    void *kargs[] = {&a};
    PDE_CUDA_TRY(cudaLaunchKernel(kern, dim3(grid), dim3(32 * kAdjWarps), kargs, 0, c.st));
    if ((rc = cuda_last_error())) return rc;
    const float scale = c.sch.dts[s] / c.sch.h2[s];   // IEEE fp32 division, as gprepare_kernel's __fdiv_rn
    const float *base = axis ? c.bb : c.ab, *tc = axis ? c.btc : c.atc;
    const long long cells = (long long)cnn(d);
    sred_kernel<<<launch_grid(c, reinterpret_cast<const void *>(sred_kernel), cells), 256, 0, c.st>>>(
        d, (int)nb, axis, c.sch.t[s], scale, X, base, tc, gmaps[2 * axis], gmaps[2 * axis + 1]);
    return cuda_last_error();
}

static int chan_grad(Ctx &c, const float *G, const float *X, long long nb, double *part) {
    const int C = c.d.C;
    sdot_kernel<<<dim3(kChanParts, C * C), 256, 0, c.st>>>(G, X, C, (size_t)c.d.N * c.d.N, (int)nb, part);
    return cuda_last_error();
}

int backward(const pde_adi_desc &d, const pde_adi_schedule &sch, const float *ab, const float *bb, const float *atc,
             const float *btc, const float *u, const float *gout, const float *chan, const float *skipw, float *gin,
             float *g_ab, float *g_bb, float *g_atc, float *g_btc, float *g_chan, float *g_skip, void *ws, size_t ws_bytes,
             cudaStream_t st) {
    if (!g_ab || !g_bb || !g_atc || !g_btc || (d.chan_op && !g_chan) || (d.skip && !g_skip)) return PDE_ERR_INVALID;
    const size_t CNN = cnn(d);
    PDE_CUDA_TRY(cudaMemsetAsync(g_ab, 0, CNN * sizeof(float), st));
    PDE_CUDA_TRY(cudaMemsetAsync(g_bb, 0, CNN * sizeof(float), st));
    PDE_CUDA_TRY(cudaMemsetAsync(g_atc, 0, CNN * sizeof(float), st));
    PDE_CUDA_TRY(cudaMemsetAsync(g_btc, 0, CNN * sizeof(float), st));
    if (d.B == 0) {
        if (d.chan_op) PDE_CUDA_TRY(cudaMemsetAsync(g_chan, 0, (size_t)d.C * d.C * sizeof(float), st));
        if (d.skip) PDE_CUDA_TRY(cudaMemsetAsync(g_skip, 0, sizeof(float), st));
        return PDE_OK;
    }
    if (!u || !gout || (d.chan_op && !chan) || (d.skip && !skipw) || !maps_ok(d, ab, bb, atc, btc)) return PDE_ERR_INVALID;
    const Layout lay = backward_layout(d);
    if (!ws || ws_bytes < lay.total || (reinterpret_cast<uintptr_t>(ws) & 255u)) return PDE_ERR_WORKSPACE;
    DeviceProps props;
    int rc = query_props(&props);
    if (rc) return rc;
    const long long chunk = chunk_of(d);
    if (debug_enabled()) print_plan("bwd", d, chunk, lay.total);
    char *w = static_cast<char *>(ws);
    double *chan_part = reinterpret_cast<double *>(w + lay.chan), *skip_part = reinterpret_cast<double *>(w + lay.skip);
    if (d.chan_op) PDE_CUDA_TRY(cudaMemsetAsync(chan_part, 0, lay.skip - lay.chan, st));
    if (d.skip) PDE_CUDA_TRY(cudaMemsetAsync(skip_part, 0, lay.tab - lay.skip, st));
    Ctx c{d, sch, ab, bb, atc, btc, chan, reinterpret_cast<float4 *>(w + lay.tab), st, props.sm_count, -1};
    float *state = reinterpret_cast<float *>(w + lay.state);
    float *const gmaps[4] = {g_ab, g_atc, g_bb, g_btc};
    const int sps = sweeps_per_step(d), steps = d.steps;
    const size_t slab = (size_t)chunk * CNN;   // one state plane set of the chunk
    auto Z = [&](int k) { return state + (size_t)(k - 1) * slab; };       // state after step k, k = 1 ... steps
    auto Y = [&](int j) { return state + (size_t)(steps + j) * slab; };   // output of sweep j of the replayed step
    float *G = state + (size_t)(steps + sps) * slab;                      // the adjoint
    for (long long b0 = 0; b0 < d.B; b0 += chunk) {
        const long long nb = d.B - b0 < chunk ? d.B - b0 : chunk;
        const float *u0 = u + (size_t)b0 * CNN, *go = gout + (size_t)b0 * CNN;
        // forward: the state at the end of every step
        for (int step = 0; step < steps; ++step) {
            const float *cur = step ? Z(step) : u0;
            float *dst = Z(step + 1);
            if (d.chan_op == 1) {
                if ((rc = mix(c, cur, dst, nb, false))) return rc;
                cur = dst;
            }
            for (int k = 0; k < sps; ++k) {
                if ((rc = sweep(c, step * sps + k, cur, dst, nb))) return rc;
                cur = dst;
            }
            if (d.chan_op == 2 && (rc = mix(c, dst, dst, nb, false))) return rc;
        }
        const long long n = nb * (long long)CNN;
        sinit_kernel<<<kSkipParts, 256, 0, st>>>(go, u0, steps ? Z(steps) : u0, G, n, skipw, d.skip, skip_part);
        if ((rc = cuda_last_error())) return rc;
        for (int step = steps - 1; step >= 0; --step) {
            const float *src = step ? Z(step) : u0;
            // replay the step; without a post-step mix the last sweep's output is the kept end state
            const int nrep = d.chan_op == 2 ? sps : sps - 1;
            const float *cur = src;
            if (d.chan_op == 1) {
                if ((rc = mix(c, src, Y(0), nb, false))) return rc;
                cur = Y(0);
            }
            for (int j = 0; j < nrep; ++j) {
                if ((rc = sweep(c, step * sps + j, cur, Y(j), nb))) return rc;
                cur = Y(j);
            }
            if (d.chan_op == 2) {
                if ((rc = chan_grad(c, G, Y(sps - 1), nb, chan_part))) return rc;
                if ((rc = mix(c, G, G, nb, true))) return rc;
            }
            for (int j = sps - 1; j >= 0; --j) {
                float *X = j < nrep ? Y(j) : Z(step + 1);
                if ((rc = adjoint(c, step * sps + j, G, X, nb, gmaps))) return rc;
            }
            if (d.chan_op == 1) {
                if ((rc = chan_grad(c, G, src, nb, chan_part))) return rc;
                if ((rc = mix(c, G, G, nb, true))) return rc;
            }
        }
        if (gin) {
            sgin_kernel<<<launch_grid(c, reinterpret_cast<const void *>(sgin_kernel), n), 256, 0, st>>>(G, go, gin + (size_t)b0 * CNN, n,
                                                                                                       skipw, d.skip);
            if ((rc = cuda_last_error())) return rc;
        }
    }
    if (d.chan_op || d.skip) {
        sfin_kernel<<<(d.C * d.C + 255) / 256, 256, 0, st>>>(d.C, chan_part, skip_part, skipw, d.chan_op ? g_chan : nullptr,
                                                             d.skip ? g_skip : nullptr);
        if ((rc = cuda_last_error())) return rc;
    }
    return PDE_OK;
}

}  // namespace stream
}  // namespace adi
}  // namespace pde

using namespace pde;
using namespace pde::adi;

extern "C" size_t pde_adi_stream_forward_workspace_bytes(const pde_adi_desc *d) {
    return stream::validate(d) == PDE_OK ? stream::forward_bytes(*d) : 0;
}

extern "C" size_t pde_adi_stream_backward_workspace_bytes(const pde_adi_desc *d) {
    return stream::validate(d) == PDE_OK ? stream::backward_layout(*d).total : 0;
}

extern "C" int pde_adi_stream_forward(const pde_adi_desc *d, const pde_adi_schedule *sched, const float *alpha_base,
                                      const float *beta_base, const float *alpha_time_coeff, const float *beta_time_coeff,
                                      const float *u, const float *chan, const float *skip_weight, float *out, void *workspace,
                                      size_t workspace_bytes, void *stream) {
    int rc = stream::validate(d);
    if (rc) return rc;
    if (!sched) return PDE_ERR_INVALID;
    return stream::forward(*d, *sched, alpha_base, beta_base, alpha_time_coeff, beta_time_coeff, u, chan, skip_weight, out,
                           workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

extern "C" int pde_adi_stream_backward(const pde_adi_desc *d, const pde_adi_schedule *sched, const float *alpha_base,
                                       const float *beta_base, const float *alpha_time_coeff, const float *beta_time_coeff,
                                       const float *u, const float *gout, const float *chan, const float *skip_weight,
                                       float *gin, float *g_alpha_base, float *g_beta_base, float *g_alpha_time_coeff,
                                       float *g_beta_time_coeff, float *g_chan, float *g_skip_weight, void *workspace,
                                       size_t workspace_bytes, void *stream) {
    int rc = stream::validate(d);
    if (rc) return rc;
    if (!sched) return PDE_ERR_INVALID;
    return stream::backward(*d, *sched, alpha_base, beta_base, alpha_time_coeff, beta_time_coeff, u, gout, chan, skip_weight,
                            gin, g_alpha_base, g_beta_base, g_alpha_time_coeff, g_beta_time_coeff, g_chan, g_skip_weight,
                            workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}
