// Implicit ADI layers with PDE_MAX_CHANNELS < C <= PDE_ADI_MAX_CHANNELS channels (5 ... 64), any plane edge
// 2 ... 128 while one sample's planes fit a block's shared memory (C * N * (N | 1) * 4 bytes <= 200 KB).
//
// The channel-aware reference layers take any channel count (SVHN.py:13, cifar10.py:25, cifar_2version.py:25);
// applied to CNN feature maps rather than to the RGB image they see 8 ... 64 channels.  This is the
// run-time-sized path of adi_generic.cu (DESIGN.md section 4.9) with two changes:
//
//   * a slot's threads STRIDE over the C * N lines of a sweep instead of owning one each, so C * N is no
//     longer bounded by the block size (the history / accumulator layouts, the tables of gprepare_kernel and
//     the line routines of adi_lines.cuh are the generic path's, unchanged; the thread that writes a line's
//     history is still the one that reads it back);
//   * the channel op is a C x C product per pixel: M is staged once in shared memory (row pitch padded to 4,
//     zeros beyond C, read as float4 broadcasts), a thread owns pixels and keeps a pixel's C inputs in
//     registers (an array of CB >= C, CB = 8, 16, 32, 64: one instantiation per bucket) before it writes
//     the first output.  Its adjoint stages M^T in the same place.  The channel gradient sum_p g uin^T is a
//     small GEMM per sample and step: a thread owns a 4 x 4 (c, d) block and a share of the pixels, sums
//     its products in double for the whole kernel, and the block's partials are reduced in fixed order
//     (per-block partials, then wfinish_kernel in block order: bit-reproducible).
//
// DESIGN.md section 4.10 has the measured numbers.
#include "adi_lines.cuh"

namespace pde {
namespace adi {
namespace wide {

using generic::Line;
using generic::kMaxN;
using generic::kMaxTileBytes;
using generic::kMaxWorkspaceBytes;
using generic::pitch_of;
using generic::tile_bytes;

constexpr int kGT = 4;                                    // edge of a thread's block of the channel gradient

__host__ __device__ inline int mat_pitch(int C) { return (C + 3) & ~3; }
__host__ __device__ inline int gm_edge(int C) { return (C + kGT - 1) / kGT; }
static size_t mat_floats(const pde_adi_desc &d) { return d.chan_op ? (size_t)d.C * mat_pitch(d.C) : 0; }
// register array of a pixel's channels
static int bucket_of(int C) { return C <= 8 ? 8 : (C <= 16 ? 16 : (C <= 32 ? 32 : 64)); }
// 64 channels in registers plus 16 double accumulators: half the block keeps the backward pass below 128 registers
__host__ __device__ constexpr int max_threads(int CB) { return CB >= 64 ? 256 : 512; }

bool serves(const pde_adi_desc &d) {
    if (d.C <= PDE_MAX_CHANNELS || d.C > PDE_ADI_MAX_CHANNELS || d.N < 2 || d.N > kMaxN) return false;
    return tile_bytes(d) <= kMaxTileBytes;
}

// ------------------------------------------------------------------------------------------
// block shape: K slots of `tps` threads (a slot = one sample in flight)
// ------------------------------------------------------------------------------------------
struct Shape {
    int CB, tps, K, threads;
    size_t smem;
};

static Shape shape_of(const pde_adi_desc &d, bool bwd) {
    Shape s;
    s.CB = bucket_of(d.C);
    const int maxt = max_threads(s.CB);
    int tps = d.C * d.N < maxt ? d.C * d.N : maxt;
    const int nb = gm_edge(d.C) * gm_edge(d.C);
    if (tps < nb) tps = nb;   // every block of the channel gradient has a thread (tiny planes)
    int K = maxt / tps;
    const int by_smem = (int)((100u * 1024u) / tile_bytes(d));
    if (K > by_smem) K = by_smem;
    if (K > 8) K = 8;
    if (K < 1) K = 1;
    s.tps = tps;
    s.K = K;
    s.threads = ((K * tps + 31) / 32) * 32;
    size_t work = (size_t)K * tile_bytes(d);
    if (bwd && d.chan_op) {   // after the last sample the tiles hold the per-thread gradient blocks
        const size_t red = (size_t)K * tps * kGT * kGT * sizeof(double);
        if (red > work) work = red;
    }
    s.smem = mat_floats(d) * sizeof(float) + work;
    return s;
}

struct WArgs {
    pde_adi_desc d;
    int S, sps, need_gin;
    int K, tps;              // slots per block, threads per slot
    const Header *hdr;       // per-sweep dt / h^2 and time
    const float4 *tab;       // (r, 1/pivot, r/pivot, mask) at [S][C][i][line] (generic::prepare)
    const float *u, *gout, *chan, *skipw;
    float *out, *gin;
    float2 *acc;             // per slot:  [alpha | beta][C][i][line] of (base, time coefficient)
    float *hist;             // per slot:  [S][C][i][line]         output of every sweep
    float *ins;              // per slot:  [steps][C][row][col]    state at the start of every step (pre-step mix only)
    double *part_chan;       // per block: [C][C]
    double *part_skip;       // per block
};

__device__ __forceinline__ Line my_slot(const WArgs &a) {
    Line t;
    t.cn = a.tps;
    t.active = (int)threadIdx.x < a.K * a.tps;
    t.slot = t.active ? threadIdx.x / a.tps : 0;
    t.within = t.active ? threadIdx.x - t.slot * a.tps : 0;
    t.c = 0;   // a thread has no line of its own here
    t.l = 0;
    return t;
}

// ms[o][i] (row pitch mat_pitch(C), zeros beyond C) <- M[o][i], or M[i][o] for the adjoint.  Whole block.
__device__ __forceinline__ void stage_matrix(float *__restrict__ ms, const float *__restrict__ mat, int C, bool transposed) {
    const int CP = mat_pitch(C);
    for (int q = threadIdx.x; q < C * CP; q += blockDim.x) {
        const int o = q / CP, i = q - o * CP;
        ms[q] = i < C ? __ldg(mat + (transposed ? i * C + o : o * C + i)) : 0.0f;
    }
}

// u[o][p] <- sum_i ms[o][i] u[i][p] for every pixel of the slot's tile (cifar10.py:65-72 before a step,
// SVHN.py:78-86 after it; with ms = M^T the adjoint g <- M^T g).  Sums in the order of adi_generic.cu's
// mix_pixels (i = 0, 1, ... from 0.0f; the padding adds exact zeros).  keep != nullptr: the inputs go there
// first ([c][row][col], the backward pass needs them).
template <int CB>
__device__ __forceinline__ void apply_matrix(float *__restrict__ tile, const float *__restrict__ ms, float *__restrict__ keep,
                                             const Line &t, int C, int N, int P) {
    const int NN = N * N, CP = mat_pitch(C), plane = N * P;
    for (int p = t.within; p < NN; p += t.cn) {
        const int row = p / N, col = p - row * N;
        float *px = tile + row * P + col;
        float v[CB];
#pragma unroll
        for (int c = 0; c < CB; ++c) {
            v[c] = c < C ? px[c * plane] : 0.0f;
            if (keep && c < C) keep[(size_t)c * NN + p] = v[c];
        }
        for (int o = 0; o < C; ++o) {
            const float4 *mr = reinterpret_cast<const float4 *>(ms + o * CP);
            float acc = 0.0f;
#pragma unroll
            for (int i = 0; i < CB; i += 4)
                if (i < C) {
                    const float4 m4 = mr[i / 4];
                    acc = fmaf(m4.x, v[i], acc);
                    acc = fmaf(m4.y, v[i + 1], acc);
                    acc = fmaf(m4.z, v[i + 2], acc);
                    acc = fmaf(m4.w, v[i + 3], acc);
                }
            px[o * plane] = acc;
        }
    }
}

// forward trajectory of the slot's sample in its tile; the backward kernel passes its history slices
template <int CB>
__device__ __forceinline__ void run_sample(const WArgs &a, const float *ms, float *tile, const Line &t, bool valid, float *hist,
                                           float *ins) {
    const pde_adi_desc &d = a.d;
    const int N = d.N, C = d.C, P = pitch_of(N), CN = C * N;
    const size_t NN = (size_t)N * N;
    for (int step = 0; step < d.steps; ++step) {
        if (d.chan_op == 1) {
            if (valid) apply_matrix<CB>(tile, ms, ins ? ins + (size_t)step * C * NN : nullptr, t, C, N, P);
            __syncthreads();
        }
        for (int k = 0; k < a.sps; ++k) {
            const int s = step * a.sps + k, axis = sweep_axis(k);
            if (valid)
                for (int ln = t.within; ln < CN; ln += t.cn) {
                    const int c = ln / N, l = ln - c * N;
                    const size_t lo = ((size_t)(s * C + c) * N) * N + l;
                    float *line = tile + (size_t)c * N * P + (axis ? l : l * P);
                    generic::sweep_line(line, axis ? P : 1, N, a.tab + lo, hist ? hist + lo : nullptr);
                }
            __syncthreads();
        }
        if (d.chan_op == 2) {
            if (valid) apply_matrix<CB>(tile, ms, nullptr, t, C, N, P);
            __syncthreads();
        }
    }
}

template <int CB>
__global__ void __launch_bounds__(max_threads(CB)) wfwd_kernel(const WArgs a) {
    extern __shared__ __align__(16) float wsmem[];
    const pde_adi_desc &d = a.d;
    const int N = d.N, C = d.C, P = pitch_of(N), NN = N * N, K = a.K;
    const Line t = my_slot(a);
    float *ms = wsmem;
    float *tile = wsmem + (d.chan_op ? C * mat_pitch(C) : 0) + (size_t)t.slot * C * N * P;
    if (d.chan_op) stage_matrix(ms, a.chan, C, false);
    const float sig = d.skip ? generic::sigmoid_of(a.skipw) : 0.0f;
    for (long long b0 = (long long)blockIdx.x * K; b0 < d.B; b0 += (long long)gridDim.x * K) {
        const long long b = b0 + t.slot;
        const bool valid = t.active && b < d.B;
        const float *u0 = a.u + (size_t)b * C * NN;
        if (valid) generic::planes_to_tile(u0, tile, t, C, N, P);
        __syncthreads();
        run_sample<CB>(a, ms, tile, t, valid, nullptr, nullptr);
        if (valid) {
            float *o = a.out + (size_t)b * C * NN;
            for (int q = t.within; q < C * NN; q += t.cn) {
                const int c = q / NN, rem = q - c * NN, row = rem / N, col = rem - row * N;
                float v = tile[(c * N + row) * P + col];
                if (d.skip) v = sig * __ldg(u0 + q) + (1.0f - sig) * v;   // SVHN.py:74
                __stcs(o + q, v);
            }
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------
// channel gradient: gM[c][d] += sum_p g[c][p] uin[d][p].  Thread (blk, pg) of a slot owns the kGT x kGT block
// blk of gM and the pixels pg, pg + npg, ...; consecutive threads take consecutive pixels of the same block
// (coalesced uin, conflict-free tile).  `uin` is the input of the channel op: the step's start state
// ([c][row][col], transposed == 0) or the output of the step's last sweep in its own line coordinates
// (x sweep: [c][col][row], transposed == 1).
// ------------------------------------------------------------------------------------------
struct GmPart {
    int blk, pg, npg, c0, d0;
    bool on;
};

__device__ __forceinline__ GmPart gm_part(const Line &t, int C) {
    const int e = gm_edge(C), nb = e * e;
    GmPart g;
    g.npg = t.cn / nb;
    g.on = t.active && t.within < g.npg * nb;
    g.blk = g.on ? t.within / g.npg : 0;
    g.pg = g.on ? t.within - g.blk * g.npg : 0;
    g.c0 = (g.blk / e) * kGT;
    g.d0 = (g.blk % e) * kGT;
    return g;
}

__device__ __forceinline__ void chan_grad(const float *__restrict__ tile, const float *uin, int transposed,
                                          double (&gm)[kGT * kGT], const GmPart &gp, int C, int N, int P) {
    if (!gp.on) return;
    const int NN = N * N, plane = N * P;
    for (int p = gp.pg; p < NN; p += gp.npg) {
        const int hi = p / N, lo = p - hi * N;
        const int row = transposed ? lo : hi, col = transposed ? hi : lo;
        float g[kGT], x[kGT];
#pragma unroll
        for (int k = 0; k < kGT; ++k) {
            g[k] = gp.c0 + k < C ? tile[(gp.c0 + k) * plane + row * P + col] : 0.0f;
            x[k] = gp.d0 + k < C ? uin[(size_t)(gp.d0 + k) * NN + p] : 0.0f;
        }
#pragma unroll
        for (int k = 0; k < kGT; ++k)
#pragma unroll
            for (int j = 0; j < kGT; ++j) gm[k * kGT + j] += (double)g[k] * (double)x[j];
    }
}

template <int CB>
__global__ void __launch_bounds__(max_threads(CB)) wbwd_kernel(const WArgs a) {
    extern __shared__ __align__(16) float wsmem[];
    __shared__ double red[512 / 32];
    const pde_adi_desc &d = a.d;
    const int N = d.N, C = d.C, P = pitch_of(N), NN = N * N, K = a.K, CN = C * N;
    const size_t CNN = (size_t)C * NN;
    const Line t = my_slot(a);
    float *ms = wsmem;
    float *work = wsmem + (d.chan_op ? C * mat_pitch(C) : 0);
    float *tile = work + (size_t)t.slot * C * N * P;
    const float sig = d.skip ? generic::sigmoid_of(a.skipw) : 0.0f;
    const size_t vb = (size_t)blockIdx.x * K + t.slot;       // the slot's slices of the workspace
    float2 *acc = a.acc + vb * 2 * CNN;
    float *hist = a.hist + vb * a.S * CNN;
    float *ins = a.ins ? a.ins + vb * d.steps * CNN : nullptr;
    const GmPart gp = gm_part(t, C);
    double gm[kGT * kGT];
#pragma unroll
    for (int q = 0; q < kGT * kGT; ++q) gm[q] = 0.0;
    double gskip = 0.0;
    if (t.active)
        for (size_t q = t.within; q < 2 * CNN; q += t.cn) acc[q] = make_float2(0.0f, 0.0f);
    __syncthreads();

    for (long long b0 = (long long)blockIdx.x * K; b0 < d.B; b0 += (long long)gridDim.x * K) {
        const long long b = b0 + t.slot;
        const bool valid = t.active && b < d.B;
        const float *u0 = a.u + (size_t)b * CNN, *go = a.gout + (size_t)b * CNN;
        if (d.chan_op) stage_matrix(ms, a.chan, C, false);
        if (valid) generic::planes_to_tile(u0, tile, t, C, N, P);
        __syncthreads();
        run_sample<CB>(a, ms, tile, t, valid, hist, ins);
        if (d.chan_op) stage_matrix(ms, a.chan, C, true);   // the adjoint's matrix from here on
        // the tile turns from the final state into the adjoint of the last step's output
        if (valid)
            for (int q = t.within; q < C * NN; q += t.cn) {
                const int c = q / NN, rem = q - c * NN, row = rem / N, col = rem - row * N;
                float *cell = tile + (c * N + row) * P + col;
                float gv = __ldcs(go + q);
                if (d.skip) {   // out = sig u0 + (1 - sig) uF  (SVHN.py:74)
                    gskip += (double)gv * ((double)__ldg(u0 + q) - (double)*cell);
                    gv *= 1.0f - sig;
                }
                *cell = gv;
            }
        __syncthreads();
        for (int step = d.steps - 1; step >= 0; --step) {
            if (d.chan_op == 2) {
                const int sl = step * a.sps + a.sps - 1;
                if (valid) chan_grad(tile, hist + (size_t)sl * CNN, sweep_axis(a.sps - 1) == 0, gm, gp, C, N, P);
                __syncthreads();
                if (valid) apply_matrix<CB>(tile, ms, nullptr, t, C, N, P);
                __syncthreads();
            }
            for (int k = a.sps - 1; k >= 0; --k) {
                const int s = step * a.sps + k, axis = sweep_axis(k);
                // the next slice to be reversed on its way from HBM into L2 (one thread per slot)
                if (valid && t.within == 0 && s > 0) generic::prefetch_slice_l2(hist + (size_t)(s - 1) * CNN, CNN * sizeof(float));
                if (valid) {
                    const float scale = __ldg(&a.hdr->scale[s]), tt = __ldg(&a.hdr->t[s]);
                    for (int ln = t.within; ln < CN; ln += t.cn) {
                        const int c = ln / N, l = ln - c * N;
                        const size_t lo = ((size_t)c * N) * N + l;
                        float *line = tile + (size_t)c * N * P + (axis ? l : l * P);
                        generic::reverse_line(line, axis ? P : 1, N, a.tab + (size_t)s * CNN + lo, hist + (size_t)s * CNN + lo,
                                              acc + (size_t)(axis ? 1 : 0) * CNN + lo, d.smooth != 0, scale, tt);
                    }
                }
                __syncthreads();
            }
            if (d.chan_op == 1) {
                if (valid) chan_grad(tile, ins + (size_t)step * CNN, 0, gm, gp, C, N, P);
                __syncthreads();
                if (valid) apply_matrix<CB>(tile, ms, nullptr, t, C, N, P);
                __syncthreads();
            }
        }
        if (a.need_gin && valid) {
            float *gi = a.gin + (size_t)b * CNN;
            for (int q = t.within; q < C * NN; q += t.cn) {
                const int c = q / NN, rem = q - c * NN, row = rem / N, col = rem - row * N;
                float v = tile[(c * N + row) * P + col];
                if (d.skip) v = fmaf(sig, __ldcs(go + q), v);
                __stcs(gi + q, v);
            }
        }
        __syncthreads();
    }
    if (d.chan_op) {
        // the block's partial of gM: every (slot, pixel share) block parked in shared memory, then summed in
        // fixed order (slot, pixel share) per entry
        const int e = gm_edge(C), nb = e * e, npg = gp.npg;
        double *part = reinterpret_cast<double *>(work);
        if (gp.on)
#pragma unroll
            for (int q = 0; q < kGT * kGT; ++q) part[((size_t)(t.slot * npg + gp.pg) * nb + gp.blk) * (kGT * kGT) + q] = gm[q];
        __syncthreads();
        for (int q = threadIdx.x; q < C * C; q += blockDim.x) {
            const int c = q / C, dd = q - c * C;
            const int blk = (c / kGT) * e + dd / kGT, k = (c % kGT) * kGT + dd % kGT;
            double s = 0.0;
            for (int w = 0; w < K * npg; ++w) s += part[((size_t)w * nb + blk) * (kGT * kGT) + k];
            a.part_chan[(size_t)blockIdx.x * C * C + q] = s;
        }
    }
    if (d.skip) {
        const double s = generic::block_sum(gskip, red);
        if (threadIdx.x == 0) a.part_skip[blockIdx.x] = s;
    }
}

// ------------------------------------------------------------------------------------------
// finish: the slots' accumulators summed in double, in slot order; alpha kinds come back from line
// coordinates ([c][col][row]) to the map's own order.  Channel partials: C * C per block, block order.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) wfinish_kernel(const __grid_constant__ pde_adi_desc d, int nblk, int nslots,
                                                      const float2 *__restrict__ acc, const double *__restrict__ part_chan,
                                                      const double *__restrict__ part_skip, const float *skipw,
                                                      float *g_ab, float *g_atc, float *g_bb, float *g_btc, float *g_chan,
                                                      float *g_skip) {
    const int N = d.N, C = d.C, NN = N * N;
    const size_t CNN = (size_t)C * NN, CC = (size_t)C * C;
    const size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (id < 2 * CNN) {
        const int beta = id >= CNN;
        const size_t rem = id - (beta ? CNN : 0);
        const int c = (int)(rem / NN), i = (int)((rem % NN) / N), l = (int)(rem % N);
        double s0 = 0.0, s1 = 0.0;
        for (int b = 0; b < nslots; ++b) {
            const float2 v = acc[(size_t)b * 2 * CNN + id];
            s0 += (double)v.x;
            s1 += (double)v.y;
        }
        const size_t q = beta ? ((size_t)c * N + i) * N + l : ((size_t)c * N + l) * N + i;
        (beta ? g_bb : g_ab)[q] = (float)s0;
        (beta ? g_btc : g_atc)[q] = (float)s1;
    } else if (id < 2 * CNN + CC) {
        if (d.chan_op) {
            const size_t q = id - 2 * CNN;
            double s = 0.0;
            for (int b = 0; b < nblk; ++b) s += part_chan[(size_t)b * CC + q];
            g_chan[q] = (float)s;
        }
    } else if (id == 2 * CNN + CC) {
        if (d.skip) {
            double s = 0.0;
            for (int b = 0; b < nblk; ++b) s += part_skip[b];
            const float sg = generic::sigmoid_of(skipw);
            g_skip[0] = (float)(s * (double)sg * (1.0 - (double)sg));
        }
    }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
static const void *fwd_kernel_for(int CB) {
    switch (CB) {
        case 8: return reinterpret_cast<const void *>(wfwd_kernel<8>);
        case 16: return reinterpret_cast<const void *>(wfwd_kernel<16>);
        case 32: return reinterpret_cast<const void *>(wfwd_kernel<32>);
        default: return reinterpret_cast<const void *>(wfwd_kernel<64>);
    }
}

static const void *bwd_kernel_for(int CB) {
    switch (CB) {
        case 8: return reinterpret_cast<const void *>(wbwd_kernel<8>);
        case 16: return reinterpret_cast<const void *>(wbwd_kernel<16>);
        case 32: return reinterpret_cast<const void *>(wbwd_kernel<32>);
        default: return reinterpret_cast<const void *>(wbwd_kernel<64>);
    }
}

struct Plan {
    Shape sh;
    int grid, per_sm;
    size_t acc_floats, hist_floats, ins_floats;   // totals over the grid's slots
    size_t bytes;
};

static size_t align256(size_t n) { return (n + 255u) & ~(size_t)255u; }

// Workspace: per slot in flight the history of all S sweeps (S C N^2 floats), the step inputs of the pre-step
// mix and the accumulators, so the backward pass replays a sample once and walks it back without a second
// replay.  It grows with C; above 1 GB the grid shrinks and blocks loop over more samples (DESIGN.md 4.10).
static int plan_backward(const pde_adi_desc &d, Plan *p) {
    DeviceProps props;
    int rc = query_props(&props);
    if (rc) return rc;
    p->sh = shape_of(d, true);
    if (p->sh.smem > (size_t)props.max_smem_optin) return PDE_ERR_UNSUPPORTED;
    p->per_sm = 1;
    rc = cached_occupancy(bwd_kernel_for(p->sh.CB), p->sh.threads, p->sh.smem, &p->per_sm);
    if (rc) return rc;
    const int K = p->sh.K;
    const size_t CNN = (size_t)d.C * d.N * d.N;
    const int S = d.steps * sweeps_per_step(d);
    const size_t per_block = ((size_t)4 + S + (d.chan_op == 1 ? d.steps : 0)) * CNN * sizeof(float) * K;
    long long grid = (long long)props.sm_count * p->per_sm;
    const long long by_batch = ((long long)d.B + K - 1) / K;
    if (grid > by_batch) grid = by_batch;
    const long long cap = (long long)(kMaxWorkspaceBytes / per_block);
    if (grid > cap) grid = cap;
    if (grid < 1) grid = 1;
    p->grid = (int)grid;
    const size_t slots = (size_t)p->grid * K;
    p->acc_floats = slots * 4 * CNN;
    p->hist_floats = slots * S * CNN;
    p->ins_floats = d.chan_op == 1 ? slots * d.steps * CNN : 0;
    p->bytes = align256(p->acc_floats * sizeof(float)) + align256(p->hist_floats * sizeof(float)) +
               align256(p->ins_floats * sizeof(float)) + align256((size_t)p->grid * ((size_t)d.C * d.C + 1) * sizeof(double)) +
               256;
    return PDE_OK;
}

size_t workspace_bytes(const pde_adi_desc &d) {
    Plan p;
    return plan_backward(d, &p) == PDE_OK ? p.bytes : 0;
}

static void fill_common(WArgs *a, const pde_adi_desc &d, const Shape &sh, const char *tables) {
    a->d = d;
    a->K = sh.K;
    a->tps = sh.tps;
    a->sps = sweeps_per_step(d);
    a->S = d.steps * a->sps;
    a->hdr = reinterpret_cast<const Header *>(tables);
    a->tab = reinterpret_cast<const float4 *>(tables + kHeaderBytes);
}

int forward(const pde_adi_desc &d, const char *tables, const float *u, const float *chan, const float *skipw, float *out,
            cudaStream_t st) {
    DeviceProps props;
    int rc = query_props(&props);
    if (rc) return rc;
    const Shape sh = shape_of(d, false);
    if (sh.smem > (size_t)props.max_smem_optin) return PDE_ERR_UNSUPPORTED;
    const void *kern = fwd_kernel_for(sh.CB);
    int per_sm = 1;
    rc = cached_occupancy(kern, sh.threads, sh.smem, &per_sm);
    if (rc) return rc;
    WArgs a{};
    fill_common(&a, d, sh, tables);
    a.u = u; a.chan = chan; a.skipw = skipw; a.out = out;
    long long grid = (long long)props.sm_count * per_sm;
    if (grid > ((long long)d.B + sh.K - 1) / sh.K) grid = ((long long)d.B + sh.K - 1) / sh.K;
    if (debug_enabled())
        fprintf(stderr, "[pde_b200] wide fwd plan: N=%d C=%d chan_op=%d wfwd<%d> K=%d threads=%d smem=%zu occ=%d grid=%lld\n", d.N,
                d.C, d.chan_op, sh.CB, sh.K, sh.threads, sh.smem, per_sm, grid);
    void *kargs[] = {&a};
    PDE_CUDA_TRY(cudaLaunchKernel(kern, dim3((unsigned)grid), dim3(sh.threads), kargs, sh.smem, st));
    return cuda_last_error();
}

int backward(const pde_adi_desc &d, const char *tables, const float *u, const float *gout, const float *chan,
             const float *skipw, float *gin, float *g_ab, float *g_bb, float *g_atc, float *g_btc, float *g_chan,
             float *g_skip, void *workspace, size_t ws_bytes, cudaStream_t st) {
    Plan p;
    int rc = plan_backward(d, &p);
    if (rc) return rc;
    if (!workspace || ws_bytes < p.bytes) return PDE_ERR_WORKSPACE;
    if (debug_enabled())
        fprintf(stderr, "[pde_b200] wide bwd plan: N=%d C=%d chan_op=%d wbwd<%d> K=%d threads=%d smem=%zu occ=%d grid=%d ws=%zu\n",
                d.N, d.C, d.chan_op, p.sh.CB, p.sh.K, p.sh.threads, p.sh.smem, p.per_sm, p.grid, p.bytes);
    char *w = reinterpret_cast<char *>((reinterpret_cast<uintptr_t>(workspace) + 255u) & ~(uintptr_t)255u);
    WArgs a{};
    fill_common(&a, d, p.sh, tables);
    a.need_gin = gin != nullptr;
    a.u = u; a.gout = gout; a.chan = chan; a.skipw = skipw; a.gin = gin;
    a.acc = reinterpret_cast<float2 *>(w);
    w += align256(p.acc_floats * sizeof(float));
    a.hist = reinterpret_cast<float *>(w);
    w += align256(p.hist_floats * sizeof(float));
    a.ins = p.ins_floats ? reinterpret_cast<float *>(w) : nullptr;
    w += align256(p.ins_floats * sizeof(float));
    a.part_chan = reinterpret_cast<double *>(w);
    a.part_skip = a.part_chan + (size_t)p.grid * d.C * d.C;
    void *kargs[] = {&a};
    PDE_CUDA_TRY(cudaLaunchKernel(bwd_kernel_for(p.sh.CB), dim3(p.grid), dim3(p.sh.threads), kargs, p.sh.smem, st));
    rc = cuda_last_error();
    if (rc) return rc;
    const size_t outs = 2 * (size_t)d.C * d.N * d.N + (size_t)d.C * d.C + 1;
    wfinish_kernel<<<(unsigned)((outs + 255) / 256), 256, 0, st>>>(d, p.grid, p.grid * p.sh.K, a.acc, a.part_chan, a.part_skip,
                                                                  skipw, g_ab, g_atc, g_bb, g_btc, g_chan, g_skip);
    return cuda_last_error();
}

}  // namespace wide
}  // namespace adi
}  // namespace pde
