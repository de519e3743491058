// Implicit ADI layers on plane sizes the specialised kernels are not built for.
//
// The reference classes take any `size` (mnist_test.py:12, SVHN.py:13, cifar10.py:25 ...); adi.cu and
// adi_split.cu hold a line (or half a line) of a sample PAIR in registers and are therefore compiled per
// plane edge (8 ... 32).  Everything else -- any edge from 2 to 128, odd ones included, as long as the
// planes of one sample fit one block's shared memory -- is served here, with the plane edge a run-time
// value:
//
//   * a block works on a few samples at a time ("slots": ~256 threads; all channels of a sample stay
//     together, so the 3x3 channel ops are block-local), one thread per (channel, line); a sample's state
//     lives in a shared-memory tile with an odd row pitch, so that walking along rows (x sweeps: lane =
//     row) and along columns (y sweeps) are both free of bank conflicts; a sweep is two in-place passes
//     over the thread's line (elimination, back substitution), one __syncthreads() per change of
//     orientation;
//   * tables, history and gradient accumulators are all stored in LINE coordinates [c][i][line]
//     (i = position along the sweep, line fastest): whatever the axis, consecutive threads touch
//     consecutive addresses.  A cell's four table values travel as one float4 (r, 1/pivot, r/pivot, mask),
//     its two accumulators (base, time coefficient) as one float2, and all indices inside the line loops
//     are 32-bit: the first version spent 60 % of its instructions on 64-bit address arithmetic;
//   * the backward pass keeps no checkpoints from the forward call: the block replays the sample's
//     trajectory, parks the output of every sweep in its own slice of the workspace (the thread that
//     writes a line is the one that reads it back), then walks the sweeps in reverse: transposed solve
//     through the same factors, lambda . (L x), smoothing^T, clamp mask, accumulate into the slot's
//     fp32 accumulators (one slice per slot, summed in double and in fixed order by gfinish_kernel).
//
// Same arithmetic as the whole-line kernels (fp32 FMA recurrences on 1 / pivot; the pivots themselves
// op for op the reference's, without contraction); tests/test_gpu_parity.py::test_cuda_generic_plane_sizes.
// This is the generality path, not the fast one: the sizes the scripts use (28, 32) never get here.
#include "adi_lines.cuh"   // sweep_line, reverse_line, planes_to_tile ... (shared with adi_wide.cu)

namespace pde {
namespace adi {
namespace generic {

constexpr int kMaxThreads = 384;   // 3 x 128 or 4 x 96 lines (x 168 registers of gbwd_kernel<4>: one block's worth)
constexpr int kChanSlots = PDE_MAX_CHANNELS * PDE_MAX_CHANNELS;

// samples a block works on at a time: enough for ~256 threads while the tiles stay below half an SM's shared memory
static int slots_per_block(const pde_adi_desc &d) {
    int k = 256 / (d.C * d.N);
    const int by_smem = (int)((100u * 1024u) / tile_bytes(d));
    if (k > by_smem) k = by_smem;
    if (k > 8) k = 8;
    return k < 1 ? 1 : k;
}
static int block_threads(const pde_adi_desc &d, int K) { return ((K * d.C * d.N + 31) / 32) * 32; }

bool serves(const pde_adi_desc &d) {
    switch (d.N) {
        case 8: case 12: case 16: case 20: case 24: case 28: case 32: return false;   // adi.cu / adi_split.cu
        default: break;
    }
    if (d.N < 2 || d.N > kMaxN || d.C < 1 || d.C > PDE_MAX_CHANNELS) return false;
    return block_threads(d, 1) <= kMaxThreads && tile_bytes(d) <= kMaxTileBytes;
}

size_t tables_bytes(const pde_adi_desc &d) { return (size_t)kHeaderBytes + 4 * table_elems(d) * sizeof(float); }

// ------------------------------------------------------------------------------------------
// tables: one thread per (sweep, channel, line), the whole line serially (the pivot recurrence is
// serial anyway).  One float4 (r, 1 / pivot, r / pivot, clamp mask) per cell at [s][c][i][line].
// Reference arithmetic: get_alpha_beta_at_time mnist_test.py:33-42 / cifar10.py:53-63,
// smooth_coefficients mnist_test.py:135-149, rows mnist_test.py:83-93, pivots mnist_test.py:169,177-181.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) gprepare_kernel(const __grid_constant__ pde_adi_desc d,
                                                       const __grid_constant__ pde_adi_schedule sch,
                                                       const float *__restrict__ ab, const float *__restrict__ bb,
                                                       const float *__restrict__ atc, const float *__restrict__ btc,
                                                       char *tables) {
    const int N = d.N, C = d.C, sps = sweeps_per_step(d), S = d.steps * sps;
    const int id = blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= S * C * N) return;
    const int l = id % N, c = (id / N) % C, s = id / (C * N);
    const int axis = sweep_axis(s % sps);
    const float *base = axis ? bb : ab, *tc = axis ? btc : atc;
    const float tt = sch.t[s], dts = sch.dts[s], h2 = sch.h2[s];
    const float third = __fdiv_rn(1.0f, 3.0f);
    float4 *tq = reinterpret_cast<float4 *>(tables + kHeaderBytes) + ((size_t)(s * C + c) * N) * N + l;

    auto coef = [&](int i, bool *inside) {
        const size_t q = axis == 0 ? ((size_t)c * N + l) * N + i : ((size_t)c * N + i) * N + l;
        const float raw = __fadd_rn(__ldg(base + q), __fmul_rn(__ldg(tc + q), tt));
        bool m = raw >= d.cmin;
        float k = raw < d.cmin ? d.cmin : raw;
        if (d.has_max) {
            m = m && raw <= d.cmax;
            k = k > d.cmax ? d.cmax : k;
        }
        *inside = m;
        return k;
    };
    if (l == 0 && c == 0) {
        Header *hdr = reinterpret_cast<Header *>(tables);
        hdr->scale[s] = __fdiv_rn(dts, h2);
        hdr->t[s] = tt;
    }
    bool m_cur, m_next = false;
    float k_cur = coef(0, &m_cur), k_prev = k_cur, cst = 0.0f;
    for (int i = 0; i < N; ++i) {
        const float k_next = i + 1 < N ? coef(i + 1, &m_next) : k_cur;   // replicate padding at both ends
        float ks = k_cur;
        if (d.smooth) ks = __fadd_rn(__fadd_rn(__fmul_rn(k_prev, third), __fmul_rn(k_cur, third)), __fmul_rn(k_next, third));
        const float r = __fdiv_rn(__fmul_rn(ks, dts), h2);
        const float diag = (i == 0 || i == N - 1) ? __fadd_rn(1.0f, r) : __fadd_rn(1.0f, __fmul_rn(2.0f, r));
        const float dn = i == 0 ? __fadd_rn(diag, d.eps) : __fadd_rn(__fsub_rn(diag, __fmul_rn(-r, cst)), d.eps);
        cst = __fdiv_rn(-r, dn);
        tq[i * N] = make_float4(r, __fdiv_rn(1.0f, dn), __fdiv_rn(r, dn), m_cur ? 1.0f : 0.0f);
        k_prev = k_cur; k_cur = k_next; m_cur = m_next;
    }
}

// ------------------------------------------------------------------------------------------
// pieces shared by the forward and the backward kernel
// ------------------------------------------------------------------------------------------
struct GArgs {
    pde_adi_desc d;
    int S, sps, need_gin;
    int K;                   // samples a block works on at a time (slots)
    const Header *hdr;       // per-sweep dt / h^2 and time (the backward entry points get no schedule)
    const float4 *tab;       // (r, 1/pivot, r/pivot, mask) at [S][C][i][line]
    const float *u, *gout, *chan, *skipw;
    float *out, *gin;
    float2 *acc;             // per slot:  [alpha | beta][C][i][line] of (base, time coefficient)
    float *hist;             // per slot:  [S][C][i][line]         output of every sweep
    float *ins;              // per slot:  [steps][C][row][col]    state at the start of every step (pre-step mix only)
    double *part_chan;       // per block: [C][C]
    double *part_skip;       // per block
};

// slot q's threads are the C * N threads [q C N, (q + 1) C N), one per (channel, line) (struct Line: adi_lines.cuh)
__device__ __forceinline__ Line my_line(const pde_adi_desc &d, int K) {
    Line t;
    t.cn = d.C * d.N;
    t.active = (int)threadIdx.x < K * t.cn;
    t.slot = t.active ? threadIdx.x / t.cn : 0;
    t.within = t.active ? threadIdx.x - t.slot * t.cn : 0;
    t.c = t.within / d.N;
    t.l = t.within - t.c * d.N;
    return t;
}

// u[c][p] <- sum_d M[c][d] u[d][p] for every pixel (cifar10.py:65-72 before a step, SVHN.py:78-86 after it);
// keep != nullptr: the unmixed planes go there first ([c][row][col], the backward pass needs them)
__device__ __forceinline__ void mix_pixels(float *__restrict__ tile, const float *__restrict__ mat, float *__restrict__ keep,
                                           const Line &t, int C, int N, int P) {
    const int NN = N * N;
    float m[kChanSlots];   // m[c * PDE_MAX_CHANNELS + d]: static indices only, stays in registers
#pragma unroll
    for (int c = 0; c < PDE_MAX_CHANNELS; ++c)
#pragma unroll
        for (int dd = 0; dd < PDE_MAX_CHANNELS; ++dd) m[c * PDE_MAX_CHANNELS + dd] = (c < C && dd < C) ? __ldg(mat + c * C + dd) : 0.0f;
    for (int p = t.within; p < NN; p += t.cn) {
        const int row = p / N, col = p - row * N;
        float v[PDE_MAX_CHANNELS];
#pragma unroll
        for (int c = 0; c < PDE_MAX_CHANNELS; ++c)
            if (c < C) {
                v[c] = tile[(c * N + row) * P + col];
                if (keep) keep[(size_t)c * NN + p] = v[c];
            }
#pragma unroll
        for (int c = 0; c < PDE_MAX_CHANNELS; ++c)
            if (c < C) {
                float acc = 0.0f;
#pragma unroll
                for (int dd = 0; dd < PDE_MAX_CHANNELS; ++dd)
                    if (dd < C) acc = fmaf(m[c * PDE_MAX_CHANNELS + dd], v[dd], acc);
                tile[(c * N + row) * P + col] = acc;
            }
    }
}

// forward trajectory of the slot's sample in its tile; the backward kernel passes its history slices
__device__ __forceinline__ void run_sample(const GArgs &a, float *tile, const Line &t, bool valid, float *hist, float *ins) {
    const pde_adi_desc &d = a.d;
    const int N = d.N, C = d.C, P = pitch_of(N);
    const size_t NN = (size_t)N * N;
    for (int step = 0; step < d.steps; ++step) {
        if (d.chan_op == 1) {
            if (valid) mix_pixels(tile, a.chan, ins ? ins + (size_t)step * C * NN : nullptr, t, C, N, P);
            __syncthreads();
        }
        for (int k = 0; k < a.sps; ++k) {
            const int s = step * a.sps + k, axis = sweep_axis(k);
            if (valid) {
                const float4 *tq = a.tab + ((size_t)(s * C + t.c) * N) * N + t.l;
                float *line = tile + (size_t)t.c * N * P + (axis ? t.l : t.l * P);
                sweep_line(line, axis ? P : 1, N, tq, hist ? hist + ((size_t)(s * C + t.c) * N) * N + t.l : nullptr);
            }
            __syncthreads();
        }
        if (d.chan_op == 2) {
            if (valid) mix_pixels(tile, a.chan, nullptr, t, C, N, P);
            __syncthreads();
        }
    }
}

__global__ void __launch_bounds__(kMaxThreads) gfwd_kernel(const GArgs a) {
    extern __shared__ __align__(16) float gsmem[];
    const pde_adi_desc &d = a.d;
    const int N = d.N, C = d.C, P = pitch_of(N), NN = N * N, K = a.K;
    const Line t = my_line(d, K);
    float *tile = gsmem + (size_t)t.slot * C * N * P;
    const float sig = d.skip ? sigmoid_of(a.skipw) : 0.0f;
    for (long long b0 = (long long)blockIdx.x * K; b0 < d.B; b0 += (long long)gridDim.x * K) {
        const long long b = b0 + t.slot;
        const bool valid = t.active && b < d.B;
        const float *u0 = a.u + (size_t)b * C * NN;
        if (valid) planes_to_tile(u0, tile, t, C, N, P);
        __syncthreads();
        run_sample(a, tile, t, valid, nullptr, nullptr);
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

// g[c][p] <- sum_c M[c][d] g[c][p] and gM[c][d] += sum_p g[c][p] uin[d][p].  `uin` is the input of the
// channel op: the step's start state ([c][row][col], transposed == 0) or the output of the step's last
// sweep in its own line coordinates (x sweep: [c][col][row], transposed == 1).
template <int C>
__device__ __forceinline__ void mix_pixels_adjoint(float *__restrict__ tile, const float *__restrict__ mat,
                                                   const float *__restrict__ uin, int transposed, double (&gm)[C * C],
                                                   const Line &t, int N, int P) {
    const int NN = N * N;
    float m[C * C];
#pragma unroll
    for (int q = 0; q < C * C; ++q) m[q] = __ldg(mat + q);
    for (int p = t.within; p < NN; p += t.cn) {
        // p walks the history in its storage order; (row, col) follows
        const int hi = p / N, lo = p - hi * N;
        const int row = transposed ? lo : hi, col = transposed ? hi : lo;
        float g[C], x[C];
#pragma unroll
        for (int c = 0; c < C; ++c) {
            g[c] = tile[(c * N + row) * P + col];
            x[c] = uin[(size_t)c * NN + p];
        }
#pragma unroll
        for (int c = 0; c < C; ++c)
#pragma unroll
            for (int dd = 0; dd < C; ++dd) gm[c * C + dd] += (double)g[c] * (double)x[dd];
#pragma unroll
        for (int dd = 0; dd < C; ++dd) {
            float acc = 0.0f;
#pragma unroll
            for (int c = 0; c < C; ++c) acc = fmaf(m[c * C + dd], g[c], acc);
            tile[(dd * N + row) * P + col] = acc;
        }
    }
}

// (one instantiation per channel count: the C x C channel-gradient sums are per-thread doubles)
template <int C>
__global__ void __maxnreg__(C <= 3 ? 128 : 168) gbwd_kernel(const GArgs a) {
    extern __shared__ __align__(16) float gsmem[];
    __shared__ double red[kMaxThreads / 32];
    const pde_adi_desc &d = a.d;
    const int N = d.N, P = pitch_of(N), NN = N * N, K = a.K;
    const size_t CNN = (size_t)C * NN;
    const Line t = my_line(d, K);
    float *tile = gsmem + (size_t)t.slot * C * N * P;
    const float sig = d.skip ? sigmoid_of(a.skipw) : 0.0f;
    const size_t vb = (size_t)blockIdx.x * K + t.slot;       // the slot's slices of the workspace
    float2 *acc = a.acc + vb * 2 * CNN;
    float *hist = a.hist + vb * a.S * CNN;
    float *ins = a.ins ? a.ins + vb * d.steps * CNN : nullptr;
    double gm[C * C];
#pragma unroll
    for (int q = 0; q < C * C; ++q) gm[q] = 0.0;
    double gskip = 0.0;
    if (t.active)
        for (size_t q = t.within; q < 2 * CNN; q += t.cn) acc[q] = make_float2(0.0f, 0.0f);
    __syncthreads();

    for (long long b0 = (long long)blockIdx.x * K; b0 < d.B; b0 += (long long)gridDim.x * K) {
        const long long b = b0 + t.slot;
        const bool valid = t.active && b < d.B;
        const float *u0 = a.u + (size_t)b * CNN, *go = a.gout + (size_t)b * CNN;
        if (valid) planes_to_tile(u0, tile, t, C, N, P);
        __syncthreads();
        run_sample(a, tile, t, valid, hist, ins);
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
                if (valid) mix_pixels_adjoint<C>(tile, a.chan, hist + (size_t)sl * CNN, sweep_axis(a.sps - 1) == 0, gm, t, N, P);
                __syncthreads();
            }
            for (int k = a.sps - 1; k >= 0; --k) {
                const int s = step * a.sps + k, axis = sweep_axis(k);
                // the next slice to be reversed on its way from HBM into L2 (one thread per slot; -3 ... -11 % of the kernel)
                if (valid && t.within == 0 && s > 0) prefetch_slice_l2(hist + (size_t)(s - 1) * CNN, CNN * sizeof(float));
                if (valid) {
                    const size_t lo = ((size_t)t.c * N) * N + t.l;
                    float *line = tile + (size_t)t.c * N * P + (axis ? t.l : t.l * P);
                    const float scale = __ldg(&a.hdr->scale[s]), tt = __ldg(&a.hdr->t[s]);
                    reverse_line(line, axis ? P : 1, N, a.tab + (size_t)s * CNN + lo, hist + (size_t)s * CNN + lo,
                                 acc + (size_t)(axis ? 1 : 0) * CNN + lo, d.smooth != 0, scale, tt);
                }
                __syncthreads();
            }
            if (d.chan_op == 1) {
                if (valid) mix_pixels_adjoint<C>(tile, a.chan, ins + (size_t)step * CNN, 0, gm, t, N, P);
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
#pragma unroll
        for (int q = 0; q < C * C; ++q) {
            const double s = block_sum(gm[q], red);
            if (threadIdx.x == 0) a.part_chan[(size_t)blockIdx.x * kChanSlots + q] = s;
        }
    }
    if (d.skip) {
        const double s = block_sum(gskip, red);
        if (threadIdx.x == 0) a.part_skip[blockIdx.x] = s;
    }
}

// ------------------------------------------------------------------------------------------
// finish: the slots' accumulators summed in double, in slot order; alpha kinds come back from line
// coordinates ([c][col][row]) to the map's own order
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gfinish_kernel(const __grid_constant__ pde_adi_desc d, int nblk, int nslots,
                                                      const float2 *__restrict__ acc, const double *__restrict__ part_chan,
                                                      const double *__restrict__ part_skip, const float *skipw,
                                                      float *g_ab, float *g_atc, float *g_bb, float *g_btc, float *g_chan,
                                                      float *g_skip) {
    const int N = d.N, C = d.C, NN = N * N;
    const size_t CNN = (size_t)C * NN;
    const size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (id < 2 * CNN) {
        // id walks the accumulators in storage order (coalesced reads); the alpha stores are the transposed ones
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
    } else if (id < 2 * CNN + (size_t)C * C) {
        if (d.chan_op) {
            const int q = (int)(id - 2 * CNN);
            double s = 0.0;
            for (int b = 0; b < nblk; ++b) s += part_chan[(size_t)b * kChanSlots + q];
            g_chan[q] = (float)s;
        }
    } else if (id == 2 * CNN + (size_t)C * C) {
        if (d.skip) {
            double s = 0.0;
            for (int b = 0; b < nblk; ++b) s += part_skip[b];
            const float sg = sigmoid_of(skipw);
            g_skip[0] = (float)(s * (double)sg * (1.0 - (double)sg));
        }
    }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
struct Plan {
    int threads, grid, K;
    size_t smem;
    size_t acc_floats, hist_floats, ins_floats;   // totals over the grid's slots
    size_t bytes;
};

static size_t align256(size_t n) { return (n + 255u) & ~(size_t)255u; }

static const void *bwd_kernel_for(int C) {
    switch (C) {
        case 1: return reinterpret_cast<const void *>(gbwd_kernel<1>);
        case 2: return reinterpret_cast<const void *>(gbwd_kernel<2>);
        case 3: return reinterpret_cast<const void *>(gbwd_kernel<3>);
        default: return reinterpret_cast<const void *>(gbwd_kernel<4>);
    }
}

static int plan_backward(const pde_adi_desc &d, Plan *p) {
    DeviceProps props;
    int rc = query_props(&props);
    if (rc) return rc;
    p->K = slots_per_block(d);
    p->threads = block_threads(d, p->K);
    p->smem = p->K * tile_bytes(d);
    int per_sm = 1;
    rc = cached_occupancy(bwd_kernel_for(d.C), p->threads, p->smem, &per_sm);
    if (rc) return rc;
    const size_t CNN = (size_t)d.C * d.N * d.N;
    const int S = d.steps * sweeps_per_step(d);
    const size_t per_block = ((size_t)4 + S + (d.chan_op == 1 ? d.steps : 0)) * CNN * sizeof(float) * p->K;
    long long grid = (long long)props.sm_count * per_sm;
    const long long by_batch = ((long long)d.B + p->K - 1) / p->K;
    if (grid > by_batch) grid = by_batch;
    const long long cap = (long long)(kMaxWorkspaceBytes / per_block);
    if (grid > cap) grid = cap;
    if (grid < 1) grid = 1;
    p->grid = (int)grid;
    const size_t slots = (size_t)p->grid * p->K;
    p->acc_floats = slots * 4 * CNN;
    p->hist_floats = slots * S * CNN;
    p->ins_floats = d.chan_op == 1 ? slots * d.steps * CNN : 0;
    p->bytes = align256(p->acc_floats * sizeof(float)) + align256(p->hist_floats * sizeof(float)) +
               align256(p->ins_floats * sizeof(float)) + align256((size_t)p->grid * (kChanSlots + 1) * sizeof(double)) + 256;
    return PDE_OK;
}

size_t workspace_bytes(const pde_adi_desc &d) {
    Plan p;
    return plan_backward(d, &p) == PDE_OK ? p.bytes : 0;
}

int prepare(const pde_adi_desc &d, const pde_adi_schedule &sch, const float *ab, const float *bb, const float *atc,
            const float *btc, char *tables, cudaStream_t st) {
    const int lines = d.steps * sweeps_per_step(d) * d.C * d.N;
    if (lines == 0) return PDE_OK;
    gprepare_kernel<<<(lines + 127) / 128, 128, 0, st>>>(d, sch, ab, bb, atc, btc, tables);
    return cuda_last_error();
}

int forward(const pde_adi_desc &d, const char *tables, const float *u, const float *chan, const float *skipw, float *out,
            cudaStream_t st) {
    DeviceProps props;
    int rc = query_props(&props);
    if (rc) return rc;
    const int K = slots_per_block(d), threads = block_threads(d, K);
    const size_t smem = K * tile_bytes(d);
    int per_sm = 1;
    rc = cached_occupancy(reinterpret_cast<const void *>(gfwd_kernel), threads, smem, &per_sm);
    if (rc) return rc;
    GArgs a{};
    a.d = d;
    a.K = K;
    a.sps = sweeps_per_step(d);
    a.S = d.steps * a.sps;
    a.hdr = reinterpret_cast<const Header *>(tables);
    a.tab = reinterpret_cast<const float4 *>(tables + kHeaderBytes);
    a.u = u; a.chan = chan; a.skipw = skipw; a.out = out;
    long long grid = (long long)props.sm_count * per_sm;
    if (grid > ((long long)d.B + K - 1) / K) grid = ((long long)d.B + K - 1) / K;
    gfwd_kernel<<<(int)grid, threads, smem, st>>>(a);
    return cuda_last_error();
}

int backward(const pde_adi_desc &d, const char *tables, const float *u, const float *gout, const float *chan,
             const float *skipw, float *gin, float *g_ab, float *g_bb, float *g_atc, float *g_btc, float *g_chan,
             float *g_skip, void *workspace, size_t ws_bytes, cudaStream_t st) {
    Plan p;
    int rc = plan_backward(d, &p);
    if (rc) return rc;
    if (!workspace || ws_bytes < p.bytes) return PDE_ERR_WORKSPACE;
    char *w = reinterpret_cast<char *>((reinterpret_cast<uintptr_t>(workspace) + 255u) & ~(uintptr_t)255u);
    GArgs a{};
    a.d = d;
    a.sps = sweeps_per_step(d);
    a.S = d.steps * a.sps;
    a.need_gin = gin != nullptr;
    a.K = p.K;
    a.hdr = reinterpret_cast<const Header *>(tables);
    a.tab = reinterpret_cast<const float4 *>(tables + kHeaderBytes);
    a.u = u; a.gout = gout; a.chan = chan; a.skipw = skipw; a.gin = gin;
    a.acc = reinterpret_cast<float2 *>(w);
    w += align256(p.acc_floats * sizeof(float));
    a.hist = reinterpret_cast<float *>(w);
    w += align256(p.hist_floats * sizeof(float));
    a.ins = p.ins_floats ? reinterpret_cast<float *>(w) : nullptr;
    w += align256(p.ins_floats * sizeof(float));
    a.part_chan = reinterpret_cast<double *>(w);
    a.part_skip = a.part_chan + (size_t)p.grid * kChanSlots;
    void *kargs[] = {&a};
    PDE_CUDA_TRY(cudaLaunchKernel(bwd_kernel_for(d.C), dim3(p.grid), dim3(p.threads), kargs, p.smem, st));
    rc = cuda_last_error();
    if (rc) return rc;
    const size_t outs = 2 * (size_t)d.C * d.N * d.N + (size_t)d.C * d.C + 1;
    gfinish_kernel<<<(unsigned)((outs + 255) / 256), 256, 0, st>>>(d, p.grid, p.grid * p.K, a.acc, a.part_chan, a.part_skip, skipw, g_ab,
                                                                  g_atc, g_bb, g_btc, g_chan, g_skip);
    return cuda_last_error();
}

}  // namespace generic
}  // namespace adi
}  // namespace pde
