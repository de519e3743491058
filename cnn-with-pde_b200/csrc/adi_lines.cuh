// Line routines of the run-time-sized implicit kernels: adi_generic.cu (C <= 4, one thread per line) and
// adi_wide.cu (5 ... 64 channels, threads stride over the lines).  Both keep a sample's planes in a
// shared-memory tile with an odd row pitch and store tables, history and accumulators in LINE
// coordinates [c][i][line]; see the head of adi_generic.cu.
#pragma once
#include "adi_common.cuh"

namespace pde {
namespace adi {
namespace generic {

constexpr int kMaxN = 128;
constexpr size_t kMaxTileBytes = 200u * 1024u;             // one sample's planes in one block's shared memory
constexpr size_t kMaxWorkspaceBytes = (size_t)1 << 30;    // history slices: the grid shrinks to stay below it

// odd row pitch of a sample's tile: rows (x sweeps) and columns (y sweeps) are both free of bank conflicts
__host__ __device__ inline int pitch_of(int N) { return N | 1; }
inline size_t tile_bytes(const pde_adi_desc &d) { return (size_t)d.C * d.N * pitch_of(d.N) * sizeof(float); }

// A block works on K samples at a time ("slots": small planes would leave a block with one or two warps);
// slot q's threads are the `cn` threads [q cn, (q + 1) cn).  Everything a slot touches -- its tile, its
// history and accumulator slices -- is its own; only the barriers are block-wide.
struct Line {
    int slot, within, c, l;
    int cn;          // threads of a slot
    bool active;     // the thread belongs to a slot
};

__device__ __forceinline__ float sigmoid_of(const float *skipw) { return 1.0f / (1.0f + expf(-__ldg(skipw))); }

// sample planes -> tile (coalesced global side, [c][row][col] with row pitch P in shared memory)
__device__ __forceinline__ void planes_to_tile(const float *__restrict__ g, float *__restrict__ tile, const Line &t, int C,
                                               int N, int P) {
    const int NN = N * N;
    for (int q = t.within; q < C * NN; q += t.cn) {
        const int c = q / NN, rem = q - c * NN, row = rem / N, col = rem - row * N;
        tile[(c * N + row) * P + col] = __ldcs(g + q);
    }
}

// One line of one sweep's factor tables: coefficient maps -> clamp -> replicate smoothing -> r -> Thomas pivots,
// one float4 (r, 1 / pivot, r / pivot, clamp mask) per cell at tq[i * N].  Reference arithmetic, without
// contraction: get_alpha_beta_at_time mnist_test.py:33-42 / cifar10.py:53-63, smooth_coefficients
// mnist_test.py:135-149, rows mnist_test.py:83-93, pivots mnist_test.py:169,177-181.  axis 0 reads the alpha maps
// along row l, axis 1 the beta maps along column l.  This is gprepare_kernel's body (adi_generic.cu) op for op, used
// by adi_stream.cu; gprepare_kernel keeps its inline copy because calling this routine changes its machine code
// (register allocation), and the existing kernels' code is kept as it was.
__device__ __forceinline__ void prepare_line(const pde_adi_desc &d, int axis, int c, int l, float tt, float dts, float h2,
                                             const float *__restrict__ ab, const float *__restrict__ bb,
                                             const float *__restrict__ atc, const float *__restrict__ btc, float4 *tq) {
    const int N = d.N;
    const float *base = axis ? bb : ab, *tc = axis ? btc : atc;
    const float third = __fdiv_rn(1.0f, 3.0f);
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

constexpr int kChunk = 4;   // cells whose loads are issued together, ahead of the dependent recurrence

// L2 prefetch of a contiguous region by one thread (TMA bulk prefetch: no registers, no shared memory).  The
// instruction wants a 16-byte aligned address and size; slices of odd planes are neither, so the region is
// shrunk to the aligned pieces it contains, starting from the aligned address below it (still inside the
// workspace: the history region itself starts on a 256-byte boundary).
__device__ __forceinline__ void prefetch_slice_l2(const void *p, size_t bytes) {
    const uintptr_t a = reinterpret_cast<uintptr_t>(p), a0 = a & ~(uintptr_t)15;
    const char *b = reinterpret_cast<const char *>(a0);
    bytes = (size_t)(a + bytes - a0);
    constexpr size_t kPiece = 16384;
    for (size_t off = 0; off < bytes; off += kPiece) {
        const unsigned n = (unsigned)((bytes - off < kPiece ? bytes - off : kPiece) & ~(size_t)15);
        if (n) asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(b + off), "r"(n) : "memory");
    }
}

// One implicit sweep of the thread's line, in place: d*_i = (d_i + r_i d*_{i-1}) / pivot_i, then
// x_i = d*_i + (r_i / pivot_i) x_{i+1} (thomas_solver_batch, mnist_test.py:151-198).  hist != nullptr: the
// result also goes to hist[i * N] (line coordinates, this thread's column of the slice).
__device__ __forceinline__ void sweep_line(float *__restrict__ line, int step, int N, const float4 *__restrict__ tq,
                                           float *__restrict__ hist) {
    float ds = line[0] * __ldg(&tq[0].y);
    line[0] = ds;
    for (int i0 = 1; i0 < N; i0 += kChunk) {
        float4 q4[kChunk];
        float p4[kChunk];
#pragma unroll
        for (int k = 0; k < kChunk; ++k)
            if (i0 + k < N) {
                q4[k] = __ldg(tq + (i0 + k) * N);
                p4[k] = line[(i0 + k) * step];
            }
#pragma unroll
        for (int k = 0; k < kChunk; ++k)
            if (i0 + k < N) {
                ds = fmaf(q4[k].x, ds, p4[k]) * q4[k].y;
                line[(i0 + k) * step] = ds;
            }
    }
    float x = ds;
    if (hist) hist[(N - 1) * N] = x;
    for (int i0 = N - 2; i0 >= 0; i0 -= kChunk) {
        float e4[kChunk], p4[kChunk];
#pragma unroll
        for (int k = 0; k < kChunk; ++k)
            if (i0 - k >= 0) {
                e4[k] = __ldg(&tq[(i0 - k) * N].z);
                p4[k] = line[(i0 - k) * step];
            }
#pragma unroll
        for (int k = 0; k < kChunk; ++k)
            if (i0 - k >= 0) {
                x = fmaf(e4[k], x, p4[k]);
                line[(i0 - k) * step] = x;
                if (hist) hist[(i0 - k) * N] = x;
            }
    }
}

// Adjoint of one sweep on the thread's line, in place on g: w_i = g_i + e_{i-1} w_{i-1};
// lambda_i = (w_i + r_{i+1} lambda_{i+1}) / pivot_i (the transposed system through the same factors), and on
// the way down dL/dr_i = lambda_i (L x)_i with x the sweep's OUTPUT -> (smoothing^T: a window of three
// products) -> dt / h^2 -> clamp mask = the contribution gc_i of this sweep to the line's base accumulator
// (times the sweep's time: to its time-coefficient accumulator).
// `x` is the thread's column of the history slice and `acc` its column of the slot's accumulators: both were last
// written by this very thread, earlier in this kernel -- plain loads, never the read-only path (hence no
// `const __restrict__` on x).
__device__ __forceinline__ void reverse_line(float *__restrict__ g, int step, int N, const float4 *__restrict__ tq,
                                             const float *x, float2 *__restrict__ acc, bool smooth, float scale, float tt) {
    float w = g[0];
    for (int i0 = 1; i0 < N; i0 += kChunk) {
        float e4[kChunk], p4[kChunk];
#pragma unroll
        for (int k = 0; k < kChunk; ++k)
            if (i0 + k < N) {
                e4[k] = __ldg(&tq[(i0 + k - 1) * N].z);
                p4[k] = g[(i0 + k) * step];
            }
#pragma unroll
        for (int k = 0; k < kChunk; ++k)
            if (i0 + k < N) {
                w = fmaf(e4[k], w, p4[k]);
                g[(i0 + k) * step] = w;
            }
    }
    const float wgt = smooth ? scale * (1.0f / 3.0f) : scale;
    const float4 qn = __ldg(tq + (N - 1) * N);
    float r_up = qn.x, m_up = qn.w;       // r and mask of cell i + 1 while the loop is at i
    float lam = w * qn.y;
    g[(N - 1) * step] = lam;
    float xc = x[(N - 1) * N], xm = x[(N - 2) * N], xp;
    float gs1 = lam * (xm - xc);          // gs_{i+1} while the loop is at i
    float gs2 = gs1;                      // gs_{i+2}; at the far end the replicated term is the cell's own
    for (int i0 = N - 2; i0 >= 0; i0 -= kChunk) {
        float4 q4[kChunk];
        float p4[kChunk], x4[kChunk];
        float2 a4[kChunk];
#pragma unroll
        for (int k = 0; k < kChunk; ++k) {
            const int i = i0 - k;
            if (i >= 0) {
                q4[k] = __ldg(tq + i * N);
                p4[k] = g[i * step];
                x4[k] = i > 0 ? x[(i - 1) * N] : 0.0f;
                a4[k] = acc[(i + 1) * N];
            }
        }
#pragma unroll
        for (int k = 0; k < kChunk; ++k) {
            const int i = i0 - k;
            if (i >= 0) {
                lam = fmaf(r_up, lam, p4[k]) * q4[k].y;
                g[i * step] = lam;
                xp = xc; xc = xm; xm = x4[k];
                const float lx = i > 0 ? (xm - xc) + (xp - xc) : xp - xc;
                const float gs0 = lam * lx;
                const float gc = (smooth ? (gs2 + gs1) + gs0 : gs1) * wgt * m_up;   // cell i + 1
                acc[(i + 1) * N] = make_float2(a4[k].x + gc, fmaf(gc, tt, a4[k].y));
                gs2 = gs1; gs1 = gs0;
                r_up = q4[k].x; m_up = q4[k].w;
            }
        }
    }
    // cell 0: gs_{-1} is the cell's own (replicate padding)
    const float gc = (smooth ? (gs2 + gs1) + gs1 : gs1) * wgt * m_up;
    const float2 a0 = acc[0];
    acc[0] = make_float2(a0.x + gc, fmaf(gc, tt, a0.y));
}

// sum of v over the block, in warp order (red: one double per warp)
__device__ __forceinline__ double block_sum(double v, double *red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFullMask, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
    if (threadIdx.x == 0)
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[w];
    return s;   // valid on thread 0
}

}  // namespace generic
}  // namespace adi
}  // namespace pde
