// Implicit operator-split (ADI) diffusion layers, forward and adjoint, for sm_100a.
//
// Reference behaviour (what is computed): mnist_test.py:33-198, fashion_mnist.py:40-196,
// SVHN.py:38-230, cifar10.py:53-211, cifar_2version.py:52-187.  How it is computed here is
// unrelated to the reference's op stream:
//
//   * pde_adi_prepare   one small kernel turns the four coefficient maps into factorised
//                       Thomas tables (r, 1/pivot, r/pivot, clamp mask) per sweep, ONCE per
//                       call, shared by the whole batch (the reference refactorises every
//                       line of every sample).
//   * adi_fwd_kernel    one warp owns channel c of PB samples; a lane owns one line of the
//                       plane and keeps it in registers through the Thomas recurrences; the
//                       plane lives in a padded shared-memory tile that is only used to turn
//                       rows into columns between sweeps.  All num_steps run on-chip: one HBM
//                       read and one HBM write per cell.
//   * adi_bwd_kernel    recomputes the forward trajectory, checkpointing the state at the
//                       end of every step in an L2-resident scratch, then walks the sweeps
//                       backwards: transposed-tridiagonal solve for the adjoint, lambda*(Lx)
//                       accumulated per pixel into lane-private shared-memory maps, and the
//                       sweep input rebuilt as x_in = (A + eps I) x_out.  When the rebuild
//                       would amplify rounding noise (device-computed bound), the kernel
//                       switches to exact per-sweep checkpoints instead.
//   * adi_finish_kernel sums the per-warp gradient partials in double (deterministic).
#include "adi_common.cuh"

namespace pde {
namespace adi {

template <int N>
struct Geo {
    static_assert(N % 4 == 0 && N >= 8 && N <= 32, "plane edge must be a multiple of 4 in [8, 32]");
    // A tile interleaves two samples as float2.  Row stride ST (in float2) with ST / 2 odd: the
    // 128-bit row accesses of 8 consecutive lanes hit 8 distinct 16-byte bank groups, and the
    // 64-bit column accesses (lane == column) of a half warp are 128 contiguous bytes.
    static constexpr int ST = N + 2;
    static constexpr int WORDS = 2 * N * ST;   // floats per tile
    static constexpr int Q = N / 4;
};

// ------------------------------------------------------------------------------------------
// prepare: coefficient map -> clamp -> smoothing -> r -> pivots, ONE launch per call.  A block
// owns a sweep, a thread one (channel, line) of it; op-for-op the fp32 arithmetic of the reference
// (no FMA contraction).  The thread writes its line into the tables of both implementations:
//   whole-line (adi.cu):        [s][c][i/4][line][i%4], one-sided Thomas pivots (the reference's);
//   half-line  (adi_split.cu):  [s][c][k/4][mirrored line][half][k%4], twisted pivots: top-down
//                               for cells 0 .. H-1 (the same values), bottom-up for N-1 .. H+1,
//                               and cell H closes both; written only when the call can be served
//                               by those kernels.
// The block reduces the sweep's largest r and "some cell clamped" and writes its header entries;
// nothing crosses blocks (the consumers fold them into the call-wide flags: header_flags).
// ------------------------------------------------------------------------------------------
constexpr int kPrepareThreads = 256;

template <int N>
__device__ __forceinline__ void prepare_body(const pde_adi_desc &d, const pde_adi_schedule &sch, const SlotMap &sm,
                                             const float *__restrict__ ab, const float *__restrict__ bb,
                                             const float *__restrict__ atc, const float *__restrict__ btc, char *tables,
                                             int want_split, const int s) {
    // Three phases per sweep.  (1) every cell in parallel: raw coefficient -> clamp (-> mask) -> smoothing ->
    // r = (k dt) / h^2; (2) one thread per line and direction: the pivot recurrences, the only serial part
    // (top-down for the reference's one-sided elimination, bottom-up for the far half of the twisted one);
    // (3) every cell in parallel: 1 / pivot, r / pivot and the table stores.  Cells are addressed in LINE
    // order [c][line][i] (i along the sweep) in shared memory.
    constexpr int H = N / 2, HQ = (H + 3) / 4, NN = N * N;
    extern __shared__ __align__(16) float prep_smem[];
    __shared__ float s_rmax[kPrepareThreads / 32];
    const int sps = sweeps_per_step(d), C = d.C, cells = C * NN;
    float *kap = prep_smem, *rr = kap + cells, *den = rr + cells, *den2 = den + cells;   // den2: bottom-up pivots
    unsigned char *inside = reinterpret_cast<unsigned char *>(den2 + cells);
    const int tid = threadIdx.x;
    const int axis = sweep_axis(s % sps);
    const float *base = axis ? bb : ab, *tc = axis ? btc : atc;
    const float tt = sch.t[s], dts = sch.dts[s], h2 = sch.h2[s];
    const float third = __fdiv_rn(1.0f, 3.0f);
    Header *hdr = reinterpret_cast<Header *>(tables);
    float *f = reinterpret_cast<float *>(tables + kHeaderBytes);
    const size_t T = table_elems(d);

    // ---- (1a) clamped coefficient, in line order.  The map is read in its own (row-major) order: coalesced.
    int any_clamped = 0;
    for (int q = tid; q < cells; q += kPrepareThreads) {
        const int c = q / NN, row = (q % NN) / N, col = q % N;
        const float raw = __fadd_rn(__ldg(base + q), __fmul_rn(__ldg(tc + q), tt));
        bool m = raw >= d.cmin;
        float k = raw < d.cmin ? d.cmin : raw;
        if (d.has_max) {
            m = m && raw <= d.cmax;
            k = k > d.cmax ? d.cmax : k;
        }
        // x sweeps: line = row, i = col; y sweeps: line = col, i = row
        const int lo = axis == 0 ? (c * N + row) * N + col : (c * N + col) * N + row;
        kap[lo] = k;
        inside[lo] = m ? 1 : 0;
        any_clamped |= m ? 0 : 1;
    }
    __syncthreads();
    // ---- (1b) r_i from the (smoothed) coefficient: (k dt) / h^2, op for op mnist_test.py:83,135-149
    float rmax = 0.0f;
    for (int q = tid; q < cells; q += kPrepareThreads) {
        const int i = q % N;
        float ks = kap[q];
        if (d.smooth)
            ks = __fadd_rn(__fadd_rn(__fmul_rn(kap[i > 0 ? q - 1 : q], third), __fmul_rn(kap[q], third)),
                           __fmul_rn(kap[i < N - 1 ? q + 1 : q], third));
        const float r = __fdiv_rn(__fmul_rn(ks, dts), h2);
        rr[q] = r;
        rmax = fmaxf(rmax, fabsf(r));
    }
    __syncthreads();
    // ---- (2) pivots.  Thread (line, 0): top-down over the whole line (mnist_test.py:165-185, c*_i = -r_i / den_i);
    // thread (line, 1): bottom-up over cells N-1 .. H+1 (twisted factorisation, adi_split.cu).
    auto diag = [&](int i, float r) {
        return (i == 0 || i == N - 1) ? __fadd_rn(1.0f, r) : __fadd_rn(1.0f, __fmul_rn(2.0f, r));
    };
    for (int job = tid; job < 2 * C * N; job += kPrepareThreads) {
        const int dir = job / (C * N), lo = (job % (C * N)) * N;
        if (dir == 0) {
            float cst = 0.0f;
#pragma unroll 4
            for (int i = 0; i < N; ++i) {
                const float r = rr[lo + i];
                const float dn = i == 0 ? __fadd_rn(diag(i, r), d.eps) : __fadd_rn(__fsub_rn(diag(i, r), __fmul_rn(-r, cst)), d.eps);
                cst = __fdiv_rn(-r, dn);
                den[lo + i] = dn;
            }
        } else if (want_split) {
            float ast = 0.0f;
#pragma unroll 4
            for (int i = N - 1; i > H; --i) {
                const float r = rr[lo + i];
                const float dn = i == N - 1 ? __fadd_rn(diag(i, r), d.eps) : __fadd_rn(__fsub_rn(diag(i, r), __fmul_rn(-r, ast)), d.eps);
                ast = __fdiv_rn(-r, dn);
                den2[lo + i] = dn;
            }
            den2[lo + H] = ast;   // c* of cell H + 1 seen from below, for the closing cell
        }
    }
    __syncthreads();
    // ---- (3) tables.  Whole-line layout [s][c][i/4][line][i%4]: one float4 per (line, i/4).
    {
        float *tr = f, *tinv = f + T, *te = f + 2 * T, *tm = f + 3 * T;
        for (int q4 = tid; q4 < cells / 4; q4 += kPrepareThreads) {
            const int c = q4 / (NN / 4), line = (q4 % (NN / 4)) % N, iq = (q4 % (NN / 4)) / N;   // consecutive threads: consecutive lines
            const int lo = (c * N + line) * N + 4 * iq;
            float4 vr, vi, ve, vm;
            float *pr = &vr.x, *pi = &vi.x, *pe = &ve.x, *pm = &vm.x;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float r = rr[lo + k], dn = den[lo + k];
                pr[k] = r;
                pi[k] = __fdiv_rn(1.0f, dn);
                pe[k] = __fdiv_rn(r, dn);
                pm[k] = inside[lo + k] ? 1.0f : 0.0f;
            }
            const size_t o = (((size_t)s * C + c) * (N / 4) + iq) * N * 4 + (size_t)line * 4;
            *reinterpret_cast<float4 *>(tr + o) = vr;
            *reinterpret_cast<float4 *>(tinv + o) = vi;
            *reinterpret_cast<float4 *>(te + o) = ve;
            *reinterpret_cast<float4 *>(tm + o) = vm;
        }
    }
    if (want_split) {
        // half-line layout [s][c][k/4][mirrored line][half][k%4] (k = cell counted from the half's plane edge):
        // near half = the top-down pivots of cells 0 .. H-1, far half = the bottom-up ones of N-1 .. H+1 and the
        // closing cell H: den_H = diag - (-r_H) c*_{H-1} - (-r_H) a*_{H+1} + eps
        const size_t TS = split::stab_floats_per_table(d);
        float *sr = f + 4 * T, *sinv = sr + TS, *se = sr + 2 * TS, *smk = sr + 3 * TS;
        for (int q4 = tid; q4 < C * N * 2 * HQ; q4 += kPrepareThreads) {
            const int h = q4 % 2, R = (q4 / 2) % N, kq = (q4 / (2 * N)) % HQ, c = q4 / (2 * N * HQ);
            const int line = split::mirror(R, N);   // mirror is an involution: table row R holds line mirror(R)
            const int lo = (c * N + line) * N;
            float4 vr, vi, ve, vm;
            float *pr = &vr.x, *pi = &vi.x, *pe = &ve.x, *pm = &vm.x;
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                const int k = 4 * kq + kk;
                if (k < H) {
                    const int i = h ? N - 1 - k : k;
                    const float r = rr[lo + i];
                    float dn;
                    if (!h) dn = den[lo + i];
                    else if (i > H) dn = den2[lo + i];
                    else {
                        const float cst_h = __fdiv_rn(-rr[lo + H - 1], den[lo + H - 1]);
                        dn = __fadd_rn(__fsub_rn(__fsub_rn(diag(H, r), __fmul_rn(-r, cst_h)), __fmul_rn(-r, den2[lo + H])), d.eps);
                    }
                    pr[kk] = r;
                    pi[kk] = __fdiv_rn(1.0f, dn);
                    pe[kk] = __fdiv_rn(r, dn);
                    pm[kk] = inside[lo + i] ? 1.0f : 0.0f;
                } else {
                    pr[kk] = 0.0f; pi[kk] = 0.0f; pe[kk] = 0.0f; pm[kk] = 0.0f;
                }
            }
            const size_t o = ((((size_t)s * C + c) * HQ + kq) * N + R) * 8 + h * 4;
            *reinterpret_cast<float4 *>(sr + o) = vr;
            *reinterpret_cast<float4 *>(sinv + o) = vi;
            *reinterpret_cast<float4 *>(se + o) = ve;
            *reinterpret_cast<float4 *>(smk + o) = vm;
        }
    }
    // the sweep's header entries
    const int any = __syncthreads_or(any_clamped);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) rmax = fmaxf(rmax, __shfl_xor_sync(kFullMask, rmax, o));
    if ((tid & 31) == 0) s_rmax[tid >> 5] = rmax;
    __syncthreads();
    if (tid == 0) {
        float m = 0.0f;
        for (int w = 0; w < kPrepareThreads / 32; ++w) m = fmaxf(m, s_rmax[w]);
        hdr->rmax_bits[s] = __float_as_uint(m);
        hdr->clamped[s] = any ? 1 : 0;
        hdr->scale[s] = __fdiv_rn(dts, h2);
        hdr->t[s] = tt;
        hdr->slot[s] = sm.slot[s];
        if (s == 0) hdr->nslots = sm.nslots;
    }
    if (s == 0)
        for (int u = tid; u < sm.nslots; u += kPrepareThreads) hdr->rep[u] = sm.rep[u];
}

template <int N>
__global__ void __launch_bounds__(kPrepareThreads) prepare_kernel(const __grid_constant__ pde_adi_desc d,
                                                      const __grid_constant__ pde_adi_schedule sch,
                                                      const __grid_constant__ SlotMap sm, const float *__restrict__ ab,
                                                      const float *__restrict__ bb, const float *__restrict__ atc,
                                                      const float *__restrict__ btc, char *tables, int want_split) {
    prepare_body<N>(d, sch, sm, ab, bb, atc, btc, tables, want_split, blockIdx.x);
}

// the tables of several layers in one launch (the kernel parameters hold every layer's schedule: ~3 KB each)
struct PrepareJob {
    pde_adi_desc d;
    pde_adi_schedule sch;
    SlotMap sm;
    const float *ab, *bb, *atc, *btc;
    char *tables;
    int s_begin;   // first block of this layer
};
struct PrepareMulti {
    int n, want_split;
    PrepareJob job[PDE_MAX_BRANCHES];
};
template <int N>
__global__ void __launch_bounds__(kPrepareThreads) prepare_multi_kernel(const __grid_constant__ PrepareMulti m) {
    int j = m.n - 1;
    while (j > 0 && (int)blockIdx.x < m.job[j].s_begin) --j;
    const PrepareJob &job = m.job[j];
    prepare_body<N>(job.d, job.sch, job.sm, job.ab, job.bb, job.atc, job.btc, job.tables, m.want_split,
                    (int)blockIdx.x - job.s_begin);
}

// ------------------------------------------------------------------------------------------
// tile helpers.  A tile holds the same plane of TWO samples, interleaved cell by cell as float2
// (lo = sample 2k, hi = sample 2k+1), N rows of ST float2.
// ------------------------------------------------------------------------------------------
template <int N>
__device__ __forceinline__ void planes_to_tile(const float *__restrict__ ga, const float *__restrict__ gb,
                                               float *tile, int lane, bool va, bool vb) {
    constexpr int ST = Geo<N>::ST;
    const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int q0 = 0; q0 < N * N / 4; q0 += 32) {
        const int q = q0 + lane;
        if (q < N * N / 4) {
            const float4 a = va ? ld_stream(reinterpret_cast<const float4 *>(ga) + q) : zero;
            const float4 b = vb ? ld_stream(reinterpret_cast<const float4 *>(gb) + q) : zero;
            const int idx = 4 * q, r = idx / N, cc = idx % N;
            float4 *dst = reinterpret_cast<float4 *>(&tile[(r * ST + cc) * 2]);
            dst[0] = make_float4(a.x, b.x, a.y, b.y);
            dst[1] = make_float4(a.z, b.z, a.w, b.w);
        }
    }
}

// out = tile                      (ua == nullptr)
// out = sig * u0 + om * tile      (skip epilogue, or gin = g + sig * gout with om == 1)
template <int N>
__device__ __forceinline__ void tile_to_planes(const float *tile, float *__restrict__ ga, float *__restrict__ gb,
                                               int lane, bool va, bool vb, const float *__restrict__ ua,
                                               const float *__restrict__ ub, float sig, float om) {
    constexpr int ST = Geo<N>::ST;
#pragma unroll
    for (int q0 = 0; q0 < N * N / 4; q0 += 32) {
        const int q = q0 + lane;
        if (q < N * N / 4) {
            const int idx = 4 * q, r = idx / N, cc = idx % N;
            const float4 *src = reinterpret_cast<const float4 *>(&tile[(r * ST + cc) * 2]);
            const float4 v0 = src[0], v1 = src[1];
            float4 a = make_float4(v0.x, v0.z, v1.x, v1.z), b = make_float4(v0.y, v0.w, v1.y, v1.w);
            if (va) {
                if (ua) {
                    const float4 w = ld_stream(reinterpret_cast<const float4 *>(ua) + q);
                    a.x = fmaf(om, a.x, sig * w.x); a.y = fmaf(om, a.y, sig * w.y);
                    a.z = fmaf(om, a.z, sig * w.z); a.w = fmaf(om, a.w, sig * w.w);
                }
                st_stream(reinterpret_cast<float4 *>(ga) + q, a);
            }
            if (vb) {
                if (ub) {
                    const float4 w = ld_stream(reinterpret_cast<const float4 *>(ub) + q);
                    b.x = fmaf(om, b.x, sig * w.x); b.y = fmaf(om, b.y, sig * w.y);
                    b.z = fmaf(om, b.z, sig * w.z); b.w = fmaf(om, b.w, sig * w.w);
                }
                st_stream(reinterpret_cast<float4 *>(gb) + q, b);
            }
        }
    }
}

// The line owned by lane t: AX == 0 -> row t (128-bit accesses, two cells of both samples each),
// AX == 1 -> column t (64-bit accesses).
template <int N, int AX>
__device__ __forceinline__ void ld_line(const float *tile, int t, f2 (&x)[N]) {
    constexpr int ST = Geo<N>::ST;
    if (AX == 0) {
#pragma unroll
        for (int j = 0; j < N / 2; ++j) {
            const ulonglong2 v = *reinterpret_cast<const ulonglong2 *>(&tile[(t * ST + 2 * j) * 2]);
            x[2 * j].v = v.x;
            x[2 * j + 1].v = v.y;
        }
    } else {
#pragma unroll
        for (int i = 0; i < N; ++i) x[i].v = *reinterpret_cast<const unsigned long long *>(&tile[(i * ST + t) * 2]);
    }
}
template <int N, int AX>
__device__ __forceinline__ void st_line(float *tile, int t, const f2 (&x)[N]) {
    constexpr int ST = Geo<N>::ST;
    if (AX == 0) {
#pragma unroll
        for (int j = 0; j < N / 2; ++j) {
            ulonglong2 v;
            v.x = x[2 * j].v;
            v.y = x[2 * j + 1].v;
            *reinterpret_cast<ulonglong2 *>(&tile[(t * ST + 2 * j) * 2]) = v;
        }
    } else {
#pragma unroll
        for (int i = 0; i < N; ++i) *reinterpret_cast<unsigned long long *>(&tile[(i * ST + t) * 2]) = x[i].v;
    }
}

// x[p][i] = sum_d mat[d * mstride] * tile_d[p][row t][i]   over the C channel tiles of a group.
// mstride == 1 walks a row of the matrix (forward mix), mstride == C a column (adjoint).
template <int N, int NP>
__device__ __forceinline__ void mix_rows(const float *group_tiles, int C, const float *__restrict__ mat, int mstride,
                                         int t, f2 (&x)[NP][N]) {
    constexpr int WORDS = Geo<N>::WORDS;
    const f2 zero = f2_bc(0.0f);
#pragma unroll
    for (int p = 0; p < NP; ++p)
#pragma unroll
        for (int i = 0; i < N; ++i) x[p][i] = zero;
    for (int dd = 0; dd < C; ++dd) {
        const float m = __ldg(mat + dd * mstride);
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            f2 row[N];
            ld_line<N, 0>(group_tiles + ((size_t)dd * NP + p) * WORDS, t, row);
#pragma unroll
            for (int i = 0; i < N; ++i) x[p][i] = f2_fmas(m, row[i], x[p][i]);
        }
    }
}

template <int N>
__device__ __forceinline__ void prefetch_tables(const float4 *ta, const float4 *tb, const float4 *tc) {
#pragma unroll
    for (int q = 0; q < N / 4; ++q) {
        prefetch_l1(ta + q * N);
        prefetch_l1(tb + q * N);
        if (tc) prefetch_l1(tc + q * N);
    }
}

template <int N>
__device__ __forceinline__ void prefetch_plane_l2(const float *g, int lane) {
#pragma unroll
    for (int off = lane * 32; off < N * N; off += 32 * 32) prefetch_l2(g + off);
}

// ------------------------------------------------------------------------------------------
// Thomas solve of (A + eps I) x = d for the NP sample pairs a lane holds (same coefficients for
// all of them: the factorisation is batch independent).  With inv = 1/pivot and e = r/pivot = -c*:
//   d*_i = inv_i d_i + e_i d*_{i-1}         x_i = d*_i + e_i x_{i+1}
// ------------------------------------------------------------------------------------------
template <int N, int NP>
__device__ __forceinline__ void thomas_solve(f2 (&x)[NP][N], const float4 *__restrict__ tinv,
                                             const float4 *__restrict__ te) {
    float e[N];
    float4 iv_n = __ldg(tinv), ev_n = __ldg(te);
#pragma unroll
    for (int q = 0; q < N / 4; ++q) {
        const float4 iv = iv_n, ev = ev_n;
        if (q + 1 < N / 4) {   // the next chunk's coefficients are in flight while this one computes
            iv_n = __ldg(tinv + (q + 1) * N);
            ev_n = __ldg(te + (q + 1) * N);
        }
        const float ivs[4] = {iv.x, iv.y, iv.z, iv.w}, evs[4] = {ev.x, ev.y, ev.z, ev.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int i = 4 * q + k;
            e[i] = evs[k];
#pragma unroll
            for (int p = 0; p < NP; ++p)
                x[p][i] = (i == 0) ? f2_muls(ivs[k], x[p][0]) : f2_fmas(evs[k], x[p][i - 1], f2_muls(ivs[k], x[p][i]));
        }
    }
#pragma unroll
    for (int i = N - 2; i >= 0; --i)
#pragma unroll
        for (int p = 0; p < NP; ++p) x[p][i] = f2_fmas(e[i], x[p][i + 1], x[p][i]);
}

__device__ __forceinline__ void group_sync(int C, int group) {
    if (C == 1)
        __syncwarp();
    else
        named_barrier(1 + group, C * 32);
}

// ------------------------------------------------------------------------------------------
// forward: one warp owns channel c of 2 * NP samples
// ------------------------------------------------------------------------------------------
template <int N, int NP>
__global__ void fwd_kernel(const Args a) {
    constexpr int WORDS = Geo<N>::WORDS;
    extern __shared__ __align__(16) float smem[];
    const pde_adi_desc &d = a.d;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int C = d.C, group = warp / C, c = warp % C;
    const bool active = lane < N;
    const int t = active ? lane : N - 1;
    float *gtiles = smem + (size_t)group * C * NP * WORDS;  // [C][NP][WORDS]
    float *my = gtiles + (size_t)c * NP * WORDS;
    const Tables T = split_tables(a.tables, d);
    const size_t plane = (size_t)N * N;
    float sig = 0.0f;
    if (d.skip) sig = 1.0f / (1.0f + expf(-__ldg(a.skipw)));
    const float om = 1.0f - sig;

    for (int item = blockIdx.x * a.G + group; item < a.nitems; item += gridDim.x * a.G) {
        const int b0 = item * 2 * NP;
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            const int ba = b0 + 2 * p, bb = ba + 1;
            const bool va = ba < d.B, vb = bb < d.B;
            planes_to_tile<N>(a.u + ((size_t)(va ? ba : 0) * C + c) * plane, a.u + ((size_t)(vb ? bb : 0) * C + c) * plane,
                              my + p * WORDS, lane, va, vb);
        }
        __syncwarp();
        f2 x[NP][N];
        bool in_regs = false;  // x holds the state as rows
        for (int step = 0; step < d.steps; ++step) {
            const int s0 = step * a.sps;
            if (d.chan_op == 1) {
                if (in_regs && active) {
#pragma unroll
                    for (int p = 0; p < NP; ++p) st_line<N, 0>(my + p * WORDS, t, x[p]);
                }
                group_sync(C, group);
                mix_rows<N, NP>(gtiles, C, a.chan + c * C, 1, t, x);
                group_sync(C, group);
            } else if (!in_regs) {
#pragma unroll
                for (int p = 0; p < NP; ++p) ld_line<N, 0>(my + p * WORDS, t, x[p]);
            }
            {   // x sweep
                const size_t o = ((size_t)s0 * C + c) * (N / 4) * N + t;
                thomas_solve<N, NP>(x, reinterpret_cast<const float4 *>(T.inv) + o,
                                    reinterpret_cast<const float4 *>(T.e) + o);
            }
            if (active) {
#pragma unroll
                for (int p = 0; p < NP; ++p) st_line<N, 0>(my + p * WORDS, t, x[p]);
            }
            __syncwarp();
#pragma unroll
            for (int p = 0; p < NP; ++p) ld_line<N, 1>(my + p * WORDS, t, x[p]);
            {   // y sweep
                const size_t o = ((size_t)(s0 + 1) * C + c) * (N / 4) * N + t;
                thomas_solve<N, NP>(x, reinterpret_cast<const float4 *>(T.inv) + o,
                                    reinterpret_cast<const float4 *>(T.e) + o);
            }
            if (active) {
#pragma unroll
                for (int p = 0; p < NP; ++p) st_line<N, 1>(my + p * WORDS, t, x[p]);
            }
            __syncwarp();
            in_regs = false;
            if (a.sps == 3) {
#pragma unroll
                for (int p = 0; p < NP; ++p) ld_line<N, 0>(my + p * WORDS, t, x[p]);
                const size_t o = ((size_t)(s0 + 2) * C + c) * (N / 4) * N + t;
                thomas_solve<N, NP>(x, reinterpret_cast<const float4 *>(T.inv) + o,
                                    reinterpret_cast<const float4 *>(T.e) + o);
                in_regs = true;
            }
            if (d.chan_op == 2) {
                if (in_regs && active) {
#pragma unroll
                    for (int p = 0; p < NP; ++p) st_line<N, 0>(my + p * WORDS, t, x[p]);
                }
                group_sync(C, group);
                mix_rows<N, NP>(gtiles, C, a.chan + c * C, 1, t, x);
                group_sync(C, group);
                in_regs = true;
            }
        }
        if (in_regs && active) {
#pragma unroll
            for (int p = 0; p < NP; ++p) st_line<N, 0>(my + p * WORDS, t, x[p]);
        }
        __syncwarp();
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            const int ba = b0 + 2 * p, bb = ba + 1;
            const bool va = ba < d.B, vb = bb < d.B;
            const size_t oa = ((size_t)(va ? ba : 0) * C + c) * plane, ob = ((size_t)(vb ? bb : 0) * C + c) * plane;
            tile_to_planes<N>(my + p * WORDS, a.out + oa, a.out + ob, lane, va, vb, d.skip ? a.u + oa : nullptr,
                              d.skip ? a.u + ob : nullptr, sig, om);
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------
// backward: one warp owns channel c of one sample pair
// ------------------------------------------------------------------------------------------

// checkpoint a lane's line: scratch pair [i * 32 + lane] (coalesced 256 B per element index);
// a slot is read back in the orientation it was written in
template <int N>
__device__ __forceinline__ void ck_store(float *slot, int lane, const f2 (&x)[N]) {
    unsigned long long *s = reinterpret_cast<unsigned long long *>(slot);
#pragma unroll
    for (int i = 0; i < N; ++i) __stcg(&s[i * 32 + lane], x[i].v);   // L2 only: keep L1 for the tables
}
template <int N>
__device__ __forceinline__ void ck_load(const float *slot, int lane, f2 (&x)[N]) {
    const unsigned long long *s = reinterpret_cast<const unsigned long long *>(slot);
#pragma unroll
    for (int i = 0; i < N; ++i) x[i].v = __ldcg(&s[i * 32 + lane]);
}

// Per-pixel gradient accumulators live in TMEM: 128 columns per warp = {A0, A1, B0, B1} x 32,
// lane = line.  acc0 += z, acc1 += t * z for the kind (alpha / beta) of the sweep.
template <int N>
__device__ __forceinline__ void tmem_accumulate(uint32_t tacc, const float (&z)[N], float tt) {
    float a[32];
    tmem_wait_st();
    tmem_ld16(tacc, a);
    tmem_ld16(tacc + 16, a + 16);
    tmem_wait_ld();
#pragma unroll
    for (int i = 0; i < N; ++i) a[i] += z[i];
    tmem_st16(tacc, a);
    tmem_st16(tacc + 16, a + 16);
    tmem_ld16(tacc + 32, a);
    tmem_ld16(tacc + 48, a + 16);
    tmem_wait_ld();
#pragma unroll
    for (int i = 0; i < N; ++i) a[i] = fmaf(tt, z[i], a[i]);
    tmem_st16(tacc + 32, a);
    tmem_st16(tacc + 48, a + 16);
}

// Four consecutive cells (4q .. 4q+3) of the line owned by lane t, straight from / to the tile.
template <int N, int AX>
__device__ __forceinline__ void ld_quad(const float *tile, int t, int q, f2 (&c)[4]) {
    constexpr int ST = Geo<N>::ST;
    if (AX == 0) {
        const ulonglong2 v0 = *reinterpret_cast<const ulonglong2 *>(&tile[(t * ST + 4 * q) * 2]);
        const ulonglong2 v1 = *reinterpret_cast<const ulonglong2 *>(&tile[(t * ST + 4 * q + 2) * 2]);
        c[0].v = v0.x; c[1].v = v0.y; c[2].v = v1.x; c[3].v = v1.y;
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k)
            c[k].v = *reinterpret_cast<const unsigned long long *>(&tile[((4 * q + k) * ST + t) * 2]);
    }
}
template <int N, int AX>
__device__ __forceinline__ void st_quad(float *tile, int t, int q, const f2 (&c)[4]) {
    constexpr int ST = Geo<N>::ST;
    if (AX == 0) {
        ulonglong2 v0, v1;
        v0.x = c[0].v; v0.y = c[1].v; v1.x = c[2].v; v1.y = c[3].v;
        *reinterpret_cast<ulonglong2 *>(&tile[(t * ST + 4 * q) * 2]) = v0;
        *reinterpret_cast<ulonglong2 *>(&tile[(t * ST + 4 * q + 2) * 2]) = v1;
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k)
            *reinterpret_cast<unsigned long long *>(&tile[((4 * q + k) * ST + t) * 2]) = c[k].v;
    }
}

// One reversed sweep.  AX: orientation of the sweep (0: lane = row, 1: lane = column).
//   g: adjoint of the sweep output, in registers in orientation AX; solved in place through the
//      factorisation A = L U:
//        U^T w = g:        w_i = g_i + e_{i-1} w_{i-1}
//        L^T lambda = w:   lambda_i = inv_i (w_i + r_{i+1} lambda_{i+1})
//   xt: tile holding the sweep OUTPUT (the state is never parked in registers during the reverse
//      pass: a lane streams its line through a window of two quads).  Inside the back-substitution
//      loop, while lambda_i is fresh: (L x)_i, v_i = lambda_i (L x)_i summed over the two samples,
//      and (if `rebuild`) the sweep INPUT x_in,i = (1 + eps) x_i - r_i (L x)_i written back in place,
//      so that the tile holds the output of the previous sweep when this one returns.
//   v -> smoothing^T -> clamp mask -> TMEM accumulators of this sweep's kind.
template <int N, int AX>
__device__ __forceinline__ void reverse_sweep(f2 (&g)[N], float *xt, int t, bool active, uint32_t tacc,
                                              const float4 *tr, const float4 *tinv, const float4 *te,
                                              const float4 *tm, float scale, float tt, float onepe, bool smooth,
                                              bool rebuild, bool clamped) {
    constexpr int Q = N / 4;
    float eprev = 0.0f;
    float4 ev_n = __ldg(te);
    // the back-substitution's first coefficients and state quads are requested before the
    // forward pass starts
    float4 iv_n = __ldg(tinv + (Q - 1) * N), rv_n = __ldg(tr + (Q - 1) * N);
    f2 xc[4], xn[4];
    ld_quad<N, AX>(xt, t, Q - 1, xc);
    ld_quad<N, AX>(xt, t, Q - 2, xn);
#pragma unroll
    for (int q = 0; q < Q; ++q) {
        const float4 ev = ev_n;
        if (q + 1 < Q) ev_n = __ldg(te + (q + 1) * N);
        const float evs[4] = {ev.x, ev.y, ev.z, ev.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int i = 4 * q + k;
            if (i > 0) g[i] = f2_fmas(eprev, g[i - 1], g[i]);
            eprev = evs[k];
        }
    }
    float v[N];
    f2 xnext = f2_bc(0.0f);   // value of x_{i+1} before it was rebuilt
    float rnext = 0.0f;
#pragma unroll
    for (int q = Q - 1; q >= 0; --q) {
        const float4 iv = iv_n, rv = rv_n;
        if (q > 0) {
            iv_n = __ldg(tinv + (q - 1) * N);
            rv_n = __ldg(tr + (q - 1) * N);
        }
        const float ivs[4] = {iv.x, iv.y, iv.z, iv.w}, rvs[4] = {rv.x, rv.y, rv.z, rv.w};
        f2 xo[4];
#pragma unroll
        for (int k = 3; k >= 0; --k) {
            const int i = 4 * q + k;
            const f2 gi = f2_muls(ivs[k], g[i]);
            const f2 lam = (i == N - 1) ? gi : f2_fmas(rnext * ivs[k], g[i + 1], gi);
            g[i] = lam;
            const f2 cur = xc[k];
            f2 lx;
            if (i == N - 1)
                lx = f2_sub(xc[k - 1], cur);
            else if (i == 0)
                lx = f2_sub(xnext, cur);
            else
                lx = f2_fmas(-2.0f, cur, f2_add(k > 0 ? xc[k - 1] : xn[3], xnext));
            v[i] = f2_hsum(f2_mul(lam, lx));
            xo[k] = f2_fmas(-rvs[k], lx, f2_muls(onepe, cur));
            xnext = cur;
            rnext = rvs[k];
        }
        if (rebuild && active) st_quad<N, AX>(xt, t, q, xo);
#pragma unroll
        for (int k = 0; k < 4; ++k) xc[k] = xn[k];
        if (q >= 2) ld_quad<N, AX>(xt, t, q - 2, xn);
    }
    // smoothing^T along the line (replicate padding puts the end taps back on the end cells)
    if (smooth) {
        const float k3 = scale * (1.0f / 3.0f);
        float lo = v[0];
#pragma unroll
        for (int i = 0; i < N; ++i) {
            const float cur = v[i];
            const float hi = (i == N - 1) ? cur : v[i + 1];
            v[i] = ((lo + cur) + hi) * k3;
            lo = cur;
        }
    } else {
#pragma unroll
        for (int i = 0; i < N; ++i) v[i] *= scale;
    }
    if (clamped) {
#pragma unroll
        for (int q = 0; q < Q; ++q) {
            const float4 m = __ldg(tm + q * N);
            v[4 * q] *= m.x; v[4 * q + 1] *= m.y; v[4 * q + 2] *= m.z; v[4 * q + 3] *= m.w;
        }
    }
    tmem_accumulate<N>(tacc, v, tt);
}

// Adjoint of a channel op on the group's g tiles (rows), using the op's INPUT state in the x
// tiles:  gm[dd] += sum g_c * x_dd ;  g_c <- sum_c' mat[c'][c] g_c'.
template <int N>
__device__ __forceinline__ void chan_adjoint(float *ggt, float *gxt, int C, int c, int group,
                                             const float *__restrict__ mat, int t, bool active,
                                             float (&gm)[PDE_MAX_CHANNELS]) {
    constexpr int WORDS = Geo<N>::WORDS;
    group_sync(C, group);
    if (active) {
        f2 g[N];
        ld_line<N, 0>(ggt + (size_t)c * WORDS, t, g);
        for (int dd = 0; dd < C; ++dd) {
            f2 x[N];
            ld_line<N, 0>(gxt + (size_t)dd * WORDS, t, x);
            f2 acc = f2_bc(0.0f);
#pragma unroll
            for (int i = 0; i < N; ++i) acc = f2_fma(g[i], x[i], acc);
            gm[dd] += f2_hsum(acc);
        }
    }
    f2 gn[1][N];
    mix_rows<N, 1>(ggt, C, mat + c, C, t, gn);
    group_sync(C, group);
    if (active) st_line<N, 0>(ggt + (size_t)c * WORDS, t, gn[0]);
    __syncwarp();
}

template <int N, bool CHAN>
__global__ void __launch_bounds__(192, 1) bwd_kernel(const Args a) {
    constexpr int WORDS = Geo<N>::WORDS;
    constexpr int SLOT = 2 * N * 32;   // floats per checkpoint slot
    extern __shared__ __align__(16) float smem[];
    __shared__ uint32_t tmem_slot;
    const pde_adi_desc &d = a.d;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nwarps = blockDim.x >> 5;
    const int C = d.C, group = warp / C, c = warp % C;
    const bool active = lane < N;
    const int t = active ? lane : N - 1;
    // Two tiles per warp: the state (streamed in place by the reverse sweeps) and the adjoint
    // (transposed through its tile between sweeps of different orientation).
    float *gxt = smem + (size_t)group * C * WORDS;
    float *ggt = smem + (size_t)nwarps * WORDS + (size_t)group * C * WORDS;
    float *xt = gxt + (size_t)c * WORDS, *gt = ggt + (size_t)c * WORDS;

    // TMEM: 128 columns per warp, lane quadrant = warp % 4
    if (warp == 0) tmem_alloc(&tmem_slot, (uint32_t)a.tmem_cols);
    tmem_fence_before_sync();
    __syncthreads();
    tmem_fence_after_sync();
    const uint32_t tbase = tmem_slot + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)((warp >> 2) * 128);
    {
        float z[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) z[i] = 0.0f;
#pragma unroll
        for (int col = 0; col < 128; col += 16) tmem_st16(tbase + col, z);
        tmem_wait_st();
    }

    const Tables T = split_tables(a.tables, d);
    bool exact, any_clamped_unused;
    header_flags(T.hdr, d.steps, a.sps, &exact, &any_clamped_unused);
    // per-sweep scalars (dt/h^2, t, "some cell clamped") are read by every warp every sweep
    __shared__ float h_scale[PDE_MAX_SWEEPS], h_t[PDE_MAX_SWEEPS];
    __shared__ int h_clamped[PDE_MAX_SWEEPS];
    for (int i = threadIdx.x; i < a.S; i += blockDim.x) {
        h_scale[i] = T.hdr->scale[i];
        h_t[i] = T.hdr->t[i];
        h_clamped[i] = T.hdr->clamped[i];
    }
    constexpr int PLANE4 = N * N / 4;
    __syncthreads();
    // tables of sweep s for this lane's line
    auto sweep_tables = [&](int s, const float4 *&pr, const float4 *&pinv, const float4 *&pe) {
        const size_t o = ((size_t)s * C + c) * PLANE4 + t;
        pr = reinterpret_cast<const float4 *>(T.r) + o;
        pinv = reinterpret_cast<const float4 *>(T.inv) + o;
        pe = reinterpret_cast<const float4 *>(T.e) + o;
    };
    // pull the table rows of a sweep into L1 one sweep ahead
    auto prefetch_sweep = [&](int s, bool with_r) {
        if (s < 0 || s >= a.S) return;
        const size_t o = ((size_t)s * C + c) * PLANE4 + t;
        prefetch_tables<N>(reinterpret_cast<const float4 *>(T.inv) + o, reinterpret_cast<const float4 *>(T.e) + o,
                           with_r ? reinterpret_cast<const float4 *>(T.r) + o : nullptr);
    };
    const size_t plane = (size_t)N * N;
    const int wg = blockIdx.x * nwarps + warp;
    float *scratch = a.scratch + (size_t)wg * a.S * SLOT;
    float sig = 0.0f;
    if (d.skip) sig = 1.0f / (1.0f + expf(-__ldg(a.skipw)));
    const float om = 1.0f - sig;
    const float onepe = 1.0f + d.eps;
    const bool smooth = d.smooth != 0;
    float gm[PDE_MAX_CHANNELS] = {0.f, 0.f, 0.f, 0.f};
    float gw = 0.0f;
    const int sps = a.sps;
    const int last_ax = (sps == 3) ? 0 : 1;  // orientation of the state after the last sweep of a step

    for (int item = blockIdx.x * a.G + group; item < a.nitems; item += gridDim.x * a.G) {
        const int ba = item * 2, bb = ba + 1;
        const bool va = ba < d.B, vb = bb < d.B;
        const size_t oa = ((size_t)(va ? ba : 0) * C + c) * plane, ob = ((size_t)(vb ? bb : 0) * C + c) * plane;
        f2 x[1][N];
        int x_ax = -1;   // orientation of x in registers (0 rows, 1 columns), -1: the tile holds it
        auto x_store = [&](int ax) {
            if (active) {
                if (ax == 0) st_line<N, 0>(xt, t, x[0]);
                else st_line<N, 1>(xt, t, x[0]);
            }
        };
        auto x_load = [&](int ax) {
            if (ax == 0) ld_line<N, 0>(xt, t, x[0]);
            else ld_line<N, 1>(xt, t, x[0]);
        };
        // ------------------------------ phase 1: forward trajectory with checkpoints
        planes_to_tile<N>(a.u + oa, a.u + ob, xt, lane, va, vb);
        __syncwarp();
        for (int step = 0; step < d.steps; ++step) {
            if (CHAN && d.chan_op == 1) {
                if (x_ax >= 0) {
                    __syncwarp();
                    x_store(x_ax);
                }
                group_sync(C, group);
                mix_rows<N, 1>(gxt, C, a.chan + c * C, 1, t, x);
                group_sync(C, group);
                x_ax = 0;
            }
            // straight-line x, y, (x) sweeps: a loop over the sweeps of a step keeps ptxas from
            // scheduling the next sweep's coefficient loads across the transposition
            const int s0 = step * sps;
            const float4 *pr, *pinv, *pe;
            if (x_ax != 0) {
                if (x_ax >= 0) {
                    __syncwarp();
                    x_store(x_ax);
                    __syncwarp();
                }
                x_load(0);
            }
            prefetch_sweep(s0 + 1, false);
            sweep_tables(s0, pr, pinv, pe);
            thomas_solve<N, 1>(x, pinv, pe);
            if (exact) ck_store<N>(scratch + (size_t)s0 * SLOT, lane, x[0]);
            x_store(0);
            __syncwarp();
            x_load(1);
            prefetch_sweep(s0 + 2, false);
            sweep_tables(s0 + 1, pr, pinv, pe);
            thomas_solve<N, 1>(x, pinv, pe);
            x_ax = 1;
            if (exact || sps == 2) ck_store<N>(scratch + (size_t)(s0 + 1) * SLOT, lane, x[0]);
            if (sps == 3) {
                x_store(1);
                __syncwarp();
                x_load(0);
                prefetch_sweep(s0 + 3, false);
                sweep_tables(s0 + 2, pr, pinv, pe);
                thomas_solve<N, 1>(x, pinv, pe);
                x_ax = 0;
                ck_store<N>(scratch + (size_t)(s0 + 2) * SLOT, lane, x[0]);
            }
            if (CHAN && d.chan_op == 2) {
                __syncwarp();
                x_store(x_ax);
                group_sync(C, group);
                mix_rows<N, 1>(gxt, C, a.chan + c * C, 1, t, x);
                group_sync(C, group);
                x_ax = 0;
            }
        }
        // the skip epilogue needs the FINAL state (after the last coupling): park it in the x tile
        if (d.skip && x_ax >= 0) {
            __syncwarp();
            x_store(x_ax);
        }
        __syncwarp();
        // ------------------------------ phase 2: reverse
        {   // the next item's input planes start their trip from HBM to L2 now
            const int nb = (item + gridDim.x * a.G) * 2;
#pragma unroll
            for (int p = 0; p < 2; ++p)
                if (nb + p < d.B) {
                    prefetch_plane_l2<N>(a.u + ((size_t)(nb + p) * C + c) * plane, lane);
                    prefetch_plane_l2<N>(a.gout + ((size_t)(nb + p) * C + c) * plane, lane);
                }
        }
        planes_to_tile<N>(a.gout + oa, a.gout + ob, gt, lane, va, vb);
        __syncwarp();
        if (d.skip) {
            // out = sig u0 + om uF:  dL/dw += sig' * sum gout (u0 - uF),  g <- om * gout
            if (active) {
                f2 accw = f2_bc(0.0f);
                f2 gl[N], uf[N];
                ld_line<N, 0>(gt, t, gl);
                ld_line<N, 0>(xt, t, uf);
                const float2 zero2 = make_float2(0.f, 0.f);
#pragma unroll
                for (int j = 0; j < N / 2; ++j) {
                    const float2 wa = va ? __ldg(reinterpret_cast<const float2 *>(a.u + oa + (size_t)t * N) + j) : zero2;
                    const float2 wb = vb ? __ldg(reinterpret_cast<const float2 *>(a.u + ob + (size_t)t * N) + j) : zero2;
                    accw = f2_fma(gl[2 * j], f2_sub(f2_make(wa.x, wb.x), uf[2 * j]), accw);
                    accw = f2_fma(gl[2 * j + 1], f2_sub(f2_make(wa.y, wb.y), uf[2 * j + 1]), accw);
                    gl[2 * j] = f2_muls(om, gl[2 * j]);
                    gl[2 * j + 1] = f2_muls(om, gl[2 * j + 1]);
                }
                st_line<N, 0>(gt, t, gl);
                gw += f2_hsum(accw);
            }
            __syncwarp();
        }
        auto g_store = [&](const f2 (&g)[N], int ax) {
            if (active) {
                if (ax == 0) st_line<N, 0>(gt, t, g);
                else st_line<N, 1>(gt, t, g);
            }
        };
        // checkpoint slot -> x tile (a slot is read back in the orientation it was written in)
        auto ck_to_xt = [&](int slot, int ax) {
            f2 xs[N];
            ck_load<N>(scratch + (size_t)slot * SLOT, lane, xs);
            __syncwarp();   // every lane is done with the previous content of the tile
            if (active) {
                if (ax == 0) st_line<N, 0>(xt, t, xs);
                else st_line<N, 1>(xt, t, xs);
            }
        };
        // the reversed sweeps of one step; g sits in registers in orientation g_ax (-1: in its tile)
        auto reverse_step = [&](f2 (&g)[N], int &g_ax, int step) {
            for (int k = sps - 1; k >= 0; --k) {
                const int s = step * sps + k, ax = sweep_axis(k);
                if (exact && k != sps - 1) ck_to_xt(s, ax);
                if (g_ax != ax) {
                    if (g_ax >= 0) g_store(g, g_ax);
                    __syncwarp();
                    if (ax == 0) ld_line<N, 0>(gt, t, g);
                    else ld_line<N, 1>(gt, t, g);
                    g_ax = ax;
                } else {
                    __syncwarp();
                }
                const float4 *pr, *pinv, *pe;
                sweep_tables(s, pr, pinv, pe);
                prefetch_sweep(s - 1, true);
                const float4 *pm = reinterpret_cast<const float4 *>(T.msk) + ((size_t)s * C + c) * PLANE4 + t;
                const float scale = h_scale[s], tt = h_t[s];
                const bool clamped = h_clamped[s] != 0;
                const bool rebuild = !exact && k > 0;
                if (ax == 0)
                    reverse_sweep<N, 0>(g, xt, t, active, tbase, pr, pinv, pe, pm, scale, tt, onepe, smooth, rebuild, clamped);
                else
                    reverse_sweep<N, 1>(g, xt, t, active, tbase + 64u, pr, pinv, pe, pm, scale, tt, onepe, smooth, rebuild, clamped);
            }
        };
        if (CHAN) {
            // a channel op sits at one end of every step and works on the group's tiles: the adjoint
            // lives in registers only inside a step
            for (int step = d.steps - 1; step >= 0; --step) {
                // state after the last sweep of this step = input of the post-step coupling
                ck_to_xt(step * sps + sps - 1, last_ax);
                if (d.chan_op == 2) {
                    __syncwarp();
                    chan_adjoint<N>(ggt, gxt, C, c, group, a.chan, t, active, gm);
                }
                {
                    f2 g[N];
                    int g_ax = -1;
                    reverse_step(g, g_ax, step);
                    g_store(g, g_ax);
                }
                if (d.chan_op == 1) {
                    // adjoint of the pre-step mix: needs g (rows) and the mix INPUT = state before
                    // this step = checkpoint of the previous step (or u) in the group's tiles
                    if (step > 0) {
                        ck_to_xt(step * sps - 1, last_ax);
                    } else {
                        __syncwarp();
                        planes_to_tile<N>(a.u + oa, a.u + ob, xt, lane, va, vb);
                    }
                    __syncwarp();
                    chan_adjoint<N>(ggt, gxt, C, c, group, a.chan, t, active, gm);
                }
            }
        } else {
            f2 g[N];
            int g_ax = -1;
            for (int step = d.steps - 1; step >= 0; --step) {
                ck_to_xt(step * sps + sps - 1, last_ax);
                reverse_step(g, g_ax, step);
            }
            if (g_ax >= 0) g_store(g, g_ax);
        }
        __syncwarp();
        if (a.need_gin)
            tile_to_planes<N>(gt, a.gin + oa, a.gin + ob, lane, va, vb, d.skip ? a.gout + oa : nullptr,
                              d.skip ? a.gout + ob : nullptr, sig, 1.0f);
        __syncwarp();
        // the next item's phase 1 mixes through the group's x tiles: nobody may still read them
        if (CHAN) group_sync(C, group);
    }
    // ------------------------------ per-warp partials: TMEM -> global (cell order [row][col])
    tmem_wait_st();
    float *pm = a.part_maps + (size_t)wg * 4 * plane;
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
        float av[32];
        tmem_ld16(tbase + kk * 32, av);
        tmem_ld16(tbase + kk * 32 + 16, av + 16);
        tmem_wait_ld();
        if (active) {
            if (kk < 2) {   // lane = row
#pragma unroll
                for (int q = 0; q < N / 4; ++q)
                    *reinterpret_cast<float4 *>(pm + kk * plane + (size_t)t * N + 4 * q) =
                        make_float4(av[4 * q], av[4 * q + 1], av[4 * q + 2], av[4 * q + 3]);
            } else {        // lane = column
#pragma unroll
                for (int i = 0; i < N; ++i) pm[kk * plane + (size_t)i * N + t] = av[i];
            }
        }
    }
#pragma unroll
    for (int dd = 0; dd < PDE_MAX_CHANNELS; ++dd) {
        const float sgm = warp_sum(active ? gm[dd] : 0.0f);
        if (lane == 0) a.part_chan[(size_t)wg * PDE_MAX_CHANNELS + dd] = sgm;
    }
    const float sgw = warp_sum(gw);
    if (lane == 0) a.part_skip[wg] = sgw;
    tmem_fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_slot, (uint32_t)a.tmem_cols);
}

// Sum the per-warp partials (double accumulation, fixed order => deterministic).  A block covers
// 32 output elements; its 8 warps each sum an interleaved slice of the partials (independent loads,
// unrolled) and the 8 slice sums are combined in a fixed order through shared memory.
constexpr int kFinishCells = 32, kFinishSlices = 8;
__device__ __forceinline__ void finish_body(const pde_adi_desc &d, int nwarps_total, int nsets_small,
                                            const float *__restrict__ part_maps, const float *__restrict__ part_chan,
                                            const float *__restrict__ part_skip, const float *__restrict__ skipw, float *g_ab,
                                            float *g_atc, float *g_bb, float *g_btc, float *g_chan, float *g_skip,
                                            const unsigned bid) {
    __shared__ double red[kFinishSlices][kFinishCells];
    const int C = d.C, N = d.N;
    const size_t plane = (size_t)N * N;
    const size_t total = 4 * (size_t)C * plane;
    const int lane = threadIdx.x % kFinishCells, slice = threadIdx.x / kFinishCells;
    const size_t idx = (size_t)bid * kFinishCells + lane;
    double acc = 0.0;
    int kind = 0, c = 0;
    size_t cell = 0;
    if (idx < total) {
        kind = (int)(idx / (C * plane));
        c = (int)((idx / plane) % C);
        cell = idx % plane;
        const int per_c = (nwarps_total - c + C - 1) / C;   // warps that own channel c: c, c + C, ...
        double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
        int j = slice;
        for (; j + 3 * kFinishSlices < per_c; j += 4 * kFinishSlices) {
            a0 += (double)part_maps[((size_t)(c + (size_t)C * j) * 4 + kind) * plane + cell];
            a1 += (double)part_maps[((size_t)(c + (size_t)C * (j + kFinishSlices)) * 4 + kind) * plane + cell];
            a2 += (double)part_maps[((size_t)(c + (size_t)C * (j + 2 * kFinishSlices)) * 4 + kind) * plane + cell];
            a3 += (double)part_maps[((size_t)(c + (size_t)C * (j + 3 * kFinishSlices)) * 4 + kind) * plane + cell];
        }
        for (; j < per_c; j += kFinishSlices)
            a0 += (double)part_maps[((size_t)(c + (size_t)C * j) * 4 + kind) * plane + cell];
        acc = (a0 + a1) + (a2 + a3);
    }
    red[slice][lane] = acc;
    __syncthreads();
    if (slice == 0 && idx < total) {
        double sum = 0.0;
#pragma unroll
        for (int q = 0; q < kFinishSlices; ++q) sum += red[q][lane];
        float *dst = kind == 0 ? g_ab : kind == 1 ? g_atc : kind == 2 ? g_bb : g_btc;
        dst[(size_t)c * plane + cell] = (float)sum;
    }
    if (bid == 0) {
        // channel-matrix and skip-weight partials: a warp per output, lanes stride over the partial sets
        // (hundreds to thousands of them), fixed shuffle tree: deterministic, and not one serial thread
        const int warp = threadIdx.x >> 5, ln = threadIdx.x & 31;
        constexpr int kWarps = kFinishCells * kFinishSlices / 32;
        if (g_chan)
            for (int q = warp; q < C * C; q += kWarps) {
                const int cc = q / C, dd = q % C;
                double a = 0.0;
                for (int w = cc + C * ln; w < nsets_small; w += C * 32) a += (double)part_chan[(size_t)w * PDE_MAX_CHANNELS + dd];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(kFullMask, a, o);
                if (ln == 0) g_chan[cc * C + dd] = (float)a;
            }
        if (g_skip && warp == kWarps - 1) {
            double a = 0.0;
            for (int w = ln; w < nsets_small; w += 32) a += (double)part_skip[w];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(kFullMask, a, o);
            if (ln == 0) {
                const double sg = 1.0 / (1.0 + exp(-(double)skipw[0]));
                g_skip[0] = (float)(a * sg * (1.0 - sg));
            }
        }
    }
}

__global__ void __launch_bounds__(kFinishCells *kFinishSlices)
    finish_kernel(pde_adi_desc d, int nwarps_total, int nsets_small, const float *__restrict__ part_maps,
                  const float *__restrict__ part_chan, const float *__restrict__ part_skip,
                  const float *__restrict__ skipw, float *g_ab, float *g_atc, float *g_bb, float *g_btc,
                  float *g_chan, float *g_skip) {
    finish_body(d, nwarps_total, nsets_small, part_maps, part_chan, part_skip, skipw, g_ab, g_atc, g_bb, g_btc, g_chan,
                g_skip, blockIdx.x);
}

struct FinishMulti {
    int n, blocks_per_job;
    FinishJob job[PDE_MAX_BRANCHES];
};
__global__ void __launch_bounds__(kFinishCells *kFinishSlices) finish_multi_kernel(const __grid_constant__ FinishMulti m) {
    const FinishJob &j = m.job[blockIdx.x / m.blocks_per_job];
    finish_body(j.d, j.nsets_maps, j.nsets_small, j.part_maps, j.part_chan, j.part_skip, j.skipw, j.g_ab, j.g_atc, j.g_bb,
                j.g_btc, j.g_chan, j.g_skip, blockIdx.x % m.blocks_per_job);
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
static int validate(const pde_adi_desc *d) {
    if (!d) return PDE_ERR_INVALID;
    if (d->B < 0 || d->C < 1 || d->N < 2 || d->steps < 0) return PDE_ERR_INVALID;
    if (d->chan_op < 0 || d->chan_op > 2) return PDE_ERR_INVALID;
    if (d->steps * sweeps_per_step(*d) > PDE_MAX_SWEEPS) return PDE_ERR_UNSUPPORTED;
    if (d->C > PDE_MAX_CHANNELS) return wide::serves(*d) ? PDE_OK : PDE_ERR_UNSUPPORTED;   // adi_wide.cu
    switch (d->N) {
        case 8: case 12: case 16: case 20: case 24: case 28: case 32: break;   // kernels compiled per plane edge
        default:
            if (!generic::serves(*d)) return PDE_ERR_UNSUPPORTED;              // adi_generic.cu: edge at run time
    }
    return PDE_OK;
}

static int groups_per_block(int C) { return C >= 3 ? 1 : (C == 2 ? 2 : 4); }

static int tile_words(int N) { return 2 * N * (N + 2); }   // one tile = one sample pair

struct BwdPlan {
    int G, warps, blocks_per_sm, grid, nitems, tile_sets, tmem_cols;
    size_t smem, scratch_floats, maps_floats, chan_floats, skip_floats;
};

static int bwd_groups(int C) { return C == 1 ? 4 : (C == 2 ? 2 : (C == 3 ? 2 : 1)); }

template <int N>
static const void *bwd_kernel_ptr(bool chan) {
    return chan ? reinterpret_cast<const void *>(bwd_kernel<N, true>) : reinterpret_cast<const void *>(bwd_kernel<N, false>);
}

static const void *bwd_kernel_for(int N, bool chan) {
    switch (N) {
        case 8: return bwd_kernel_ptr<8>(chan);
        case 12: return bwd_kernel_ptr<12>(chan);
        case 16: return bwd_kernel_ptr<16>(chan);
        case 20: return bwd_kernel_ptr<20>(chan);
        case 24: return bwd_kernel_ptr<24>(chan);
        case 28: return bwd_kernel_ptr<28>(chan);
        case 32: return bwd_kernel_ptr<32>(chan);
        default: return nullptr;
    }
}

static int plan_bwd(const pde_adi_desc *d, BwdPlan *p) {
    DeviceProps props;
    int rc = query_props(&props);
    if (rc) return rc;
    p->G = bwd_groups(d->C);
    p->warps = p->G * d->C;
    p->tile_sets = 2;
    p->tmem_cols = p->warps <= 4 ? 128 : (p->warps <= 8 ? 256 : 512);
    p->smem = (size_t)p->tile_sets * p->warps * tile_words(d->N) * sizeof(float);
    if (p->smem > (size_t)props.max_smem_optin || p->warps > 16) return PDE_ERR_UNSUPPORTED;
    const void *kern = bwd_kernel_for(d->N, d->chan_op != 0);
    if (!kern) return PDE_ERR_UNSUPPORTED;
    // Residency from first principles: the occupancy calculator answers 1 block / SM for kernels
    // that allocate tensor memory, whatever their footprint.
    KernelInfo fa;
    rc = kernel_info(kern, p->smem, &fa);
    if (rc) return rc;
    const int threads = p->warps * 32;
    const int regs_per_warp = ((fa.regs + 7) / 8) * 8 * 32;
    const int by_regs = 65536 / (regs_per_warp * p->warps);
    const int by_smem = (int)((size_t)(228 * 1024) / (p->smem + fa.static_smem + 1024));
    const int by_threads = 2048 / threads;
    const int by_tmem = 512 / p->tmem_cols;
    int occ = by_regs;
    if (by_smem < occ) occ = by_smem;
    if (by_threads < occ) occ = by_threads;
    if (by_tmem < occ) occ = by_tmem;
    p->blocks_per_sm = occ;
    if (debug_enabled())
        fprintf(stderr, "[pde_b200] bwd plan: N=%d C=%d warps=%d smem=%zu regs=%d by_regs=%d by_smem=%d by_tmem=%d\n",
                d->N, d->C, p->warps, p->smem, fa.regs, by_regs, by_smem, by_tmem);
    if (p->blocks_per_sm < 1) p->blocks_per_sm = 1;
    p->nitems = (d->B + 1) / 2;
    int want = (p->nitems + p->G - 1) / p->G;
    int cap = props.sm_count * p->blocks_per_sm;
    p->grid = want < cap ? want : cap;
    if (p->grid < 1) p->grid = 1;
    const size_t S = (size_t)d->steps * sweeps_per_step(*d);
    const size_t nw = (size_t)p->grid * p->warps;
    p->scratch_floats = nw * (S > 0 ? S : 1) * 2 * d->N * 32;
    p->maps_floats = nw * 4 * d->N * d->N;
    p->chan_floats = nw * PDE_MAX_CHANNELS;
    p->skip_floats = nw;
    return PDE_OK;
}

template <int N>
static int launch_fwd(const Args &a, int NP, int sm_count, int threads, size_t smem, cudaStream_t st) {
    auto go = [&](auto kern) -> int {
        // persistent grid: exactly the blocks that are resident at once (registers included)
        int per_sm = 1;
        int rc = cached_occupancy(reinterpret_cast<const void *>(kern), threads, smem, &per_sm);
        if (rc) return rc;
        const int want = (a.nitems + a.G - 1) / a.G, cap = sm_count * per_sm;
        kern<<<want < cap ? want : cap, threads, smem, st>>>(a);
        return cuda_last_error();
    };
    return NP == 1 ? go(fwd_kernel<N, 1>) : go(fwd_kernel<N, 2>);
}

static int launch_bwd(const Args &a, const BwdPlan &p, cudaStream_t st) {
    const void *kern = bwd_kernel_for(a.d.N, a.d.chan_op != 0);
    if (!kern) return PDE_ERR_UNSUPPORTED;
    void *params[] = {const_cast<Args *>(&a)};
    PDE_CUDA_TRY(cudaLaunchKernel(kern, dim3(p.grid), dim3(p.warps * 32), params, p.smem, st));
    return cuda_last_error();
}

#define PDE_DISPATCH_N(N_, CALL)                     \
    switch (N_) {                                    \
        case 8: rc = CALL<8>; break;                 \
        case 12: rc = CALL<12>; break;               \
        case 16: rc = CALL<16>; break;               \
        case 20: rc = CALL<20>; break;               \
        case 24: rc = CALL<24>; break;               \
        case 28: rc = CALL<28>; break;               \
        case 32: rc = CALL<32>; break;               \
        default: rc = PDE_ERR_UNSUPPORTED;           \
    }

void launch_finish(const pde_adi_desc &d, int nsets_maps, int nsets_small, const float *part_maps,
                   const float *part_chan, const float *part_skip, const float *skipw, float *g_ab, float *g_atc,
                   float *g_bb, float *g_btc, float *g_chan, float *g_skip, cudaStream_t st) {
    const size_t total = 4 * (size_t)d.C * d.N * d.N;
    finish_kernel<<<(unsigned)((total + kFinishCells - 1) / kFinishCells), kFinishCells * kFinishSlices, 0, st>>>(
        d, nsets_maps, nsets_small, part_maps, part_chan, part_skip, skipw, g_ab, g_atc, g_bb, g_btc, g_chan, g_skip);
}

void launch_finish_multi(int n, const FinishJob *jobs, cudaStream_t st) {
    FinishMulti m{};
    m.n = n;
    const size_t total = 4 * (size_t)jobs[0].d.C * jobs[0].d.N * jobs[0].d.N;   // the jobs agree in C and N
    m.blocks_per_job = (int)((total + kFinishCells - 1) / kFinishCells);
    for (int i = 0; i < n; ++i) m.job[i] = jobs[i];
    finish_multi_kernel<<<(unsigned)(n * m.blocks_per_job), kFinishCells * kFinishSlices, 0, st>>>(m);
}

}  // namespace adi
}  // namespace pde

using namespace pde;
using namespace pde::adi;

extern "C" size_t pde_adi_tables_bytes(const pde_adi_desc *d) {
    if (validate(d) != PDE_OK) return 0;
    if (generic::serves(*d) || wide::serves(*d)) return generic::tables_bytes(*d);   // one table layout for both
    // header | tables of adi.cu | tables of adi_split.cu (always reserved: the size does not depend
    // on which implementation a call ends up using)
    return (size_t)kHeaderBytes + (4 * table_elems(*d) + split::table_floats(*d)) * sizeof(float);
}

static size_t legacy_workspace_bytes(const pde_adi_desc *d) {
    BwdPlan p;
    if (plan_bwd(d, &p) != PDE_OK) return 0;
    return (p.scratch_floats + p.maps_floats + p.chan_floats + p.skip_floats) * sizeof(float) + 256;
}

extern "C" size_t pde_adi_checkpoint_bytes(const pde_adi_desc *d) {
    if (validate(d) != PDE_OK) return 0;
    if (generic::serves(*d) || wide::serves(*d)) return 0;   // their backward pass replays the trajectory
    return split::supported(*d) ? split::checkpoint_bytes(*d) : 0;
}

extern "C" size_t pde_adi_backward_saved_workspace_bytes(const pde_adi_desc *d) {
    if (validate(d) != PDE_OK) return 0;
    if (generic::serves(*d)) return generic::workspace_bytes(*d);
    if (wide::serves(*d)) return wide::workspace_bytes(*d);
    if (split::supported(*d)) return split::workspace_bytes(*d);
    return legacy_workspace_bytes(d);
}

extern "C" size_t pde_adi_backward_workspace_bytes(const pde_adi_desc *d) {
    if (validate(d) != PDE_OK) return 0;
    if (generic::serves(*d)) return generic::workspace_bytes(*d);
    if (wide::serves(*d)) return wide::workspace_bytes(*d);
    if (split::supported(*d)) return split::workspace_bytes(*d) + split::checkpoint_bytes(*d) + 256;
    return legacy_workspace_bytes(d);
}

// sweeps with the same axis, time, time step and spacing share their tables
static void make_slot_map(const pde_adi_desc &d, const pde_adi_schedule &sch, SlotMap *m) {
    const int sps = sweeps_per_step(d), S = d.steps * sps;
    int nslots = 0;
    for (int s = 0; s < S; ++s) {
        int u = -1;
        for (int q = 0; q < s && u < 0; ++q)
            if (sweep_axis(q % sps) == sweep_axis(s % sps) && sch.t[q] == sch.t[s] && sch.dts[q] == sch.dts[s] &&
                sch.h2[q] == sch.h2[s])
                u = m->slot[q];
        if (u < 0) {
            u = nslots++;
            m->rep[u] = (short)s;
        }
        m->slot[s] = (short)u;
    }
    m->nslots = nslots;
}

// kap, r, top-down pivots, bottom-up pivots (floats) + the clamp mask (bytes), all C * N * N cells of a sweep
static size_t prepare_smem_bytes(int C, int N) { return (size_t)C * N * N * (4 * sizeof(float) + 1) + 16; }

template <int N>
static int launch_prepare(const pde_adi_desc &d, const pde_adi_schedule &sch, const SlotMap &sm, const float *ab,
                          const float *bb, const float *atc, const float *btc, char *tables, int want_split,
                          cudaStream_t st) {
    const int S = d.steps * sweeps_per_step(d);
    const size_t smem = prepare_smem_bytes(d.C, N);
    int rc = kernel_info(reinterpret_cast<const void *>(prepare_kernel<N>), smem, nullptr);
    if (rc) return rc;
    prepare_kernel<N><<<S, kPrepareThreads, smem, st>>>(d, sch, sm, ab, bb, atc, btc, tables, want_split);
    return cuda_last_error();
}

extern "C" int pde_adi_prepare(const pde_adi_desc *d, const pde_adi_schedule *sched, const float *ab,
                               const float *bb, const float *atc, const float *btc, void *tables,
                               void *stream) {
    int rc = validate(d);
    if (rc) return rc;
    if (!sched || !ab || !bb || !atc || !btc || !tables) return PDE_ERR_INVALID;
    if (reinterpret_cast<uintptr_t>(tables) & 255u) return PDE_ERR_WORKSPACE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int S = d->steps * sweeps_per_step(*d);
    if (S == 0) return PDE_OK;   // zero steps: identity, no tables
    if (generic::serves(*d) || wide::serves(*d))   // gprepare_kernel is channel-count agnostic
        return generic::prepare(*d, *sched, ab, bb, atc, btc, static_cast<char *>(tables), st);
    SlotMap sm;
    make_slot_map(*d, *sched, &sm);
    const int want_split = split::supported(*d) ? 1 : 0;
    char *tb = static_cast<char *>(tables);
    switch (d->N) {
        case 8: rc = launch_prepare<8>(*d, *sched, sm, ab, bb, atc, btc, tb, 0, st); break;
        case 12: rc = launch_prepare<12>(*d, *sched, sm, ab, bb, atc, btc, tb, 0, st); break;
        case 16: rc = launch_prepare<16>(*d, *sched, sm, ab, bb, atc, btc, tb, 0, st); break;
        case 20: rc = launch_prepare<20>(*d, *sched, sm, ab, bb, atc, btc, tb, 0, st); break;
        case 24: rc = launch_prepare<24>(*d, *sched, sm, ab, bb, atc, btc, tb, 0, st); break;
        case 28: rc = launch_prepare<28>(*d, *sched, sm, ab, bb, atc, btc, tb, want_split, st); break;
        case 32: rc = launch_prepare<32>(*d, *sched, sm, ab, bb, atc, btc, tb, want_split, st); break;
        default: rc = PDE_ERR_UNSUPPORTED;
    }
    return rc;
}

// ---------------------------------------------------------------------------- several layers, one launch
static int multi_validate(int n, const pde_adi_desc *d) {
    if (n < 1 || n > PDE_MAX_BRANCHES || !d) return PDE_ERR_INVALID;
    for (int i = 0; i < n; ++i) {
        const int rc = validate(&d[i]);
        if (rc) return rc;
        if (generic::serves(d[i]) || wide::serves(d[i])) return PDE_ERR_UNSUPPORTED;   // single-layer calls only
    }
    if (d[0].B == 0) return PDE_OK;
    return split::multi_compatible(n, d) ? PDE_OK : PDE_ERR_UNSUPPORTED;
}

extern "C" int pde_adi_multi_prepare(int n, const pde_adi_desc *d, const pde_adi_schedule *sched,
                                     const float *const *ab, const float *const *bb, const float *const *atc,
                                     const float *const *btc, void *const *tables, void *stream) {
    int rc = multi_validate(n, d);
    if (rc) return rc;
    if (!sched || !ab || !bb || !atc || !btc || !tables) return PDE_ERR_INVALID;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    PrepareMulti m{};
    m.want_split = 1;
    int blocks = 0;
    for (int i = 0; i < n; ++i) {
        if (!ab[i] || !bb[i] || !atc[i] || !btc[i] || !tables[i]) return PDE_ERR_INVALID;
        if (reinterpret_cast<uintptr_t>(tables[i]) & 255u) return PDE_ERR_WORKSPACE;
        const int S = d[i].steps * sweeps_per_step(d[i]);
        if (S == 0) continue;
        PrepareJob &j = m.job[m.n++];
        j.d = d[i];
        j.sch = sched[i];
        make_slot_map(d[i], sched[i], &j.sm);
        j.ab = ab[i]; j.bb = bb[i]; j.atc = atc[i]; j.btc = btc[i];
        j.tables = static_cast<char *>(tables[i]);
        j.s_begin = blocks;
        blocks += S;
    }
    if (blocks == 0) return PDE_OK;
    const size_t smem = prepare_smem_bytes(d[0].C, d[0].N);
    if (d[0].N == 28) {
        rc = kernel_info(reinterpret_cast<const void *>(prepare_multi_kernel<28>), smem, nullptr);
        if (rc) return rc;
        prepare_multi_kernel<28><<<blocks, kPrepareThreads, smem, st>>>(m);
    } else if (d[0].N == 32) {
        rc = kernel_info(reinterpret_cast<const void *>(prepare_multi_kernel<32>), smem, nullptr);
        if (rc) return rc;
        prepare_multi_kernel<32><<<blocks, kPrepareThreads, smem, st>>>(m);
    } else {
        return PDE_ERR_UNSUPPORTED;
    }
    return cuda_last_error();
}

extern "C" int pde_adi_multi_forward_train(int n, const pde_adi_desc *d, const void *const *tables, const float *u,
                                           const float *const *chan, const float *const *skipw, float *const *out,
                                           void *const *ckpt, void *stream) {
    int rc = multi_validate(n, d);
    if (rc) return rc;
    if (d[0].B == 0) return PDE_OK;
    if (!tables || !u || !out || !ckpt || !aligned16(u)) return PDE_ERR_INVALID;
    for (int i = 0; i < n; ++i) {
        if (!tables[i] || !out[i] || !ckpt[i] || !aligned16(out[i])) return PDE_ERR_INVALID;
        if (d[i].chan_op && (!chan || !chan[i])) return PDE_ERR_INVALID;
        if (d[i].skip && (!skipw || !skipw[i])) return PDE_ERR_INVALID;
    }
    return split::forward_multi(n, d, tables, u, chan, skipw, out, ckpt, static_cast<cudaStream_t>(stream));
}

extern "C" int pde_adi_multi_backward_saved(int n, const pde_adi_desc *d, const void *const *tables, const float *u,
                                            const float *const *gout, const float *const *chan,
                                            const float *const *skipw, const void *const *ckpt, float *const *gin,
                                            float *const *g_ab, float *const *g_bb, float *const *g_atc,
                                            float *const *g_btc, float *const *g_chan, float *const *g_skip,
                                            void *const *workspace, const size_t *workspace_bytes, void *stream) {
    int rc = multi_validate(n, d);
    if (rc) return rc;
    if (!g_ab || !g_bb || !g_atc || !g_btc) return PDE_ERR_INVALID;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    for (int i = 0; i < n; ++i) {
        if (!g_ab[i] || !g_bb[i] || !g_atc[i] || !g_btc[i]) return PDE_ERR_INVALID;
        if (d[i].chan_op && (!g_chan || !g_chan[i])) return PDE_ERR_INVALID;
        if (d[i].skip && (!g_skip || !g_skip[i])) return PDE_ERR_INVALID;
    }
    if (d[0].B == 0) {
        for (int i = 0; i < n; ++i) {
            const size_t mapb = (size_t)d[i].C * d[i].N * d[i].N * sizeof(float);
            PDE_CUDA_TRY(cudaMemsetAsync(g_ab[i], 0, mapb, st));
            PDE_CUDA_TRY(cudaMemsetAsync(g_bb[i], 0, mapb, st));
            PDE_CUDA_TRY(cudaMemsetAsync(g_atc[i], 0, mapb, st));
            PDE_CUDA_TRY(cudaMemsetAsync(g_btc[i], 0, mapb, st));
            if (g_chan && g_chan[i]) PDE_CUDA_TRY(cudaMemsetAsync(g_chan[i], 0, (size_t)d[i].C * d[i].C * sizeof(float), st));
            if (g_skip && g_skip[i]) PDE_CUDA_TRY(cudaMemsetAsync(g_skip[i], 0, sizeof(float), st));
        }
        return PDE_OK;
    }
    if (!tables || !u || !gout || !ckpt || !workspace || !workspace_bytes || !aligned16(u)) return PDE_ERR_INVALID;
    for (int i = 0; i < n; ++i) {
        if (!tables[i] || !gout[i] || !aligned16(gout[i]) || (gin && gin[i] && !aligned16(gin[i]))) return PDE_ERR_INVALID;
        if (d[i].chan_op && (!chan || !chan[i])) return PDE_ERR_INVALID;
        if (d[i].skip && (!skipw || !skipw[i])) return PDE_ERR_INVALID;
    }
    return split::backward_multi(n, d, tables, u, gout, chan, skipw, ckpt, gin, g_ab, g_bb, g_atc, g_btc, g_chan, g_skip,
                                 workspace, workspace_bytes, st);
}

extern "C" int pde_adi_forward_train(const pde_adi_desc *d, const void *tables, const float *u, const float *chan,
                                     const float *skipw, float *out, void *ckpt, void *stream) {
    int rc = validate(d);
    if (rc) return rc;
    if (d->B == 0) return PDE_OK;   // an empty batch (a rank with no samples) is a no-op: its pointers may be NULL
    if (!tables || !u || !out) return PDE_ERR_INVALID;
    if (d->chan_op && !chan) return PDE_ERR_INVALID;
    if (d->skip && !skipw) return PDE_ERR_INVALID;
    if (generic::serves(*d))   // scalar accesses: no alignment requirement (odd plane edges)
        return generic::forward(*d, static_cast<const char *>(tables), u, chan, skipw, out, static_cast<cudaStream_t>(stream));
    if (wide::serves(*d))
        return wide::forward(*d, static_cast<const char *>(tables), u, chan, skipw, out, static_cast<cudaStream_t>(stream));
    if (!aligned16(u) || !aligned16(out)) return PDE_ERR_INVALID;
    // with checkpoints to write: the half-line kernel (its backward twin needs them); plain
    // inference: the whole-line kernel below, which is the faster forward (DESIGN.md section 4)
    if (ckpt && split::supported(*d))
        return split::forward(*d, static_cast<const char *>(tables), u, chan, skipw, out, static_cast<float *>(ckpt),
                              static_cast<cudaStream_t>(stream));
    DeviceProps props;
    rc = query_props(&props);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    Args a{};
    a.d = *d;
    a.sps = sweeps_per_step(*d);
    a.S = d->steps * a.sps;
    a.G = groups_per_block(d->C);
    // a warp advances NP sample pairs; small batches spread over more warps instead
    // measured: two pairs per warp win for the single-channel 28 x 28 layers (coefficient rows shared
    // by four samples), one pair for the three-channel 32 x 32 ones (254 registers cost residency)
    int NP = d->C == 1 ? 2 : 1;
    if (NP == 2 && (d->B + 3) / 4 < props.sm_count * 4 * a.G) NP = 1;
    if (tune_np(*d) == 1 || tune_np(*d) == 2) NP = tune_np(*d);
    a.nitems = (d->B + 2 * NP - 1) / (2 * NP);
    a.tables = static_cast<const char *>(tables);
    a.u = u; a.chan = chan; a.skipw = skipw; a.out = out;
    const int warps = a.G * d->C;
    const size_t smem = (size_t)warps * NP * tile_words(d->N) * sizeof(float);
    switch (d->N) {
        case 8: rc = launch_fwd<8>(a, NP, props.sm_count, warps * 32, smem, st); break;
        case 12: rc = launch_fwd<12>(a, NP, props.sm_count, warps * 32, smem, st); break;
        case 16: rc = launch_fwd<16>(a, NP, props.sm_count, warps * 32, smem, st); break;
        case 20: rc = launch_fwd<20>(a, NP, props.sm_count, warps * 32, smem, st); break;
        case 24: rc = launch_fwd<24>(a, NP, props.sm_count, warps * 32, smem, st); break;
        case 28: rc = launch_fwd<28>(a, NP, props.sm_count, warps * 32, smem, st); break;
        case 32: rc = launch_fwd<32>(a, NP, props.sm_count, warps * 32, smem, st); break;
        default: rc = PDE_ERR_UNSUPPORTED;
    }
    return rc;
}

extern "C" int pde_adi_forward(const pde_adi_desc *d, const void *tables, const float *u, const float *chan,
                               const float *skipw, float *out, void *stream) {
    return pde_adi_forward_train(d, tables, u, chan, skipw, out, nullptr, stream);
}

extern "C" int pde_adi_backward(const pde_adi_desc *d, const void *tables, const float *u, const float *gout,
                                const float *chan, const float *skipw, float *gin, float *g_ab, float *g_bb,
                                float *g_atc, float *g_btc, float *g_chan, float *g_skip, void *workspace,
                                size_t workspace_bytes, void *stream) {
    return pde_adi_backward_saved(d, tables, u, gout, chan, skipw, nullptr, gin, g_ab, g_bb, g_atc, g_btc, g_chan,
                                  g_skip, workspace, workspace_bytes, stream);
}

extern "C" int pde_adi_backward_saved(const pde_adi_desc *d, const void *tables, const float *u, const float *gout,
                                      const float *chan, const float *skipw, const void *ckpt, float *gin,
                                      float *g_ab, float *g_bb, float *g_atc, float *g_btc, float *g_chan,
                                      float *g_skip, void *workspace, size_t workspace_bytes, void *stream) {
    int rc = validate(d);
    if (rc) return rc;
    if (!g_ab || !g_bb || !g_atc || !g_btc) return PDE_ERR_INVALID;
    if (d->chan_op && !g_chan) return PDE_ERR_INVALID;
    if (d->skip && !g_skip) return PDE_ERR_INVALID;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (d->B == 0) {
        // empty batch (a rank without samples): every gradient is exactly zero; u / gout / gin may be NULL
        const size_t mapb = (size_t)d->C * d->N * d->N * sizeof(float);
        PDE_CUDA_TRY(cudaMemsetAsync(g_ab, 0, mapb, st));
        PDE_CUDA_TRY(cudaMemsetAsync(g_bb, 0, mapb, st));
        PDE_CUDA_TRY(cudaMemsetAsync(g_atc, 0, mapb, st));
        PDE_CUDA_TRY(cudaMemsetAsync(g_btc, 0, mapb, st));
        if (g_chan) PDE_CUDA_TRY(cudaMemsetAsync(g_chan, 0, (size_t)d->C * d->C * sizeof(float), st));
        if (g_skip) PDE_CUDA_TRY(cudaMemsetAsync(g_skip, 0, sizeof(float), st));
        return PDE_OK;
    }
    if (!tables || !u || !gout) return PDE_ERR_INVALID;
    if (d->chan_op && !chan) return PDE_ERR_INVALID;
    if (d->skip && !skipw) return PDE_ERR_INVALID;
    if (generic::serves(*d))
        return generic::backward(*d, static_cast<const char *>(tables), u, gout, chan, skipw, gin, g_ab, g_bb, g_atc, g_btc,
                                 g_chan, g_skip, workspace, workspace_bytes, st);
    if (wide::serves(*d))
        return wide::backward(*d, static_cast<const char *>(tables), u, gout, chan, skipw, gin, g_ab, g_bb, g_atc, g_btc,
                              g_chan, g_skip, workspace, workspace_bytes, st);
    if (!aligned16(u) || !aligned16(gout) || (gin && !aligned16(gin))) return PDE_ERR_INVALID;
    if (d->B > 0 && split::supported(*d)) {
        const char *tb = static_cast<const char *>(tables);
        if (ckpt)
            return split::backward(*d, tb, u, gout, chan, skipw, static_cast<const float *>(ckpt), gin, g_ab, g_bb, g_atc,
                                   g_btc, g_chan, g_skip, workspace, workspace_bytes, st);
        // no checkpoints from the forward call: make them first, at the head of the workspace
        const size_t ckb = split::checkpoint_bytes(*d) + 256;
        if (!workspace || workspace_bytes < ckb + split::workspace_bytes(*d)) return PDE_ERR_WORKSPACE;
        rc = split::forward(*d, tb, u, chan, skipw, nullptr, static_cast<float *>(workspace), st);
        if (rc) return rc;
        return split::backward(*d, tb, u, gout, chan, skipw, static_cast<const float *>(workspace), gin, g_ab, g_bb,
                               g_atc, g_btc, g_chan, g_skip, static_cast<char *>(workspace) + ckb, workspace_bytes - ckb, st);
    }
    BwdPlan p;
    rc = plan_bwd(d, &p);
    if (rc) return rc;
    const size_t need = (p.scratch_floats + p.maps_floats + p.chan_floats + p.skip_floats) * sizeof(float) + 256;
    if (!workspace || workspace_bytes < need) return PDE_ERR_WORKSPACE;
    float *ws = reinterpret_cast<float *>((reinterpret_cast<uintptr_t>(workspace) + 255u) & ~(uintptr_t)255u);
    Args a{};
    a.d = *d;
    a.sps = sweeps_per_step(*d);
    a.S = d->steps * a.sps;
    a.G = p.G;
    a.nitems = p.nitems;
    a.need_gin = gin != nullptr;
    a.tile_sets = p.tile_sets;
    a.tmem_cols = p.tmem_cols;
    a.tables = static_cast<const char *>(tables);
    a.u = u; a.gout = gout; a.chan = chan; a.skipw = skipw; a.gin = gin;
    a.scratch = ws;
    a.part_maps = ws + p.scratch_floats;
    a.part_chan = a.part_maps + p.maps_floats;
    a.part_skip = a.part_chan + p.chan_floats;
    const int nw = p.grid * p.warps;
    rc = launch_bwd(a, p, st);
    if (rc) return rc;
    launch_finish(*d, nw, nw, a.part_maps, a.part_chan, a.part_skip, skipw, g_ab, g_atc, g_bb, g_btc, g_chan, g_skip, st);
    return cuda_last_error();
}
