// Implicit ADI layers, second implementation: HALF a line per thread, twisted factorisation.
//
// Same mathematics as adi.cu (reference: mnist_test.py:33-198, fashion_mnist.py:40-196,
// SVHN.py:38-230, cifar10.py:53-211, cifar_2version.py:52-187); different mapping onto the SM
// (DESIGN.md section 4.0 has the measurements behind every choice):
//
//   * A tridiagonal system can be eliminated from BOTH ends towards the middle ("twisted"
//     factorisation): two independent recurrences of half the length and one exchange where they
//     meet.  Here the two halves of a line belong to two threads of a warp (lanes l and l ^ P), so
//     a thread keeps N/2 cells of one sample pair in registers, the dependent chains are half as
//     long and an SM holds twice the warps of adi.cu for the same number of samples in flight.
//   * Everything is addressed in MIRRORED coordinates: a half line is indexed from the plane edge
//     (k = 0) to the junction (k = H-1) in both halves, so both threads of a line run the same
//     instruction stream; rows and columns of the tile are stored in that order too.
//   * A block advances groups of P sample pairs of every channel; every lane of a warp is busy for
//     any plane edge that is a multiple of 32 / (2 P).  The transposition between x and y sweeps goes
//     through a shared-memory tile as in adi.cu, but across the warps of the block: one
//     __syncthreads() per change of orientation.
//   * Forward: every sweep is a phase in which a thread applies its coefficients (staged in shared
//     memory by TMA one phase ahead) to its half line of Q groups in turn; it optionally writes the
//     state at the end of every step as a tile image (the "checkpoints": HBM is idle in these kernels).
//   * Backward: starts from those checkpoints instead of recomputing the trajectory; checkpoint
//     tiles arrive by TMA bulk copies one step ahead, the next item's gout planes by bulk copies too, the
//     coefficients by TMA one sweep ahead; gradient accumulators live in tensor memory.
//   * Plane I/O (u, out, gout, grad_input) is one TMA bulk copy per plane into / out of a tile slot in
//     natural layout; the first and last sweeps convert in registers (nat_ld_half / nat_st_half).
#include "adi_common.cuh"

namespace pde {
namespace adi {
namespace split {

template <int N, int P>
struct SG {
    static_assert(N % 4 == 0 && N >= 8 && N <= 32, "plane edge must be a multiple of 4 in [8, 32]");
    static_assert(P == 1 || P == 2 || P == 4 || P == 8, "pairs per block");
    static constexpr int H = N / 2;                 // cells per half line
    static constexpr int HQ = (H + 3) / 4;          // float4 chunks of a half line in the tables
    static constexpr int HCH = H / 2;               // 16-byte tile chunks (2 cells x 2 samples) per half row
    static constexpr int PADC = (HCH % 2 == 0) ? 1 : 0;   // keeps the two halves of a row in different bank halves
    static constexpr int HS = HCH + PADC;           // chunk stride between the halves of a row
    static constexpr int NC = 2 * HS;               // chunks per tile row
    static constexpr int LPW = 16 / P;              // lines per warp
    static constexpr int WPC = (N + LPW - 1) / LPW; // warps per channel
    static constexpr int RS = NC * P * 4;           // floats per tile row
    static constexpr int HPAD = 16;                 // 64 bytes between the two halves of the rows: a half warp
                                                    // reading a column touches rows of both halves
    static constexpr int TILE = N * RS + HPAD;      // floats per tile: P sample pairs of one channel
    static constexpr int QS = N * 2;                // float4 stride between the chunks of a table row
    // With four pairs, the planes of a group also sit in a tile slot in natural (NCHW) layout, one
    // plane per sample, as bulk copies bring them in and take them out.  Plane pitch: N * N + 4 floats,
    // so that the half-row reads of make_lane's lane map (LDS.64) spread over the banks: 2 wavefronts
    // for 28 x 28 (N * N = 784 = 16 mod 32 puts the four pairs' sample a in one bank: 4 wavefronts);
    // 32 x 32: 4 instead of 16, as two lines of a half warp then share their banks whatever the pitch.
    static constexpr int NPITCH = N * N + 4;
    // tile slot: a tile, or a group's planes if they need more (28 x 28, four pairs: 64 bytes more)
    static constexpr int SLOT = TILE > 2 * P * NPITCH ? TILE : 2 * P * NPITCH;
    // x sets keep the checkpoint image size: there the layer input goes unpadded when the pitch
    // would not fit
    static constexpr int XPITCH = 2 * P * NPITCH <= TILE ? NPITCH : N * N;
    static_assert(TILE % 4 == 0 && SLOT % 4 == 0 && NPITCH % 4 == 0, "16-byte aligned tiles and planes");
};

// float offset of (mirrored) row R of a tile
template <int N, int P>
__device__ __forceinline__ int row_off(int R) {
    return R * SG<N, P>::RS + (R >= SG<N, P>::H ? SG<N, P>::HPAD : 0);
}

// ------------------------------------------------------------------------------------------
// tile: N rows (mirrored order) x NC chunks x P pairs x {cell 2m, cell 2m+1} x {sample a, b}
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ f2 shfl_xor_f2(f2 a, int m) {
    const float lo = __shfl_xor_sync(kFullMask, f2_lo(a), m);
    const float hi = __shfl_xor_sync(kFullMask, f2_hi(a), m);
    return f2_make(lo, hi);
}

struct Lane {
    int c, wi, pp, h, R, tid_c;
    int b0, b1;   // float offsets of the thread's half row / half column inside a tile
    int tab;      // float4 offset of its coefficients inside the tables of one sweep
    bool active;
};

// AX == 0: the thread's half row (row R, half h); AX == 1: its half column (column R, rows of half h)
template <int N, int P, int AX>
__device__ __forceinline__ int half_base_of(int R, int h, int pp) {
    using G = SG<N, P>;
    if (AX == 0) return row_off<N, P>(R) + (h * G::HS * P + pp) * 4;
    const int hc = R >= G::H ? 1 : 0, kc = R - hc * G::H;
    return h * (G::H * G::RS + G::HPAD) + ((hc * G::HS + (kc >> 1)) * P + pp) * 4 + (kc & 1) * 2;
}
template <int N, int P, int AX>
__device__ __forceinline__ int half_base(const Lane &t) {
    return AX == 0 ? t.b0 : t.b1;
}

template <int N, int P, int AX>
__device__ __forceinline__ void ld_half(const float *tile, const Lane &t, f2 (&x)[N / 2]) {
    using G = SG<N, P>;
    const float *b = tile + half_base<N, P, AX>(t);
    if (AX == 0) {
#pragma unroll
        for (int m = 0; m < G::HCH; ++m) {
            const ulonglong2 v = *reinterpret_cast<const ulonglong2 *>(b + m * P * 4);
            x[2 * m].v = v.x;
            x[2 * m + 1].v = v.y;
        }
    } else {
#pragma unroll
        for (int k = 0; k < G::H; ++k) x[k].v = *reinterpret_cast<const unsigned long long *>(b + k * G::RS);
    }
}
template <int N, int P, int AX>
__device__ __forceinline__ void st_half(float *tile, const Lane &t, const f2 (&x)[N / 2]) {
    using G = SG<N, P>;
    float *b = tile + half_base<N, P, AX>(t);
    if (AX == 0) {
#pragma unroll
        for (int m = 0; m < G::HCH; ++m) {
            ulonglong2 v;
            v.x = x[2 * m].v;
            v.y = x[2 * m + 1].v;
            *reinterpret_cast<ulonglong2 *>(b + m * P * 4) = v;
        }
    } else {
#pragma unroll
        for (int k = 0; k < G::H; ++k) *reinterpret_cast<unsigned long long *>(b + k * G::RS) = x[k].v;
    }
}

// Two pairs per group (one block per SM, nothing hides the barriers of the bulk-copy path): planes of the
// block's P sample pairs (channel c) <-> tile by the threads.  A thread moves two adjacent cells of
// both samples of a pair per step; consecutive lanes take consecutive pairs, then consecutive
// cells.  All global loads of a thread are issued before the first one is used.
template <int N, int P>
struct PlaneIO {
    using G = SG<N, P>;
    static constexpr int F2 = N * N / 2;
    static constexpr int NTHR = G::WPC * 32;
    static constexpr int IT = (P * F2 + NTHR - 1) / NTHR;

    __device__ static __forceinline__ int tile_off(int f, int pp, bool &hc) {
        const int i = f / (N / 2), j0 = 2 * (f % (N / 2));
        hc = j0 >= G::H;
        const int m = hc ? (N - 2 - j0) / 2 : j0 / 2;
        return row_off<N, P>(mirror(i, N)) + (((hc ? G::HS : 0) + m) * P + pp) * 4;
    }

    // Which pair, cell pair and tile slot a thread handles in step `it` of a plane copy.  When a step
    // of the block advances a whole number of plane rows (all shipped sizes but 28 x 28 with two pairs),
    // the pair and the column part are per-thread constants and only the row moves: no divisions in
    // the loops.
    static constexpr bool REGULAR = (NTHR % P == 0) && ((NTHR / P) % (N / 2) == 0);
    static constexpr int FSTEP = NTHR / P, RSTEP = FSTEP / (N / 2);
    struct Thread {
        int pp, f0, i0, colo;
        bool hc;
    };
    __device__ static __forceinline__ Thread thread(int tid_c) {
        Thread th;
        th.pp = tid_c % P;
        th.f0 = tid_c / P;
        th.i0 = th.f0 / (N / 2);
        const int j0 = 2 * (th.f0 % (N / 2));
        th.hc = j0 >= G::H;
        const int m = th.hc ? (N - 2 - j0) / 2 : j0 / 2;
        th.colo = (((th.hc ? G::HS : 0) + m) * P + th.pp) * 4;
        return th;
    }
    struct Slot {
        int pp, f, off;
        bool hc, in;
    };
    __device__ static __forceinline__ Slot slot(const Thread &th, int tid_c, int it) {
        Slot sl;
        if (REGULAR) {
            sl.pp = th.pp;
            sl.f = th.f0 + it * FSTEP;
            sl.hc = th.hc;
            const int i = th.i0 + it * RSTEP;
            sl.in = i < N;
            sl.off = row_off<N, P>(mirror(i < N ? i : 0, N)) + th.colo;
        } else {
            const int idx = tid_c + it * NTHR;
            sl.pp = idx % P;
            sl.f = idx / P;
            sl.in = idx < P * F2;
            sl.off = tile_off(sl.in ? sl.f : 0, sl.pp, sl.hc);
        }
        return sl;
    }

    __device__ static __forceinline__ void to_tile(const float *__restrict__ g, float *tile, int item, int c, int C, int B,
                                                   int tid_c) {
        const float2 zero = make_float2(0.f, 0.f);
        const Thread th = thread(tid_c);
        float2 a[IT], b[IT];
#pragma unroll
        for (int it = 0; it < IT; ++it) {
            const Slot sl = slot(th, tid_c, it);
            const int ba = (item * P + sl.pp) * 2, bb = ba + 1;
            a[it] = (sl.in && ba < B) ? __ldcs(reinterpret_cast<const float2 *>(g + ((size_t)ba * C + c) * (N * N)) + sl.f) : zero;
            b[it] = (sl.in && bb < B) ? __ldcs(reinterpret_cast<const float2 *>(g + ((size_t)bb * C + c) * (N * N)) + sl.f) : zero;
        }
#pragma unroll
        for (int it = 0; it < IT; ++it) {
            const Slot sl = slot(th, tid_c, it);
            if (sl.in)
                *reinterpret_cast<float4 *>(tile + sl.off) = sl.hc ? make_float4(a[it].y, b[it].y, a[it].x, b[it].x)
                                                                   : make_float4(a[it].x, b[it].x, a[it].y, b[it].y);
        }
    }

    // out = tile                    (w == nullptr)
    // out = sig * w + om * tile     (skip epilogue: w = u0;  grad_input: w = gout, om = 1)
    __device__ static __forceinline__ void from_tile(const float *tile, float *__restrict__ g, int item, int c, int C,
                                                     int B, int tid_c, const float *__restrict__ w, float sig, float om) {
        const float2 zero = make_float2(0.f, 0.f);
        const Thread th = thread(tid_c);
        float2 wa[IT], wb[IT];
        if (w) {
#pragma unroll
            for (int it = 0; it < IT; ++it) {
                const Slot sl = slot(th, tid_c, it);
                const int ba = (item * P + sl.pp) * 2, bb = ba + 1;
                wa[it] = (sl.in && ba < B) ? __ldcs(reinterpret_cast<const float2 *>(w + ((size_t)ba * C + c) * (N * N)) + sl.f) : zero;
                wb[it] = (sl.in && bb < B) ? __ldcs(reinterpret_cast<const float2 *>(w + ((size_t)bb * C + c) * (N * N)) + sl.f) : zero;
            }
        }
#pragma unroll
        for (int it = 0; it < IT; ++it) {
            const Slot sl = slot(th, tid_c, it);
            if (sl.in) {
                const int f = sl.f;
                const bool hc = sl.hc;
                const int ba = (item * P + sl.pp) * 2, bb = ba + 1;
                const float4 v = *reinterpret_cast<const float4 *>(tile + sl.off);
                float2 a = hc ? make_float2(v.z, v.x) : make_float2(v.x, v.z);
                float2 b = hc ? make_float2(v.w, v.y) : make_float2(v.y, v.w);
                if (w) {
                    a.x = fmaf(om, a.x, sig * wa[it].x);
                    a.y = fmaf(om, a.y, sig * wa[it].y);
                    b.x = fmaf(om, b.x, sig * wb[it].x);
                    b.y = fmaf(om, b.y, sig * wb[it].y);
                }
                if (ba < B) __stcs(reinterpret_cast<float2 *>(g + ((size_t)ba * C + c) * (N * N)) + f, a);
                if (bb < B) __stcs(reinterpret_cast<float2 *>(g + ((size_t)bb * C + c) * (N * N)) + f, b);
            }
        }
    }
};

// ------------------------------------------------------------------------------------------
// Plane I/O with four pairs per group.  The 2P planes of a group travel between global memory and a tile
// slot by TMA bulk copies, one per plane, in natural layout: sample s of channel c at
// slot + c * cstride + s * pitch.  Samples beyond the batch are not copied; zero_tail clears them.
// The sweep that first reads a group takes its half row from the natural layout (nat_ld_half) and,
// after a barrier, stores it in tile layout; the last sweep does the reverse (nat_st_half).
// ------------------------------------------------------------------------------------------
template <int N, int P>
__device__ __forceinline__ int group_valid(long long grp, int B) {   // samples of group grp inside the batch
    const long long v = (long long)B - grp * 2 * P;
    return v <= 0 ? 0 : (v >= 2 * P ? 2 * P : (int)v);
}

// one thread: bulk loads of the group's valid planes, completing on `bar` (the caller expects the bytes)
template <int N, int P>
__device__ __forceinline__ void planes_load(float *slot, int cstride, int pitch, const float *__restrict__ g, long long grp,
                                            int C, int B, uint64_t *bar) {
    const int nv = group_valid<N, P>(grp, B);
    for (int c = 0; c < C; ++c)
        for (int s = 0; s < nv; ++s)
            tma_load_1d(slot + c * cstride + s * pitch, g + ((size_t)(grp * 2 * P + s) * C + c) * (N * N),
                        (uint32_t)(N * N * sizeof(float)), bar);
}

// one thread: bulk stores of the group's valid planes, as one bulk group
template <int N, int P>
__device__ __forceinline__ void planes_store(float *__restrict__ g, const float *slot, int cstride, int pitch, long long grp,
                                             int C, int B) {
    const int nv = group_valid<N, P>(grp, B);
    for (int c = 0; c < C; ++c)
        for (int s = 0; s < nv; ++s)
            tma_store_1d(g + ((size_t)(grp * 2 * P + s) * C + c) * (N * N), slot + c * cstride + s * pitch,
                         (uint32_t)(N * N * sizeof(float)));
    bulk_commit();
}

// every thread of the block: zero planes nv .. 2P-1 of every channel (samples beyond the batch)
template <int N, int P>
__device__ __forceinline__ void zero_tail(float *slot, int cstride, int pitch, int C, int nv) {
    constexpr int F4 = N * N / 4;
    const int per_c = (2 * P - nv) * F4;
    for (int i = threadIdx.x; i < C * per_c; i += blockDim.x) {
        const int c = i / per_c, r = i - c * per_c;
        *reinterpret_cast<float4 *>(slot + c * cstride + (nv + r / F4) * pitch + 4 * (r % F4)) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
}

// The thread's half row (row mirror(R), near or far half, cells from the plane edge) of its sample
// pair, from / to the natural layout.  Cells 2m, 2m+1 are columns 2m, 2m+1 (near) or N-1-2m, N-2-2m (far).
template <int N, int P, int PITCH>
__device__ __forceinline__ void nat_ld_half(const float *slot, const Lane &t, f2 (&x)[N / 2]) {
    const float *pa = slot + 2 * t.pp * PITCH + mirror(t.R, N) * N, *pb = pa + PITCH;
#pragma unroll
    for (int m = 0; m < N / 4; ++m) {
        const int j = t.h ? N - 2 - 2 * m : 2 * m;
        const float2 va = *reinterpret_cast<const float2 *>(pa + j), vb = *reinterpret_cast<const float2 *>(pb + j);
        x[2 * m] = t.h ? f2_make(va.y, vb.y) : f2_make(va.x, vb.x);
        x[2 * m + 1] = t.h ? f2_make(va.x, vb.x) : f2_make(va.y, vb.y);
    }
}
// plane = x                   (w == nullptr)
// plane = om * x + sig * w    (skip blend, w the same cells of a global plane set: out w = u, om = 1 - sig;
//                              grad_input w = gout, om = 1)
template <int N, int P, int PITCH>
__device__ __forceinline__ void nat_st_half(float *slot, const Lane &t, const f2 (&x)[N / 2], const float *__restrict__ w,
                                            long long grp, int c, int C, int B, float sig, float om) {
    const int i = mirror(t.R, N);
    float *pa = slot + 2 * t.pp * PITCH + i * N, *pb = pa + PITCH;
    const long long ba = grp * 2 * P + 2 * t.pp, bb = ba + 1;
    const float *wa = w + ((size_t)ba * C + c) * (N * N) + i * N, *wb = w + ((size_t)bb * C + c) * (N * N) + i * N;
    const float2 zero = make_float2(0.f, 0.f);
#pragma unroll
    for (int m = 0; m < N / 4; ++m) {
        const int j = t.h ? N - 2 - 2 * m : 2 * m;
        const float lo_a = f2_lo(x[2 * m]), lo_b = f2_hi(x[2 * m]), hi_a = f2_lo(x[2 * m + 1]), hi_b = f2_hi(x[2 * m + 1]);
        float2 a = t.h ? make_float2(hi_a, lo_a) : make_float2(lo_a, hi_a);
        float2 b = t.h ? make_float2(hi_b, lo_b) : make_float2(lo_b, hi_b);
        if (w) {
            const float2 va = ba < B ? __ldg(reinterpret_cast<const float2 *>(wa + j)) : zero;
            const float2 vb = bb < B ? __ldg(reinterpret_cast<const float2 *>(wb + j)) : zero;
            a.x = fmaf(om, a.x, sig * va.x);
            a.y = fmaf(om, a.y, sig * va.y);
            b.x = fmaf(om, b.x, sig * vb.x);
            b.y = fmaf(om, b.y, sig * vb.y);
        }
        *reinterpret_cast<float2 *>(pa + j) = a;
        *reinterpret_cast<float2 *>(pb + j) = b;
    }
}

// Rows of a tile slot that holds a group's planes -> the same slot in tile layout (the caller has
// passed a barrier since the planes arrived; a barrier must follow before other threads read)
template <int N, int P, int PITCH>
__device__ __forceinline__ void planes_to_rows(float *slot, const Lane &t) {
    f2 x[N / 2];
    nat_ld_half<N, P, PITCH>(slot, t, x);
    __syncthreads();   // every thread has read its rows in natural layout
    if (t.active) st_half<N, P, 0>(slot, t, x);
}

// the thread's coefficients of one table for one sweep: HQ float4, the same address for the P
// threads that own this half line in different sample pairs
template <int N, int P>
__device__ __forceinline__ void ld_coef(const float4 *__restrict__ p, float (&v)[4 * SG<N, P>::HQ]) {
    using G = SG<N, P>;
#pragma unroll
    for (int q = 0; q < G::HQ; ++q) {
        const float4 a = __ldg(p + q * G::QS);
        v[4 * q] = a.x; v[4 * q + 1] = a.y; v[4 * q + 2] = a.z; v[4 * q + 3] = a.w;
    }
}

// x[k] = sum_d mat[d * mstride] * (half row of channel d)
template <int N, int P>
__device__ __forceinline__ void mix_rows(const float *tiles, int cstride, int C, const float *__restrict__ mat,
                                         int mstride, const Lane &t, f2 (&x)[N / 2]) {
    using G = SG<N, P>;
    const f2 zero = f2_bc(0.0f);
#pragma unroll
    for (int k = 0; k < G::H; ++k) x[k] = zero;
    for (int dd = 0; dd < C; ++dd) {
        const float m = __ldg(mat + dd * mstride);
        f2 row[G::H];
        ld_half<N, P, 0>(tiles + (size_t)dd * cstride, t, row);
#pragma unroll
        for (int k = 0; k < G::H; ++k) x[k] = f2_fmas(m, row[k], x[k]);
    }
}

// ------------------------------------------------------------------------------------------
// (A + eps I) x = d by twisted elimination.  Each half, cells numbered from its edge:
//   d*_k = inv_k d_k + e_k d*_{k-1}                         k = 0 .. H-1
//   the far half owns the closing cell: x = d*_{H-1} + e_{H-1} (near half's d*_{H-1})
//   the near half's last cell:          x = d*_{H-1} + e_{H-1} (that x)
//   x_k = d*_k + e_k x_{k+1}                               k = H-2 .. 0
// ------------------------------------------------------------------------------------------
template <int N, int P, int NP>
__device__ __forceinline__ void solve(f2 (&x)[NP][N / 2], const float (&iv)[4 * SG<N, P>::HQ],
                                      const float (&e)[4 * SG<N, P>::HQ], bool far) {
    constexpr int H = N / 2;
#pragma unroll
    for (int p = 0; p < NP; ++p) x[p][0] = f2_muls(iv[0], x[p][0]);
#pragma unroll
    for (int k = 1; k < H; ++k)
#pragma unroll
        for (int p = 0; p < NP; ++p) x[p][k] = f2_fmas(e[k], x[p][k - 1], f2_muls(iv[k], x[p][k]));
    f2 o[NP];
#pragma unroll
    for (int p = 0; p < NP; ++p) o[p] = shfl_xor_f2(x[p][H - 1], P);
#pragma unroll
    for (int p = 0; p < NP; ++p) x[p][H - 1] = f2_fmas(far ? e[H - 1] : 0.0f, o[p], x[p][H - 1]);
#pragma unroll
    for (int p = 0; p < NP; ++p) o[p] = shfl_xor_f2(x[p][H - 1], P);
#pragma unroll
    for (int p = 0; p < NP; ++p) x[p][H - 1] = f2_fmas(far ? 0.0f : e[H - 1], o[p], x[p][H - 1]);
#pragma unroll
    for (int k = H - 2; k >= 0; --k)
#pragma unroll
        for (int p = 0; p < NP; ++p) x[p][k] = f2_fmas(e[k], x[p][k + 1], x[p][k]);
}

// L2 prefetch of a contiguous region by one thread (TMA bulk prefetch: no registers, no smem)
__device__ __forceinline__ void prefetch_region_l2(const void *p, size_t bytes) {
    const char *b = static_cast<const char *>(p);
    constexpr size_t kChunk = 16384;
    for (size_t off = 0; off < bytes; off += kChunk) {
        const unsigned n = (unsigned)((bytes - off < kChunk ? bytes - off : kChunk) & ~(size_t)15);
        if (n) asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(b + off), "r"(n) : "memory");
    }
}

template <int N, int P>
__device__ __forceinline__ Lane make_lane() {
    using G = SG<N, P>;
    Lane t;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    t.c = warp / G::WPC;
    t.wi = warp % G::WPC;
    t.pp = lane % P;
    t.h = (lane / P) & 1;
    const int line = t.wi * G::LPW + lane / (2 * P);
    t.active = line < N;
    t.tid_c = threadIdx.x - t.c * G::WPC * 32;
    t.R = t.active ? line : N - 1;
    t.b0 = half_base_of<N, P, 0>(t.R, t.h, t.pp);
    t.b1 = half_base_of<N, P, 1>(t.R, t.h, t.pp);
    t.tab = (t.c * G::HQ * N + t.R) * 2 + t.h;
    return t;
}

// per-thread pointer (float4 units) into a split table for sweep s
template <int N, int P>
__device__ __forceinline__ size_t tab_off(int s, int C, const Lane &t) {
    using G = SG<N, P>;
    return (size_t)(s * (C * G::HQ * N * 2) + t.tab);
}

// P == 4 serves the single-channel layers (one channel per block), P == 2 up to three channels
template <int N, int P>
constexpr int max_threads() { return P >= 4 ? SG<N, P>::WPC * 32 : SG<N, P>::WPC * 32 * 3; }
// P == 4: two blocks of 7-8 warps per SM.  The register file is split over the four schedulers
// (16 K registers each) and a block's warps are dealt round-robin, so two blocks put four warps on a
// scheduler: 128 registers per thread, not 65536 / threads.

// ------------------------------------------------------------------------------------------
// forward.  A block owns Q groups of P sample pairs (all channels).  Every sweep is one PHASE: the
// thread loads its coefficients once and applies them to its half line of the Q groups in turn
// (the state lives in the tiles between phases), so the coefficient traffic is amortised over Q.
// The closing half sweep of a Strang step and the opening one of the next run back to back on
// the registers (same orientation).
// ------------------------------------------------------------------------------------------
// One warp folds the per-sweep header entries into the flags the backward kernel reads.  Not inlined:
// the forward kernels' register allocation has no slack for it (12 - 24 bytes of spills when inlined).
__device__ __noinline__ void write_ck_flags(const Header *hdr, int steps, int sps, CkFlags *out) {
    bool ex, anyc;
    header_flags(hdr, steps, sps, &ex, &anyc);
    if ((threadIdx.x & 31) == 0) {
        out->mode_exact = ex ? 1 : 0;
        out->any_clamped = anyc ? 1 : 0;
    }
}

// MIX1: instantiation for layers with a pre-step channel mix (chan_op == 1), which runs inside the
// first sweep phase of a step; the others keep the plain schedule (and their register allocation).
template <int N, int P, int Q, bool MIX1>
__device__ __forceinline__ void sfwd_body(const Args &a, const int bid, const int nblk) {
    using G = SG<N, P>;
    constexpr int H = G::H, TILE = G::TILE, SLOT = G::SLOT, NPI = G::NPITCH, HQ4 = 4 * G::HQ;
    constexpr bool BULK = P >= 4;   // plane I/O by bulk copies (see PlaneIO)
    extern __shared__ __align__(128) float smem[];
    __shared__ __align__(8) uint64_t cbar[2];
    __shared__ __align__(8) uint64_t ubar;   // the planes of an item's Q groups
    __shared__ short h_slot[PDE_MAX_SWEEPS];
    const pde_adi_desc &d = a.d;
    const Lane t = make_lane<N, P>();
    const int C = d.C, nthr = blockDim.x;
    const bool far = t.h == 1;
    const int SET = C * Q * SLOT;   // floats per tile set: Q groups of every channel
    // coefficient stage: 1/pivot and r/pivot of one sweep (all channels), double buffered, filled
    // by TMA one phase ahead
    const int CT = C * G::HQ * N * 2 * 4;
    float *cbuf = smem + SET;
    const size_t T = stab_floats_per_table(d);
    float sig = 0.0f;
    if (d.skip) sig = 1.0f / (1.0f + expf(-__ldg(a.skipw)));
    const float om = 1.0f - sig;
    const int sps = a.sps, S = a.S;
    {
        const Header *hdr = reinterpret_cast<const Header *>(a.tables);
        for (int i = threadIdx.x; i < S; i += nthr) h_slot[i] = hdr->slot[i];
        // the call-wide flags of the backward pass travel with the checkpoints
        if (a.ck_flags && bid == 0 && threadIdx.x < 32) write_ck_flags(hdr, d.steps, sps, a.ck_flags);
    }
    if (threadIdx.x == 0) {
        mbar_init(&cbar[0], 1);
        mbar_init(&cbar[1], 1);
        mbar_init(&ubar, 1);
        mbar_fence_init();
    }
    __syncthreads();
    uint32_t cphase = 0u;
    auto c_fill = [&](int b, int s) {   // call after a barrier that ends every read of buffer b
        if (threadIdx.x == 0) {
            fence_proxy_async();
            const uint32_t bytes = (uint32_t)(CT * sizeof(float));
            mbar_expect_tx(&cbar[b], 2 * bytes);
            tma_load_1d(cbuf + (size_t)(2 * b) * CT, a.stab + T + (size_t)s * CT, bytes, &cbar[b]);
            tma_load_1d(cbuf + (size_t)(2 * b + 1) * CT, a.stab + 2 * T + (size_t)s * CT, bytes, &cbar[b]);
        }
    };
    const size_t plane = (size_t)N * N;
    // thread 0: u planes of group q of item `it` -> tile slot q (natural layout); the fill of group 0
    // expects the bytes of the whole item.  Call after a barrier that ends every use of slot q.
    auto u_fill = [&](int it, int q) {
        fence_proxy_async();
        if (q == 0) {
            const int nv = group_valid<N, Q * P>(it, d.B);   // samples of the item
            mbar_expect_tx(&ubar, (uint32_t)(nv * C * plane * sizeof(float)));
        }
        planes_load<N, P>(smem + q * SLOT, Q * SLOT, NPI, a.u, (long long)it * Q + q, C, d.B, &ubar);
    };
    uint32_t uphase = 0u;
    int cb = 0;
    if (bid < a.nitems) {
        c_fill(0, 0);
        if (BULK && threadIdx.x == 0)
            for (int q = 0; q < Q; ++q) u_fill(bid, q);
    }
    // Four pairs per group serve only layers without channel ops (make_plan): the first sweep, on rows,
    // reads the planes from the natural layout; a last sweep on rows (Strang) writes the output planes,
    // the last column sweep of a Lie step leaves that to a pass of its own.
    const bool nat_first = BULK;
    const bool nat_last = BULK && sps == 3;

    for (int item = bid; item < a.nitems; item += nblk) {
        const int next_item = item + nblk;
        float *set = smem;
        float *my = set + (size_t)t.c * Q * SLOT;   // this channel's Q tiles
        if (threadIdx.x == 0) {   // the next item's planes start their trip from HBM to L2 now
            const long long nb = (long long)next_item * Q * 2 * P;
            if (nb < d.B) {
                const long long ns = (d.B - nb) < 2 * P * Q ? (d.B - nb) : 2 * P * Q;
                prefetch_region_l2(a.u + (size_t)nb * C * plane, (size_t)ns * C * plane * sizeof(float));
            }
        }
        __syncthreads();   // the previous item's output planes have been read out of the tiles
        if (!BULK) {
#pragma unroll 1
            for (int q = 0; q < Q; ++q) PlaneIO<N, P>::to_tile(a.u, my + q * SLOT, item * Q + q, t.c, C, d.B, t.tid_c);
        } else {
            for (int q = 0; q < Q; ++q) {
                const int nv = group_valid<N, P>((long long)item * Q + q, d.B);
                if (nv < 2 * P) zero_tail<N, P>(set + q * SLOT, Q * SLOT, NPI, C, nv);
            }
            mbar_wait(&ubar, uphase);
            uphase ^= 1u;
        }
        // tile q -> output planes: the thread's half row x of group q (row orientation) goes to the
        // natural layout in place, then out by bulk stores; the slot is refilled with the next item's
        // group as soon as the store has read it (refill of q - 1 behind the store of q)
        auto emit = [&](int q, const f2 (&x)[H]) {
            __syncthreads();   // every thread has read tile q
            if (t.active)
                nat_st_half<N, P, NPI>(my + q * SLOT, t, x, d.skip ? a.u : nullptr, (long long)item * Q + q, t.c, C, d.B, sig, om);
            fence_proxy_async();
            __syncthreads();
            if (threadIdx.x == 0) {
                if (a.out) planes_store<N, P>(a.out, set + q * SLOT, Q * SLOT, NPI, (long long)item * Q + q, C, d.B);
                else bulk_commit();
                if (next_item < a.nitems) {
                    if (q > 0) {
                        bulk_wait_read<1>();
                        u_fill(next_item, q - 1);
                    }
                    if (q == Q - 1) {
                        bulk_wait_read<0>();
                        u_fill(next_item, q);
                    }
                }
            }
        };
        // u <- M u over the channels of every group (rows); leaves the tiles in row orientation
        auto mix_phase = [&]() {
            __syncthreads();
#pragma unroll 1
            for (int q = 0; q < Q; ++q) {
                f2 x[H];
                mix_rows<N, P>(set + q * SLOT, Q * SLOT, C, a.chan + t.c * C, 1, t, x);
                __syncthreads();
                if (t.active) st_half<N, P, 0>(my + q * SLOT, t, x);
            }
        };
        int s = 0;
        while (s < S) {
            const int k = s % sps, step = s / sps, ax = sweep_axis(k);
            // the pre-step mix (cifar) runs inside the step's first sweep phase: mixed rows go from the
            // tiles of all channels into registers, through the sweep and only then back to the tile
            const bool mix_first = MIX1 && k == 0 && d.chan_op == 1;
            if (!MIX1 && k == 0 && d.chan_op == 1) mix_phase();
            // the next sweep has the same orientation and (Strang: same time, time step, spacing) the same tables
            const bool fuse = sps == 3 && k == 2 && s + 1 < S && d.chan_op == 0 && h_slot[s] == h_slot[s + 1];
            const int s_next = s + (fuse ? 2 : 1);
            // phase boundary: the tiles change orientation and every thread has taken its coefficients
            // out of the other stage
            __syncthreads();
            {
                const int ns = s_next < S ? s_next : (next_item < a.nitems ? 0 : -1);
                if (ns >= 0) c_fill(cb ^ 1, ns);
            }
            mbar_wait(&cbar[cb], (cphase >> cb) & 1u);
            cphase ^= 1u << cb;
            float iv[HQ4], e[HQ4];
            {
                const float4 *ci = reinterpret_cast<const float4 *>(cbuf + (size_t)(2 * cb) * CT) + t.tab;
                const float4 *ce = reinterpret_cast<const float4 *>(cbuf + (size_t)(2 * cb + 1) * CT) + t.tab;
#pragma unroll
                for (int q = 0; q < G::HQ; ++q) {
                    const float4 a4 = ci[q * G::QS], b4 = ce[q * G::QS];
                    iv[4 * q] = a4.x; iv[4 * q + 1] = a4.y; iv[4 * q + 2] = a4.z; iv[4 * q + 3] = a4.w;
                    e[4 * q] = b4.x; e[4 * q + 1] = b4.y; e[4 * q + 2] = b4.z; e[4 * q + 3] = b4.w;
                }
            }
            cb ^= 1;
            if (MIX1 && mix_first) {
                f2 xm[Q][H];
#pragma unroll
                for (int q = 0; q < Q; ++q) mix_rows<N, P>(set + q * SLOT, Q * SLOT, C, a.chan + t.c * C, 1, t, xm[q]);
                __syncthreads();   // every channel has read every tile of the item
#pragma unroll
                for (int q = 0; q < Q; ++q) {
                    f2 x[1][H];
#pragma unroll
                    for (int kk = 0; kk < H; ++kk) x[0][kk] = xm[q][kk];
                    solve<N, P, 1>(x, iv, e, far);
                    if (t.active) st_half<N, P, 0>(my + q * SLOT, t, x[0]);
                }
                s = s_next;
                continue;
            }
            const bool from_planes = nat_first && s == 0, to_planes = nat_last && s_next >= S;
#pragma unroll 1
            for (int q = 0; q < Q; ++q) {
                float *tile = my + q * SLOT;
                f2 x[1][H];
                if (from_planes) nat_ld_half<N, P, NPI>(tile, t, x[0]);
                else if (ax == 0) ld_half<N, P, 0>(tile, t, x[0]);
                else ld_half<N, P, 1>(tile, t, x[0]);
                solve<N, P, 1>(x, iv, e, far);
                if (k == sps - 1 && a.ckpt && t.active) {
                    // state after the last sweep of the step, written as a tile image: the backward
                    // kernel brings it back with one bulk copy per step
                    float *ck = a.ckpt + (((size_t)(item * Q + q) * d.steps + step) * C + t.c) * TILE;
                    if (ax == 0) {
#pragma unroll
                        for (int m = 0; m < G::HCH; ++m) {
                            ulonglong2 v;
                            v.x = x[0][2 * m].v;
                            v.y = x[0][2 * m + 1].v;
                            __stcs(reinterpret_cast<ulonglong2 *>(ck + t.b0 + m * P * 4), v);
                        }
                    } else {
#pragma unroll
                        for (int kk = 0; kk < H; ++kk)
                            __stcs(reinterpret_cast<unsigned long long *>(ck + t.b1 + kk * G::RS), x[0][kk].v);
                    }
                }
                if (fuse) solve<N, P, 1>(x, iv, e, far);
                if (to_planes) {
                    emit(q, x[0]);
                    continue;
                }
                if (from_planes) __syncthreads();   // every thread has read the group's planes
                if (t.active) {
                    if (ax == 0) st_half<N, P, 0>(tile, t, x[0]);
                    else st_half<N, P, 1>(tile, t, x[0]);
                }
            }
            if (k == sps - 1 && d.chan_op == 2) mix_phase();
            s = s_next;
        }
        if (!BULK) {
            __syncthreads();
            if (a.out) {
#pragma unroll 1
                for (int q = 0; q < Q; ++q)
                    PlaneIO<N, P>::from_tile(my + q * SLOT, a.out, item * Q + q, t.c, C, d.B, t.tid_c, d.skip ? a.u : nullptr,
                                             sig, om);
            }
        } else if (!nat_last) {
            __syncthreads();
#pragma unroll 1
            for (int q = 0; q < Q; ++q) {
                f2 x[H];
                ld_half<N, P, 0>(my + q * SLOT, t, x);
                emit(q, x);
            }
        }
    }
    if (BULK && threadIdx.x == 0) bulk_wait_all();   // the output stores are complete before the block ends
}

template <int N, int P, int Q, bool MIX1>
__global__ void __launch_bounds__(max_threads<N, P>(), P >= 4 ? 2 : 1) sfwd_kernel(const Args a) {
    sfwd_body<N, P, Q, MIX1>(a, blockIdx.x, gridDim.x);
}

// Several layers applied to the SAME input in one launch (the three PDE branches of cifar10's
// MultiScaleExtractor, cifar10.py:272-274; the two of cifar_2version's HybridPDEExtractor,
// cifar_2version.py:287-288).  The resident blocks are dealt to the branches in proportion to their
// work (sweeps per item): blocks blk_begin[b] .. blk_begin[b + 1] - 1 walk the items of branch b.
struct MultiArgs {
    int n;
    int blk_begin[PDE_MAX_BRANCHES + 1];
    Args a[PDE_MAX_BRANCHES];
};

__device__ __forceinline__ int multi_branch_of(const MultiArgs &m, int *bid, int *nblk) {
    int b = m.n - 1;
    while (b > 0 && (int)blockIdx.x < m.blk_begin[b]) --b;
    *bid = (int)blockIdx.x - m.blk_begin[b];
    *nblk = m.blk_begin[b + 1] - m.blk_begin[b];
    return b;
}

template <int N, int P, int Q, bool MIX1>
__global__ void __launch_bounds__(max_threads<N, P>(), P >= 4 ? 2 : 1) sfwd_multi_kernel(const __grid_constant__ MultiArgs m) {
    int bid, nblk;
    const int b = multi_branch_of(m, &bid, &nblk);
    sfwd_body<N, P, Q, MIX1>(m.a[b], bid, nblk);
}

// ------------------------------------------------------------------------------------------
// backward
// ------------------------------------------------------------------------------------------

// Per-pixel gradient accumulators in TMEM: 64 columns per warp = {A0, A1, B0, B1} x 16, one TMEM
// lane per thread.  acc0 += m0 * z, acc1 += m1 * z (m0 = dt/h^2, m1 = t dt/h^2) for the kind (alpha / beta) of the sweep.
__device__ __forceinline__ void tmem_accumulate16(uint32_t tacc, const float (&z)[16], float m0, float m1) {
    float a0[16], a1[16];
    tmem_wait_st();
    tmem_ld16(tacc, a0);
    tmem_ld16(tacc + 16, a1);
    tmem_wait_ld();
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        a0[i] = fmaf(m0, z[i], a0[i]);
        a1[i] = fmaf(m1, z[i], a1[i]);
    }
    tmem_st16(tacc, a0);
    tmem_st16(tacc + 16, a1);
}

// Two adjacent cells (2m, 2m+1) of the thread's half line, straight from / to a tile.
template <int N, int P, int AX>
__device__ __forceinline__ void ld_duo(const float *tile, const Lane &t, int m, f2 &lo, f2 &hi) {
    using G = SG<N, P>;
    if (AX == 0) {
        const ulonglong2 v = *reinterpret_cast<const ulonglong2 *>(tile + t.b0 + m * P * 4);
        lo.v = v.x;
        hi.v = v.y;
    } else {
        lo.v = *reinterpret_cast<const unsigned long long *>(tile + t.b1 + (2 * m) * G::RS);
        hi.v = *reinterpret_cast<const unsigned long long *>(tile + t.b1 + (2 * m + 1) * G::RS);
    }
}
template <int N, int P, int AX>
__device__ __forceinline__ void st_duo(float *tile, const Lane &t, int m, f2 lo, f2 hi) {
    using G = SG<N, P>;
    if (AX == 0) {
        ulonglong2 v;
        v.x = lo.v;
        v.y = hi.v;
        *reinterpret_cast<ulonglong2 *>(tile + t.b0 + m * P * 4) = v;
    } else {
        *reinterpret_cast<unsigned long long *>(tile + t.b1 + (2 * m) * G::RS) = lo.v;
        *reinterpret_cast<unsigned long long *>(tile + t.b1 + (2 * m + 1) * G::RS) = hi.v;
    }
}

// One reversed sweep for the thread's half line of ONE group (orientation AX); the coefficients
// are in registers and serve all groups of the block.
//   gt: tile with the adjoint of the sweep output -> adjoint of the sweep input
//       w_k = g_k + e_{k-1} w_{k-1};  the far half's closing cell also takes e w of the near half's last cell
//       lambda_{H-1} = inv w (far) | inv (w + r lambda of the closing cell) (near)
//       lambda_k = inv_k (w_k + r_{k+1} lambda_{k+1})
//   xt: tile with the sweep OUTPUT -> (if rebuilt) the sweep INPUT x_in = (1 + eps) x - r (L x);
//       the state is streamed through a window of two cell pairs, results leave as soon as they exist
//   vacc_k += lambda_k (L x)_k summed over the two samples
template <int N, int P, int AX>
__device__ __forceinline__ void reverse_core(float *gt, float *xt, const Lane &t, float (&vacc)[16],
                                             const float (&r)[4 * SG<N, P>::HQ], const float (&iv)[4 * SG<N, P>::HQ],
                                             float onepe, bool far, bool rebuild) {
    using G = SG<N, P>;
    constexpr int H = N / 2, HCH = G::HCH;
    f2 g[H];
    ld_half<N, P, AX>(gt, t, g);
    f2 c_lo, c_hi, n_lo, n_hi;
    ld_duo<N, P, AX>(xt, t, HCH - 1, c_lo, c_hi);
    if (HCH >= 2) ld_duo<N, P, AX>(xt, t, HCH - 2, n_lo, n_hi);
    // e_k = r_k / pivot_k is rebuilt as r_k * inv_k (scalar, off the dependent chain) instead of
    // being loaded: a third less coefficient traffic and 16 registers less
#pragma unroll
    for (int k = 1; k < H; ++k) g[k] = f2_fmas(r[k - 1] * iv[k - 1], g[k - 1], g[k]);
    {
        const f2 z = shfl_xor_f2(f2_muls(r[H - 1] * iv[H - 1], g[H - 1]), P);
        g[H - 1] = f2_fmas(far ? 1.0f : 0.0f, z, g[H - 1]);
    }
    f2 lam = f2_muls(iv[H - 1], g[H - 1]);
    {
        const f2 z = shfl_xor_f2(f2_muls(r[H - 1], lam), P);
        lam = f2_fmas(far ? 0.0f : iv[H - 1], z, lam);
    }
    f2 xnext = shfl_xor_f2(c_hi, P);   // the cell across the junction (sweep output)
    const bool wr = rebuild && t.active;
#pragma unroll
    for (int m = HCH - 1; m >= 0; --m) {
        const int k1 = 2 * m + 1, k0 = 2 * m;
        // cell k1
        if (k1 < H - 1) lam = f2_fmas(r[k1 + 1] * iv[k1], lam, f2_muls(iv[k1], g[k1]));
        const f2 lam1 = lam;
        f2 lx = f2_fmas(-2.0f, c_hi, f2_add(c_lo, xnext));
        vacc[k1] += f2_hsum(f2_mul(lam, lx));
        const f2 o_hi = f2_fmas(-r[k1], lx, f2_muls(onepe, c_hi));
        xnext = c_hi;
        // cell k0
        lam = f2_fmas(r[k0 + 1] * iv[k0], lam, f2_muls(iv[k0], g[k0]));
        lx = (m == 0) ? f2_sub(xnext, c_lo) : f2_fmas(-2.0f, c_lo, f2_add(n_hi, xnext));
        vacc[k0] += f2_hsum(f2_mul(lam, lx));
        const f2 o_lo = f2_fmas(-r[k0], lx, f2_muls(onepe, c_lo));
        xnext = c_lo;
        if (t.active) st_duo<N, P, AX>(gt, t, m, lam, lam1);
        if (wr) st_duo<N, P, AX>(xt, t, m, o_lo, o_hi);
        c_lo = n_lo;
        c_hi = n_hi;
        if (m >= 2) ld_duo<N, P, AX>(xt, t, m - 2, n_lo, n_hi);
    }
}

// The smoothing adjoint along a half line: v_k <- (v_{k-1} + v_k + v_{k+1}) / 3, with the replicate
// padding's end taps put back on the edge cell (k = 0) and the neighbour across the junction
// (k = H-1) fetched from the other half.
template <int N, int P>
__device__ __forceinline__ void smooth_adjoint(float (&v)[16]) {
    constexpr int H = N / 2;
    const float third = 1.0f / 3.0f;
    const float vj = __shfl_xor_sync(kFullMask, v[H - 1], P);
    float lo = v[0];
#pragma unroll
    for (int k = 0; k < H; ++k) {
        const float cur = v[k];
        const float hi = (k == H - 1) ? vj : v[k + 1];
        v[k] = ((lo + cur) + hi) * third;
        lo = cur;
    }
}

// v (summed over the block's groups) -> smoothing^T -> clamp mask -> x dt/h^2 -> TMEM accumulators.
// When no sweep of the call has a clamped cell, the mask is all ones and the (linear) smoothing
// adjoint commutes with the sums over sweeps and samples: it is then applied once, to the
// accumulators, when the kernel ends (`smooth_now` false).
template <int N, int P>
__device__ __forceinline__ void reverse_finish(float (&v)[16], uint32_t tacc, const float4 *tm, float scale, float tt,
                                               bool smooth_now, bool clamped) {
    using G = SG<N, P>;
    constexpr int H = G::H;
    if (smooth_now) smooth_adjoint<N, P>(v);
    if (clamped) {
        float m[4 * G::HQ];
        ld_coef<N, P>(tm, m);
#pragma unroll
        for (int k = 0; k < H; ++k) v[k] *= m[k];
    }
    tmem_accumulate16(tacc, v, scale, tt * scale);
}

// Adjoint of a channel op on one group.  On entry (after a barrier) the g tiles hold the adjoint of
// the op's output as rows, the x tiles the op's INPUT:
//   gm[dd] += sum g_c x_dd ;  g_c <- sum_c' mat[c'][c] g_c'.
template <int N, int P>
__device__ __forceinline__ void chan_adjoint(float *ggt, const float *gxt, int cstride, int C,
                                             const float *__restrict__ mat, const Lane &t,
                                             float (&gm)[PDE_MAX_CHANNELS]) {
    using G = SG<N, P>;
    constexpr int H = G::H;
    {
        f2 g[H];
        ld_half<N, P, 0>(ggt + (size_t)t.c * cstride, t, g);
        for (int dd = 0; dd < C; ++dd) {
            f2 x[H];
            ld_half<N, P, 0>(gxt + (size_t)dd * cstride, t, x);
            f2 acc = f2_bc(0.0f);
#pragma unroll
            for (int k = 0; k < H; ++k) acc = f2_fma(g[k], x[k], acc);
            if (t.active) gm[dd] += f2_hsum(acc);
        }
    }
    f2 gn[H];
    mix_rows<N, P>(ggt, cstride, C, mat + t.c, C, t, gn);
    __syncthreads();
    if (t.active) st_half<N, P, 0>(ggt + (size_t)t.c * cstride, t, gn);
}

// Backward kernel.  One group of P sample pairs (all channels) per block iteration; both tile sets
// are double buffered and filled asynchronously one stage ahead:
//   x tiles: TMA bulk copies of the checkpoints (the forward kernel wrote them as tile images),
//            stream (item, last step) ... (item, step 0), (next item, last step) ...
//   g tiles: the next item's gout planes by TMA bulk copies while the current item is reversed.
template <int N, int P, bool CHAN>
__device__ __forceinline__ void sbwd_body(const Args &a, const int bid, const int nblk) {
    using G = SG<N, P>;
    constexpr int H = G::H, TILE = G::TILE, SLOT = G::SLOT, NPI = G::NPITCH, XPI = G::XPITCH, HQ4 = 4 * G::HQ;
    // the channel ops read x and g tile sets with one channel stride
    static_assert(!CHAN || SLOT == TILE, "channel ops need tiles and g slots of one size");
    extern __shared__ __align__(128) float smem[];
    __shared__ uint32_t tmem_slot;
    __shared__ __align__(8) uint64_t xbar[2];
    __shared__ __align__(8) uint64_t gbar[2];
    const pde_adi_desc &d = a.d;
    const Lane t = make_lane<N, P>();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int C = d.C, nthr = blockDim.x;
    const bool far = t.h == 1;
    const int CS = TILE;                 // channel stride inside an x tile set (a checkpoint image)
    const int SET = C * TILE;            // floats per x tile set
    const int GSET = C * SLOT;           // floats per g set (channel stride SLOT)
    // four pairs: second g set, the next item's gout arrives while this one is reversed; plane I/O by bulk
    // copies (see PlaneIO)
    constexpr bool GDB = P >= 4;
    // tile sets by offset from the one shared-memory base (pointer arrays indexed at run time would
    // end up in local memory and turn every tile access into a generic load)
    auto xset = [&](int b) { return smem + b * SET; };
    auto gset = [&](int b) { return smem + 2 * SET + (GDB ? b : 0) * GSET; };
    // coefficient stage: r and 1/pivot of one sweep (all channels), double buffered, filled by TMA
    // one sweep ahead -- the tables do not survive in what is left of L1 beside the tiles
    const int CT = C * G::HQ * N * 2 * 4;   // floats per table per sweep
    float *cbuf = smem + 2 * SET + (GDB ? 2 : 1) * GSET;
    __shared__ __align__(8) uint64_t cbar[2];

    if (warp == 0) tmem_alloc(&tmem_slot, (uint32_t)a.tmem_cols);
    if (threadIdx.x == 0) {
        mbar_init(&xbar[0], 1);
        mbar_init(&xbar[1], 1);
        mbar_init(&gbar[0], 1);
        mbar_init(&gbar[1], 1);
        mbar_init(&cbar[0], 1);
        mbar_init(&cbar[1], 1);
        mbar_fence_init();
    }
    const Header *hdr = reinterpret_cast<const Header *>(a.tables);
    tmem_fence_before_sync();
    __syncthreads();
    tmem_fence_after_sync();
    const uint32_t tbase = tmem_slot + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)((warp >> 2) * 64);
    {
        float z[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) z[i] = 0.0f;
#pragma unroll
        for (int col = 0; col < 64; col += 16) tmem_st16(tbase + col, z);
        tmem_wait_st();
    }
    const bool exact = a.ck_flags->mode_exact != 0;
    const size_t T = stab_floats_per_table(d);
    const float4 *tab_r = reinterpret_cast<const float4 *>(a.stab);
    const float4 *tab_inv = reinterpret_cast<const float4 *>(a.stab + T);
    const float4 *tab_e = reinterpret_cast<const float4 *>(a.stab + 2 * T);
    const float4 *tab_m = reinterpret_cast<const float4 *>(a.stab + 3 * T);
    const size_t plane = (size_t)N * N;
    const size_t ck_step = (size_t)SET;   // floats per (group, step): a tile image per channel
    float sig = 0.0f;
    if (d.skip) sig = 1.0f / (1.0f + expf(-__ldg(a.skipw)));
    const float om = 1.0f - sig;
    const float onepe = 1.0f + d.eps;
    const bool smooth = d.smooth != 0;
    const bool defer_smooth = smooth && a.ck_flags->any_clamped == 0;   // see reverse_finish
    float gm[PDE_MAX_CHANNELS] = {0.f, 0.f, 0.f, 0.f};
    float gw = 0.0f;
    const int sps = a.sps;
    const int last_ax = (sps == 3) ? 0 : 1;
    // exact mode: outputs of the first sps-1 sweeps of the step being reversed, per block
    const size_t scr_slot = (size_t)H * nthr;
    unsigned long long *sweep_scr =
        reinterpret_cast<unsigned long long *>(a.scratch) + (size_t)bid * 2 * scr_slot + threadIdx.x;
    // the layer input is needed in the spare x buffer at step 0 (pre-step mix adjoint, exact
    // recomputation): the first checkpoint of the next item then waits for the end of the item
    const bool defer_cross = exact || (CHAN && d.chan_op == 1);

    // ---- asynchronous x stream
    uint32_t xphase = 0u;      // bit b: parity the next wait on buffer b expects
    uint32_t xpending = 0u;    // bit b: a fill of buffer b has not been waited for yet
    auto x_fill = [&](int b, int item, int step) {   // call after a barrier that ends every use of buffer b
        if (threadIdx.x == 0) {
            fence_proxy_async();
            const uint32_t bytes = (uint32_t)(SET * sizeof(float));
            mbar_expect_tx(&xbar[b], bytes);
            tma_load_1d(xset(b), a.ckpt + ((size_t)item * d.steps + step) * ck_step, bytes, &xbar[b]);
        }
        xpending |= 1u << b;
    };
    auto x_wait = [&](int b) {
        if (xpending & (1u << b)) {
            mbar_wait(&xbar[b], (xphase >> b) & 1u);
            xphase ^= 1u << b;
            xpending &= ~(1u << b);
        }
    };
    uint32_t cphase = 0u;
    auto c_fill = [&](int b, int s) {   // call after a barrier that ends every read of buffer b
        if (threadIdx.x == 0) {
            fence_proxy_async();
            const uint32_t bytes = (uint32_t)(CT * sizeof(float));
            mbar_expect_tx(&cbar[b], 2 * bytes);
            tma_load_1d(cbuf + (size_t)(2 * b) * CT, a.stab + (size_t)s * CT, bytes, &cbar[b]);
            tma_load_1d(cbuf + (size_t)(2 * b + 1) * CT, a.stab + T + (size_t)s * CT, bytes, &cbar[b]);
        }
    };
    // the layer input of group `it`, natural layout (pitch XPI), into x set b: exact recomputation and
    // the pre-step mix adjoint need it at step 0
    auto u_xfill = [&](int b, int it) {   // call after a barrier that ends every use of buffer b
        if (threadIdx.x == 0) {
            fence_proxy_async();
            mbar_expect_tx(&xbar[b], (uint32_t)(group_valid<N, P>(it, d.B) * C * plane * sizeof(float)));
            planes_load<N, P>(xset(b), CS, XPI, a.u, it, C, d.B, &xbar[b]);
        }
        xpending |= 1u << b;
    };
    auto u_xrows = [&](int b, int it) {   // after x_wait(b): the layer input as rows of x set b
        const int nv = group_valid<N, P>(it, d.B);
        if (nv < 2 * P) zero_tail<N, P>(xset(b), CS, XPI, C, nv);
        __syncthreads();
        planes_to_rows<N, P, XPI>(xset(b) + (size_t)t.c * CS, t);
        __syncthreads();
    };
    // gout planes of group `it` -> g set b, natural layout; the slot's previous grad_input store must
    // have been read out first
    uint32_t gphase = 0u;
    auto g_fill = [&](int b, int it) {   // call after a barrier that ends every use of set b
        if (threadIdx.x == 0) {
            bulk_wait_read<0>();
            fence_proxy_async();
            mbar_expect_tx(&gbar[b], (uint32_t)(group_valid<N, P>(it, d.B) * C * plane * sizeof(float)));
            planes_load<N, P>(gset(b), SLOT, NPI, a.gout, it, C, d.B, &gbar[b]);
        }
    };
    int xb = 0, gb = 0, cb = 0;
    if (bid < a.nitems) {
        x_fill(0, bid, d.steps - 1);
        c_fill(0, a.S - 1);
        if (GDB) g_fill(0, bid);
    }

    for (int item = bid; item < a.nitems; item += nblk) {
        const int next_item = item + nblk;
        float *ggt = gset(gb), *gt = ggt + (size_t)t.c * SLOT;
        __syncthreads();   // the previous item's grad_input has been written; nobody reads the other g set
        if (GDB) {
            if (next_item < a.nitems) g_fill(gb ^ 1, next_item);
            const int nv = group_valid<N, P>(item, d.B);
            if (nv < 2 * P) zero_tail<N, P>(ggt, SLOT, NPI, C, nv);
            mbar_wait(&gbar[gb], (gphase >> gb) & 1u);
            gphase ^= 1u << gb;
            __syncthreads();
            planes_to_rows<N, P, NPI>(gt, t);
        } else {
            PlaneIO<N, P>::to_tile(a.gout, gt, item, t.c, C, d.B, t.tid_c);
            __syncthreads();
        }
        // Which orientation last touched a tile set, and whether a barrier has passed since: a thread
        // only reads and writes its own half line within one orientation, so a barrier is needed
        // exactly when the orientation changes (2 = block-wide access pattern).
        int x_last = 2, g_last = GDB ? 0 : 2;
        bool x_sync = true, g_sync = !GDB;
        auto bar = [&]() {
            __syncthreads();
            x_sync = true;
            g_sync = true;
        };
        auto touch_x = [&](int o) {
            if ((x_last != o || o == 2) && !x_sync) bar();
            x_last = o;
            x_sync = false;
        };
        auto touch_g = [&](int o) {
            if ((g_last != o || o == 2) && !g_sync) bar();
            g_last = o;
            g_sync = false;
        };
        auto adjoint_chan = [&](const float *gx) {   // gx: tile set with the op's input (read only)
            touch_g(2);
            bar();
            chan_adjoint<N, P>(ggt, gx, CS, C, a.chan, t, gm);
            g_last = 0;
            g_sync = false;
        };

        if (d.skip) {
            // out = sig u0 + om uF:  dL/dw += sig' * sum gout (u0 - uF),  g <- om * gout
            x_wait(xb);
            f2 uf[H], gl[H];
            if (d.chan_op == 2) mix_rows<N, P>(xset(xb), CS, C, a.chan + t.c * C, 1, t, uf);   // uF = K (last state)
            else ld_half<N, P, 0>(xset(xb) + (size_t)t.c * CS, t, uf);
            touch_g(0);
            ld_half<N, P, 0>(gt, t, gl);
            if (t.active) {
                f2 accw = f2_bc(0.0f);
                const int i = mirror(t.R, N);
                const float2 zero2 = make_float2(0.f, 0.f);
                const int ba = (item * P + t.pp) * 2, bb = ba + 1;
#pragma unroll
                for (int m = 0; m < G::HCH; ++m) {
                    // cells k = 2m, 2m+1 of the half row: columns 2m, 2m+1 (near) or N-1-2m, N-2-2m (far)
                    const int j0 = t.h ? N - 2 - 2 * m : 2 * m;
                    const float2 wa = ba < d.B ? __ldg(reinterpret_cast<const float2 *>(a.u + ((size_t)ba * C + t.c) * plane + (size_t)i * N + j0)) : zero2;
                    const float2 wb = bb < d.B ? __ldg(reinterpret_cast<const float2 *>(a.u + ((size_t)bb * C + t.c) * plane + (size_t)i * N + j0)) : zero2;
                    const f2 u0 = t.h ? f2_make(wa.y, wb.y) : f2_make(wa.x, wb.x);
                    const f2 u1 = t.h ? f2_make(wa.x, wb.x) : f2_make(wa.y, wb.y);
                    accw = f2_fma(gl[2 * m], f2_sub(u0, uf[2 * m]), accw);
                    accw = f2_fma(gl[2 * m + 1], f2_sub(u1, uf[2 * m + 1]), accw);
                    gl[2 * m] = f2_muls(om, gl[2 * m]);
                    gl[2 * m + 1] = f2_muls(om, gl[2 * m + 1]);
                }
                st_half<N, P, 0>(gt, t, gl);
                gw += f2_hsum(accw);
            }
            x_last = 0;   // rows of the x set were read (all channels if coupled)
            x_sync = false;
        }

        for (int step = d.steps - 1; step >= 0; --step) {
            float *gxt = xset(xb), *xt = gxt + (size_t)t.c * CS;       // state after the last sweep of `step`
            float *gxs = xset(xb ^ 1), *xs = gxs + (size_t)t.c * CS;   // spare: the stage ahead
            // every use of the spare buffer (previous step) ends here; start the stage ahead
            bar();
            if (step > 0) x_fill(xb ^ 1, item, step - 1);
            else if (GDB && defer_cross) u_xfill(xb ^ 1, item);
            else if (!defer_cross && next_item < a.nitems) x_fill(xb ^ 1, next_item, d.steps - 1);
            x_wait(xb);
            if (exact) {
                // recompute the sweeps of this step from its input (spare buffer), keeping every sweep output
                f2 x[1][H];
                if (GDB || step > 0) x_wait(xb ^ 1);
                if (GDB && step == 0) u_xrows(xb ^ 1, item);
                if (!GDB && step == 0) {
                    PlaneIO<N, P>::to_tile(a.u, xs, item, t.c, C, d.B, t.tid_c);
                    __syncthreads();
                }
                if (CHAN && (d.chan_op == 1 || (d.chan_op == 2 && step > 0))) {
                    mix_rows<N, P>(gxs, CS, C, a.chan + t.c * C, 1, t, x[0]);
                    __syncthreads();   // every thread has read the spare set before it is used as scratch
                } else if (step > 0 && last_ax == 1) {
                    ld_half<N, P, 0>(xs, t, x[0]);
                    __syncthreads();
                } else {
                    ld_half<N, P, 0>(xs, t, x[0]);
                }
                for (int k = 0; k + 1 < sps; ++k) {
                    const int s = step * sps + k;
                    float iv[HQ4], e[HQ4];
                    ld_coef<N, P>(tab_inv + tab_off<N, P>(s, C, t), iv);
                    ld_coef<N, P>(tab_e + tab_off<N, P>(s, C, t), e);
                    if (k == 1) {
                        if (t.active) st_half<N, P, 0>(xs, t, x[0]);
                        __syncthreads();
                        ld_half<N, P, 1>(xs, t, x[0]);
                    }
                    solve<N, P, 1>(x, iv, e, far);
#pragma unroll
                    for (int kk = 0; kk < H; ++kk) __stcg(sweep_scr + ((size_t)k * H + kk) * nthr, x[0][kk].v);
                }
                __syncthreads();
                if (step > 0) x_fill(xb ^ 1, item, step - 1);   // the spare buffer was used as scratch
                x_last = 2;
                x_sync = true;
            }
            // adjoint of the post-step coupling: its input is the state after the last sweep
            if (CHAN && d.chan_op == 2) {
                adjoint_chan(gxt);
                x_last = 0;
                x_sync = false;
            }
            for (int k = sps - 1; k >= 0; --k) {
                const int s = step * sps + k, ax = sweep_axis(k);
                const size_t o = tab_off<N, P>(s, C, t);
                // per-sweep scalars straight from the header (shared memory is full)
                const float sw_scale = __ldg(&hdr->scale[s]), sw_t = __ldg(&hdr->t[s]);
                const bool sw_clamped = __ldg(&hdr->clamped[s]) != 0;
                // every thread has its registers loaded from the other coefficient buffer (previous sweep)
                bar();
                {
                    const int ns = s > 0 ? s - 1 : (next_item < a.nitems ? a.S - 1 : -1);
                    if (ns >= 0) c_fill(cb ^ 1, ns);
                }
                mbar_wait(&cbar[cb], (cphase >> cb) & 1u);
                cphase ^= 1u << cb;
                float r[HQ4], iv[HQ4];
                {
                    const float4 *cr = reinterpret_cast<const float4 *>(cbuf + (size_t)(2 * cb) * CT) + t.tab;
                    const float4 *ci = reinterpret_cast<const float4 *>(cbuf + (size_t)(2 * cb + 1) * CT) + t.tab;
#pragma unroll
                    for (int q = 0; q < G::HQ; ++q) {
                        const float4 a4 = cr[q * G::QS], b4 = ci[q * G::QS];
                        r[4 * q] = a4.x; r[4 * q + 1] = a4.y; r[4 * q + 2] = a4.z; r[4 * q + 3] = a4.w;
                        iv[4 * q] = b4.x; iv[4 * q + 1] = b4.y; iv[4 * q + 2] = b4.z; iv[4 * q + 3] = b4.w;
                    }
                }
                cb ^= 1;
                const bool rebuild = !exact && k > 0;
                touch_g(ax);
                touch_x(ax);
                float vacc[16];
#pragma unroll
                for (int kk = 0; kk < 16; ++kk) vacc[kk] = 0.0f;
                if (exact && k != sps - 1) {   // this sweep's output comes back from the block's scratch
                    f2 x[H];
#pragma unroll
                    for (int kk = 0; kk < H; ++kk) x[kk].v = __ldcg(sweep_scr + ((size_t)k * H + kk) * nthr);
                    if (t.active) {
                        if (ax == 0) st_half<N, P, 0>(xt, t, x);
                        else st_half<N, P, 1>(xt, t, x);
                    }
                }
                if (ax == 0) reverse_core<N, P, 0>(gt, xt, t, vacc, r, iv, onepe, far, rebuild);
                else reverse_core<N, P, 1>(gt, xt, t, vacc, r, iv, onepe, far, rebuild);
                reverse_finish<N, P>(vacc, tbase + (ax ? 32u : 0u), tab_m + o, sw_scale, sw_t, smooth && !defer_smooth, sw_clamped);
            }
            if (CHAN && d.chan_op == 1) {
                // adjoint of the pre-step mix: needs g (rows) and the mix INPUT = state before this step
                // (two pairs per group only: CHAN is never instantiated with four)
                if (step > 0) {
                    x_wait(xb ^ 1);
                } else {
                    bar();
                    PlaneIO<N, P>::to_tile(a.u, xs, item, t.c, C, d.B, t.tid_c);
                }
                adjoint_chan(gxs);
            }
            xb ^= 1;
        }
        if (!GDB) {
            touch_g(2);
            if (a.need_gin)
                PlaneIO<N, P>::from_tile(gt, a.gin, item, t.c, C, d.B, t.tid_c, d.skip ? a.gout : nullptr, sig, 1.0f);
        } else if (a.need_gin) {   // the g rows -> natural layout (+ skip blend) -> bulk stores
            touch_g(0);
            f2 x[H];
            ld_half<N, P, 0>(gt, t, x);
            __syncthreads();   // every thread has read its rows of the g set
            if (t.active) nat_st_half<N, P, NPI>(gt, t, x, d.skip ? a.gout : nullptr, item, t.c, C, d.B, sig, 1.0f);
            fence_proxy_async();
            __syncthreads();
            if (threadIdx.x == 0) planes_store<N, P>(a.gin, ggt, SLOT, NPI, item, C, d.B);
        }
        if (defer_cross && next_item < a.nitems) {
            __syncthreads();   // the layer input in the spare buffer has been consumed
            x_fill(xb, next_item, d.steps - 1);
        }
        if (GDB) gb ^= 1;
    }

    if (GDB && threadIdx.x == 0) bulk_wait_all();   // the grad_input stores are complete before the block ends

    // ------------------------------ partials: TMEM -> sum over the P pairs -> global [row][col]
    tmem_wait_st();
    float *pm = a.part_maps + ((size_t)bid * C + t.c) * 4 * plane;
    const int L = mirror(t.R, N);   // the line's position in the plane
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
        float av[16];
        tmem_ld16(tbase + kk * 16, av);
        tmem_wait_ld();
        if (defer_smooth) smooth_adjoint<N, P>(av);
#pragma unroll
        for (int o = 1; o < P; o <<= 1)
#pragma unroll
            for (int k = 0; k < H; ++k) av[k] += __shfl_xor_sync(kFullMask, av[k], o);
        if (t.active && t.pp == 0) {
#pragma unroll
            for (int k = 0; k < H; ++k) {
                const int along = t.h ? N - 1 - k : k;
                const size_t cell = kk < 2 ? (size_t)L * N + along : (size_t)along * N + L;
                pm[kk * plane + cell] = av[k];
            }
        }
    }
    const size_t set = ((size_t)bid * G::WPC + t.wi) * C + t.c;
#pragma unroll
    for (int dd = 0; dd < PDE_MAX_CHANNELS; ++dd) {
        const float sgm = warp_sum(gm[dd]);
        if (lane == 0) a.part_chan[set * PDE_MAX_CHANNELS + dd] = sgm;
    }
    const float sgw = warp_sum(gw);
    if (lane == 0) a.part_skip[set] = sgw;
    tmem_fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_slot, (uint32_t)a.tmem_cols);
}

template <int N, int P, bool CHAN>
__global__ void __launch_bounds__(max_threads<N, P>(), P >= 4 ? 2 : 1) sbwd_kernel(const Args a) {
    sbwd_body<N, P, CHAN>(a, blockIdx.x, gridDim.x);
}

template <int N, int P, bool CHAN>
__global__ void __launch_bounds__(max_threads<N, P>(), P >= 4 ? 2 : 1) sbwd_multi_kernel(const __grid_constant__ MultiArgs m) {
    int bid, nblk;
    const int b = multi_branch_of(m, &bid, &nblk);
    sbwd_body<N, P, CHAN>(m.a[b], bid, nblk);
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
bool supported(const pde_adi_desc &d) {
    if (tune_impl(d) == PDE_ADI_TUNE_IMPL_WHOLE_LINE) return false;
    if (d.steps < 1 || d.B < 1 || d.C > 3) return false;
    if (d.N != 28 && d.N != 32) return false;
    // Training calls on 28 x 28 / 32 x 32 planes take the half-line kernels at every batch size: at the
    // reference's own batches (64 ... 512) a call is latency bound, and half the dependent chain per
    // thread plus TMA-staged coefficients is what shortens it (measured, kernels only: fashion B 256
    // 64 -> 43 us, mnist B 64 111 -> 68 us, cifar10 pde2 B 512 196 -> 170 us, svhn B 256 212 -> 162 us).
    DeviceProps props;
    return query_props(&props) == PDE_OK;
}

size_t table_floats(const pde_adi_desc &d) { return 4 * stab_floats_per_table(d); }

constexpr int kMaxQ = 4;

struct Plan {
    int P, Qf, Qb, threads, wpc, ngroups, tmem_cols;
    size_t tile_bytes, slot_bytes, scr_slot;   // one tile (P pairs of one channel); one tile slot (SG::SLOT); f2 per
                                               // sweep output of a block (exact mode)
};

template <int N, int P>
static void fill_geo(const pde_adi_desc &d, Plan *p) {
    using G = SG<N, P>;
    p->wpc = G::WPC;
    p->threads = G::WPC * 32 * d.C;
    p->tile_bytes = (size_t)G::TILE * sizeof(float);
    p->slot_bytes = (size_t)G::SLOT * sizeof(float);
    p->scr_slot = (size_t)G::H * p->threads;
}

static int make_plan(const pde_adi_desc &d, Plan *p) {
    DeviceProps props;
    int rc = query_props(&props);
    if (rc) return rc;
    const int sm = props.sm_count;
    // pairs per group: 4 for the single-channel layers once the batch fills the GPU with such groups
    p->P = 2;
    if (d.C == 1 && d.chan_op == 0) {
        const int forced = tune_p(d);
        if (forced == 4 || (forced != 2 && (d.B + 7) / 8 >= 2 * sm)) p->P = 4;
    }
    if (d.N == 28) { if (p->P == 4) fill_geo<28, 4>(d, p); else fill_geo<28, 2>(d, p); }
    else if (d.N == 32) { if (p->P == 4) fill_geo<32, 4>(d, p); else fill_geo<32, 2>(d, p); }
    else return PDE_ERR_UNSUPPORTED;
    p->ngroups = (d.B + 2 * p->P - 1) / (2 * p->P);
    // groups per forward block: as many as still leave two blocks of work per SM and fit the shared memory
    // the block may take.  The registers decide how many blocks an SM holds (128 per thread, two blocks, for
    // four pairs per group; ~168 per thread for two pairs: three blocks of 128 threads, one block of 256 or 384),
    // the tiles get what is left of 227 KB per block beside the two coefficient stages.  For the three-channel
    // layers that admits two groups (111 KB of tiles; measured at batch 65536: cifar10 pde1 forward 2.49 ->
    // 2.19 ms, pde2 3.83 -> 3.33, cifar_2version 2.98 -> 2.62, SVHN 5.05 -> 4.67).
    const size_t coef_stage = (size_t)4 * d.C * ((d.N / 2 + 3) / 4) * d.N * 2 * 16;
    const int blocks_per_sm = p->threads <= 128 ? 3 : 1;   // two pairs per group
    const size_t tile_budget = p->P == 4 ? (size_t)101 * 1024   // two blocks: 4 x 25 KB tiles + 14 KB of coefficients each
                                         : (size_t)227 * 1024 / blocks_per_sm - coef_stage - 2048;
    auto pick = [&](int qmax, size_t tiles_per_group, int forced) {
        int q = qmax;
        while (q > 1 && ((p->ngroups + q - 1) / q < 2 * sm || (size_t)q * tiles_per_group * p->slot_bytes > tile_budget)) q >>= 1;
        if (forced == 1 || forced == 2 || (forced == 4 && qmax == 4)) q = forced;
        return q;
    };
    p->Qf = pick(p->P == 4 ? 4 : 2, (size_t)d.C, tune_qf(d));
    p->Qb = 1;   // measured: the backward kernel gains nothing from sharing coefficient loads
    const int warps = p->threads / 32;
    const int blocks4 = (warps + 3) / 4;
    p->tmem_cols = blocks4 * 64 <= 64 ? 64 : (blocks4 * 64 <= 128 ? 128 : (blocks4 * 64 <= 256 ? 256 : 512));
    return PDE_OK;
}

size_t checkpoint_bytes(const pde_adi_desc &d) {
    Plan p;
    if (!supported(d) || make_plan(d, &p) != PDE_OK) return 0;
    // one tile image per (group, step, channel)
    const size_t groups = (size_t)((p.ngroups + kMaxQ - 1) / kMaxQ) * kMaxQ;
    return groups * d.steps * d.C * p.tile_bytes + 256 + kCkHeaderFloats * sizeof(float);
}

template <int N>
static const void *bwd_kernel_n(int P, bool chan) {
    if (P == 4) return reinterpret_cast<const void *>(sbwd_kernel<N, 4, false>);
    return chan ? reinterpret_cast<const void *>(sbwd_kernel<N, 2, true>)
                : reinterpret_cast<const void *>(sbwd_kernel<N, 2, false>);
}
static const void *bwd_kernel_for(int N, int P, bool chan) {
    if (N == 28) return bwd_kernel_n<28>(P, chan);
    if (N == 32) return bwd_kernel_n<32>(P, chan);
    return nullptr;
}
template <int N>
static const void *fwd_kernel_n(int P, int Q, bool mix1) {
    if (P == 4)
        return Q == 4 ? reinterpret_cast<const void *>(sfwd_kernel<N, 4, 4, false>)
                      : (Q == 2 ? reinterpret_cast<const void *>(sfwd_kernel<N, 4, 2, false>)
                                : reinterpret_cast<const void *>(sfwd_kernel<N, 4, 1, false>));
    if (mix1)
        return Q == 2 ? reinterpret_cast<const void *>(sfwd_kernel<N, 2, 2, true>)
                      : reinterpret_cast<const void *>(sfwd_kernel<N, 2, 1, true>);
    return Q == 2 ? reinterpret_cast<const void *>(sfwd_kernel<N, 2, 2, false>)
                  : reinterpret_cast<const void *>(sfwd_kernel<N, 2, 1, false>);
}
static const void *fwd_kernel_for(int N, int P, int Q, bool mix1) {
    if (N == 28) return fwd_kernel_n<28>(P, Q, mix1);
    if (N == 32) return fwd_kernel_n<32>(P, Q, mix1);
    return nullptr;
}

// the multi-branch kernels exist for the two-pairs-per-group geometry (the multi-branch models of the
// reference are three-channel: cifar10.py:253-258, cifar_2version.py:269-270)
template <int N>
static const void *fwd_multi_kernel_n(int Q, bool mix1) {
    if (mix1)
        return Q == 2 ? reinterpret_cast<const void *>(sfwd_multi_kernel<N, 2, 2, true>)
                      : reinterpret_cast<const void *>(sfwd_multi_kernel<N, 2, 1, true>);
    return Q == 2 ? reinterpret_cast<const void *>(sfwd_multi_kernel<N, 2, 2, false>)
                  : reinterpret_cast<const void *>(sfwd_multi_kernel<N, 2, 1, false>);
}
static const void *fwd_multi_kernel_for(int N, int P, int Q, bool mix1) {
    if (P != 2 || (Q != 1 && Q != 2)) return nullptr;
    if (N == 28) return fwd_multi_kernel_n<28>(Q, mix1);
    if (N == 32) return fwd_multi_kernel_n<32>(Q, mix1);
    return nullptr;
}
static const void *bwd_multi_kernel_for(int N, int P, bool chan) {
    if (P != 2) return nullptr;
    if (N == 28)
        return chan ? reinterpret_cast<const void *>(sbwd_multi_kernel<28, 2, true>)
                    : reinterpret_cast<const void *>(sbwd_multi_kernel<28, 2, false>);
    if (N == 32)
        return chan ? reinterpret_cast<const void *>(sbwd_multi_kernel<32, 2, true>)
                    : reinterpret_cast<const void *>(sbwd_multi_kernel<32, 2, false>);
    return nullptr;
}

struct BwdLaunch {
    int grid, nitems, occ;
    size_t smem;
};

static int plan_bwd_grid(const pde_adi_desc &d, const Plan &p, BwdLaunch *b, const void *kern_override = nullptr) {
    DeviceProps props;
    int rc = query_props(&props);
    if (rc) return rc;
    const void *kern = kern_override ? kern_override : bwd_kernel_for(d.N, p.P, d.chan_op != 0);
    if (!kern) return PDE_ERR_UNSUPPORTED;
    // x tile sets double buffered, g sets (tile slots) too for P == 4, two coefficient stages of two tables
    b->smem = (size_t)2 * d.C * p.tile_bytes + (size_t)(p.P >= 4 ? 2 : 1) * d.C * p.slot_bytes + (size_t)4 * d.C * ((d.N / 2 + 3) / 4) * d.N * 2 * 16;
    if (b->smem > (size_t)props.max_smem_optin) return PDE_ERR_UNSUPPORTED;
    // residency from first principles (the occupancy calculator answers 1 block / SM for kernels
    // that allocate tensor memory)
    KernelInfo fa;
    rc = kernel_info(kern, b->smem, &fa);
    if (rc) return rc;
    // registers: 16 K per scheduler, a block's warps dealt round-robin over the four schedulers
    const int warps = p.threads / 32;
    const int regs_per_warp = ((fa.regs + 7) / 8) * 8 * 32;
    int occ = 16384 / (regs_per_warp * ((warps + 3) / 4));
    const int by_smem = (int)((size_t)(228 * 1024) / (b->smem + fa.static_smem + 1024));
    const int by_threads = 2048 / p.threads;
    const int by_tmem = 512 / p.tmem_cols;
    if (by_smem < occ) occ = by_smem;
    if (by_threads < occ) occ = by_threads;
    if (by_tmem < occ) occ = by_tmem;
    if (occ < 1) occ = 1;
    b->occ = occ;
    b->nitems = p.ngroups;
    if (debug_enabled())
        fprintf(stderr, "[pde_b200] split bwd plan: N=%d C=%d P=%d threads=%d smem=%zu regs=%d occ=%d tmem=%d\n", d.N,
                d.C, p.P, p.threads, b->smem, fa.regs, occ, p.tmem_cols);
    const int cap = props.sm_count * occ;
    b->grid = b->nitems < cap ? b->nitems : cap;
    if (b->grid < 1) b->grid = 1;
    return PDE_OK;
}

struct WsLayout {
    size_t scratch_floats, maps_floats, chan_floats, skip_floats;
    int nsets_maps, nsets_small;
};

static void ws_layout(const pde_adi_desc &d, const Plan &p, int grid, WsLayout *w) {
    w->scratch_floats = (size_t)grid * 2 * p.scr_slot * 2;   // two sweep outputs per block (exact mode)
    w->nsets_maps = grid * d.C;
    w->nsets_small = grid * p.wpc * d.C;
    w->maps_floats = (size_t)w->nsets_maps * 4 * d.N * d.N;
    w->chan_floats = (size_t)w->nsets_small * PDE_MAX_CHANNELS;
    w->skip_floats = (size_t)w->nsets_small;
}

size_t workspace_bytes(const pde_adi_desc &d) {
    Plan p;
    BwdLaunch b;
    if (!supported(d) || make_plan(d, &p) != PDE_OK) return 0;
    if (plan_bwd_grid(d, p, &b) != PDE_OK) return 0;
    WsLayout w;
    ws_layout(d, p, b.grid, &w);
    return (w.scratch_floats + w.maps_floats + w.chan_floats + w.skip_floats) * sizeof(float) + 512;
}

static void fill_args(const pde_adi_desc &d, const char *tables, Args *a) {
    a->d = d;
    a->sps = sweeps_per_step(d);
    a->S = d.steps * a->sps;
    a->G = 1;
    a->tables = tables;
    a->stab = reinterpret_cast<const float *>(tables + kHeaderBytes) + 4 * table_elems(d);
}

int forward(const pde_adi_desc &d, const char *tables, const float *u, const float *chan, const float *skipw,
            float *out, float *ckpt, cudaStream_t st) {
    if (!aligned16(u) || !aligned16(out)) return PDE_ERR_UNSUPPORTED;   // planes move by bulk copies
    Plan p;
    int rc = make_plan(d, &p);
    if (rc) return rc;
    DeviceProps props;
    rc = query_props(&props);
    if (rc) return rc;
    const void *kern = fwd_kernel_for(d.N, p.P, p.Qf, d.chan_op == 1);
    if (!kern) return PDE_ERR_UNSUPPORTED;
    // Qf groups of tiles, two coefficient stages of two tables
    const size_t smem = (size_t)d.C * p.Qf * p.slot_bytes + (size_t)4 * d.C * ((d.N / 2 + 3) / 4) * d.N * 2 * 16;
    if (smem > (size_t)props.max_smem_optin) return PDE_ERR_UNSUPPORTED;
    int per_sm = 1;
    rc = cached_occupancy(kern, p.threads, smem, &per_sm);
    if (rc) return rc;
    Args a{};
    fill_args(d, tables, &a);
    a.nitems = (p.ngroups + p.Qf - 1) / p.Qf;
    a.u = u; a.chan = chan; a.skipw = skipw; a.out = out;
    if (ckpt) {   // [CkFlags, 256 bytes][tile images]
        float *base = reinterpret_cast<float *>((reinterpret_cast<uintptr_t>(ckpt) + 255u) & ~(uintptr_t)255u);
        a.ck_flags = reinterpret_cast<CkFlags *>(base);
        a.ckpt = base + kCkHeaderFloats;
    }
    const int cap = props.sm_count * per_sm;
    const int grid = a.nitems < cap ? a.nitems : cap;
    if (debug_enabled())
        fprintf(stderr, "[pde_b200] split fwd plan: N=%d C=%d P=%d Q=%d threads=%d smem=%zu occ=%d grid=%d\n", d.N, d.C, p.P,
                p.Qf, p.threads, smem, per_sm, grid);
    void *params[] = {&a};
    PDE_CUDA_TRY(cudaLaunchKernel(kern, dim3(grid), dim3(p.threads), params, smem, st));
    return cuda_last_error();
}

int backward(const pde_adi_desc &d, const char *tables, const float *u, const float *gout, const float *chan,
             const float *skipw, const float *ckpt, float *gin, float *g_ab, float *g_bb, float *g_atc, float *g_btc,
             float *g_chan, float *g_skip, void *workspace, size_t workspace_bytes_, cudaStream_t st) {
    if (!aligned16(u) || !aligned16(gout) || !aligned16(gin)) return PDE_ERR_UNSUPPORTED;   // planes move by bulk copies
    Plan p;
    BwdLaunch b;
    int rc = make_plan(d, &p);
    if (rc) return rc;
    rc = plan_bwd_grid(d, p, &b);
    if (rc) return rc;
    WsLayout w;
    ws_layout(d, p, b.grid, &w);
    const size_t need = (w.scratch_floats + w.maps_floats + w.chan_floats + w.skip_floats) * sizeof(float) + 512;
    if (!workspace || workspace_bytes_ < need || !ckpt) return PDE_ERR_WORKSPACE;
    float *ws = reinterpret_cast<float *>((reinterpret_cast<uintptr_t>(workspace) + 255u) & ~(uintptr_t)255u);
    Args a{};
    fill_args(d, tables, &a);
    a.nitems = b.nitems;
    a.need_gin = gin != nullptr;
    a.tmem_cols = p.tmem_cols;
    a.u = u; a.gout = gout; a.chan = chan; a.skipw = skipw; a.gin = gin;
    {
        float *base = const_cast<float *>(reinterpret_cast<const float *>((reinterpret_cast<uintptr_t>(ckpt) + 255u) & ~(uintptr_t)255u));
        a.ck_flags = reinterpret_cast<CkFlags *>(base);
        a.ckpt = base + kCkHeaderFloats;
    }
    a.scratch = ws;
    a.part_maps = ws + w.scratch_floats;
    a.part_chan = a.part_maps + w.maps_floats;
    a.part_skip = a.part_chan + w.chan_floats;
    const void *kern = bwd_kernel_for(d.N, p.P, d.chan_op != 0);
    void *params[] = {&a};
    PDE_CUDA_TRY(cudaLaunchKernel(kern, dim3(b.grid), dim3(p.threads), params, b.smem, st));
    rc = cuda_last_error();
    if (rc) return rc;
    launch_finish(d, w.nsets_maps, w.nsets_small, a.part_maps, a.part_chan, a.part_skip, skipw, g_ab, g_atc, g_bb, g_btc,
                  g_chan, g_skip, st);
    return cuda_last_error();
}

// ------------------------------------------------------------------------------------------
// several layers on the same input, one launch per pass
// ------------------------------------------------------------------------------------------
bool multi_compatible(int n, const pde_adi_desc *d) {
    if (n < 2 || n > PDE_MAX_BRANCHES || !d) return false;
    for (int i = 0; i < n; ++i) {
        if (!supported(d[i])) return false;
        if (d[i].B != d[0].B || d[i].C != d[0].C || d[i].N != d[0].N || d[i].chan_op != d[0].chan_op ||
            d[i].skip != d[0].skip || d[i].tuning != d[0].tuning)
            return false;
    }
    Plan p;
    if (make_plan(d[0], &p) != PDE_OK) return false;
    return fwd_multi_kernel_for(d[0].N, p.P, p.Qf, d[0].chan_op == 1) != nullptr &&
           bwd_multi_kernel_for(d[0].N, p.P, d[0].chan_op != 0) != nullptr;
}

// Deal `total` resident blocks to the branches in proportion to their work per item (sweeps, plus the
// item's load / store), at most `nitems` each; fills m->blk_begin and returns the grid size.
static int deal_blocks(int n, const pde_adi_desc *d, int total, int nitems, MultiArgs *m) {
    double w[PDE_MAX_BRANCHES], wsum = 0.0;
    for (int i = 0; i < n; ++i) {
        w[i] = d[i].steps * sweeps_per_step(d[i]) + 3.0;
        wsum += w[i];
    }
    int used = 0, nb[PDE_MAX_BRANCHES];
    for (int i = 0; i < n; ++i) {
        nb[i] = (int)(total * w[i] / wsum);
        if (nb[i] > nitems) nb[i] = nitems;
        if (nb[i] < 1) nb[i] = 1;
        used += nb[i];
    }
    for (bool grew = true; grew && used < total;) {   // hand out what rounding and the caps left over, heaviest first
        grew = false;
        int best = -1;
        for (int i = 0; i < n; ++i)
            if (nb[i] < nitems && (best < 0 || w[i] / nb[i] > w[best] / nb[best])) best = i;
        if (best >= 0) {
            ++nb[best];
            ++used;
            grew = true;
        }
    }
    m->blk_begin[0] = 0;
    for (int i = 0; i < n; ++i) m->blk_begin[i + 1] = m->blk_begin[i] + nb[i];
    return m->blk_begin[n];
}

static float *ck_images(void *ckpt, CkFlags **flags) {   // [CkFlags, 256 bytes][tile images]
    float *base = reinterpret_cast<float *>((reinterpret_cast<uintptr_t>(ckpt) + 255u) & ~(uintptr_t)255u);
    *flags = reinterpret_cast<CkFlags *>(base);
    return base + kCkHeaderFloats;
}

int forward_multi(int n, const pde_adi_desc *d, const void *const *tables, const float *u, const float *const *chan,
                  const float *const *skipw, float *const *out, void *const *ckpt, cudaStream_t st) {
    if (!aligned16(u)) return PDE_ERR_UNSUPPORTED;   // planes move by bulk copies
    for (int i = 0; i < n; ++i)
        if (!aligned16(out[i])) return PDE_ERR_UNSUPPORTED;
    Plan p;
    int rc = make_plan(d[0], &p);
    if (rc) return rc;
    DeviceProps props;
    rc = query_props(&props);
    if (rc) return rc;
    const void *kern = fwd_multi_kernel_for(d[0].N, p.P, p.Qf, d[0].chan_op == 1);
    if (!kern) return PDE_ERR_UNSUPPORTED;
    const size_t smem = (size_t)d[0].C * p.Qf * p.slot_bytes + (size_t)4 * d[0].C * ((d[0].N / 2 + 3) / 4) * d[0].N * 2 * 16;
    if (smem > (size_t)props.max_smem_optin) return PDE_ERR_UNSUPPORTED;
    int per_sm = 1;
    rc = cached_occupancy(kern, p.threads, smem, &per_sm);
    if (rc) return rc;
    MultiArgs m{};
    m.n = n;
    const int nitems = (p.ngroups + p.Qf - 1) / p.Qf;
    for (int i = 0; i < n; ++i) {
        Args &a = m.a[i];
        fill_args(d[i], static_cast<const char *>(tables[i]), &a);
        a.nitems = nitems;
        a.u = u;
        a.chan = chan ? chan[i] : nullptr;
        a.skipw = skipw ? skipw[i] : nullptr;
        a.out = out[i];
        if (ckpt && ckpt[i]) a.ckpt = ck_images(ckpt[i], &a.ck_flags);
    }
    const int grid = deal_blocks(n, d, props.sm_count * per_sm, nitems, &m);   // the branches share the resident set
    if (debug_enabled())
        fprintf(stderr, "[pde_b200] split fwd multi plan: n=%d N=%d C=%d chan_op=%d P=%d Q=%d threads=%d smem=%zu occ=%d grid=%d\n", n,
                d[0].N, d[0].C, d[0].chan_op, p.P, p.Qf, p.threads, smem, per_sm, grid);
    void *params[] = {&m};
    PDE_CUDA_TRY(cudaLaunchKernel(kern, dim3(grid), dim3(p.threads), params, smem, st));
    return cuda_last_error();
}

int backward_multi(int n, const pde_adi_desc *d, const void *const *tables, const float *u, const float *const *gout,
                   const float *const *chan, const float *const *skipw, const void *const *ckpt, float *const *gin,
                   float *const *g_ab, float *const *g_bb, float *const *g_atc, float *const *g_btc, float *const *g_chan,
                   float *const *g_skip, void *const *workspace, const size_t *workspace_bytes_, cudaStream_t st) {
    if (!aligned16(u)) return PDE_ERR_UNSUPPORTED;   // planes move by bulk copies
    for (int i = 0; i < n; ++i)
        if (!aligned16(gout[i]) || (gin && !aligned16(gin[i]))) return PDE_ERR_UNSUPPORTED;
    Plan p;
    BwdLaunch b;
    int rc = make_plan(d[0], &p);
    if (rc) return rc;
    const void *kern = bwd_multi_kernel_for(d[0].N, p.P, d[0].chan_op != 0);
    if (!kern) return PDE_ERR_UNSUPPORTED;
    rc = plan_bwd_grid(d[0], p, &b, kern);
    if (rc) return rc;
    DeviceProps props;
    rc = query_props(&props);
    if (rc) return rc;
    MultiArgs m{};
    m.n = n;
    const int grid = deal_blocks(n, d, props.sm_count * b.occ, b.nitems, &m);
    if (debug_enabled())
        fprintf(stderr, "[pde_b200] split bwd multi plan: n=%d N=%d C=%d chan_op=%d P=%d occ=%d grid=%d\n", n, d[0].N, d[0].C,
                d[0].chan_op, p.P, b.occ, grid);
    FinishJob jobs[PDE_MAX_BRANCHES];
    for (int i = 0; i < n; ++i) {
        WsLayout w;
        ws_layout(d[i], p, m.blk_begin[i + 1] - m.blk_begin[i], &w);
        const size_t need = (w.scratch_floats + w.maps_floats + w.chan_floats + w.skip_floats) * sizeof(float) + 512;
        if (!workspace || !workspace[i] || workspace_bytes_[i] < need || !ckpt || !ckpt[i]) return PDE_ERR_WORKSPACE;
        float *ws = reinterpret_cast<float *>((reinterpret_cast<uintptr_t>(workspace[i]) + 255u) & ~(uintptr_t)255u);
        Args &a = m.a[i];
        fill_args(d[i], static_cast<const char *>(tables[i]), &a);
        a.nitems = b.nitems;
        a.need_gin = gin && gin[i];
        a.tmem_cols = p.tmem_cols;
        a.u = u;
        a.gout = gout[i];
        a.chan = chan ? chan[i] : nullptr;
        a.skipw = skipw ? skipw[i] : nullptr;
        a.gin = gin ? gin[i] : nullptr;
        a.ckpt = ck_images(const_cast<void *>(ckpt[i]), &a.ck_flags);
        a.scratch = ws;
        a.part_maps = ws + w.scratch_floats;
        a.part_chan = a.part_maps + w.maps_floats;
        a.part_skip = a.part_chan + w.chan_floats;
        jobs[i] = FinishJob{d[i], w.nsets_maps, w.nsets_small, a.part_maps, a.part_chan, a.part_skip, a.skipw,
                            g_ab[i], g_atc[i], g_bb[i], g_btc[i], g_chan ? g_chan[i] : nullptr, g_skip ? g_skip[i] : nullptr};
    }
    void *params[] = {&m};
    PDE_CUDA_TRY(cudaLaunchKernel(kern, dim3(grid), dim3(p.threads), params, b.smem, st));
    rc = cuda_last_error();
    if (rc) return rc;
    launch_finish_multi(n, jobs, st);
    return cuda_last_error();
}

}  // namespace split
}  // namespace adi
}  // namespace pde
