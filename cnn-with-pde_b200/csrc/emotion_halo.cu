// emotion_recognition.PDELayer on planes the whole-plane kernels of explicit.cu cannot hold: N x N planes with
// 65 <= N <= 4096 and 0 ... 16 steps, element-aligned fp32 I/O.
//
// Forward, one launch.  A block owns a kTH x kTW tile of output cells of one sample and reads the tile's window
// from u0: the tile plus K cells of halo on every side.  Window cells on the reflected ghost ring (row -1 = row 1,
// row N = row N - 2, the same for columns) hold their frozen values in both shared-memory buffers and are never
// written; cells beyond the ring are zero and never read (the update of a plane cell reads plane cells and ring
// cells, never a corner).  Step s updates the plane cells of window cells [s, WH - s) x [s, WW - s) from the
// previous buffer only (Jacobi), so after K steps exactly the tile is valid; the last step writes the tile
// straight to the output.
//
// Backward, per chunk of samples (workspace layout in `layout`):
//   1. replay: the forward kernel, run for K - 1 steps, writes each step's tile into the workspace (u^1 .. u^{K-1});
//   2. K single-step adjoint launches, k = K - 1 ... 0: lambda^k from lambda^{k+1} (zero outside the plane) and
//      u^k (ghosts from u0), emo_bwd_kernel's arithmetic.  lambda^k overwrites u^{k+1}, which no later step reads;
//      lambda^0 is grad_input before the ghost terms;
//   3. the adjoint that flows into the frozen ghost ring is summed over the steps in four N-vectors per sample and
//      added to grad_input at rows 1 / N - 2 and columns 1 / N - 2 at the end (fold kernel);
//   4. dA_i = sum lambda d2_row u per row, dB_j per column: fp32 within a step and tile, added into double partials
//      that one block owns per (sample slot, tile), summed in a fixed order across tiles, slots and chunks, then
//      weighted by {1, sin 2 pi y, sin 4 pi y} / {1, cos 2 pi x, cos 4 pi x} in double: bit-reproducible.
// Coefficients come from emo_profile, the routine every emotion kernel uses.  Indices into planes are 64-bit.
//
// I/O type T (fp32 or bf16) is that of u0, gout, out and grad_input only: windows, replayed states, adjoint planes,
// edge sums and partials are fp32 / double in both.  In bf16 the adjoint kernel meets T at k = Nt - 1 (lambda^Nt =
// gout) and at k = 0 (u^0, and lambda^0 = grad_input).  lambda^0 is rounded on its store except at the cells the
// fold adds ghost-ring terms to (rows and columns 1 and N - 2): their fp32 values wait in a side buffer
// [slot][4][N] until the fold adds those terms and rounds, so grad_input is rounded once, as in the fp32 order.
#include <cstdio>
#include <type_traits>

#include "common.cuh"
#include "emo_profile.cuh"
#include "emotion_halo.cuh"

namespace pde {
namespace halo {

using expl::emo_profile;
using expl::io_ldg;
using expl::io_round;
using expl::io_stcs;

constexpr int kThreads = 256, kWarps = kThreads / 32;
constexpr int kTH = 32, kTW = 64;      // output tile: a warp per row, 64 fp32 columns = two 128-byte lines
constexpr int kMaxChunk = 512;         // sample slots per backward chunk (bounds the partial sums' finish)

struct FwdArgs {
    pde_emo_desc d;
    const void *u0;        // I/O type
    const float *w6, *xs, *ys;
    void *out;             // forward: u^K, I/O type
    float *hist;           // replay: u^s of slot b at hist + (s - 1) * hstride + b * N^2, s = 1 ... K
    size_t hstride;
    int K, ntw, ntiles;
    long long nitems;      // (sample, tile) items, tile fastest
};

struct AdjArgs {
    pde_emo_desc d;
    const float *w6, *xs, *ys;
    const void *u0;        // the chunk's layer input: the ghost ring of every state (I/O type)
    const void *uk;        // u^k of the chunk's slots (slot stride N^2): u0 at k = 0, else an fp32 plane
    const void *lin;       // lambda^{k+1}: gout at k = Nt - 1, else an fp32 plane
    void *lout;            // lambda^k (NULL: not needed): grad_input at k = 0, else an fp32 plane
    float *edge;           // [slot][top | bottom | left | right][N] (NULL: no grad_input)
    float *side;           // bf16 grad_input: [slot][row 1 | row N - 2 | column 1 | column N - 2][N] fp32 lambda^0
    double *pa, *pb;       // [slot][tile column][N] row sums, [slot][tile row][N] column sums
    int ntw, nth, ntiles;
    long long nitems;
};

// a_i of the window rows and b_j of the window columns; zero outside the plane
__device__ __forceinline__ void load_coeffs(const pde_emo_desc &d, const float *w6, const float *xs, const float *ys,
                                            int gr0, int gc0, int WH, int WW, float *sa, float *sb) {
    for (int t = threadIdx.x; t < WH + WW; t += kThreads) {
        const int g = t < WH ? gr0 + t : gc0 + t - WH;
        float av = 0.0f, bv = 0.0f;
        if ((unsigned)g < (unsigned)d.N) emo_profile(d, w6, xs, ys, g, &av, &bv);
        if (t < WH) sa[t] = av;
        else sb[t - WH] = bv;
    }
}

// window cell (i, j) <- plane cell (gr0 + i, gc0 + j): plane cells from `in`, ghost-ring cells (corners excluded)
// reflected from `ring`, or zero where `ring` is NULL; every other cell zero.  Into w0, and w1 when set.
template <typename TI, typename TR>
__device__ __forceinline__ void load_window(float *w0, float *w1, const TI *in, const TR *ring, int gr0, int gc0,
                                            int WH, int WW, int N) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = warp; i < WH; i += kWarps) {
        const int gr = gr0 + i;
        const bool rin = (unsigned)gr < (unsigned)N, rg = gr == -1 || gr == N;
        const int sr = gr == -1 ? 1 : (gr == N ? N - 2 : gr);
        for (int j = lane; j < WW; j += 32) {
            const int gc = gc0 + j;
            const bool cin = (unsigned)gc < (unsigned)N, cg = gc == -1 || gc == N;
            const int sc = gc == -1 ? 1 : (gc == N ? N - 2 : gc);
            float v = 0.0f;
            if (rin && cin) v = io_ldg(in + (size_t)gr * N + gc);
            else if (ring && ((rin && cg) || (rg && cin))) v = io_ldg(ring + (size_t)sr * N + sc);
            w0[i * WW + j] = v;
            if (w1) w1[i * WW + j] = v;
        }
    }
}

// one explicit step of the plane cells among window cells [lo, WH - lo) x [lo, WW - lo), in emo_step's
// arithmetic: into dst when set, and the tile's cells (window cells [K, K + kTH) x [K, K + kTW)) into the plane g
// when set (streaming stores for the layer output)
template <bool kStream, typename TG>
__device__ __forceinline__ void fwd_step(const float *src, float *dst, TG *g, int lo, int K, int WH, int WW, int gr0,
                                         int gc0, int N, const float *sa, const float *sb) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = lo + warp; i < WH - lo; i += kWarps) {
        const int gr = gr0 + i;
        if ((unsigned)gr >= (unsigned)N) continue;
        const float ai = sa[i];
        const bool row_tile = i >= K && i < K + kTH;
        for (int j = lo + lane; j < WW - lo; j += 32) {
            const int gc = gc0 + j;
            if ((unsigned)gc >= (unsigned)N) continue;
            const float *p = src + i * WW + j;
            const float ct = p[0], two = 2.0f * ct;
            const float dr = (p[WW] - two) + p[-WW];
            const float dc = (p[1] - two) + p[-1];
            const float v = fmaf(sb[j], dc, fmaf(ai, dr, ct));
            if (dst) dst[i * WW + j] = v;
            if (g && row_tile && j >= K && j < K + kTW) {
                if (kStream) io_stcs(g + (size_t)gr * N + gc, v);
                else g[(size_t)gr * N + gc] = io_round<TG>(v);
            }
        }
    }
}

// kReplay = false: the layer forward (K = Nt >= 1 steps into out); true: the backward's replay (K = Nt - 1 >= 1
// steps, every state into hist, fp32).  T: the I/O type of u0 and out
template <bool kReplay, typename T>
__global__ void __launch_bounds__(kThreads) emo_halo_fwd_kernel(const FwdArgs a) {
    extern __shared__ __align__(16) float smem[];
    const int N = a.d.N, K = a.K, WH = kTH + 2 * K, WW = kTW + 2 * K;
    float *sa = smem, *sb = smem + WH, *w0 = sb + WW, *w1 = w0 + WH * WW;   // w1: only touched when K > 1
    const size_t NN = (size_t)N * N;
    for (long long item = blockIdx.x; item < a.nitems; item += gridDim.x) {
        const long long b = item / a.ntiles;
        const int tile = (int)(item - b * a.ntiles);
        const int gr0 = (tile / a.ntw) * kTH - K, gc0 = (tile % a.ntw) * kTW - K;
        const T *u = static_cast<const T *>(a.u0) + (size_t)b * NN;
        __syncthreads();   // the previous item is done with shared memory
        load_coeffs(a.d, a.w6, a.xs, a.ys, gr0, gc0, WH, WW, sa, sb);
        load_window(w0, K > 1 ? w1 : nullptr, u, u, gr0, gc0, WH, WW, N);
        __syncthreads();
        const float *src = w0;
        float *dst = w1;
        for (int s = 1; s <= K; ++s) {
            if constexpr (kReplay) {
                float *g = a.hist + (size_t)(s - 1) * a.hstride + (size_t)b * NN;
                fwd_step<false>(src, s < K ? dst : nullptr, g, s, K, WH, WW, gr0, gc0, N, sa, sb);
            } else {
                T *g = s == K ? static_cast<T *>(a.out) + (size_t)b * NN : nullptr;
                fwd_step<true>(src, s < K ? dst : nullptr, g, s, K, WH, WW, gr0, gc0, N, sa, sb);
            }
            if (s < K) {
                __syncthreads();
                float *t = const_cast<float *>(src);
                src = dst;
                dst = t;
            }
        }
    }
}

// One reversed step on a tile: lambda^k = M^T lambda^{k+1} with lambda zero outside the plane, what flows into the
// ghost ring, and this step's dA / dB terms.  Arithmetic of emo_bwd_kernel.  T: the I/O type; kLinIO: lambda^{k+1}
// is gout (k = Nt - 1); kFirst: k = 0 (u^k is u0, lambda^k is grad_input).  fp32 I/O uses <float, false, false> for
// every k: all its planes have one type.
template <typename T, bool kLinIO, bool kFirst>
__global__ void __launch_bounds__(kThreads) emo_halo_adj_kernel(const AdjArgs a) {
    using TL = std::conditional_t<kLinIO, T, float>;
    using TU = std::conditional_t<kFirst, T, float>;
    constexpr bool kSide = kFirst && sizeof(T) == 2;   // lambda^0's fold cells stay fp32 until the fold
    constexpr int WH = kTH + 2, WW = kTW + 2;
    __shared__ float L[WH * WW], U[WH * WW], sa[WH], sb[WW];
    __shared__ float red[kWarps][kTW];
    const int N = a.d.N, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const size_t NN = (size_t)N * N;
    for (long long item = blockIdx.x; item < a.nitems; item += gridDim.x) {
        const long long b = item / a.ntiles;
        const int tile = (int)(item - b * a.ntiles), tr = tile / a.ntw, tc = tile % a.ntw;
        const int gr0 = tr * kTH - 1, gc0 = tc * kTW - 1;
        __syncthreads();   // the previous item is done with shared memory
        load_coeffs(a.d, a.w6, a.xs, a.ys, gr0, gc0, WH, WW, sa, sb);
        load_window<TL, TL>(L, nullptr, static_cast<const TL *>(a.lin) + (size_t)b * NN, nullptr, gr0, gc0, WH, WW, N);
        load_window(U, nullptr, static_cast<const TU *>(a.uk) + (size_t)b * NN, static_cast<const T *>(a.u0) + (size_t)b * NN,
                    gr0, gc0, WH, WW, N);
        __syncthreads();
        float *e = a.edge ? a.edge + (size_t)b * 4 * N : nullptr;
        float fB[2] = {0.0f, 0.0f};
#pragma unroll
        for (int y = 0; y < kTH / kWarps; ++y) {
            const int i = 1 + warp + y * kWarps, gr = gr0 + i;
            float fA = 0.0f;
            if (gr < N) {
                const float am = sa[i - 1], ai = sa[i], ap = sa[i + 1];
#pragma unroll
                for (int x = 0; x < 2; ++x) {
                    const int j = 1 + lane + 32 * x, gc = gc0 + j;
                    if (gc >= N) continue;
                    const float *pl = L + i * WW + j, *pu = U + i * WW + j;
                    const float lct = pl[0], uct = pu[0], two = 2.0f * uct;
                    const float dr = (pu[WW] - two) + pu[-WW], dc = (pu[1] - two) + pu[-1];
                    fA = fmaf(lct, dr, fA);
                    fB[x] = fmaf(lct, dc, fB[x]);
                    const float al = ai * lct, blv = sb[j] * lct;
                    float nv = (lct - 2.0f * al) - 2.0f * blv;
                    nv = fmaf(am, pl[-WW], nv);
                    nv = fmaf(ap, pl[WW], nv);
                    nv = fmaf(sb[j - 1], pl[-1], nv);
                    nv = fmaf(sb[j + 1], pl[1], nv);
                    if (a.lout) {
                        if (kSide && a.side && (gr == 1 || gr == N - 2 || gc == 1 || gc == N - 2)) {
                            float *sd = a.side + (size_t)b * 4 * N;
                            if (gr == 1) sd[gc] = nv;
                            if (gr == N - 2) sd[N + gc] = nv;
                            if (gc == 1) sd[2 * N + gr] = nv;
                            if (gc == N - 2) sd[3 * N + gr] = nv;
                        } else {
                            static_cast<TU *>(a.lout)[(size_t)b * NN + (size_t)gr * N + gc] = io_round<TU>(nv);
                        }
                    }
                    if (e) {   // a_0 lam(0, j) / a_{N-1} lam(N-1, j) / b_0 lam(i, 0) / b_{N-1} lam(i, N-1): ghost ring
                        if (gr == 0) e[gc] += al;
                        if (gr == N - 1) e[N + gc] += al;
                        if (gc == 0) e[2 * N + gr] += blv;
                        if (gc == N - 1) e[3 * N + gr] += blv;
                    }
                }
            }
            fA = warp_sum(fA);
            if (lane == 0 && gr < N) a.pa[((size_t)b * a.ntw + tc) * N + gr] += (double)fA;
        }
        red[warp][lane] = fB[0];
        red[warp][lane + 32] = fB[1];
        __syncthreads();
        if (tid < kTW) {
            const int gc = gc0 + 1 + tid;
            if (gc < N) {
                float s = 0.0f;
                for (int w = 0; w < kWarps; ++w) s += red[w][tid];
                a.pb[((size_t)b * a.nth + tr) * N + gc] += (double)s;
            }
        }
    }
}

// grad_input += the ghost ring's adjoint through the reflection: rows 1 / N - 2 first, then columns 1 / N - 2
// (the order of emo_bwd_kernel); a thread per edge cell.  fp32 adds to grad_input in place; bf16 takes lambda^0 of
// the cell from the side buffer and rounds the sum on its store
template <typename T>
__global__ void emo_halo_fold_kernel(int N, long long ncells, const float *__restrict__ edge,
                                     const float *__restrict__ side, T *gin) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= ncells) return;
    const long long b = idx / (4 * N);
    const int t = (int)(idx - b * 4 * N), sd = t / N, q = t - sd * N;
    const float *e = edge + (size_t)b * 4 * N;
    T *g = gin + (size_t)b * N * N;
    auto lam0 = [&](int i, int j) {
        if constexpr (sizeof(T) == 4) return g[(size_t)i * N + j];
        else return side[(size_t)b * 4 * N + t];
    };
    int i, j;
    float v;
    if (sd < 2) {
        i = sd == 0 ? 1 : N - 2;
        j = q;
        v = lam0(i, j) + e[sd * N + j];
        if (j == 1) v += e[2 * N + i];
        if (j == N - 2) v += e[3 * N + i];
    } else {
        if (q == 1 || q == N - 2) return;   // done with the rows above
        i = q;
        j = sd == 2 ? 1 : N - 2;
        v = lam0(i, j) + e[sd * N + i];
    }
    g[(size_t)i * N + j] = io_round<T>(v);
}

// tot[i] = dA_i (i < N), tot[N + j] = dB_j: double, summed over slots then tiles in a fixed order
__global__ void emo_halo_sum_kernel(int N, int nslots, int ntw, int nth, const double *__restrict__ pa,
                                    const double *__restrict__ pb, double *tot) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= 2 * N) return;
    const bool rows = q < N;
    const int i = rows ? q : q - N, nt = rows ? ntw : nth;
    const double *p = rows ? pa : pb;
    double s = 0.0;
    for (int b = 0; b < nslots; ++b)
        for (int t = 0; t < nt; ++t) s += p[((size_t)b * nt + t) * N + i];
    tot[q] = s;
}

// the six scalar gradients, in double, reduced over the block in a fixed order
constexpr int kFinishThreads = 256;
__global__ void __launch_bounds__(kFinishThreads) emo_halo_finish_kernel(pde_emo_desc d, const double *__restrict__ tot,
                                                                         const float *__restrict__ xs,
                                                                         const float *__restrict__ ys, float *g_w6) {
    __shared__ double red[6][kFinishThreads];
    const int t = threadIdx.x;
    const float two_pi = (float)(2.0 * 3.141592653589793), four_pi = (float)(4.0 * 3.141592653589793);
    const double ka = (double)d.half_dt / (double)d.dx2, kb = (double)d.dt / (double)d.dy2;
    double g[6] = {0, 0, 0, 0, 0, 0};
    for (int q = t; q < d.N; q += kFinishThreads) {
        const double s1 = (double)sinf(__fmul_rn(two_pi, ys[q])), s2 = (double)sinf(__fmul_rn(four_pi, ys[q]));
        const double c1 = (double)cosf(__fmul_rn(two_pi, xs[q])), c2 = (double)cosf(__fmul_rn(four_pi, xs[q]));
        const double A = tot[q], B = tot[d.N + q];
        g[0] += ka * A; g[1] += ka * A * s1; g[2] += ka * A * s2;
        g[3] += kb * B; g[4] += kb * B * c1; g[5] += kb * B * c2;
    }
    for (int k = 0; k < 6; ++k) red[k][t] = g[k];
    __syncthreads();
    for (int o = kFinishThreads / 2; o > 0; o >>= 1) {
        if (t < o)
            for (int k = 0; k < 6; ++k) red[k][t] += red[k][t + o];
        __syncthreads();
    }
    if (t < 6) g_w6[t] = (float)red[t][0];
}

// ------------------------------------------------------------------------------------------ host
// Backward workspace, from a 256-byte aligned base: tot [2N] doubles, pa [chunk][ntw][N] and pb [chunk][nth][N]
// doubles, edges [chunk][4][N] floats, state / adjoint planes [Nt][chunk][N][N] floats (none for Nt <= 1), and for
// bf16 I/O the side buffer [chunk][4][N] floats.  chunk = the sample slots whose share of the fp32 layout fits
// kHaloWorkspaceCap, at least 1, at most min(B, kMaxChunk): the same in both I/O types, so that the partial sums
// are added in the same order.
struct Layout {
    int ntw, nth, ntiles, planes;
    long long chunk;
    size_t pa, pb, edge, plane, side, bytes;
};

static Layout layout(const pde_emo_desc *d, int io_bytes) {
    Layout l;
    const size_t N = (size_t)d->N, NN = N * N;
    l.ntw = (d->N + kTW - 1) / kTW;
    l.nth = (d->N + kTH - 1) / kTH;
    l.ntiles = l.ntw * l.nth;
    l.planes = d->Nt >= 2 ? d->Nt : 0;
    const size_t slot = (size_t)l.planes * NN * sizeof(float) + 4 * N * sizeof(float) + (size_t)(l.ntw + l.nth) * N * sizeof(double);
    long long c = (long long)(kHaloWorkspaceCap / slot);
    if (c > kMaxChunk) c = kMaxChunk;
    if (c > d->B) c = d->B;
    if (c < 1) c = 1;
    l.chunk = c;
    l.pa = 2 * N * sizeof(double);
    l.pb = l.pa + (size_t)c * l.ntw * N * sizeof(double);
    l.edge = l.pb + (size_t)c * l.nth * N * sizeof(double);
    l.plane = l.edge + (size_t)c * 4 * N * sizeof(float);
    l.side = l.plane + (size_t)c * l.planes * NN * sizeof(float);
    l.bytes = 256 + l.side + (io_bytes == 2 ? (size_t)c * 4 * N * sizeof(float) : 0);
    return l;
}

size_t emo_halo_workspace_bytes(const pde_emo_desc *d, int io_bytes) { return layout(d, io_bytes).bytes; }

struct Launch {
    const void *kern;
    size_t smem;
    int regs, per_sm;
    long long grid;
};

static int plan_launch(const void *kern, size_t smem, long long nitems, const DeviceProps &props, Launch *p) {
    p->kern = kern;
    p->smem = smem;
    KernelInfo ki;
    int rc = kernel_info(kern, smem, &ki);
    if (rc) return rc;
    rc = cached_occupancy(kern, kThreads, smem, &p->per_sm);
    if (rc) return rc;
    p->regs = ki.regs;
    p->grid = (long long)props.sm_count * p->per_sm;   // persistent blocks stride over the items
    if (p->grid > nitems) p->grid = nitems;
    return PDE_OK;
}

template <typename T>
static int plan_fwd(const FwdArgs &a, bool replay, const DeviceProps &props, Launch *p) {
    const size_t WH = kTH + 2 * a.K, WW = kTW + 2 * a.K;
    const size_t smem = (WH + WW + (a.K > 1 ? 2 : 1) * WH * WW) * sizeof(float);
    const void *kern = replay ? reinterpret_cast<const void *>(emo_halo_fwd_kernel<true, T>)
                              : reinterpret_cast<const void *>(emo_halo_fwd_kernel<false, T>);
    return plan_launch(kern, smem, a.nitems, props, p);
}

static int launch(const Launch &p, void *args, cudaStream_t st) {
    void *kargs[] = {args};
    PDE_CUDA_TRY(cudaLaunchKernel(p.kern, dim3((unsigned)p.grid), dim3(kThreads), kargs, p.smem, st));
    return cuda_last_error();
}

static FwdArgs fwd_args(const pde_emo_desc *d, const void *u0, const float *w6, const float *xs, const float *ys, int K,
                        long long nsamples) {
    FwdArgs a{};
    a.d = *d; a.u0 = u0; a.w6 = w6; a.xs = xs; a.ys = ys; a.K = K;
    a.ntw = (d->N + kTW - 1) / kTW;
    a.ntiles = a.ntw * ((d->N + kTH - 1) / kTH);
    a.nitems = nsamples * a.ntiles;
    return a;
}

// the adjoint kernel of reversed step k: fp32 I/O has one for every k
template <typename T>
static const void *adj_kernel(bool lin_io, bool first) {
    if constexpr (sizeof(T) == 4) {
        return reinterpret_cast<const void *>(emo_halo_adj_kernel<float, false, false>);
    } else {
        if (lin_io) return first ? reinterpret_cast<const void *>(emo_halo_adj_kernel<T, true, true>)
                                 : reinterpret_cast<const void *>(emo_halo_adj_kernel<T, true, false>);
        return first ? reinterpret_cast<const void *>(emo_halo_adj_kernel<T, false, true>)
                     : reinterpret_cast<const void *>(emo_halo_adj_kernel<T, false, false>);
    }
}

template <typename T>
int emo_halo_forward(const pde_emo_desc *d, const T *u0, const float *w6, const float *xs, const float *ys, T *out,
                     const DeviceProps &props, cudaStream_t st) {
    const size_t bytes = (size_t)d->B * d->N * d->N * sizeof(T);
    if (d->Nt == 0) {
        if (debug_enabled()) fprintf(stderr, "[pde_b200] emotion halo fwd plan: B=%d N=%d Nt=0 copy\n", d->B, d->N);
        PDE_CUDA_TRY(cudaMemcpyAsync(out, u0, bytes, cudaMemcpyDeviceToDevice, st));
        return PDE_OK;
    }
    FwdArgs a = fwd_args(d, u0, w6, xs, ys, d->Nt, d->B);
    a.out = out;
    Launch p;
    int rc = plan_fwd<T>(a, false, props, &p);
    if (rc) return rc;
    if (debug_enabled())
        fprintf(stderr, "[pde_b200] emotion halo fwd plan: B=%d N=%d Nt=%d tile=%dx%d window=%dx%d smem=%zu regs=%d "
                "occ=%d grid=%lld items=%lld\n", d->B, d->N, d->Nt, kTH, kTW, kTH + 2 * d->Nt, kTW + 2 * d->Nt, p.smem,
                p.regs, p.per_sm, p.grid, a.nitems);
    return launch(p, &a, st);
}

template <typename T>
int emo_halo_backward(const pde_emo_desc *d, const T *u0, const T *gout, const float *w6, const float *xs,
                      const float *ys, T *gin, float *g_w6, void *workspace, size_t workspace_bytes,
                      const DeviceProps &props, cudaStream_t st) {
    const Layout l = layout(d, (int)sizeof(T));
    if (!workspace || workspace_bytes < l.bytes) return PDE_ERR_WORKSPACE;
    char *base = reinterpret_cast<char *>((reinterpret_cast<uintptr_t>(workspace) + 255u) & ~(uintptr_t)255u);
    double *tot = reinterpret_cast<double *>(base), *pa = reinterpret_cast<double *>(base + l.pa),
           *pb = reinterpret_cast<double *>(base + l.pb);
    float *edge = reinterpret_cast<float *>(base + l.edge), *planes = reinterpret_cast<float *>(base + l.plane);
    float *side = sizeof(T) == 2 ? reinterpret_cast<float *>(base + l.side) : nullptr;
    const int N = d->N, Nt = d->Nt;
    const size_t NN = (size_t)N * N;
    const long long B = d->B, chunk = l.chunk;
    int rc;
    PDE_CUDA_TRY(cudaMemsetAsync(pa, 0, (size_t)chunk * (l.ntw + l.nth) * N * sizeof(double), st));   // pa, pb
    if (Nt == 0 && gin) PDE_CUDA_TRY(cudaMemcpyAsync(gin, gout, (size_t)B * NN * sizeof(T), cudaMemcpyDeviceToDevice, st));
    auto plane = [&](int p) { return planes + (size_t)p * chunk * NN; };
    Launch rp{}, ap{};
    AdjArgs q{};
    q.d = *d; q.w6 = w6; q.xs = xs; q.ys = ys; q.pa = pa; q.pb = pb;
    q.ntw = l.ntw; q.nth = l.nth; q.ntiles = l.ntiles;
    for (long long b0 = 0; Nt > 0 && b0 < B; b0 += chunk) {
        const long long nb = B - b0 < chunk ? B - b0 : chunk;
        const T *u = u0 + (size_t)b0 * NN, *g = gout + (size_t)b0 * NN;
        T *gi = gin ? gin + (size_t)b0 * NN : nullptr;
        if (gi) PDE_CUDA_TRY(cudaMemsetAsync(edge, 0, (size_t)nb * 4 * N * sizeof(float), st));
        if (Nt >= 2) {   // u^1 ... u^{Nt-1} into planes 0 ... Nt - 2
            FwdArgs r = fwd_args(d, u, w6, xs, ys, Nt - 1, nb);
            r.hist = planes;
            r.hstride = (size_t)chunk * NN;
            if ((rc = plan_fwd<T>(r, true, props, &rp))) return rc;
            if ((rc = launch(rp, &r, st))) return rc;
        }
        q.u0 = u;
        q.edge = gi ? edge : nullptr;
        q.side = gi ? side : nullptr;
        q.nitems = nb * l.ntiles;
        for (int k = Nt - 1; k >= 0; --k) {
            q.uk = k == 0 ? static_cast<const void *>(u) : plane(k - 1);
            q.lin = k + 1 == Nt ? static_cast<const void *>(g) : plane(k + 1 == Nt - 1 ? Nt - 1 : k + 1);
            q.lout = k == 0 ? static_cast<void *>(gi) : plane(k == Nt - 1 ? Nt - 1 : k);
            if ((rc = plan_launch(adj_kernel<T>(k + 1 == Nt, k == 0), 0, q.nitems, props, &ap))) return rc;
            if ((rc = launch(ap, &q, st))) return rc;
        }
        if (gi) {
            const long long ncells = nb * 4 * N;
            emo_halo_fold_kernel<T><<<(unsigned)((ncells + 255) / 256), 256, 0, st>>>(N, ncells, edge, side, gi);
            if ((rc = cuda_last_error())) return rc;
        }
    }
    if (debug_enabled())
        fprintf(stderr, "[pde_b200] emotion halo bwd plan: B=%d N=%d Nt=%d tile=%dx%d chunk=%lld workspace=%zu "
                "replay: window=%dx%d smem=%zu regs=%d grid=%lld; adjoint: smem=%d regs=%d grid=%lld; gin=%d\n",
                d->B, N, Nt, kTH, kTW, chunk, l.bytes, kTH + 2 * (Nt > 1 ? Nt - 1 : 0), kTW + 2 * (Nt > 1 ? Nt - 1 : 0),
                rp.smem, rp.regs, rp.grid, (int)((2 * (kTH + 2) * (kTW + 2) + (kTH + 2) + (kTW + 2) + kWarps * kTW) * 4),
                ap.regs, ap.grid, gin != nullptr);
    const int nslots = (int)(chunk < B ? chunk : B);
    emo_halo_sum_kernel<<<(2 * N + 255) / 256, 256, 0, st>>>(N, nslots, l.ntw, l.nth, pa, pb, tot);
    if ((rc = cuda_last_error())) return rc;
    emo_halo_finish_kernel<<<1, kFinishThreads, 0, st>>>(*d, tot, xs, ys, g_w6);
    return cuda_last_error();
}

template int emo_halo_forward<float>(const pde_emo_desc *, const float *, const float *, const float *, const float *,
                                     float *, const DeviceProps &, cudaStream_t);
template int emo_halo_forward<__nv_bfloat16>(const pde_emo_desc *, const __nv_bfloat16 *, const float *, const float *,
                                             const float *, __nv_bfloat16 *, const DeviceProps &, cudaStream_t);
template int emo_halo_backward<float>(const pde_emo_desc *, const float *, const float *, const float *, const float *,
                                      const float *, float *, float *, void *, size_t, const DeviceProps &, cudaStream_t);
template int emo_halo_backward<__nv_bfloat16>(const pde_emo_desc *, const __nv_bfloat16 *, const __nv_bfloat16 *,
                                              const float *, const float *, const float *, __nv_bfloat16 *, float *, void *,
                                              size_t, const DeviceProps &, cudaStream_t);

}  // namespace halo
}  // namespace pde
