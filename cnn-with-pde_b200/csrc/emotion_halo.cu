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
#include <cstdio>

#include "common.cuh"
#include "emo_profile.cuh"
#include "emotion_halo.cuh"

namespace pde {
namespace halo {

using expl::emo_profile;

constexpr int kThreads = 256, kWarps = kThreads / 32;
constexpr int kTH = 32, kTW = 64;      // output tile: a warp per row, 64 fp32 columns = two 128-byte lines
constexpr int kMaxChunk = 512;         // sample slots per backward chunk (bounds the partial sums' finish)

struct FwdArgs {
    pde_emo_desc d;
    const float *u0, *w6, *xs, *ys;
    float *out;            // forward: u^K
    float *hist;           // replay: u^s of slot b at hist + (s - 1) * hstride + b * N^2, s = 1 ... K
    size_t hstride;
    int K, ntw, ntiles;
    long long nitems;      // (sample, tile) items, tile fastest
};

struct AdjArgs {
    pde_emo_desc d;
    const float *w6, *xs, *ys;
    const float *u0;       // the chunk's layer input: the ghost ring of every state
    const float *uk;       // u^k of the chunk's slots (slot stride N^2)
    const float *lin;      // lambda^{k+1}
    float *lout;           // lambda^k (NULL: not needed)
    float *edge;           // [slot][top | bottom | left | right][N] (NULL: no grad_input)
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
__device__ __forceinline__ void load_window(float *w0, float *w1, const float *in, const float *ring, int gr0, int gc0,
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
            if (rin && cin) v = __ldg(in + (size_t)gr * N + gc);
            else if (ring && ((rin && cg) || (rg && cin))) v = __ldg(ring + (size_t)sr * N + sc);
            w0[i * WW + j] = v;
            if (w1) w1[i * WW + j] = v;
        }
    }
}

// one explicit step of the plane cells among window cells [lo, WH - lo) x [lo, WW - lo), in emo_step's
// arithmetic: into dst when set, and the tile's cells (window cells [K, K + kTH) x [K, K + kTW)) into the plane g
// when set (streaming stores for the layer output)
template <bool kStream>
__device__ __forceinline__ void fwd_step(const float *src, float *dst, float *g, int lo, int K, int WH, int WW, int gr0,
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
                if (kStream) __stcs(g + (size_t)gr * N + gc, v);
                else g[(size_t)gr * N + gc] = v;
            }
        }
    }
}

// kReplay = false: the layer forward (K = Nt >= 1 steps into out); true: the backward's replay (K = Nt - 1 >= 1
// steps, every state into hist)
template <bool kReplay>
__global__ void __launch_bounds__(kThreads) emo_halo_fwd_kernel(const FwdArgs a) {
    extern __shared__ __align__(16) float smem[];
    const int N = a.d.N, K = a.K, WH = kTH + 2 * K, WW = kTW + 2 * K;
    float *sa = smem, *sb = smem + WH, *w0 = sb + WW, *w1 = w0 + WH * WW;   // w1: only touched when K > 1
    const size_t NN = (size_t)N * N;
    for (long long item = blockIdx.x; item < a.nitems; item += gridDim.x) {
        const long long b = item / a.ntiles;
        const int tile = (int)(item - b * a.ntiles);
        const int gr0 = (tile / a.ntw) * kTH - K, gc0 = (tile % a.ntw) * kTW - K;
        const float *u = a.u0 + (size_t)b * NN;
        __syncthreads();   // the previous item is done with shared memory
        load_coeffs(a.d, a.w6, a.xs, a.ys, gr0, gc0, WH, WW, sa, sb);
        load_window(w0, K > 1 ? w1 : nullptr, u, u, gr0, gc0, WH, WW, N);
        __syncthreads();
        const float *src = w0;
        float *dst = w1;
        for (int s = 1; s <= K; ++s) {
            float *g = kReplay ? a.hist + (size_t)(s - 1) * a.hstride + (size_t)b * NN
                               : (s == K ? a.out + (size_t)b * NN : nullptr);
            fwd_step<!kReplay>(src, s < K ? dst : nullptr, g, s, K, WH, WW, gr0, gc0, N, sa, sb);
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
// ghost ring, and this step's dA / dB terms.  Arithmetic of emo_bwd_kernel.
__global__ void __launch_bounds__(kThreads) emo_halo_adj_kernel(const AdjArgs a) {
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
        load_window(L, nullptr, a.lin + (size_t)b * NN, nullptr, gr0, gc0, WH, WW, N);
        load_window(U, nullptr, a.uk + (size_t)b * NN, a.u0 + (size_t)b * NN, gr0, gc0, WH, WW, N);
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
                    if (a.lout) a.lout[(size_t)b * NN + (size_t)gr * N + gc] = nv;
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
// (the order of emo_bwd_kernel); a thread per edge cell
__global__ void emo_halo_fold_kernel(int N, long long ncells, const float *__restrict__ edge, float *gin) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= ncells) return;
    const long long b = idx / (4 * N);
    const int t = (int)(idx - b * 4 * N), side = t / N, q = t - side * N;
    const float *e = edge + (size_t)b * 4 * N;
    float *g = gin + (size_t)b * N * N;
    int i, j;
    float v;
    if (side < 2) {
        i = side == 0 ? 1 : N - 2;
        j = q;
        v = g[(size_t)i * N + j] + e[side * N + j];
        if (j == 1) v += e[2 * N + i];
        if (j == N - 2) v += e[3 * N + i];
    } else {
        if (q == 1 || q == N - 2) return;   // done with the rows above
        i = q;
        j = side == 2 ? 1 : N - 2;
        v = g[(size_t)i * N + j] + e[side * N + i];
    }
    g[(size_t)i * N + j] = v;
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
// doubles, edges [chunk][4][N] floats, state / adjoint planes [Nt][chunk][N][N] floats (none for Nt <= 1).
// chunk = the sample slots whose share fits kHaloWorkspaceCap, at least 1, at most min(B, kMaxChunk).
struct Layout {
    int ntw, nth, ntiles, planes;
    long long chunk;
    size_t pa, pb, edge, plane, bytes;
};

static Layout layout(const pde_emo_desc *d) {
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
    l.bytes = 256 + l.plane + (size_t)c * l.planes * NN * sizeof(float);
    return l;
}

size_t emo_halo_workspace_bytes(const pde_emo_desc *d) { return layout(d).bytes; }

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

static int plan_fwd(const FwdArgs &a, bool replay, const DeviceProps &props, Launch *p) {
    const size_t WH = kTH + 2 * a.K, WW = kTW + 2 * a.K;
    const size_t smem = (WH + WW + (a.K > 1 ? 2 : 1) * WH * WW) * sizeof(float);
    const void *kern = replay ? reinterpret_cast<const void *>(emo_halo_fwd_kernel<true>)
                              : reinterpret_cast<const void *>(emo_halo_fwd_kernel<false>);
    return plan_launch(kern, smem, a.nitems, props, p);
}

static int launch(const Launch &p, void *args, cudaStream_t st) {
    void *kargs[] = {args};
    PDE_CUDA_TRY(cudaLaunchKernel(p.kern, dim3((unsigned)p.grid), dim3(kThreads), kargs, p.smem, st));
    return cuda_last_error();
}

static FwdArgs fwd_args(const pde_emo_desc *d, const float *u0, const float *w6, const float *xs, const float *ys, int K,
                        long long nsamples) {
    FwdArgs a{};
    a.d = *d; a.u0 = u0; a.w6 = w6; a.xs = xs; a.ys = ys; a.K = K;
    a.ntw = (d->N + kTW - 1) / kTW;
    a.ntiles = a.ntw * ((d->N + kTH - 1) / kTH);
    a.nitems = nsamples * a.ntiles;
    return a;
}

int emo_halo_forward(const pde_emo_desc *d, const float *u0, const float *w6, const float *xs, const float *ys,
                     float *out, const DeviceProps &props, cudaStream_t st) {
    const size_t bytes = (size_t)d->B * d->N * d->N * sizeof(float);
    if (d->Nt == 0) {
        if (debug_enabled()) fprintf(stderr, "[pde_b200] emotion halo fwd plan: B=%d N=%d Nt=0 copy\n", d->B, d->N);
        PDE_CUDA_TRY(cudaMemcpyAsync(out, u0, bytes, cudaMemcpyDeviceToDevice, st));
        return PDE_OK;
    }
    FwdArgs a = fwd_args(d, u0, w6, xs, ys, d->Nt, d->B);
    a.out = out;
    Launch p;
    int rc = plan_fwd(a, false, props, &p);
    if (rc) return rc;
    if (debug_enabled())
        fprintf(stderr, "[pde_b200] emotion halo fwd plan: B=%d N=%d Nt=%d tile=%dx%d window=%dx%d smem=%zu regs=%d "
                "occ=%d grid=%lld items=%lld\n", d->B, d->N, d->Nt, kTH, kTW, kTH + 2 * d->Nt, kTW + 2 * d->Nt, p.smem,
                p.regs, p.per_sm, p.grid, a.nitems);
    return launch(p, &a, st);
}

int emo_halo_backward(const pde_emo_desc *d, const float *u0, const float *gout, const float *w6, const float *xs,
                      const float *ys, float *gin, float *g_w6, void *workspace, size_t workspace_bytes,
                      const DeviceProps &props, cudaStream_t st) {
    const Layout l = layout(d);
    if (!workspace || workspace_bytes < l.bytes) return PDE_ERR_WORKSPACE;
    char *base = reinterpret_cast<char *>((reinterpret_cast<uintptr_t>(workspace) + 255u) & ~(uintptr_t)255u);
    double *tot = reinterpret_cast<double *>(base), *pa = reinterpret_cast<double *>(base + l.pa),
           *pb = reinterpret_cast<double *>(base + l.pb);
    float *edge = reinterpret_cast<float *>(base + l.edge), *planes = reinterpret_cast<float *>(base + l.plane);
    const int N = d->N, Nt = d->Nt;
    const size_t NN = (size_t)N * N;
    const long long B = d->B, chunk = l.chunk;
    int rc;
    PDE_CUDA_TRY(cudaMemsetAsync(pa, 0, (size_t)chunk * (l.ntw + l.nth) * N * sizeof(double), st));   // pa, pb
    if (Nt == 0 && gin) PDE_CUDA_TRY(cudaMemcpyAsync(gin, gout, (size_t)B * NN * sizeof(float), cudaMemcpyDeviceToDevice, st));
    auto plane = [&](int p) { return planes + (size_t)p * chunk * NN; };
    Launch rp{}, ap{};
    AdjArgs q{};
    q.d = *d; q.w6 = w6; q.xs = xs; q.ys = ys; q.pa = pa; q.pb = pb;
    q.ntw = l.ntw; q.nth = l.nth; q.ntiles = l.ntiles;
    for (long long b0 = 0; Nt > 0 && b0 < B; b0 += chunk) {
        const long long nb = B - b0 < chunk ? B - b0 : chunk;
        const float *u = u0 + (size_t)b0 * NN, *g = gout + (size_t)b0 * NN;
        float *gi = gin ? gin + (size_t)b0 * NN : nullptr;
        if (gi) PDE_CUDA_TRY(cudaMemsetAsync(edge, 0, (size_t)nb * 4 * N * sizeof(float), st));
        if (Nt >= 2) {   // u^1 ... u^{Nt-1} into planes 0 ... Nt - 2
            FwdArgs r = fwd_args(d, u, w6, xs, ys, Nt - 1, nb);
            r.hist = planes;
            r.hstride = (size_t)chunk * NN;
            if ((rc = plan_fwd(r, true, props, &rp))) return rc;
            if ((rc = launch(rp, &r, st))) return rc;
        }
        q.u0 = u;
        q.edge = gi ? edge : nullptr;
        q.nitems = nb * l.ntiles;
        if ((rc = plan_launch(reinterpret_cast<const void *>(emo_halo_adj_kernel), 0, q.nitems, props, &ap))) return rc;
        for (int k = Nt - 1; k >= 0; --k) {
            q.uk = k == 0 ? u : plane(k - 1);
            q.lin = k + 1 == Nt ? g : plane(k + 1 == Nt - 1 ? Nt - 1 : k + 1);
            q.lout = k == 0 ? gi : plane(k == Nt - 1 ? Nt - 1 : k);
            if ((rc = launch(ap, &q, st))) return rc;
        }
        if (gi) {
            const long long ncells = nb * 4 * N;
            emo_halo_fold_kernel<<<(unsigned)((ncells + 255) / 256), 256, 0, st>>>(N, ncells, edge, gi);
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

}  // namespace halo
}  // namespace pde
