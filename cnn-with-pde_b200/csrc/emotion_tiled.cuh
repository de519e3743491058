// Register-tiled kernels for emotion_recognition.PDELayer (emotion_recognition.py:76-97) when the
// plane edge is a multiple of 16 (the reference model: 48 x 48).  Included by explicit.cu.
//
// A warp owns one plane: half h of the warp (lanes 16h .. 16h+15) holds rows h*N/2 .. of the plane,
// lane `sub` of the half holds CW = N / 16 adjacent columns of those RH = N / 2 rows in registers
// (72 registers for the reference model; every lane is busy).  One explicit step updates a lane's
// rows top to bottom in place (the old row above is carried in registers); per step the two halves
// swap their facing rows once (shfl_xor 16), and per row the only traffic is two warp shuffles for
// the left / right neighbours across lanes plus broadcast shared-memory reads (one per four rows)
// of the row coefficient and of the frozen left / right ghost column for the plane-edge lanes.
// The frozen top / bottom ghost rows live in registers.  All Nt steps run on-chip: one HBM read and
// one HBM write per cell per call.
//
// Backward: the forward steps are replayed into a per-warp history in global memory laid out
// [k][row][column][lane] (each access a coalesced 128 bytes) -- half the trajectory at a time, each
// half replayed from the layer input right before it is reversed, so that the history of the warps in
// flight (8 per SM x 46 KB = 54 MB for the reference model) stays in L2; the reverse pass keeps the
// adjoint plane in registers, streams u^k back row by row a few rows ahead of its use, and accumulates
//   dA_i += lam * d2_row u^k, weighted on the fly by {1, sin 2 pi y_i, sin 4 pi y_i}  (3 registers),
//   dB_j += lam * d2_col u^k per owned column                                        (CW registers),
// in fp32 within a step and in double across steps and planes.  What flows into the frozen ghost ring is summed
// over the steps (top / bottom rows in registers, left / right columns in shared memory by the edge
// lanes) and folded back through the reflection at the end.
//
// Planes in HBM (u0, gout, out, gin) are fp32 or bf16 (template T): a bf16 cell is widened on load (the frozen
// ghosts with it), a result is rounded once on its store (grad_input after the ghost-ring fold); registers, the
// history and every sum are fp32 / double in both instantiations.
#pragma once

namespace pde {
namespace expl {

constexpr int kTileWarps = 4;          // warps per block
constexpr int kTilePartDoubles = 3 + kEmoMaxN;   // per-warp partials: A weighted sums, B per column

__device__ __forceinline__ float shfl_up1(float v) { return __shfl_up_sync(kFullMask, v, 1); }
__device__ __forceinline__ float shfl_dn1(float v) { return __shfl_down_sync(kFullMask, v, 1); }
__device__ __forceinline__ float shfl_x16(float v) { return __shfl_xor_sync(kFullMask, v, 16); }

struct TileShared {
    float a[kEmoMaxN + 8];     // a[1 + i] = a_i, zero padded at both ends
    float b[kEmoMaxN + 8];     // b[1 + j] = b_j, zero padded
    float s1[kEmoMaxN], s2[kEmoMaxN];                 // sin 2 pi y_i, sin 4 pi y_i
    float ghost[kTileWarps][2][kEmoMaxN];             // [warp][left | right][row]: frozen u ghost columns
    float gadj[kTileWarps][kEmoMaxN / 2][32];         // [warp][local row][lane]: adjoint sums of the ghost columns
                                                      // (every lane keeps a slot so the update has no branch;
                                                      // only the plane-edge lanes' slots are read back)
};

__device__ __forceinline__ void tile_coefficients(const EmoArgs &a, TileShared &sh, int N) {
    const int tid = threadIdx.x;
    if (tid < N) {
        float av, bv;
        emo_profile(a.d, a.w6, a.xs, a.ys, tid, &av, &bv);
        sh.a[tid + 1] = av;
        sh.b[tid + 1] = bv;
        const float two_pi = (float)(2.0 * 3.141592653589793), four_pi = (float)(4.0 * 3.141592653589793);
        sh.s1[tid] = sinf(__fmul_rn(two_pi, a.ys[tid]));
        sh.s2[tid] = sinf(__fmul_rn(four_pi, a.ys[tid]));
    }
    if (tid == 0) {
        sh.a[0] = sh.a[N + 1] = 0.f;
        sh.b[0] = sh.b[N + 1] = 0.f;
    }
    __syncthreads();
}

// Geometry of a lane: half h owns rows r0 .. r0 + RH - 1, columns j0 .. j0 + CW - 1.
template <int N>
struct Tile {
    static constexpr int CW = N / 16, RH = N / 2;
};

// load a lane's block of the plane and capture the frozen ghosts (reflect padding of u^0):
// gedge = top ghost row (= row 1) in the upper half, bottom ghost row (= row N - 2) in the lower
template <int N, typename T>
__device__ __forceinline__ void tile_load(const T *__restrict__ src, int half, int sub, int r0, int j0,
                                          float (&u)[N / 2][N / 16], float (&gedge)[N / 16], float *gl, float *gr) {
    constexpr int CW = Tile<N>::CW, RH = Tile<N>::RH;
#pragma unroll
    for (int r = 0; r < RH; ++r)
#pragma unroll
        for (int c = 0; c < CW; ++c) u[r][c] = io_ldg(src + (r0 + r) * N + j0 + c);
#pragma unroll
    for (int c = 0; c < CW; ++c) gedge[c] = half == 0 ? u[1][c] : u[RH - 2][c];
    // left ghost = column 1, right ghost = column N - 2 of u^0
    if (sub == 1 / CW) {
#pragma unroll
        for (int r = 0; r < RH; ++r) gl[r0 + r] = u[r][1 % CW];
    }
    if (sub == (N - 2) / CW) {
#pragma unroll
        for (int r = 0; r < RH; ++r) gr[r0 + r] = u[r][(N - 2) % CW];
    }
    __syncwarp();
}

// one explicit step, in place; identical arithmetic (association, FMA use) to emo_step
template <int N>
__device__ __forceinline__ void tile_step(float (&u)[N / 2][N / 16], const float (&gedge)[N / 16],
                                          const float (&b)[N / 16], const float *sa_r0, const float *gl_r0,
                                          const float *gr_r0, int half, int sub) {
    constexpr int CW = Tile<N>::CW, RH = Tile<N>::RH;
    float up[CW], below[CW];
#pragma unroll
    for (int c = 0; c < CW; ++c) {
        const float facing_top = shfl_x16(u[0][c]);        // lower half's first row, seen from the upper half
        const float facing_bot = shfl_x16(u[RH - 1][c]);   // upper half's last row, seen from the lower half
        up[c] = half == 0 ? gedge[c] : facing_bot;
        below[c] = half == 0 ? facing_top : gedge[c];
    }
    float ai[4], gls[4], grs[4];
#pragma unroll
    for (int r = 0; r < RH; ++r) {
        if ((r & 3) == 0) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                ai[k] = sa_r0[r + k];
                gls[k] = gl_r0[r + k];
                grs[k] = gr_r0[r + k];
            }
        }
        float lfv = shfl_up1(u[r][CW - 1]);
        float rtv = shfl_dn1(u[r][0]);
        if (sub == 0) lfv = gls[r & 3];
        if (sub == 15) rtv = grs[r & 3];
        float nv[CW];
#pragma unroll
        for (int c = 0; c < CW; ++c) {
            const float ct = u[r][c];
            const float dn = (r < RH - 1) ? u[r + 1][c] : below[c];
            const float lf = (c > 0) ? u[r][c - 1] : lfv;
            const float rt = (c < CW - 1) ? u[r][c + 1] : rtv;
            // (dn - 2 ct) + up: 2 ct is exact, so the fused form rounds exactly like emo_step's
            const float dr = fmaf(-2.0f, ct, dn) + up[c];
            const float dc = fmaf(-2.0f, ct, rt) + lf;
            nv[c] = fmaf(b[c], dc, fmaf(ai[r & 3], dr, ct));
        }
#pragma unroll
        for (int c = 0; c < CW; ++c) {
            up[c] = u[r][c];
            u[r][c] = nv[c];
        }
    }
}

template <int N, typename T>
__global__ void __launch_bounds__(kTileWarps * 32) emo_fwd_tiled(const EmoArgs a) {
    constexpr int CW = Tile<N>::CW, RH = Tile<N>::RH;
    __shared__ __align__(16) TileShared sh;
    tile_coefficients(a, sh, N);
    const int lane = threadIdx.x & 31, half = lane >> 4, sub = lane & 15;
    // broadcast: tells the compiler the warp index (and every loop bound made of it) is warp-uniform, so the
    // shuffles inside the plane loop need no WARPSYNC.COLLECTIVE / ENDCOLLECTIVE wrappers (4 extra instructions each)
    const int warp = __shfl_sync(kFullMask, (int)(threadIdx.x >> 5), 0);
    const int r0 = half * RH, j0 = sub * CW;
    float b[CW];
#pragma unroll
    for (int c = 0; c < CW; ++c) b[c] = sh.b[1 + j0 + c];
    float *gl = sh.ghost[warp][0], *gr = sh.ghost[warp][1];
    for (int plane = blockIdx.x * kTileWarps + warp; plane < a.d.B; plane += gridDim.x * kTileWarps) {
        const size_t off = (size_t)plane * N * N;
        float u[RH][CW], gedge[CW];
        tile_load<N>(static_cast<const T *>(a.u0) + off, half, sub, r0, j0, u, gedge, gl, gr);
#pragma unroll 1
        for (int k = 0; k < a.d.Nt; ++k) tile_step<N>(u, gedge, b, sh.a + 1 + r0, gl + r0, gr + r0, half, sub);
        T *o = static_cast<T *>(a.out) + off;
#pragma unroll
        for (int r = 0; r < RH; ++r)
#pragma unroll
            for (int c = 0; c < CW; ++c) io_stcs(o + (r0 + r) * N + j0 + c, u[r][c]);
        __syncwarp();   // the ghost columns are rewritten by the next plane
    }
}

template <int N, typename T>
__global__ void __launch_bounds__(kTileWarps * 32) emo_bwd_tiled(const EmoArgs a, float *hist_all, double *part) {
    constexpr int CW = Tile<N>::CW, RH = Tile<N>::RH;
    constexpr int HROW = CW * 32;               // floats per history row
    __shared__ __align__(16) TileShared sh;
    tile_coefficients(a, sh, N);
    const int lane = threadIdx.x & 31, half = lane >> 4, sub = lane & 15;
    // broadcast: tells the compiler the warp index (and every loop bound made of it) is warp-uniform, so the
    // shuffles inside the plane loop need no WARPSYNC.COLLECTIVE / ENDCOLLECTIVE wrappers (4 extra instructions each)
    const int warp = __shfl_sync(kFullMask, (int)(threadIdx.x >> 5), 0);
    const int r0 = half * RH, j0 = sub * CW;
    const int Nt = a.d.Nt, S1 = (Nt + 1) / 2;   // states per history segment
    float b[CW], bm[CW], bp[CW];
#pragma unroll
    for (int c = 0; c < CW; ++c) {
        b[c] = sh.b[1 + j0 + c];
        bm[c] = sh.b[j0 + c];        // b_{j-1}, zero left of the plane
        bp[c] = sh.b[2 + j0 + c];    // b_{j+1}, zero right of the plane
    }
    float *gl = sh.ghost[warp][0], *gr = sh.ghost[warp][1];
    float *eslot = &sh.gadj[warp][0][lane];              // this lane's column of slots, stride 32
    const int wg = blockIdx.x * kTileWarps + warp;
    float *hist = hist_all + (size_t)wg * (S1 + 1) * RH * HROW + lane;   // S1 states + the parked adjoint
    double dA0 = 0.0, dA1 = 0.0, dA2 = 0.0, dBd[CW];
#pragma unroll
    for (int c = 0; c < CW; ++c) dBd[c] = 0.0;
    const bool edge_l = sub == 0, edge_r = sub == 15;

    for (int plane = wg; plane < a.d.B; plane += gridDim.x * kTileWarps) {
        const size_t off = (size_t)plane * N * N;
        float gedge[CW];
        // ------------------------------ adjoint state
        float lam[RH][CW];   // = gout once the first segment has been replayed
#pragma unroll
        for (int r = 0; r < RH; ++r) eslot[r * 32] = 0.0f;
        float eedge[CW];
#pragma unroll
        for (int c = 0; c < CW; ++c) eedge[c] = 0.f;
        __syncwarp();
        constexpr int AHEAD = 4;    // history rows requested ahead of their use
        // The history holds HALF the trajectory at a time (one checkpoint, the layer input itself):
        // segment 1 = states S1 .. Nt-1, segment 0 = states 0 .. S1-1, each replayed from u^0 into the same
        // slots right before it is reversed.  13 forward steps instead of 9 for Nt = 10, but the history of
        // the warps in flight (54 MB instead of 109) stays in L2 instead of spilling to HBM.
#pragma unroll 1
        for (int seg = (Nt > S1 ? 1 : 0); seg >= 0; --seg) {
        const int kb = seg ? S1 : 0, ke = seg ? Nt : S1;
        // the adjoint plane waits in a spare history slot while the registers replay the forward steps
        float *park = hist + (size_t)S1 * RH * HROW;
        const bool parked = seg == 0 && Nt > S1;
        if (parked) {
#pragma unroll
            for (int r = 0; r < RH; ++r)
#pragma unroll
                for (int c = 0; c < CW; ++c) __stcg(park + (r * CW + c) * 32, lam[r][c]);
        }
        {   // ------------------------------ replay: u^kb .. u^{ke-1} into the history
            float u[RH][CW];
            tile_load<N>(static_cast<const T *>(a.u0) + off, half, sub, r0, j0, u, gedge, gl, gr);
#pragma unroll 1
            for (int k = 0; k < ke; ++k) {
                if (k >= kb) {
                    float *hk = hist + (size_t)(k - kb) * RH * HROW;
#pragma unroll
                    for (int r = 0; r < RH; ++r)
#pragma unroll
                        for (int c = 0; c < CW; ++c) __stcg(hk + (r * CW + c) * 32, u[r][c]);
                }
                if (k + 1 < ke) tile_step<N>(u, gedge, b, sh.a + 1 + r0, gl + r0, gr + r0, half, sub);
            }
        }
        if (parked) {
#pragma unroll
            for (int r = 0; r < RH; ++r)
#pragma unroll
                for (int c = 0; c < CW; ++c) lam[r][c] = __ldcg(park + (r * CW + c) * 32);
        } else {
            const T *go = static_cast<const T *>(a.gout) + off;
#pragma unroll
            for (int r = 0; r < RH; ++r)
#pragma unroll
                for (int c = 0; c < CW; ++c) lam[r][c] = io_ldcs(go + (r0 + r) * N + j0 + c);
        }
        // ------------------------------ reverse over the segment
#pragma unroll 1   // the body is 24 unrolled rows; more copies only thrash the instruction cache
        for (int k = ke - 1; k >= kb; --k) {
            const float *hk = hist + (size_t)(k - kb) * RH * HROW;
            // fp32 partial sums live for one step only (72 terms per lane); across steps and planes
            // the sums are carried in double: the six gradients are sums with heavy cancellation
            float fA0 = 0.f, fA1 = 0.f, fA2 = 0.f, fB[CW];
#pragma unroll
            for (int c = 0; c < CW; ++c) fB[c] = 0.f;
            float uh[RH][CW];
#pragma unroll
            for (int r = 0; r < AHEAD; ++r)
#pragma unroll
                for (int c = 0; c < CW; ++c) uh[r][c] = __ldcg(hk + (r * CW + c) * 32);
            // rows facing the other half: adjoint (old values) now, state when its row has arrived
            float lup[CW], lbelow[CW], uup[CW], ubelow[CW];
#pragma unroll
            for (int c = 0; c < CW; ++c) {
                const float lt = shfl_x16(lam[0][c]), lb = shfl_x16(lam[RH - 1][c]);
                lup[c] = half == 0 ? 0.0f : lb;          // the adjoint ring is zero
                lbelow[c] = half == 0 ? lt : 0.0f;
                const float ut = shfl_x16(uh[0][c]);
                ubelow[c] = half == 0 ? ut : gedge[c];
                uup[c] = gedge[c];                         // upper half; the lower half fills it in below
            }
            {   // the upper half's last row of u^k, needed by the lower half at its first row
                float ulast[CW];
#pragma unroll
                for (int c = 0; c < CW; ++c) ulast[c] = __ldcg(hk + ((RH - 1) * CW + c) * 32);
#pragma unroll
                for (int c = 0; c < CW; ++c) {
                    const float ub = shfl_x16(ulast[c]);
                    if (half == 1) uup[c] = ub;
                }
            }
            float am[4], ai[4], ap[4], gls[4], grs[4], s1v[4], s2v[4];
#pragma unroll
            for (int r = 0; r < RH; ++r) {
                if (r + AHEAD < RH) {
#pragma unroll
                    for (int c = 0; c < CW; ++c) uh[r + AHEAD][c] = __ldcg(hk + ((r + AHEAD) * CW + c) * 32);
                }
                if ((r & 3) == 0) {
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        am[q] = sh.a[r0 + r + q];
                        ai[q] = sh.a[r0 + r + q + 1];
                        ap[q] = sh.a[r0 + r + q + 2];
                        gls[q] = gl[r0 + r + q];
                        grs[q] = gr[r0 + r + q];
                        s1v[q] = sh.s1[r0 + r + q];
                        s2v[q] = sh.s2[r0 + r + q];
                    }
                }
                const int q = r & 3;
                float llf = shfl_up1(lam[r][CW - 1]), lrt = shfl_dn1(lam[r][0]);
                float ulf = shfl_up1(uh[r][CW - 1]), urt = shfl_dn1(uh[r][0]);
                if (edge_l) { llf = 0.0f; ulf = gls[q]; }
                if (edge_r) { lrt = 0.0f; urt = grs[q]; }
                float nv[CW], qa = 0.0f, blv_first = 0.0f, blv_last = 0.0f;
#pragma unroll
                for (int c = 0; c < CW; ++c) {
                    const float lct = lam[r][c], uct = uh[r][c];
                    const float ldn = (r < RH - 1) ? lam[r + 1][c] : lbelow[c];
                    const float udn = (r < RH - 1) ? uh[r + 1][c] : ubelow[c];
                    const float l_lf = (c > 0) ? lam[r][c - 1] : llf, l_rt = (c < CW - 1) ? lam[r][c + 1] : lrt;
                    const float u_lf = (c > 0) ? uh[r][c - 1] : ulf, u_rt = (c < CW - 1) ? uh[r][c + 1] : urt;
                    const float dr = fmaf(-2.0f, uct, udn) + uup[c], dc = fmaf(-2.0f, uct, u_rt) + u_lf;
                    qa = fmaf(lct, dr, qa);
                    fB[c] = fmaf(lct, dc, fB[c]);
                    const float al = ai[q] * lct, blv = b[c] * lct;
                    float v = fmaf(-2.0f, blv, fmaf(-2.0f, al, lct));   // (lct - 2 al) - 2 blv, same rounding
                    v = fmaf(am[q], lup[c], v);
                    v = fmaf(ap[q], ldn, v);
                    v = fmaf(bm[c], l_lf, v);
                    v = fmaf(bp[c], l_rt, v);
                    nv[c] = v;
                    // a_0 lam(0, j) flows into the top ghost row, a_{N-1} lam(N-1, j) into the bottom one
                    if (r == 0 && half == 0) eedge[c] += al;
                    if (r == RH - 1 && half == 1) eedge[c] += al;
                    if (c == 0) blv_first = blv;
                    if (c == CW - 1) blv_last = blv;
                }
                fA0 += qa;
                fA1 = fmaf(qa, s1v[q], fA1);
                fA2 = fmaf(qa, s2v[q], fA2);
                eslot[r * 32] += edge_r ? blv_last : blv_first;   // b_0 lam(i, 0) / b_{N-1} lam(i, N-1): ghost columns
#pragma unroll
                for (int c = 0; c < CW; ++c) {
                    lup[c] = lam[r][c];
                    uup[c] = uh[r][c];
                    lam[r][c] = nv[c];
                }
            }
            dA0 += (double)fA0; dA1 += (double)fA1; dA2 += (double)fA2;
#pragma unroll
            for (int c = 0; c < CW; ++c) dBd[c] += (double)fB[c];
        }
        }
        __syncwarp();
        if (a.need_gin) {
            T *gi = static_cast<T *>(a.gin) + off;
#pragma unroll
            for (int r = 0; r < RH; ++r)
#pragma unroll
                for (int c = 0; c < CW; ++c) {
                    float v = lam[r][c];
                    if (half == 0 && r == 1) v += eedge[c];            // row 1 <- top ghost
                    if (half == 1 && r == RH - 2) v += eedge[c];       // row N - 2 <- bottom ghost
                    if (c == 1 % CW) {        // column 1 <- left ghost (summed by the half's lane 0)
                        const float e = sh.gadj[warp][r][half * 16];
                        v += (sub == 1 / CW) ? e : 0.0f;
                    }
                    if (c == (N - 2) % CW) {  // column N - 2 <- right ghost (summed by the half's lane 15)
                        const float e = sh.gadj[warp][r][half * 16 + 15];
                        v += (sub == (N - 2) / CW) ? e : 0.0f;
                    }
                    io_stcs(gi + (r0 + r) * N + j0 + c, v);
                }
        }
        __syncwarp();
    }
    // per-warp partials (double): weighted A sums over all lanes, B per column over the two halves
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        dA0 += __shfl_xor_sync(kFullMask, dA0, o);
        dA1 += __shfl_xor_sync(kFullMask, dA1, o);
        dA2 += __shfl_xor_sync(kFullMask, dA2, o);
    }
    double *pw = part + (size_t)wg * kTilePartDoubles;
    if (lane == 0) { pw[0] = dA0; pw[1] = dA1; pw[2] = dA2; }
#pragma unroll
    for (int c = 0; c < CW; ++c) {
        const double s = dBd[c] + __shfl_xor_sync(kFullMask, dBd[c], 16);
        if (half == 0) pw[3 + j0 + c] = s;
    }
}

__global__ void emo_finish_tiled(pde_emo_desc d, int nwarps, const double *__restrict__ part,
                                 const float *__restrict__ xs, float *g_w6) {
    __shared__ double red[3 + kEmoMaxN];
    const int i = threadIdx.x;
    if (i < 3 + d.N) {
        double s = 0.0;
        for (int w = 0; w < nwarps; ++w) s += part[(size_t)w * kTilePartDoubles + i];
        red[i] = s;
    }
    __syncthreads();
    if (i == 0) {
        const float two_pi = (float)(2.0 * 3.141592653589793), four_pi = (float)(4.0 * 3.141592653589793);
        const double ka = (double)d.half_dt / (double)d.dx2, kb = (double)d.dt / (double)d.dy2;
        double g3 = 0.0, g4 = 0.0, g5 = 0.0;
        for (int q = 0; q < d.N; ++q) {
            const double c1 = (double)cosf(__fmul_rn(two_pi, xs[q])), c2 = (double)cosf(__fmul_rn(four_pi, xs[q]));
            g3 += kb * red[3 + q];
            g4 += kb * red[3 + q] * c1;
            g5 += kb * red[3 + q] * c2;
        }
        g_w6[0] = (float)(ka * red[0]);
        g_w6[1] = (float)(ka * red[1]);
        g_w6[2] = (float)(ka * red[2]);
        g_w6[3] = (float)g3;
        g_w6[4] = (float)g4;
        g_w6[5] = (float)g5;
    }
}

// ------------------------------------------------------------------------------------------ host
// warps in flight per SM during the backward pass: each owns Nt * N * N * 4 bytes of history
// (92 KB for the reference model); 8 per SM keep the whole history (109 MB) inside the 126 MB L2
static int emo_tiled_bwd_grid(const pde_emo_desc *d, int sm_count) {
    const int per_sm = 2;
    int grid = sm_count * per_sm;
    const int want = (d->B + kTileWarps - 1) / kTileWarps;
    if (grid > want) grid = want;
    return grid < 1 ? 1 : grid;
}

static size_t emo_tiled_hist_floats(const pde_emo_desc *d, int grid) {
    const int seg = (d->Nt + 1) / 2;   // the history holds half the trajectory at a time
    return (size_t)grid * kTileWarps * (seg + 1) * (d->N / 2) * (d->N / 16) * 32;   // + the parked adjoint
}

static size_t emo_tiled_workspace_bytes(const pde_emo_desc *d, int sm_count) {
    const int grid = emo_tiled_bwd_grid(d, sm_count);
    return emo_tiled_hist_floats(d, grid) * sizeof(float) + (size_t)grid * kTileWarps * kTilePartDoubles * sizeof(double) + 512;
}

template <int N, typename T>
static int emo_tiled_forward_n(const EmoArgs &a, int sm_count, cudaStream_t st) {
    int per_sm = 1;   // persistent grid: the blocks resident at once (register bound)
    int rc = cached_occupancy(reinterpret_cast<const void *>(emo_fwd_tiled<N, T>), kTileWarps * 32, 0, &per_sm);
    if (rc) return rc;
    const int want = (a.d.B + kTileWarps - 1) / kTileWarps;
    int grid = sm_count * per_sm;
    if (grid > want) grid = want;
    emo_fwd_tiled<N, T><<<grid, kTileWarps * 32, 0, st>>>(a);
    return cuda_last_error();
}

template <typename T>
static int emo_tiled_forward(const EmoArgs &a, int sm_count, cudaStream_t st) {
    switch (a.d.N) {
        case 16: return emo_tiled_forward_n<16, T>(a, sm_count, st);
        case 32: return emo_tiled_forward_n<32, T>(a, sm_count, st);
        case 48: return emo_tiled_forward_n<48, T>(a, sm_count, st);
        default: return PDE_ERR_UNSUPPORTED;
    }
}

template <typename T>
static int emo_tiled_backward(const EmoArgs &a, int sm_count, void *workspace, const float *xs, float *g_w6,
                              cudaStream_t st) {
    const int grid = emo_tiled_bwd_grid(&a.d, sm_count);
    float *hist = reinterpret_cast<float *>((reinterpret_cast<uintptr_t>(workspace) + 255u) & ~(uintptr_t)255u);
    double *part = reinterpret_cast<double *>(hist + emo_tiled_hist_floats(&a.d, grid));
    switch (a.d.N) {
        case 16: emo_bwd_tiled<16, T><<<grid, kTileWarps * 32, 0, st>>>(a, hist, part); break;
        case 32: emo_bwd_tiled<32, T><<<grid, kTileWarps * 32, 0, st>>>(a, hist, part); break;
        case 48: emo_bwd_tiled<48, T><<<grid, kTileWarps * 32, 0, st>>>(a, hist, part); break;
        default: return PDE_ERR_UNSUPPORTED;
    }
    int rc = cuda_last_error();
    if (rc) return rc;
    emo_finish_tiled<<<1, 3 + kEmoMaxN + 29, 0, st>>>(a.d, grid * kTileWarps, part, xs, g_w6);
    return cuda_last_error();
}

}  // namespace expl
}  // namespace pde
