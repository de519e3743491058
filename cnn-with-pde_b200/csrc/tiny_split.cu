// tiny_imagenet.ImprovedDiffusionLayer, the methods its forward never reaches (tiny_imagenet.py:88-233):
//   implicit_diffusion_step / solve_implicit_x / solve_implicit_y   scalar-coefficient ADI: every line
//       of every plane is the same tridiagonal system (bands -r, 1 + 2r, ends 1 + r), solved by the
//       reference's Thomas variant that clamps the pivots at stability_eps instead of shifting them;
//   diffuse_x_explicit / diffuse_y_explicit                         one explicit Neumann step per axis.
// `use_implicit` is stored and never read by the reference, so nothing calls these today; they are here
// for whoever wires the flag up.  All five maps are linear in u with constant coefficients and
// self-adjoint (symmetric bands), so the backward pass is the same kernel applied to the upstream gradient.
//
// Mapping: a plane (<= 64 x 64) sits in a padded shared-memory tile (row stride 65 floats: a thread
// walking its own row and a thread walking its own column both hit 32 distinct banks); 64 threads own
// a plane, thread t solves row t (x sweep) and then column t (y sweep) in registers.  The pivots do not
// depend on the line, the plane or the sample: one thread per axis factorises once per block.  Both
// sweeps of the ADI step run on-chip: one HBM read and one HBM write per cell.  Larger planes, up to 4096 x 4096,
// go to the line-streaming kernels of tiny_split_tiled.cu (tsplit_on_chip decides).
#include "common.cuh"
#include "tiny_split_tiled.cuh"

namespace pde {
namespace tsplit {

constexpr int kMaxN = 64;
constexpr int kStride = kMaxN + 1;
constexpr int kPlanesPerBlock = 2;
constexpr int kThreads = kMaxN * kPlanesPerBlock;

struct Args {
    pde_tiny_split_desc d;
    const float *u;
    float *out;
};

struct Factors {
    float cp[kMaxN];    // c'_i   (tiny_imagenet.py:170,178)
    float inv[kMaxN];   // 1 / clamped pivot
};

// thomas_algorithm_batch's elimination of the constant bands, once (tiny_imagenet.py:169-180)
__device__ void factorise(Factors &f, int n, float am, float bmid, float bend, float eps) {
    f.cp[0] = __fdiv_rn(am, bend);
    f.inv[0] = __fdiv_rn(1.0f, bend);
    for (int i = 1; i < n; ++i) {
        const float b = i == n - 1 ? bend : bmid;
        float denom = __fsub_rn(b, __fmul_rn(am, f.cp[i - 1]));
        denom = denom < eps ? eps : denom;
        f.cp[i] = i < n - 1 ? __fdiv_rn(am, denom) : 0.0f;
        f.inv[i] = __fdiv_rn(1.0f, denom);
    }
}

// one line of n cells at `line` with element stride `st` (floats) inside the tile
__device__ __forceinline__ void solve_line(float *line, int st, int n, float am, const Factors &f) {
    float x[kMaxN];
#pragma unroll
    for (int i = 0; i < kMaxN; ++i) x[i] = i < n ? line[i * st] : 0.0f;
    x[0] = __fmul_rn(x[0], f.inv[0]);
#pragma unroll
    for (int i = 1; i < kMaxN; ++i)
        if (i < n) x[i] = __fmul_rn(__fsub_rn(x[i], __fmul_rn(am, x[i - 1])), f.inv[i]);
#pragma unroll
    for (int i = kMaxN - 2; i >= 0; --i)
        if (i < n - 1) x[i] = __fsub_rn(x[i], __fmul_rn(f.cp[i], x[i + 1]));
#pragma unroll
    for (int i = 0; i < kMaxN; ++i)
        if (i < n) line[i * st] = x[i];
}

// u + k (Neumann second difference), tiny_imagenet.py:205-214
__device__ __forceinline__ void explicit_line(float *line, int st, int n, float k) {
    float x[kMaxN];
#pragma unroll
    for (int i = 0; i < kMaxN; ++i) x[i] = i < n ? line[i * st] : 0.0f;
    if (n < 2) return;
#pragma unroll
    for (int i = 0; i < kMaxN; ++i) {
        const float lo = x[i > 0 ? i - 1 : 0], hi = x[i < kMaxN - 1 ? i + 1 : i];
        float acc;
        if (i == 0) acc = __fsub_rn(hi, x[i]);
        else if (i == n - 1) acc = __fsub_rn(lo, x[i]);
        else acc = __fadd_rn(__fsub_rn(lo, __fmul_rn(2.0f, x[i])), hi);
        if (i < n) line[i * st] = __fadd_rn(x[i], __fmul_rn(k, acc));
    }
}

__global__ void __launch_bounds__(kThreads) tiny_split_kernel(const Args a) {
    __shared__ float tile[kPlanesPerBlock][kMaxN * kStride];
    __shared__ Factors fx, fy;
    const pde_tiny_split_desc &d = a.d;
    const int H = d.H, W = d.W, mode = d.mode;
    const int t = threadIdx.x % kMaxN, g = threadIdx.x / kMaxN;
    if (mode <= 2) {
        if (threadIdx.x == 0 && mode != 2) factorise(fx, W, d.cx[0], d.cx[1], d.cx[2], d.eps);
        if (threadIdx.x == 32 && mode != 1) factorise(fy, H, d.cy[0], d.cy[1], d.cy[2], d.eps);
    }
    __syncthreads();
    float *mine = tile[g];
    const int P = H * W;
    for (long long p0 = (long long)blockIdx.x * kPlanesPerBlock; p0 < d.B; p0 += (long long)gridDim.x * kPlanesPerBlock) {
        const long long p = p0 + g;
        const bool live = p < d.B;
        if (live) {
            const float *src = a.u + (size_t)p * P;
            for (int q = t; q < P; q += kMaxN) mine[(q / W) * kStride + (q % W)] = __ldcs(src + q);
        }
        __syncthreads();
        if (live) {
            if (mode == 0 || mode == 1) { if (t < H) solve_line(mine + t * kStride, 1, W, d.cx[0], fx); }
            else if (mode == 3) { if (t < H) explicit_line(mine + t * kStride, 1, W, d.cx[0]); }
        }
        __syncthreads();
        if (live) {
            if (mode == 0 || mode == 2) { if (t < W) solve_line(mine + t, kStride, H, d.cy[0], fy); }
            else if (mode == 4) { if (t < W) explicit_line(mine + t, kStride, H, d.cy[0]); }
        }
        __syncthreads();
        if (live) {
            float *dst = a.out + (size_t)p * P;
            for (int q = t; q < P; q += kMaxN) __stcs(dst + q, mine[(q / W) * kStride + (q % W)]);
        }
        __syncthreads();
    }
}

// the plane fits tiny_split_kernel's tile; every other plane of the domain takes the line-streaming kernels
inline bool tsplit_on_chip(const pde_tiny_split_desc *d) { return d->H <= kMaxN && d->W <= kMaxN; }

}  // namespace tsplit
}  // namespace pde

using namespace pde;

extern "C" int pde_tiny_split(const pde_tiny_split_desc *d, const float *u, float *out, void *stream) {
    if (!d || d->B < 0 || d->H < 1 || d->W < 1 || d->mode < 0 || d->mode > 4) return PDE_ERR_INVALID;
    if (d->H > tsplit_tiled::kMaxEdge || d->W > tsplit_tiled::kMaxEdge) return PDE_ERR_UNSUPPORTED;
    if (d->B == 0) return PDE_OK;
    if (!u || !out) return PDE_ERR_INVALID;
    DeviceProps props;
    int rc = query_props(&props);
    if (rc) return rc;
    if (!tsplit::tsplit_on_chip(d)) return tsplit_tiled::tiny_split_tiled(d, u, out, props, static_cast<cudaStream_t>(stream));
    int per_sm = 1;
    rc = cached_occupancy(reinterpret_cast<const void *>(tsplit::tiny_split_kernel), tsplit::kThreads, 0, &per_sm);
    if (rc) return rc;
    tsplit::Args a{};
    a.d = *d;
    a.u = u;
    a.out = out;
    const long long want = ((long long)d->B + tsplit::kPlanesPerBlock - 1) / tsplit::kPlanesPerBlock;
    const long long cap = (long long)props.sm_count * per_sm;
    const int grid = (int)(want < cap ? want : cap);
    tsplit::tiny_split_kernel<<<grid, tsplit::kThreads, 0, static_cast<cudaStream_t>(stream)>>>(a);
    return cuda_last_error();
}
