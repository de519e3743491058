// Definitions shared by the two implementations of the implicit ADI layers:
//   adi.cu        a lane owns a whole line of one sample pair (plain Thomas recurrences);
//   adi_split.cu  a thread owns HALF a line (twisted factorisation: both halves eliminate
//                 towards the middle at once), P sample pairs share a block and its
//                 coefficient loads.
#pragma once
#include <cstdio>

#include "common.cuh"

namespace pde {
namespace adi {

constexpr int kHeaderBytes = 4096;
constexpr float kAmpLimit = 256.0f;  // see DESIGN.md "reverse reconstruction"

struct Header {
    // written per sweep by prepare_kernel (one block per sweep, no cross-block step); the call-wide
    // flags the backward kernels need are folded from them by header_flags: by the half-line forward
    // kernel into the head of the checkpoint buffer (CkFlags), by the whole-line backward kernel itself
    float scale[PDE_MAX_SWEEPS];
    float t[PDE_MAX_SWEEPS];
    unsigned rmax_bits[PDE_MAX_SWEEPS];
    int clamped[PDE_MAX_SWEEPS];   // 1 if any cell of sweep s sits outside the clamp interval
    // sweeps with the same axis, time, time step and spacing have the same tables (Strang: the
    // closing half sweep of a step and the opening one of the next): slot[s] numbers the distinct
    // ones in order of first appearance, rep[u] is the first sweep of slot u (host computed)
    int nslots;
    short slot[PDE_MAX_SWEEPS];
    short rep[PDE_MAX_SWEEPS];
};
static_assert(sizeof(Header) <= kHeaderBytes, "header too large");

__host__ __device__ inline int sweeps_per_step(const pde_adi_desc &d) { return d.lie ? 2 : 3; }
// axis 0: lines along W (alpha); axis 1: lines along H (beta)
__host__ __device__ inline int sweep_axis(int k_in_step) { return k_in_step == 1 ? 1 : 0; }

__host__ __device__ inline size_t table_elems(const pde_adi_desc &d) {
    return (size_t)d.steps * sweeps_per_step(d) * d.C * d.N * d.N;
}

struct Tables {
    const Header *hdr;
    const float *r, *inv, *e, *msk;
};

__host__ __device__ inline Tables split_tables(const void *tables, const pde_adi_desc &d) {
    Tables t;
    const char *b = static_cast<const char *>(tables);
    t.hdr = reinterpret_cast<const Header *>(b);
    const float *f = reinterpret_cast<const float *>(b + kHeaderBytes);
    const size_t T = table_elems(d);
    t.r = f;
    t.inv = f + T;
    t.e = f + 2 * T;
    t.msk = f + 3 * T;
    return t;
}

// Software prefetch (no register destination).
__device__ __forceinline__ void prefetch_l1(const void *p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// head of the checkpoint buffer (first 256 bytes), written by sfwd_kernel, read by sbwd_kernel
struct CkFlags {
    int mode_exact;    // rebuilding sweep inputs would amplify rounding noise: per-sweep checkpoints
    int any_clamped;   // 1 if any cell of any sweep sits outside the clamp interval
};
constexpr int kCkHeaderFloats = 64;

struct Args {
    pde_adi_desc d;
    int S, sps, G, nitems, need_gin;
    int tile_sets, tmem_cols;
    const char *tables;
    const float *u, *gout, *chan, *skipw;
    float *out, *gin;
    float *scratch, *part_maps, *part_chan, *part_skip;
    // adi_split.cu only: split-layout tables, step checkpoints (written by the forward kernel,
    // read by the backward one) and the number of partial sets per channel
    const float *stab;
    float *ckpt;
    CkFlags *ck_flags;
};

// pde_adi_desc.tuning (include/pde_b200.h)
__host__ __device__ inline int tune_impl(const pde_adi_desc &d) { return d.tuning & 3; }
__host__ __device__ inline int tune_p(const pde_adi_desc &d) { return (d.tuning >> 2) & 7; }
__host__ __device__ inline int tune_qf(const pde_adi_desc &d) { return (d.tuning >> 5) & 7; }
__host__ __device__ inline int tune_np(const pde_adi_desc &d) { return (d.tuning >> 8) & 3; }

// The sweep -> distinct-table map, computed on the host from the schedule (kernel parameter).
struct SlotMap {
    int nslots;
    short slot[PDE_MAX_SWEEPS];
    short rep[PDE_MAX_SWEEPS];
};

// Call-wide flags from the per-sweep header entries, computed by one warp (a few loads per lane).  exact: rebuilding a sweep's input from its output would amplify rounding noise
// by more than kAmpLimit inside some step (DESIGN.md "reverse reconstruction") -> per-sweep
// checkpoints.  any_clamped: some cell of some sweep sits outside the clamp interval.
__device__ __forceinline__ void header_flags(const Header *hdr, int steps, int sps, bool *exact, bool *any_clamped) {
    const int lane = threadIdx.x & 31;
    float amp = 1.0f;
    int cl = 0;
    for (int step = lane; step < steps; step += 32) {
        float a = 1.0f;
        cl |= hdr->clamped[step * sps];
        // the first sweep of a step is never rebuilt (its input is a checkpoint)
        for (int k = 1; k < sps; ++k) {
            a *= 1.0f + 4.0f * __uint_as_float(hdr->rmax_bits[step * sps + k]);
            cl |= hdr->clamped[step * sps + k];
        }
        amp = fmaxf(amp, a);
        if (!(a == a)) amp = __int_as_float(0x7fc00000);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float other = __shfl_xor_sync(kFullMask, amp, o);
        amp = (amp == amp && other == other) ? fmaxf(amp, other) : __int_as_float(0x7fc00000);
        cl |= __shfl_xor_sync(kFullMask, cl, o);
    }
    *exact = amp > kAmpLimit || !(amp == amp);
    *any_clamped = cl != 0;
}

// adi.cu: sums the per-set gradient partials (double, fixed order).  Map partials: nsets_maps sets
// [set][kind][plane] with set % C == channel; channel / skip partials: nsets_small sets.
void launch_finish(const pde_adi_desc &d, int nsets_maps, int nsets_small, const float *part_maps,
                   const float *part_chan, const float *part_skip, const float *skipw, float *g_ab,
                   float *g_atc, float *g_bb, float *g_btc, float *g_chan, float *g_skip, cudaStream_t st);

// one layer's share of a multi-layer finish launch
struct FinishJob {
    pde_adi_desc d;
    int nsets_maps, nsets_small;
    const float *part_maps, *part_chan, *part_skip, *skipw;
    float *g_ab, *g_atc, *g_bb, *g_btc, *g_chan, *g_skip;
};
void launch_finish_multi(int n, const FinishJob *jobs, cudaStream_t st);

// adi_split.cu
namespace split {
// mirrored index of a row / column / line: 0 .. H-1 from the near edge, H .. N-1 from the far edge
// inwards (an involution)
__host__ __device__ __forceinline__ int mirror(int i, int N) {
    const int H = N / 2;
    return i < H ? i : H + (N - 1 - i);
}
// floats per table in the half-line layout [s][c][k/4][line][half][k%4] (k = mirrored cell)
__host__ __device__ inline size_t stab_floats_per_table(const pde_adi_desc &d) {
    const int H = d.N / 2, HQ = (H + 3) / 4;
    return (size_t)d.steps * sweeps_per_step(d) * d.C * HQ * d.N * 2 * 4;
}
bool supported(const pde_adi_desc &d);
size_t table_floats(const pde_adi_desc &d);             // 4 tables in the split layout
size_t checkpoint_bytes(const pde_adi_desc &d);
size_t workspace_bytes(const pde_adi_desc &d);          // partials (+ exact-mode scratch), no checkpoints
int forward(const pde_adi_desc &d, const char *tables, const float *u, const float *chan, const float *skipw,
            float *out, float *ckpt, cudaStream_t st);
int backward(const pde_adi_desc &d, const char *tables, const float *u, const float *gout, const float *chan,
             const float *skipw, const float *ckpt, float *gin, float *g_ab, float *g_bb, float *g_atc,
             float *g_btc, float *g_chan, float *g_skip, void *workspace, size_t workspace_bytes,
             cudaStream_t st);
bool multi_compatible(int n, const pde_adi_desc *d);
int forward_multi(int n, const pde_adi_desc *d, const void *const *tables, const float *u, const float *const *chan,
                  const float *const *skipw, float *const *out, void *const *ckpt, cudaStream_t st);
int backward_multi(int n, const pde_adi_desc *d, const void *const *tables, const float *u, const float *const *gout,
                   const float *const *chan, const float *const *skipw, const void *const *ckpt, float *const *gin,
                   float *const *g_ab, float *const *g_bb, float *const *g_atc, float *const *g_btc, float *const *g_chan,
                   float *const *g_skip, void *const *workspace, const size_t *workspace_bytes, cudaStream_t st);
}  // namespace split

// adi_generic.cu: every other plane edge (2 ... 128, run-time value; one block per sample, state in shared memory)
namespace generic {
bool serves(const pde_adi_desc &d);
size_t tables_bytes(const pde_adi_desc &d);
size_t workspace_bytes(const pde_adi_desc &d);          // accumulators + per-block sweep history; 0 without a device
int prepare(const pde_adi_desc &d, const pde_adi_schedule &sch, const float *ab, const float *bb, const float *atc,
            const float *btc, char *tables, cudaStream_t st);
int forward(const pde_adi_desc &d, const char *tables, const float *u, const float *chan, const float *skipw, float *out,
            cudaStream_t st);
int backward(const pde_adi_desc &d, const char *tables, const float *u, const float *gout, const float *chan,
             const float *skipw, float *gin, float *g_ab, float *g_bb, float *g_atc, float *g_btc, float *g_chan,
             float *g_skip, void *workspace, size_t workspace_bytes, cudaStream_t st);
}  // namespace generic

// adi_wide.cu: 5 ... PDE_ADI_MAX_CHANNELS channels, any edge 2 ... 128 (tables: generic::prepare / tables_bytes)
namespace wide {
bool serves(const pde_adi_desc &d);
size_t workspace_bytes(const pde_adi_desc &d);          // accumulators + per-slot sweep history; 0 without a device
int forward(const pde_adi_desc &d, const char *tables, const float *u, const float *chan, const float *skipw, float *out,
            cudaStream_t st);
int backward(const pde_adi_desc &d, const char *tables, const float *u, const float *gout, const float *chan,
             const float *skipw, float *gin, float *g_ab, float *g_bb, float *g_atc, float *g_btc, float *g_chan,
             float *g_skip, void *workspace, size_t workspace_bytes, cudaStream_t st);
}  // namespace wide

}  // namespace adi
}  // namespace pde
