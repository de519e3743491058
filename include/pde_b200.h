/*
 * include/pde_b200.h -- C ABI of libpde_b200.so, the sm_100a implementation of the PDE
 * block of MariMamgo/CNN-with-PDE (forward + hand-derived adjoint).
 *
 * The reference has no native code and therefore no FFI: the interface these entry points
 * replace is the `forward` of its seven nn.Module classes plus the autograd graph PyTorch
 * records under them.  Each group below names the reference code it stands in for; the
 * Python binding a maintainer adds (ctypes) is shown in INTEGRATION.md and implemented in
 * cnn-with-pde_b200/_cabi.py.
 *
 * Conventions
 *   - plain pointers and sizes only; every tensor pointer is a DEVICE pointer to contiguous
 *     fp32 NCHW data owned by the caller (torch's caching allocator); nothing is allocated
 *     or freed inside the library; workspaces are caller-provided;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, no call
 *     synchronises the device;
 *   - return value: 0 on success, a negative PDE_ERR_* for argument errors, a positive
 *     cudaError_t if the CUDA runtime reported one.  No exceptions cross the boundary;
 *   - re-entrant across host threads and streams; no setting lives outside the descriptors: which
 *     kernel variant serves a call is a pure function of the descriptor (its `tuning` field
 *     included) and of the device, so forward and backward of one descriptor always agree.  The
 *     only process-level state is a read-mostly cache of per-kernel launch attributes (registers,
 *     occupancy, "shared-memory limit raised"), filled on first use under a mutex;
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef PDE_B200_H
#define PDE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PDE_B200_ABI_VERSION 3

#define PDE_OK 0
#define PDE_ERR_INVALID (-1)      /* NULL pointer, negative size, inconsistent descriptor   */
#define PDE_ERR_UNSUPPORTED (-2)  /* valid for the reference but not built here (see DESIGN) */
#define PDE_ERR_WORKSPACE (-3)    /* workspace / table buffer too small or misaligned       */

#define PDE_MAX_SWEEPS 192        /* 64 Strang steps or 96 Lie steps                        */
#define PDE_MAX_CHANNELS 4        /* channels of the register-resident implicit kernels     */
#define PDE_ADI_MAX_CHANNELS 64   /* bound of pde_adi_desc.C (implicit family)              */

int pde_b200_abi_version(void);
const char *pde_b200_error_string(int code);
/* SM count, compute capability and L2 size of the current device (for the bench harness). */
int pde_b200_device_info(int *sm_count, int *cc_major, int *cc_minor, size_t *l2_bytes);

/* ---------------------------------------------------------------------------------------
 * Implicit ADI family.  Replaces DiffusionLayer.forward  mnist_test.py:44-65,
 * fashion_mnist.py:48-69, SVHN.py:49-76; EnhancedDiffusionLayer.forward cifar10.py:74-114;
 * LearnableDiffusionLayer.forward cifar_2version.py:70-104, and everything they call
 * (get_alpha_beta_at_time, diffuse_{x,y}_vectorized[_parallel], smooth_coefficients,
 * thomas_solver_batch[_optimized], apply_channel_{mixing,coupling}).
 * ------------------------------------------------------------------------------------- */
typedef struct pde_adi_desc {
    int32_t B, C, N;          /* batch, channels, plane edge H == W == N.
                                 C <= PDE_MAX_CHANNELS: N = 8, 12, ... 32 have kernels compiled
                                 for them; any other N in 2 ... 128 while C * N * (N | 1) * 4
                                 bytes <= 200 KB (one sample's planes in one block's shared
                                 memory) and C * N <= 384 (a thread per line).
                                 PDE_MAX_CHANNELS < C <= PDE_ADI_MAX_CHANNELS: any N in 2 ... 128
                                 while C * N * (N | 1) * 4 bytes <= 200 KB (e.g. C <= 48 at 32 x 32,
                                 12 at 64 x 64); no checkpoints (the backward pass replays), no
                                 pde_adi_multi_* (PDE_ERR_UNSUPPORTED)                          */
    int32_t steps;            /* num_steps                                                   */
    int32_t lie;              /* 0 Strang x(dt/2) y(dt) x(dt/2); 1 Lie x(dt/2) y(dt/2)        */
    int32_t smooth;           /* 3-tap replicate smoothing of the clamped map along the sweep */
    int32_t has_max;          /* clamp(min,max) instead of clamp(min)                        */
    int32_t chan_op;          /* 0 none, 1 pre-step u<-M u (cifar), 2 post-step u<-K u (SVHN) */
    int32_t skip;             /* out = sigmoid(w) u0 + (1-sigmoid(w)) u   (SVHN.py:74)        */
    float cmin, cmax, eps;    /* clamp bounds, stability_eps added to every Thomas pivot      */
    int32_t tuning;           /* 0 = automatic.  PDE_ADI_TUNE_* bits force a kernel variant
                                 (tests, A/B timing); results are the same for every value     */
} pde_adi_desc;

/* pde_adi_desc.tuning: implementation (bits 0-1), sample pairs per half-line group (bits 2-4),
 * groups per half-line forward block (bits 5-7), sample pairs per whole-line forward warp
 * (bits 8-9).  Invalid combinations fall back to the automatic choice. */
#define PDE_ADI_TUNE_IMPL_AUTO 0
#define PDE_ADI_TUNE_IMPL_HALF_LINE 1   /* adi_split.cu even for small batches                   */
#define PDE_ADI_TUNE_IMPL_WHOLE_LINE 2  /* adi.cu even where the half-line kernels would serve   */
#define PDE_ADI_TUNE_P(p) (((p) & 7) << 2)    /* 0 auto, 2 or 4                                  */
#define PDE_ADI_TUNE_QF(q) (((q) & 7) << 5)   /* 0 auto, 1, 2 or 4                               */
#define PDE_ADI_TUNE_NP(n) (((n) & 3) << 8)   /* 0 auto, 1 or 2                                  */

/* Per-sweep schedule, built by the host exactly as the reference accumulates it in Python
 * double (current_time += dt/2) and rounded to fp32 the way ATen rounds a Python scalar:
 * t[s] = time at which the coefficient maps are evaluated, dts[s] = time step of the sweep,
 * h2[s] = (spacing**2) of the sweep.  Length = steps * (lie ? 2 : 3) <= PDE_MAX_SWEEPS. */
typedef struct pde_adi_schedule {
    float t[PDE_MAX_SWEEPS];
    float dts[PDE_MAX_SWEEPS];
    float h2[PDE_MAX_SWEEPS];
} pde_adi_schedule;

/* Bytes of device memory for the factorised coefficient tables of one layer call. */
size_t pde_adi_tables_bytes(const pde_adi_desc *d);
/* Bytes of device workspace pde_adi_backward needs (step checkpoints + gradient partials). */
size_t pde_adi_backward_workspace_bytes(const pde_adi_desc *d);

/* Coefficient maps -> clamp -> smoothing -> r -> Thomas pivots, once per call and shared by
 * the whole batch.  Maps are [C][N][N] ((N,N) for the single-channel layers).  `tables`
 * must hold pde_adi_tables_bytes(d) bytes, 256-byte aligned. */
int pde_adi_prepare(const pde_adi_desc *d, const pde_adi_schedule *sched,
                    const float *alpha_base, const float *beta_base,
                    const float *alpha_time_coeff, const float *beta_time_coeff,
                    void *tables, void *stream);

/* u, out: [B][C][N][N].  chan: [C][C] or NULL (chan_op == 0).  skip_weight: 1 value or NULL. */
int pde_adi_forward(const pde_adi_desc *d, const void *tables, const float *u,
                    const float *chan, const float *skip_weight, float *out, void *stream);

/* Training variants of pde_adi_forward / pde_adi_backward.  Replace what autograd keeps between
 * the reference's forward and backward (mnist_test.py:44-65 and the graph recorded under it): here
 * that is the state at the end of every step ("checkpoints": pde_adi_checkpoint_bytes(d) bytes,
 * 256-byte aligned, opaque layout), so that the backward kernel does not recompute the forward
 * trajectory.  pde_adi_checkpoint_bytes returns 0 when the configuration is served by kernels
 * that rebuild the trajectory themselves (plane edges other than 28 / 32, four or more channels); ckpt may
 * then be NULL.  pde_adi_backward (no ckpt) stays valid for every configuration: it makes the
 * checkpoints itself inside its (then batch-sized) workspace.  pde_adi_backward_saved needs
 * pde_adi_backward_saved_workspace_bytes(d) bytes of workspace when ckpt != NULL and
 * pde_adi_backward_workspace_bytes(d) when ckpt == NULL. */
size_t pde_adi_checkpoint_bytes(const pde_adi_desc *d);
size_t pde_adi_backward_saved_workspace_bytes(const pde_adi_desc *d);
int pde_adi_forward_train(const pde_adi_desc *d, const void *tables, const float *u,
                          const float *chan, const float *skip_weight, float *out, void *ckpt,
                          void *stream);
int pde_adi_backward_saved(const pde_adi_desc *d, const void *tables, const float *u, const float *gout,
                           const float *chan, const float *skip_weight, const void *ckpt, float *gin,
                           float *g_alpha_base, float *g_beta_base,
                           float *g_alpha_time_coeff, float *g_beta_time_coeff,
                           float *g_chan, float *g_skip_weight,
                           void *workspace, size_t workspace_bytes, void *stream);

/* gin may be NULL (the layer is the first op of every reference model, so grad_input is
 * normally not needed).  Gradient outputs are OVERWRITTEN (not accumulated): four maps
 * [C][N][N], g_chan [C][C] (or NULL), g_skip_weight 1 value (or NULL). */
int pde_adi_backward(const pde_adi_desc *d, const void *tables, const float *u, const float *gout,
                     const float *chan, const float *skip_weight, float *gin,
                     float *g_alpha_base, float *g_beta_base,
                     float *g_alpha_time_coeff, float *g_beta_time_coeff,
                     float *g_chan, float *g_skip_weight,
                     void *workspace, size_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------------------
 * Several implicit layers applied to the SAME input, one launch per pass instead of one per layer.
 * Replaces the branch loops of MultiScaleExtractor.forward (cifar10.py:272-274: pde1, pde2, pde3 on x)
 * and HybridPDEExtractor.forward (cifar_2version.py:287-288: diffusion1, diffusion2 on x) and what
 * autograd records under them.  Arrays have n <= PDE_MAX_BRANCHES entries, one per layer; the layers
 * may differ in steps, dt, spacing and splitting but must agree in B, C, N, chan_op, skip and tuning
 * (the branches share one kernel instantiation).  PDE_ERR_UNSUPPORTED means "call the layers one by
 * one": the configuration is not served by the half-line kernels or the layers do not agree.
 * Buffer sizes are those of the single-layer queries on d[i]; outputs and grad_input are bit-identical
 * to n single-layer calls, coefficient gradients equal them up to the fp32 summation order (the
 * branches share the resident blocks, so each block sums a different subset of the batch).  gin[i] (each may be NULL, or gin == NULL) receives the gradient of branch i with
 * respect to the input; the caller (autograd) adds them up.
 * ------------------------------------------------------------------------------------- */
#define PDE_MAX_BRANCHES 4
int pde_adi_multi_prepare(int n, const pde_adi_desc *d, const pde_adi_schedule *sched,
                          const float *const *alpha_base, const float *const *beta_base,
                          const float *const *alpha_time_coeff, const float *const *beta_time_coeff,
                          void *const *tables, void *stream);
int pde_adi_multi_forward_train(int n, const pde_adi_desc *d, const void *const *tables, const float *u,
                                const float *const *chan, const float *const *skip_weight, float *const *out,
                                void *const *ckpt, void *stream);
int pde_adi_multi_backward_saved(int n, const pde_adi_desc *d, const void *const *tables, const float *u,
                                 const float *const *gout, const float *const *chan, const float *const *skip_weight,
                                 const void *const *ckpt, float *const *gin,
                                 float *const *g_alpha_base, float *const *g_beta_base,
                                 float *const *g_alpha_time_coeff, float *const *g_beta_time_coeff,
                                 float *const *g_chan, float *const *g_skip_weight,
                                 void *const *workspace, const size_t *workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------------------
 * Explicit family, frozen reflected ghost ring.  Replaces PDELayer.forward / alpha / beta
 * emotion_recognition.py:76-97.
 * ------------------------------------------------------------------------------------- */
typedef struct pde_emo_desc {
    int32_t B, N, Nt;         /* batch, plane edge (Nx == Ny == N <= 64), int(T/dt)           */
    float half_dt;            /* fp32(0.5*dt)      (scalar in alpha())                       */
    float dt;                 /* fp32(dt)          (scalar in beta())                        */
    float dx2, dy2;           /* fp32(dx**2), fp32(dy**2)                                    */
    int32_t tuning;           /* 0 = automatic; PDE_EMO_TUNE_GENERIC forces the shared-memory
                                 kernels where the register-tiled ones would serve            */
} pde_emo_desc;
#define PDE_EMO_TUNE_GENERIC 1

size_t pde_emotion_backward_workspace_bytes(const pde_emo_desc *d);
/* w6 = {alpha_w1, alpha_w2, alpha_w3, beta_w1, beta_w2, beta_w3}; xs, ys: the registered
 * buffers x (N,), y (N,).  u0, out: [B][1][N][N]. */
int pde_emotion_forward(const pde_emo_desc *d, const float *u0, const float *w6, const float *xs,
                        const float *ys, float *out, void *stream);
int pde_emotion_backward(const pde_emo_desc *d, const float *u0, const float *gout, const float *w6,
                         const float *xs, const float *ys, float *gin, float *g_w6,
                         void *workspace, size_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------------------
 * Explicit family, zero ghosts, per-channel scalars.  Replaces ImprovedDiffusionLayer.forward
 * and simple_diffusion_step, tiny_imagenet.py:34-72.
 *
 * Domain: 1 <= H, W <= 4096 (any combination: odd sizes and rectangles), 0 <= steps <= 16,
 * 1 <= C <= 1024, fp32 and bf16 I/O.  Smaller planes also take more than 16 steps where the
 * whole-plane kernels hold a plane and its step states in one block's shared memory.  Two kernel
 * families serve it, chosen per pass: the whole-plane ring kernels wherever they fit (W % 4 == 0,
 * for bf16 also H * W % 8 == 0, and the plane plus its step states within shared memory), the tiled
 * kernels everywhere else in the domain.  Anything else is PDE_ERR_UNSUPPORTED; B = 0 is a no-op
 * wherever the domain or the whole-plane kernels serve the descriptor.
 * Alignment: where the whole-plane kernels serve a pass, u / out / gout / gin must be 16-byte
 * aligned; where the tiled kernels do, element alignment is enough (4 bytes fp32, 2 bytes bf16), so a
 * batch slice such as x[1:] of a plane with W % 4 != 0 can be passed as it is.
 * pde_tiny_backward_workspace_bytes serves both I/O types: the largest of what the fp32 and bf16
 * backward passes need, 0 for a descriptor neither serves.
 * ------------------------------------------------------------------------------------- */
typedef struct pde_tiny_desc {
    int32_t B, C, H, W, steps;
    float dt, cmin, cmax, blend;  /* blend = 0.1 (tiny_imagenet.py:49)                        */
} pde_tiny_desc;

size_t pde_tiny_backward_workspace_bytes(const pde_tiny_desc *d);
int pde_tiny_forward(const pde_tiny_desc *d, const float *u, const float *alpha_base,
                     const float *channel_scaling, float *out, void *stream);
/* g_alpha_base, g_channel_scaling: [C], overwritten.  gin may be NULL. */
int pde_tiny_backward(const pde_tiny_desc *d, const float *u, const float *gout,
                      const float *alpha_base, const float *channel_scaling, float *gin,
                      float *g_alpha_base, float *g_channel_scaling,
                      void *workspace, size_t workspace_bytes, void *stream);

/* bf16-I/O variants (SURVEY.md section 8f rank 3): u, out, gout, gin are bfloat16 planes in the same NCHW
 * layout (the whole-plane kernels need H * W a multiple of 8; the tiled ones take any plane); arithmetic, parameters and parameter gradients stay fp32 and the
 * results are rounded to nearest even once, on the way out.  This is the one layer of the reference that
 * is bound by HBM bandwidth, so halving the bytes per cell is what a half-precision pipeline gains from it.
 * Workspace size: pde_tiny_backward_workspace_bytes. */
int pde_tiny_forward_bf16(const pde_tiny_desc *d, const void *u, const float *alpha_base,
                          const float *channel_scaling, void *out, void *stream);
int pde_tiny_backward_bf16(const pde_tiny_desc *d, const void *u, const void *gout,
                           const float *alpha_base, const float *channel_scaling, void *gin,
                           float *g_alpha_base, float *g_channel_scaling,
                           void *workspace, size_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------------------
 * The dormant scalar-coefficient methods of ImprovedDiffusionLayer, tiny_imagenet.py:88-233:
 * implicit_diffusion_step (:88-102), solve_implicit_x / _y (:104-157, with the clamp(denom) Thomas
 * variant of :159-190) and diffuse_x_explicit / diffuse_y_explicit (:199-233).  The reference stores
 * `use_implicit` (:21) and never reads it, so no forward reaches them; these entry points serve a
 * caller that does.  u, out: [B][H][W] planes, H, W <= 64.  All five maps are linear in u and
 * self-adjoint: the gradient with respect to u is the same call on the upstream gradient.
 * ------------------------------------------------------------------------------------- */
#define PDE_TINY_SPLIT_ADI 0          /* x solve with cx, then y solve with cy                  */
#define PDE_TINY_SPLIT_IMPLICIT_X 1
#define PDE_TINY_SPLIT_IMPLICIT_Y 2
#define PDE_TINY_SPLIT_EXPLICIT_X 3
#define PDE_TINY_SPLIT_EXPLICIT_Y 4
typedef struct pde_tiny_split_desc {
    int32_t B, H, W, mode;
    /* implicit modes: {fp32(-r), fp32(1 + 2 r), fp32(1 + r)} with r = coeff * dt / 1.0**2 evaluated in
     * double as the reference does before torch.full rounds it; explicit modes: [0] = fp32(coeff * dt) */
    float cx[3], cy[3];
    float eps;                /* stability_eps: lower clamp of the Thomas pivots                 */
} pde_tiny_split_desc;
int pde_tiny_split(const pde_tiny_split_desc *d, const float *u, float *out, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* PDE_B200_H */
