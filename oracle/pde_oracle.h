/*
 * oracle/pde_oracle.h -- TEST INFRASTRUCTURE, NOT PRODUCT.
 *
 * CPU restatement (plain C) of the PDE layers of MariMamgo/CNN-with-PDE, used only as
 * the parity checker in tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * --impl reference legs.  Nothing under cnn-with-pde_b200/ may include, link or call it.
 *
 * Pinning: the reference ships no tests or golden vectors ("parity unpinned" by the
 * reference itself, SURVEY.md section 8c).  This oracle is pinned instead against
 * fixtures generated from the reference's own Python modules imported unmodified
 * (tests/golden/make_golden.py -> tests/golden/ npz files).
 *
 * The file pde_oracle.c is compiled twice (REAL=float / REAL=double); every entry point
 * exists as <name>_f32 and <name>_f64.
 */
#ifndef PDE_ORACLE_H
#define PDE_ORACLE_H

#ifdef __cplusplus
extern "C" {
#endif

/* Implicit (ADI) family: mnist_test.py:11-198, fashion_mnist.py:18-196, SVHN.py:12-230,
 * cifar10.py:24-211, cifar_2version.py:20-187. */
typedef struct {
    int B, C, N;        /* batch, channels, plane edge (H == W == N)                       */
    int steps;          /* num_steps                                                       */
    int lie;            /* 0: Strang x(dt/2) y(dt) x(dt/2); 1: Lie x(dt/2) y(dt/2)          */
    int smooth;         /* 1: 3-tap replicate-padded mean along the sweep axis             */
    int has_max;        /* 1: clamp(min,max); 0: clamp(min) only                           */
    int chan_op;        /* 0 none; 1 pre-step u<-M u (cifar); 2 post-step u<-K u (SVHN)     */
    int skip;           /* 1: out = sig(w) u0 + (1-sig(w)) u (SVHN.py:74)                   */
    int nthreads;       /* OpenMP threads over samples (<=0: library default)              */
    double dt, hx, hy;  /* time step, spacing used by x sweeps, spacing used by y sweeps   */
    double cmin, cmax;  /* clamp bounds                                                    */
    double eps;         /* stability_eps added to every Thomas pivot                       */
} oracle_adi_desc;

/* maps are [C][N][N]; chan is [C][C] (NULL if chan_op==0); skipw is 1 value (NULL if !skip) */
int oracle_adi_forward_f32(const oracle_adi_desc *d, const float *u,
                           const float *alpha_base, const float *beta_base,
                           const float *alpha_tc, const float *beta_tc,
                           const float *chan, const float *skipw, float *out);
int oracle_adi_forward_f64(const oracle_adi_desc *d, const double *u,
                           const double *alpha_base, const double *beta_base,
                           const double *alpha_tc, const double *beta_tc,
                           const double *chan, const double *skipw, double *out);
/* gin may be NULL.  Parameter gradients are always returned in double. */
int oracle_adi_backward_f32(const oracle_adi_desc *d, const float *u, const float *gout,
                            const float *alpha_base, const float *beta_base,
                            const float *alpha_tc, const float *beta_tc,
                            const float *chan, const float *skipw, float *gin,
                            double *g_alpha_base, double *g_beta_base,
                            double *g_alpha_tc, double *g_beta_tc,
                            double *g_chan, double *g_skipw);
int oracle_adi_backward_f64(const oracle_adi_desc *d, const double *u, const double *gout,
                            const double *alpha_base, const double *beta_base,
                            const double *alpha_tc, const double *beta_tc,
                            const double *chan, const double *skipw, double *gin,
                            double *g_alpha_base, double *g_beta_base,
                            double *g_alpha_tc, double *g_beta_tc,
                            double *g_chan, double *g_skipw);

/* emotion_recognition.py:56-97.  Planes are N x N (Nx == Ny == N), C == 1. */
typedef struct {
    int B, N, Nt;
    int nthreads;
    double dt, dx, dy;  /* dx = Lx/Nx, dy = Ly/Ny                                           */
} oracle_emo_desc;

/* w = {alpha_w1, alpha_w2, alpha_w3, beta_w1, beta_w2, beta_w3}; xs, ys are the
 * registered buffers x (Nx,), y (Ny,). */
int oracle_emotion_forward_f32(const oracle_emo_desc *d, const float *u0, const float *w,
                               const float *xs, const float *ys, float *out);
int oracle_emotion_forward_f64(const oracle_emo_desc *d, const double *u0, const double *w,
                               const double *xs, const double *ys, double *out);
int oracle_emotion_backward_f32(const oracle_emo_desc *d, const float *u0, const float *gout,
                                const float *w, const float *xs, const float *ys,
                                float *gin, double *gw);
int oracle_emotion_backward_f64(const oracle_emo_desc *d, const double *u0, const double *gout,
                                const double *w, const double *xs, const double *ys,
                                double *gin, double *gw);

/* tiny_imagenet.py:14-72 (live path only). */
typedef struct {
    int B, C, H, W, steps;
    int nthreads;
    double dt, cmin, cmax, blend; /* blend = 0.1 (tiny_imagenet.py:49)                      */
} oracle_tiny_desc;

int oracle_tiny_forward_f32(const oracle_tiny_desc *d, const float *u, const float *alpha_base,
                            const float *scaling, float *out);
int oracle_tiny_forward_f64(const oracle_tiny_desc *d, const double *u, const double *alpha_base,
                            const double *scaling, double *out);
int oracle_tiny_backward_f32(const oracle_tiny_desc *d, const float *u, const float *gout,
                             const float *alpha_base, const float *scaling, float *gin,
                             double *g_alpha, double *g_scaling);
int oracle_tiny_backward_f64(const oracle_tiny_desc *d, const double *u, const double *gout,
                             const double *alpha_base, const double *scaling, double *gin,
                             double *g_alpha, double *g_scaling);

/* tiny_imagenet.py:88-233 (dormant methods: scalar-coefficient ADI step, explicit x / y splits). */
int oracle_tiny_split_f32(int B, int H, int W, int mode, const float *cx, const float *cy, float eps, int nthreads,
                          const float *u, float *out);
int oracle_tiny_split_f64(int B, int H, int W, int mode, const double *cx, const double *cy, double eps, int nthreads,
                          const double *u, double *out);

#ifdef __cplusplus
}
#endif
#endif
