/*
 * sbd.h - C ABI of libsbd.so, the B200-native (sm_100a, fp64) engine for the
 * SAPG / MYULA semi-blind TV-deblurring hot path of
 * charles-kmc/Semi-blind-image-deblurring-problems-with-TV.
 *
 * The reference has no FFI; its operator interface is MATLAB function handles
 * in the `op` struct (SAPG/SAPG_algorithm_Guassian.m:58-64) and the positional
 * signatures of the utils/ functions.  Each entry point below names the
 * reference interface (file:line) it replaces; the MEX gateway in
 * `mex/sbd_mex.c` and the ctypes binding in `sbd_b200/_lib.py` bind exactly
 * these symbols.
 *
 * Conventions
 *  - every image pointer is a HOST pointer to a MATLAB-layout (column-major)
 *    rows x cols array of IEEE doubles, caller-owned; data is copied in/out.
 *    Entry points ending in `_dev` take DEVICE pointers in the same layout.
 *  - return 0 on success, a negative SBD_E_* code on failure; nothing is ever
 *    thrown across the ABI.  `sbd_last_error` returns the text of the last
 *    failure on that context (or of the last failed sbd_create if ctx==NULL).
 *  - a context is bound to one GPU and is not re-entrant (MATLAB/Octave call
 *    MEX functions from the single interpreter thread).
 *  - there is no CPU fallback: without a usable sm_100 device sbd_create fails.
 */
#ifndef SBD_H_
#define SBD_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SBD_VERSION 100

/* error codes */
#define SBD_OK            0
#define SBD_E_INVALID    -1   /* bad argument (size, NULL pointer, unknown model ...) */
#define SBD_E_CUDA       -2   /* CUDA runtime error (text in sbd_last_error)          */
#define SBD_E_NODEVICE   -3   /* no usable GPU                                        */
#define SBD_E_NOMEM      -4   /* device allocation failed                             */
#define SBD_E_COMM       -5   /* NCCL error / communicator not initialised            */
#define SBD_E_UNSUPPORTED -6  /* e.g. FFT operators on a side with a prime factor > 7  */

/* PSF families.  psi = (w1,w2) | (alpha,beta) | (b,-) */
#define SBD_GAUSSIAN 0        /* utils/Gaussian_psf.m:2-19   */
#define SBD_MOFFAT   1        /* utils/moffat_psf.m:2-23     */
#define SBD_LAPLACE  2        /* utils/laplace_psf.m:1-15    */

/* which spatial kernel / spectrum */
#define SBD_K_PSF   0         /* normalised PSF h                                  */
#define SBD_K_DPSI0 1         /* d h / d psi[0]  (diff_fftgaus_w1 | diff_moffat_alpha | diff_laplace_b) */
#define SBD_K_DPSI1 2         /* d h / d psi[1]  (diff_fftgaus_w2 | diff_moffat_beta)                   */

/* operator selector for sbd_blur* */
#define SBD_OP_A    0         /* A   = real(ifft2(H .* fft2(x)))        run_Gaussian_demo.m:136 */
#define SBD_OP_AT   1         /* A'  = real(ifft2(conj(H) .* fft2(x)))  run_Gaussian_demo.m:137 */
#define SBD_OP_D0   2         /* dif_w1 | diff_A_alpha | diff_A_b       run_Gaussian_demo.m:138 */
#define SBD_OP_D1   3         /* dif_w2 | diff_A_beta                   run_Gaussian_demo.m:139 */

typedef struct sbd_ctx sbd_ctx;

/* ------------------------------------------------------------------------
 * Context.  rows x cols is the image size (MATLAB size(x)); the FFT-based
 * operators take every size whose sides lie in [max(psf_size, 2), 4096] and
 * have no prime factor above 7 (other sizes: SBD_E_UNSUPPORTED, naming the
 * side and its factor); the TV entry points (tvnorm, diffh/diffv, tvprox)
 * accept any size >= 2.  `max_batch` is the
 * largest number of images / Markov chains a single call will carry.
 * ---------------------------------------------------------------------- */
int sbd_create(sbd_ctx** out, int rows, int cols, int psf_size, int model,
               double phi, int max_batch, int device);
int sbd_destroy(sbd_ctx* ctx);
const char* sbd_last_error(const sbd_ctx* ctx);
int sbd_version(void);
/* number of kernels this context has launched so far (bench `gpu_launches`) */
long long sbd_launch_count(const sbd_ctx* ctx);
int sbd_synchronize(sbd_ctx* ctx);

/* ------------------------------------------------------------------------
 * PSF builders (utils/psf_gaussian.m:2-19, psf_moffat.m:2-20, psf_laplace.m:1-13
 * and the spatial part of diff_fftgaus_w1/w2.m, diff_moffat_alpha/beta.m,
 * diff_laplace_b.m).  out: psf_size x psf_size, column-major.
 * ---------------------------------------------------------------------- */
int sbd_psf_taps(sbd_ctx* ctx, const double psi[2], int which, double* out);
/* utils/resize.m:1-12 applied to the kernel above: the full rows x cols
 * complex spectrum, split into real and imaginary parts (column-major).     */
int sbd_psf_spectrum(sbd_ctx* ctx, const double psi[2], int which, double* re, double* im);

/* ------------------------------------------------------------------------
 * Blur operators - closures A, AT, dif_* of run_Gaussian_demo.m:136-139,
 * run_moffat_demo.m:134-137, run_laplace_demo.m:105-107.  batch images are
 * stored back to back.  One real forward FFT, a fused PSF multiply and one
 * inverse FFT per image (the spectrum of the PSF is generated on the fly).
 * ---------------------------------------------------------------------- */
int sbd_blur(sbd_ctx* ctx, const double* x, const double psi[2], int op, double* out, int batch);
int sbd_blur_dev(sbd_ctx* ctx, const double* d_x, const double psi[2], int op, double* d_out, int batch);

/* ------------------------------------------------------------------------
 * TV pieces.
 *  sbd_tvnorm  : utils/TVnorm.m:1-2 (periodic backward differences)
 *  sbd_diff    : SALSA/diffh.m:1-3 (axis=1) / SALSA/diffv.m:1-3 (axis=0)
 *  sbd_tvprox  : [f,px,py] = chambolle_prox_TV_stop(g,'lambda',l,'maxiter',K,
 *                'tol',tol,'tau',tau,'dualvars',[px py])
 *                utils/chambolle_prox_TV_stop.m:1-166.  dual_px/dual_py may be
 *                NULL (zero start, :68-69).  px/py/iters/err outputs may be NULL.
 *                maxiter < 1 is an error (the reference leaves MaxIter
 *                undefined, :80/:131).  Each image of the batch stops on its
 *                own `err <= tol` test exactly like the reference loop.
 *                sbd_tvprox_dev: d_f must not overlap d_g (the last fused block
 *                writes f while other blocks still read g) - SBD_E_INVALID otherwise.
 * ---------------------------------------------------------------------- */
int sbd_tvnorm(sbd_ctx* ctx, const double* x, double* out, int batch);
int sbd_diff(sbd_ctx* ctx, const double* x, int axis, double* out, int batch);
int sbd_tvprox(sbd_ctx* ctx, const double* g, double lambda, int maxiter, double tol,
               double tau, const double* dual_px, const double* dual_py,
               double* f, double* px, double* py, int* iters, double* err, int batch);
int sbd_tvprox_dev(sbd_ctx* ctx, const double* d_g, double lambda, int maxiter, double tol,
                   double tau, double* d_f, int* iters, double* err, int batch);

/* ------------------------------------------------------------------------
 * Likelihood closures evaluated in ONE pass over x (op.f, op.gradF,
 * op.grad_w1/w2 | grad_alpha/beta | grad_b, op.gradF_sigma, op.g, op.logPi:
 * run_Gaussian_demo.m:171-175,187,195).
 *   scal[0] = f          = ||y - A x||_F^2 / (2 sigma2)
 *   scal[1] = grad_psi0  = sum((D0 x).*(A x - y)) / sigma2
 *   scal[2] = grad_psi1
 *   scal[3] = gradF_sigma= ||y - A x||^2/(2 sigma2^2) - numel/(2 sigma2)
 *   scal[4] = g          = TVnorm(x)
 *   scal[5] = logPi      = -f - theta*g
 *   gradF (nullable)     = real(A'(A x - y))/sigma2, rows x cols
 * ---------------------------------------------------------------------- */
int sbd_likelihood(sbd_ctx* ctx, const double* x, const double* y, const double psi[2],
                   double sigma2, double theta, double scal[6], double* gradF);

/* ------------------------------------------------------------------------
 * Setup stage of the demo scripts, on the device (SURVEY.md 8f-2).
 *  sbd_max_eigenval : utils/max_eigenval_Gaussian_Moffat.m:1-27 / max_eigenval_Laplace.m:28-55 -
 *                     power iteration on A'A at `psi`; x0 (rows x cols, nullable) is the start
 *                     vector the reference draws with randn(im_size) (NULL -> Philox(seed)).
 *  sbd_observe      : run_Gaussian_demo.m:145-168 - Ax = A(x; psi), sigma = ||Ax - mean(Ax)||_F /
 *                     sqrt(numel * 10^(BSNR/10)), y = Ax + sigma * noise (noise nullable -> Philox).
 *                     ax_norm (nullable) receives ||Ax - mean(Ax)||_F (for sigma_min / sigma_max).
 * ---------------------------------------------------------------------- */
int sbd_max_eigenval(sbd_ctx* ctx, const double psi[2], const double* x0, double tol, int max_iter,
                     uint64_t seed, double* val, int* iters);
int sbd_observe(sbd_ctx* ctx, const double* x, const double psi[2], double bsnr, const double* noise,
                uint64_t seed, double* y, double* sigma, double* ax_norm);

/* ------------------------------------------------------------------------
 * Post-SAPG MAP estimate (SURVEY.md 8f-1): SALSA/SALSA_v2.m:156-494 as the demos configure it
 * (run_Gaussian_demo.m:210-242): ADMM with the TV prox computed by chambolle_prox_TV_stop
 * warm-started from the previous dual pair ('TVINITIALIZATION',1,'TViters',tv_iters), the
 * least-squares step invLS = real(ifft2(fft2(.) ./ (|H|^2 + mu))), zero initialisation,
 * stopping criterion 1 (relative change of the objective < tolA, at most maxiter iterations).
 *   objective [maxiter+1], distance [maxiter], mses [maxiter+1] (nullable; mses needs x_true).
 *   n_outer receives the number of outer iterations executed.
 * ---------------------------------------------------------------------- */
int sbd_salsa_tv(sbd_ctx* ctx, const double* y, const double psi[2], double tau, double mu, int maxiter,
                 double tolA, int tv_iters, const double* x_true, double* x, double* objective,
                 double* distance, double* mses, int* n_outer);

/* ------------------------------------------------------------------------
 * SAPG driver: SAPG/SAPG_algorithm_Guassian.m:7-308, SAPG_algorithm_moffat.m:7-297,
 * SAPG_algorithm_laplace.m:7-268 (warm-up MYULA + SAPG main loop + traces).
 * ---------------------------------------------------------------------- */
typedef struct sbd_params {
    /* lengths */
    int32_t samples;            /* op.samples  (total_iter)                               */
    int32_t warmup;             /* op.warmup                                               */
    int32_t burnIn;             /* op.burnIn                                               */
    int32_t n_chains;           /* chains on THIS context (1 = the reference)              */
    /* MYULA */
    double gam;                 /* c.gam*op.gamma | op.gamma          Guassian.m:31        */
    double lamb;                /* c.lam*op.lambda | op.lambda        Guassian.m:30        */
    double prox_lambda;         /* op.lambda (prox uses lambda*theta) run_Gaussian_demo.m:191 */
    int32_t chambolle_maxiter;  /* 25                                 run_Gaussian_demo.m:188 */
    int32_t pad0;
    double chambolle_tol;       /* 1e-3   chambolle_prox_TV_stop.m:78 */
    double chambolle_tau;       /* 0.249  chambolle_prox_TV_stop.m:77 */
    /* theta */
    double th_init, min_th, max_th, c_theta;
    /* PSF parameters (w1,w2 | alpha,beta | b) */
    double psi_init[2], psi_min[2], psi_max[2], c_psi[2];
    double psi_fixed[2];        /* op.w1 / op.alpha / op.b : value used when fix_psi       */
    double psi_true[2];         /* op.w1 ... : true PSF for err_psf                        */
    int32_t fix_psi[2];
    /* sigma^2 */
    double sigma2_init, sigma2_min, sigma2_max, c_sigma2;
    double sigma2_fixed;        /* Gaussian: op.sigma_init; others: op.sigma^2 (Q15)       */
    int32_t fix_sigma;
    int32_t err_psf_lag;        /* 1: Gaussian err_psf uses (w1(ii), w2(ii-1)) (Q9)        */
    /* step size delta(i) = d_scale * i^(-d_exp) / numel */
    double d_scale, d_exp;
    /* noise */
    uint64_t seed;              /* Philox key (used when `noise` == NULL)                  */
    int32_t chain_offset;       /* global id of local chain 0 (Philox stream = id)         */
    int32_t total_chains;       /* chains over all ranks (>= n_chains)                     */
    int32_t post_mean;          /* 1: accumulate posterior mean of X for ii > burnIn       */
    int32_t use_graph;          /* 1: replay each iteration from a CUDA graph; 0: eager launches;
                                   -1: automatic (graph for small problems, rows*cols*n_chains <= 2^21) */
} sbd_params;

typedef struct sbd_traces {
    /* all nullable; lengths in elements */
    double* logPiTrace_WU;      /* [warmup]                                                */
    double* thetas;             /* [samples]                                               */
    double* sigmas;             /* [samples]                                               */
    double* psi0;               /* [samples]  w1s | alphas | bs                            */
    double* psi1;               /* [samples]  w2s | betas                                  */
    double* grad_theta;         /* [samples]                                               */
    double* grad_psi0;          /* [samples]                                               */
    double* grad_psi1;          /* [samples]                                               */
    double* grad_sigma;         /* [samples]                                               */
    double* logPiTraceX;        /* [samples]                                               */
    double* gXTrace;            /* [samples]                                               */
    double* err_psf;            /* [samples]                                               */
    double* err_sample;         /* [samples]  Laplace MSE(X,x) in dB (needs x_true)        */
    double* tol_theta;          /* [samples]                                               */
    double* tol_psi0;           /* [samples]                                               */
    double* tol_psi1;           /* [samples]                                               */
    double* tol_sigma;          /* [samples]                                               */
    double* mean_theta;         /* [samples-burnIn]                                        */
    double* mean_psi0;          /* [samples-burnIn]                                        */
    double* mean_psi1;          /* [samples-burnIn]                                        */
    double* mean_sigma;         /* [samples-burnIn]                                        */
    int32_t* chambolle_iters;   /* [samples] sweeps executed by chain 0's prox             */
    double* X_warm;             /* [n_chains*rows*cols] state after warm-up                */
    double* X_last;             /* [n_chains*rows*cols] last sample                        */
    double* X_mean;             /* [rows*cols] posterior mean (post_mean=1), chain average  */
    double EB[4];               /* theta_EB, psi0_EB, psi1_EB, sigma_EB                    */
    double err_warm0;           /* Laplace err_warm(1) = MSE(X0, x)                        */
    double seconds;             /* execTimeFindParameters (device-timed, whole call)       */
    double seconds_main;        /* device time of the main loop only (samples-1 steps)     */
    long long launches_main;    /* kernels launched inside the main loop                   */
    int32_t last_samp;
    int32_t pad1;
} sbd_traces;

/* y, X0 (nullable -> y), x_true (nullable): rows x cols host images.
 * noise (nullable): [(warmup-1) + (samples-1)] x n_chains x rows x cols doubles,
 * consumed in the order the reference calls randn; NULL -> on-device Philox. */
int sbd_sapg_run(sbd_ctx* ctx, const double* y, const double* X0, const double* x_true,
                 const sbd_params* prm, const double* noise, sbd_traces* out);
/* Device-resident variant used by the throughput bench: y/X0 already in HBM. */
int sbd_sapg_run_dev(sbd_ctx* ctx, const double* d_y, const double* d_X0,
                     const sbd_params* prm, sbd_traces* out);

/* ------------------------------------------------------------------------
 * Multi-GPU: one context per GPU / process.  Chains are sharded over ranks and
 * the per-chain stochastic-gradient sums are all-gathered with NCCL at every
 * outer iteration (generalises `G_b = mean(g_b)`, SAPG_algorithm_moffat.m:170-173).
 * ---------------------------------------------------------------------- */
#define SBD_NCCL_ID_BYTES 128
int sbd_comm_unique_id(char id[SBD_NCCL_ID_BYTES]);
int sbd_comm_init(sbd_ctx* ctx, int nranks, int rank, const char id[SBD_NCCL_ID_BYTES]);
int sbd_comm_destroy(sbd_ctx* ctx);

/* per-phase device timings of the MAIN LOOP of the last sbd_sapg_run
 * (milliseconds summed over the iterations, and how many event pairs were
 * summed); names via sbd_phase_name.  Only filled after sbd_set_profile(ctx,1)
 * (or SBD_PROFILE=1): event pairs are recorded on the compute stream while the
 * iterations are enqueued and resolved after the run, so the run itself is not
 * perturbed by synchronisation. */
#define SBD_N_PHASES 8
int sbd_set_profile(sbd_ctx* ctx, int on);
int sbd_phase_times(const sbd_ctx* ctx, double ms[SBD_N_PHASES], long long calls[SBD_N_PHASES]);
const char* sbd_phase_name(int i);

/* ------------------------------------------------------------------------
 * Posterior statistics of X (no reference counterpart: the reference stubs a
 * Welford accumulator, SAPG_algorithm_Guassian.m:233-235,246,292-293).  For each
 * chain c and block size s = 2^j, j = 0 .. L-1, Welford accumulators (m_c, M2_c)
 * of the block mean over the samples X_ii, ii = burnIn+1 .. samples (the window
 * of post_mean; n = samples - burnIn per chain).  Block (I,J) covers rows
 * [I*s, min((I+1)*s, rows)) x cols [J*s, min((J+1)*s, cols)) and its mean divides
 * by the pixels it actually holds.  Per block the device returns, over the C chains
 * of this context in local chain order:
 *   mean = (sum_c m_c) / C   (at s = 1 bitwise X_mean),  within = sum_c M2_c,
 *   between = sum_c (m_c - mean)^2.
 * From these: var = (within + n*between) / (C*n - 1), std = sqrt(var), and the
 * Gelman-Rubin Rhat = sqrt(((n-1)/n * W + B/n) / W) with W = within / (C(n-1)),
 * B/n = between / (C-1) (NaN for C < 2 or n < 2).  DESIGN.md "Posterior statistics".
 * ---------------------------------------------------------------------- */
/* 0 (default): off.  L in 1..7: every following sbd_sapg_run / sbd_sapg_run_dev accumulates the posterior moments of
   X over ii = burnIn+1..samples at block sizes 1, 2, ..., 2^(L-1) (see DESIGN.md).  Requires burnIn >= 1. */
int sbd_set_posterior(sbd_ctx* ctx, int levels);
/* statistics of the last run at block size 2^level: mean, within, between are ceil(rows/s) x ceil(cols/s)
   (each nullable); n = samples per chain, chains = C on this context. */
int sbd_posterior_stats(const sbd_ctx* ctx, int level, double* mean, double* within, double* between,
                        int* n, int* chains);

/* ------------------------------------------------------------------------
 * Precision and convergence of the posterior statistics (no reference counterpart).  Over the same window and block
 * sizes, per chain c and element:
 *   batch means: batch length b (given, or floor(sqrt(n))), B = floor(n/b) batches covering the first B*b samples of
 *     the window; a Welford pair (mb_c, M2b_c) of the B batch means.  Returned over the C chains:
 *     batch_mean = sum_c mb_c / C, batch_within = sum_c M2b_c, batch_between = sum_c (mb_c - batch_mean)^2.
 *   split halves: h = floor(n/2); half 1 = the first h samples of the window, half 2 = the last h (the middle sample
 *     of an odd n belongs to neither).  Over the 2C half-chains, ordered (c, half 1), (c, half 2):
 *     half_mean = mean of the half-chain means, half_within = sum M2, half_between = sum (m_hc - half_mean)^2.
 * From these and var of sbd_posterior_stats:
 *   tau2 = b (batch_within + B batch_between) / (C B - 1)   (NaN for C B < 2),
 *   ESS = C n var / tau2,  MCSE = sqrt(tau2 / (C n)),
 *   Rhat_split = sqrt(((h-1)/h W + Bh) / W),  W = half_within / (2C(h-1)),  Bh = half_between / (2C-1)
 *                (NaN for h < 2).  DESIGN.md "Posterior statistics".
 * ---------------------------------------------------------------------- */
/* 0 (default): off.  -1: batch length floor(sqrt(n)).  b >= 1: batch length b.  Sticky, like sbd_set_posterior.
   A run with diagnostics needs sbd_set_posterior(ctx, L >= 1); b > n gives B = 0 (zero batch arrays). */
int sbd_set_posterior_diagnostics(sbd_ctx* ctx, int batch_len);
/* diagnostics of the last run at block size 2^level; arrays ceil(rows/s) x ceil(cols/s), each nullable;
   batch_len = b, n_batches = B, half_n = h of that run. */
int sbd_posterior_diagnostics(const sbd_ctx* ctx, int level,
                              double* batch_mean, double* batch_within, double* batch_between,
                              double* half_mean, double* half_within, double* half_between,
                              int* batch_len, int* n_batches, int* half_n);

/* ------------------------------------------------------------------------
 * Marginal credible intervals and the posterior median (no reference counterpart).  Over the same window and block
 * sizes, one streaming estimator per element fed the values of the C chains of this context at every step, in local
 * chain order (N = C*n values): extended P^2 (Jain & Chlamtac 1985, Raatikainen 1987) with 9 markers at the
 * probabilities {0, a/4, a/2, 1/4+a/4, 1/2, 3/4-a/4, 1-a/2, 1-a/4, 1}, a = alpha.  lower = quantile alpha/2,
 * median = 1/2, upper = 1 - alpha/2: the markers q2, q4, q6 for N >= 9; for 1 <= N < 9 the linear interpolation of the
 * N sorted values at h = (N-1)p; NaN for N = 0.  Memory does not grow with C.  DESIGN.md "Credible intervals and the
 * median".
 * ---------------------------------------------------------------------- */
/* 0 (default): off.  0 < alpha < 1: every following SAPG run accumulates the posterior quantiles alpha/2, 1/2,
   1 - alpha/2 at the block sizes of sbd_set_posterior.  Sticky.  Needs sbd_set_posterior(ctx, L >= 1). */
int sbd_set_posterior_quantiles(sbd_ctx* ctx, double alpha);
/* lower, median, upper of the last run at block size 2^level (each nullable, ceil(rows/s) x ceil(cols/s));
   alpha and count = C*n of that run. */
int sbd_posterior_quantiles(const sbd_ctx* ctx, int level, double* lower, double* median, double* upper,
                            double* alpha, long long* count);

/* ------------------------------------------------------------------------
 * Launch-geometry control (no reference counterpart: the reference has no
 * launch geometry).  Used by the parity tests to pin the production geometry
 * of the fused Chambolle kernel at sizes the oracle finishes quickly, and by
 * tuning runs.  Options (value -1 / 0 restores the automatic choice):
 *   "chamb_seg"    rows per marching-warp segment of the fused Chambolle kernel
 *   "chamb_levels" sweeps fused per launch: 4 (default), 3, 1 = single-sweep kernel
 *   "chamb_emit"   0: separate prox-output pass instead of the tail block writing f
 *   "chamb_plan33" 0: plan K = 4k+1 as 4 x k, 1 instead of 4 x (k-2), 3 x 3
 *   "chamb_errsub" sampled stop test (the sum of err_k^2 over a subset of the rows already proves err_k > tol;
 *                  exact fallback otherwise; same k, p and f): 1 whenever the caller does not ask for the value
 *                  of err (SAPG, sbd_tvprox_dev with err == NULL), 0 never, -1 automatic (large problems only)
 *   "chamb_coop"   the whole prox (all sweeps, stop test, f) as ONE cooperative launch, one warp per (row, 64-pixel
 *                  strip), blocks of an image synchronised by a barrier per sweep (tv_coop.cuh): 1 whenever the grid
 *                  fits the device, 0 never, -1 automatic (rows*cols*chains <= 2^21 and none of the options above set)
 *   "overlap"      0: launch the prox of a SAPG iteration on the main stream (serial order) instead of on its own
 *                  stream next to the statistics / scalar update / next gradient (same results either way)
 *   "pdl"          0: launch the fused Chambolle kernels without programmatic dependent launch
 *   "tv_seg"       rows per segment of the TVnorm / single-sweep / output kernels
 *   "geom_chains"  derive the geometry from this many chains instead of the batch
 * sbd_get_geometry: out = {levels, chamb_seg, chamb_grid_x, chamb_grid_y,
 *                          tv_seg, tv_grid_x, tv_grid_y, rows_line_pairs,
 *                          coop_blocks_per_image, coop_units_per_warp}   (the last two 0: the prox of `batch` images
 *                          runs the fused kernels)
 * ---------------------------------------------------------------------- */
#define SBD_N_GEOM 10
int sbd_set_option(sbd_ctx* ctx, const char* name, int value);
int sbd_get_geometry(sbd_ctx* ctx, int batch, int out[SBD_N_GEOM]);

#ifdef __cplusplus
}
#endif
#endif /* SBD_H_ */
