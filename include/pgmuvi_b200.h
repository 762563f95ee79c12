/*
 * pgmuvi_b200 - C ABI of the B200-native exact-GP training engine.
 *
 * Drop-in boundary for ONE path of ICSM/pgmuvi: spectral-mixture kernel build ->
 * Cholesky exact marginal log-likelihood -> hyper-parameter gradient -> Adam step.
 * The reference has no FFI of its own (it is pure Python on GPyTorch); each entry point
 * below cites the reference interface it replaces.  A maintainer binds these with ctypes
 * (see INTEGRATION.md); pgmuvi_b200/_lib.py is that binding.
 *
 * Conventions
 *  - plain pointers and sizes; every pointer is a DEVICE pointer unless it says "host";
 *  - all buffers are caller-owned, kernels never allocate, outputs are written in place;
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *  - return value: 0 ok, <0 bad argument / launch failure (pgm_last_error() has the text);
 *  - per-light-curve status goes to info[B]:
 *        0      Cholesky succeeded without jitter
 *        1..3   succeeded after adding jitter 1e-8*10^(k-1) (f64) / 1e-6*10^(k-1) (f32)
 *               to the diagonal (GPyTorch psd_safe_cholesky ladder, SURVEY.md A.5)
 *        -1     NaN in K~ (GPyTorch NanError): a NaN in x, in the fixed noise or in a raw
 *               parameter other than the mean, also when an earlier pivot is not positive
 *        -2     not positive definite after 3 jitter tries (GPyTorch NotPSDError)
 *    A light curve with info < 0 has NaN mll and grad_raw, and alpha_out (where an entry point
 *    has one) is NaN over [0, n_valid) and 0 beyond.
 *
 * Packed raw-parameter layout, P = 1 + Q + 2*Q*ds (+1 if PGM_FLAG_LEARN_NOISE) + NL:
 *     [ mean | w[0..Q) | mu[q*ds+k] | sigma[q*ds+k] | (learned noise) | lam[0..NL) ]
 * mirroring gpytorch's raw_constant, raw_mixture_weights [Q], raw_mixture_means [Q,1,ds],
 * raw_mixture_scales [Q,1,ds], raw_noise [1] (pgmuvi/lightcurve.py:3847-3849, 6475-6480).
 * ds = d for the plain spectral-mixture kinds; the separable kinds (d = 2, pgmuvi/gps.py:
 * 1327-1336: SM(time) * k(wavelength)) have ds = 1 and NL wavelength-kernel parameters
 *     lam = [ raw_outputscale, raw_lengthscale (, raw_alpha) ]  or  [ raw_constant ].
 */
#ifndef PGMUVI_B200_H
#define PGMUVI_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* kernel kinds: gpytorch.kernels.SpectralMixtureKernel as instantiated at
 * pgmuvi/gps.py:208 (1-D) and :305 (ard_num_dims=2). */
#define PGM_KIND_SM1D 0          /* d = 1: sum_q w_q E_q C_q                               */
#define PGM_KIND_SM_ARD_PRODSUM 1 /* d = 2: prod_d sum_q w_q E_qd C_qd  (GPyTorch order)    */
#define PGM_KIND_SM_ARD_SUMPROD 2 /* d = 2: sum_q w_q prod_d E_qd C_qd  (switchable variant) */
/* separable SM(time) * wavelength kernel, gps.py:990-1002 x 1045-1072, product at :1327-1336 */
#define PGM_KIND_SEP_RBF 3      /* ScaleKernel(RBFKernel):        os exp(-tau^2 / 2 l^2)       NL=2 */
#define PGM_KIND_SEP_MATERN15 4 /* ScaleKernel(MaternKernel 1.5): os (1+s3 r) exp(-s3 r)       NL=2 */
#define PGM_KIND_SEP_RQ 5       /* ScaleKernel(RQKernel):         os (1+tau^2/2 a l^2)^-a      NL=3 */
#define PGM_KIND_SEP_CONST 6    /* ConstantKernel (AchromaticGPModel, gps.py:1414-1415)        NL=1 */

/* N3 - stationary time kernels instead of the spectral mixture (pgmuvi/gps.py:985-990: the
 * reference's DEFAULT time kernel of the separable models is ScaleKernel(MaternKernel(1.5));
 * MaternGPModel gps.py:1131-1184).  kernel_kind = PGM_KIND_STAT(tk, wk):
 *   tk 0 ScaleKernel(RBFKernel), 1 ScaleKernel(MaternKernel(nu=1.5)),           (time)
 *      2 quasi-periodic ScaleKernel(PeriodicKernel * RBFKernel), gps.py:915-935:
 *        os exp(-2 sin^2(pi tau / p) / lambda) exp(-tau^2 / (2 l^2)), slots os, lambda, p, l
 *      3 quasi-periodic + ScaleKernel(RBFKernel) (PeriodicPlusStochasticGPModel,
 *        gps.py:1187-1236; wk = 0 only), slots os, lambda, p, l, os2, l2
 *      4 / 5 ScaleKernel(MaternKernel(nu = 0.5 | 2.5)) (MaternGPModel nu, gps.py:1166-1179;
 *        wk = 0 only), slots os, l
 *   wk 0 none (d = 1), 1 ScaleKernel(RBF), 2 ScaleKernel(Matern-1.5), 3 ScaleKernel(RQ),
 *      4 ConstantKernel                                                          (wavelength)
 * Pass Q = 0; packed layout [ mean | (noise) | time-kernel parameters (os_t, l_t | os, lambda,
 * p, l) | wavelength parameters as above ]. */
#define PGM_KIND_STAT_BASE 8
#define PGM_KIND_STAT(tk, wk) (PGM_KIND_STAT_BASE + 5 * (tk) + (wk))

/* constraint kinds: gpytorch.constraints chosen at pgmuvi/lightcurve.py:3817-4008 */
#define PGM_CON_NONE 0     /* value = raw                                         */
#define PGM_CON_SOFTPLUS 1 /* Positive / GreaterThan(lb): softplus(raw) + lb      */
#define PGM_CON_INTERVAL 2 /* Interval(lb, ub): lb + (ub - lb) * sigmoid(raw)     */
#define PGM_CON_RSOFTPLUS 3 /* ub / (softplus(raw) + lb): a Positive / GreaterThan LENGTHSCALE l seen as the
                              frequency scale 1 / (2 pi l) of a spectral-mixture component (ub = 1 / (2 pi)):
                              the flicker term SMK + ScaleKernel(RBFKernel), pgmuvi/gps.py:992-1002          */

/* flags */
#define PGM_FLAG_GRAD 1          /* also compute d MLL / d raw (loss.backward, trainers.py:181) */
#define PGM_FLAG_LEARN_NOISE 2   /* last slot is a learnable homoskedastic noise variance       */
#define PGM_FLAG_BOUNDS_PER_LC 4 /* con_lb / con_ub are [B,P] (else [P], shared)                */
#define PGM_FLAG_TF32X3 16       /* staged engine: the K~^-1 = X^T X products of the gradient run on
                                    the Blackwell tensor cores (tcgen05, 3xTF32, FP32 accumulators in
                                    tensor memory); needs pgm_staged_tf32x3_workspace_bytes          */
#define PGM_FLAG_TF32X3_CHOL 32  /* staged engine, panel schedule (n > 12800): the right-looking trailing
                                    updates C -= L_panel L_panel^T run on tcgen05 (3xTF32) as well; the MLL
                                    then carries fp32-class error (with PGM_FLAG_TF32X3 only, it is the
                                    FP64 value)                                                        */
#define PGM_FLAG_NOSYNC 64       /* staged engine: do not synchronise the stream.  All four passes of the
                                    jitter ladder are enqueued (kernels of a later pass return at once for a
                                    light curve that is already factored); `info` is final when the stream has
                                    drained.  Only where the Cholesky pass is one launch (B * N < 1024 tile rows
                                    in total and N <= 200, i.e. single GPs up to n = 12800 and small batches);
                                    other shapes return an error.  Makes a training loop over ONE GP
                                    (pgmuvi/trainers.py:177-207) a pure enqueue loop.                          */
#define PGM_FLAG_JITTER_F32 8    /* jitter ladder 1e-6, 1e-5, 1e-4 (GPyTorch's float32 cholesky_jitter)
                                    instead of 1e-8, 1e-7, 1e-6; set by the *_f32 entry points, and
                                    by f64 callers whose MODEL is float32                          */

/* optimiser kinds: torch.optim.* as selected at pgmuvi/trainers.py:141-147 */
#define PGM_OPT_SGD 0
#define PGM_OPT_ADAM 1
#define PGM_OPT_ADAMW 2

int pgm_version(void);
const char* pgm_last_error(void); /* host string, thread-local */

/* Bytes of device workspace the f64 / f32 entry points below need for light curves of up
 * to n_max points (independent of B: the workspace is per resident thread block). */
size_t pgm_workspace_bytes(int elem_size, int n_max, int d, int Q, int device);

/*
 * MLL (+ gradient) of B independent light curves.
 * Replaces, per light curve, one pass of  model(train_x) -> -ExactMarginalLogLikelihood ->
 * loss.backward()  (pgmuvi/trainers.py:179-181; gps.py:217-220, 315-318).
 *
 *  x            [B, n_max, d]  inputs (time [, wavelength]), row-major as train_x
 *  n_valid      [B] or NULL    true n per light curve (ragged batches); NULL => n_max
 *  y            [B, n_max]
 *  fixed_noise  [B, n_max] or NULL  per-point noise VARIANCE (FixedNoiseGaussianLikelihood,
 *                                   lightcurve.py:2780-2789), already clamped by the host
 *  raw          [B, P]         packed raw parameters
 *  con_kind     [P] (int32), con_lb / con_ub  [P] or [B,P]   constraint table
 *  mll          [B]   out: per-datum marginal log-likelihood  (loss = -mll)
 *  grad_raw     [B,P] out: d mll / d raw   (only with PGM_FLAG_GRAD; may be NULL otherwise)
 *  info         [B]   out: see above
 */
int pgm_sm_mll_grad_f64(const double* x, const int32_t* n_valid, const double* y,
                        const double* fixed_noise, const double* raw,
                        const int32_t* con_kind, const double* con_lb, const double* con_ub,
                        int B, int n_max, int d, int Q, int kernel_kind, int flags,
                        double* mll, double* grad_raw, int32_t* info,
                        void* workspace, size_t workspace_bytes, void* stream);

/*
 * The same call, additionally returning alpha = K~^-1 (y - c)  ([B, n_max], zero beyond n_valid;
 * needs PGM_FLAG_GRAD).  d mll / d y = -alpha / n, which is all a NON-constant mean function
 * needs: the host evaluates any mean m(x; theta_m) (gpytorch LinearMean, pgmuvi's PowerLawMean /
 * DustMean, pgmuvi/gps.py:31-171, 223-372, 617-780), passes y - m(x) with the constant slot
 * frozen at 0, and chains -alpha / n through d m / d theta_m (loss.backward, trainers.py:181).
 */
int pgm_sm_mll_grad_alpha_f64(const double* x, const int32_t* n_valid, const double* y,
                              const double* fixed_noise, const double* raw,
                              const int32_t* con_kind, const double* con_lb, const double* con_ub,
                              int B, int n_max, int d, int Q, int kernel_kind, int flags,
                              double* mll, double* grad_raw, double* alpha_out, int32_t* info,
                              void* workspace, size_t workspace_bytes, void* stream);

/*
 * N1 - exact posterior prediction at m test inputs per light curve:
 *     mean*[b, s] = c_b + K*^T alpha,     var*[b, s] = k** - || L^-1 k* ||^2    (latent f)
 * Replaces  likelihood(model(x_fine))  in eval mode (pgmuvi/lightcurve.py:9607-9640, 9862, 9937),
 * which the reference evaluates on a 10000-point grid under gpytorch.settings.fast_pred_var
 * (an approximate variance; this is the exact one).  The likelihood's homoskedastic noise is
 * NOT added here (the host adds the learned noise where the reference's likelihood would).
 * Runs the P and T phases of the staged engine, then one persistent kernel over
 * (light curve, 64-point test tile) jobs.  Arguments as pgm_sm_mll_grad_staged_f64, plus
 *   xstar [B, m, d] test inputs (same transformed units as x), mean / var [B, m] outputs.
 * Failed light curves (info < 0) get NaN.  Blocking, like the staged engine.
 */
size_t pgm_predict_workspace_bytes(int n_max, int B, int device);
int pgm_sm_predict_f64(const double* x, const int32_t* n_valid, const double* y,
                       const double* fixed_noise, const double* raw, const int32_t* con_kind,
                       const double* con_lb, const double* con_ub, int B, int n_max, int d, int Q,
                       int kernel_kind, int flags, const double* xstar, int m, double* mean,
                       double* var, int32_t* info, void* workspace, size_t workspace_bytes,
                       void* stream);

/* Persistent grid of the fused kernels for this model family on the current device (SMs x resident
 * blocks per SM): callers that balance the last wave of a batch (pgmuvi_b200/batch.py) need it.
 * -1 on a bad argument. */
int pgm_fused_grid(int d, int Q, int kernel_kind);

/*
 * Staged engine: the same quantities as pgm_sm_mll_grad_f64 (same arguments), computed stage
 * by stage over the whole device: K~ of every light curve lives in HBM as the lower triangle
 * of 64x64 tile images (right-looking blocked Cholesky + inverse + gradient contraction, one
 * output tile per thread block, one launch per dependency stage carrying B x tiles blocks).
 *   B = 1, n_max large: ONE large exact GP (BASELINE configs C3 n = 8000 / C4 n = 32768;
 *                       "single large GPs stay on one GPU");
 *   B large:            batches whose light curves are too long for one block's scratch.
 * Replaces the same reference calls (pgmuvi/trainers.py:179-181) under
 * gpytorch.settings.fast_computations(False, False, False), i.e. the exact Cholesky branch
 * the reference takes only for n <= 800 (SURVEY.md F6).
 * The call is BLOCKING: it synchronises `stream` once per Cholesky pass to learn whether any
 * light curve must repeat it with more jitter (unless PGM_FLAG_NOSYNC).  B <= 65535.
 */
size_t pgm_staged_workspace_bytes(int n_max, int B);
int pgm_sm_mll_grad_staged_f64(const double* x, const int32_t* n_valid, const double* y,
                               const double* fixed_noise, const double* raw,
                               const int32_t* con_kind, const double* con_lb,
                               const double* con_ub, int B, int n_max, int d, int Q,
                               int kernel_kind, int flags, double* mll, double* grad_raw,
                               int32_t* info, void* workspace, size_t workspace_bytes,
                               void* stream);

int pgm_sm_mll_grad_staged_alpha_f64(const double* x, const int32_t* n_valid, const double* y,
                                     const double* fixed_noise, const double* raw,
                                     const int32_t* con_kind, const double* con_lb,
                                     const double* con_ub, int B, int n_max, int d, int Q,
                                     int kernel_kind, int flags, double* mll, double* grad_raw,
                                     double* alpha_out, int32_t* info, void* workspace,
                                     size_t workspace_bytes, void* stream);

/*
 * Dense covariance K + D of each light curve, written to K_out [B, n_max, n_max] (rows /
 * columns >= n_valid are left untouched).  Replaces SpectralMixtureKernel.forward(x, x) +
 * likelihood noise (gps.py:208, 305; lightcurve.py:2786-2807).  Same device code as the
 * fused path's on-the-fly builder; exists for parity tests and the large-n path.
 */
int pgm_sm_kernel_dense_f64(const double* x, const int32_t* n_valid, const double* fixed_noise,
                            const double* raw, const int32_t* con_kind, const double* con_lb,
                            const double* con_ub, int B, int n_max, int d, int Q,
                            int kernel_kind, int flags, double* K_out, void* stream);

/*
 * One optimiser step on packed raw parameters of B light curves, in place.
 * Replaces optimizer.step() (trainers.py:182) for torch.optim.SGD / Adam / AdamW with
 * torch defaults (betas given, eps, weight_decay: Adam -> added to the gradient, AdamW ->
 * decoupled).  grad_mll is d mll / d raw as produced above; the step minimises loss = -mll.
 * `active` ([B] int32 or NULL) masks light curves that already stopped.  step counts from 1.
 */
int pgm_optim_step_f64(double* raw, const double* grad_mll, double* exp_avg, double* exp_avg_sq,
                       const int32_t* active, int B, int P, int optim_kind, double lr,
                       double beta1, double beta2, double eps, double weight_decay, int step,
                       void* stream);

/*
 * Whole training loop on device: maxiter x (MLL+grad -> optimiser step), every light curve
 * independent, no host synchronisation inside.  Replaces pgmuvi.trainers.train
 * (trainers.py:12-209) for a batch: same loss/parameter history and early-stop rule
 * (`stop and i > miniter and std(loss[-stopavg:]) < stop`, trainers.py:200-207).
 *
 *  raw           [B,P]  in: initial raw parameters; out: final
 *  loss_hist     [maxiter, B] out: loss (= -mll) evaluated before each step; NaN after stop
 *  raw_hist      [maxiter+1, B, P] or NULL  out: raw parameters, initial value first
 *  n_iter        [B] out: iterations executed per light curve
 *  opt_state     [2, B, P] scratch for exp_avg / exp_avg_sq (zeroed by the call)
 */
int pgm_sm_fit_f64(const double* x, const int32_t* n_valid, const double* y,
                   const double* fixed_noise, double* raw, const int32_t* con_kind,
                   const double* con_lb, const double* con_ub, int B, int n_max, int d, int Q,
                   int kernel_kind, int flags, int optim_kind, double lr, double beta1,
                   double beta2, double eps, double weight_decay, int maxiter, int miniter,
                   double stop, int stopavg, double* loss_hist, double* raw_hist,
                   int32_t* n_iter, int32_t* info, double* opt_state, void* workspace,
                   size_t workspace_bytes, void* stream);

/*
 * fp32 entry points: the reference's DEFAULT dtype (pgmuvi casts data to torch.float32,
 * lightcurve.py:2434-2446, 742-745; parameters and constraint bounds are fp32 unless the user
 * calls .double()).  Same arguments as the _f64 entry points with float buffers.  Storage is
 * fp32, arithmetic is fp64: inputs are widened into a staging area on device, the fp64 kernels
 * run, results are rounded once to fp32 - i.e. the results are the correctly rounded fp32
 * values of the fp64 path (north-star fp32 bar: 1e-4 relative against the fp64 oracle).
 * The workspace is the _f64 workspace rounded up to 256 bytes, followed by
 * pgm_f32_staging_bytes(...) bytes (maxiter = 0 / want_raw_hist = 0 for pgm_sm_mll_grad_f32).
 * pgm_sm_fit_f32 keeps the optimiser state and the iterates in fp64 on device for the whole
 * loop and narrows raw / loss_hist / raw_hist at the end.
 */
size_t pgm_f32_staging_bytes(int B, int n_max, int d, int Q, int kernel_kind, int flags,
                             int maxiter, int want_raw_hist);
int pgm_sm_mll_grad_f32(const float* x, const int32_t* n_valid, const float* y,
                        const float* fixed_noise, const float* raw, const int32_t* con_kind,
                        const float* con_lb, const float* con_ub, int B, int n_max, int d, int Q,
                        int kernel_kind, int flags, float* mll, float* grad_raw, int32_t* info,
                        void* workspace, size_t workspace_bytes, void* stream);
int pgm_sm_fit_f32(const float* x, const int32_t* n_valid, const float* y,
                   const float* fixed_noise, float* raw, const int32_t* con_kind,
                   const float* con_lb, const float* con_ub, int B, int n_max, int d, int Q,
                   int kernel_kind, int flags, int optim_kind, double lr, double beta1,
                   double beta2, double eps, double weight_decay, int maxiter, int miniter,
                   double stop, int stopavg, float* loss_hist, float* raw_hist, int32_t* n_iter,
                   int32_t* info, void* workspace, size_t workspace_bytes, void* stream);

/*
 * fp32 models on the Blackwell tensor cores ("TF32-refined", north star kernel 2/3).  The staged
 * engine with the third of the flops that only feeds the gradient - K~^-1 = X^T X (lauum), contracted
 * with W = alpha alpha^T - K~^-1 and dK/dtheta - as 3xTF32 tcgen05.mma products: X^T is split into
 * TF32 hi / lo operand images (hi hi + hi lo + lo hi, FP32 accumulation in tensor memory, about
 * 2^-21 relative per product), one CTA per 128x128 tile of K~^-1, contraction in FP64 straight out of
 * tensor memory (K~^-1 is never written anywhere).  The MLL value, the Cholesky factor, the solves and
 * the inverse factor stay on the FP64 path, so `mll` is the same number the _f64 entry returns; the
 * gradient is held to the fp32 acceptance of SURVEY.md section 7 (error against the fp64 oracle <=
 * max(1e-4 relative, the error of the oracle run in float32); tests/test_gpu_tf32x3.py).
 * With PGM_FLAG_TF32X3_CHOL the trailing updates of the panel-schedule Cholesky (n > 12800: 90 % of
 * the factorisation's flops) run on tcgen05 too - north star kernel (2); pgm_sm_mll_grad_tf32x3_f32
 * sets it, the _f64 entry takes it from `flags`.
 *   pgm_sm_mll_grad_staged_tf32x3_f64  double buffers, = pgm_sm_mll_grad_staged_f64 | PGM_FLAG_TF32X3
 *   pgm_sm_mll_grad_tf32x3_f32         float buffers (the reference's default dtype,
 *                                      pgmuvi/lightcurve.py:2434-2446); workspace =
 *                                      pgm_staged_tf32x3_workspace_bytes rounded up to 256 +
 *                                      pgm_f32_staging_bytes(..., 0, 0); float32 jitter ladder
 * Both replace loss = -mll(output, y); loss.backward() of pgmuvi/trainers.py:179-181.  Blocking.
 */
size_t pgm_staged_tf32x3_workspace_bytes(int n_max, int B);
int pgm_sm_mll_grad_staged_tf32x3_f64(const double* x, const int32_t* n_valid, const double* y,
                                      const double* fixed_noise, const double* raw,
                                      const int32_t* con_kind, const double* con_lb,
                                      const double* con_ub, int B, int n_max, int d, int Q,
                                      int kernel_kind, int flags, double* mll, double* grad_raw,
                                      int32_t* info, void* workspace, size_t workspace_bytes,
                                      void* stream);
int pgm_sm_mll_grad_tf32x3_f32(const float* x, const int32_t* n_valid, const float* y,
                               const float* fixed_noise, const float* raw,
                               const int32_t* con_kind, const float* con_lb, const float* con_ub,
                               int B, int n_max, int d, int Q, int kernel_kind, int flags,
                               float* mll, float* grad_raw, int32_t* info, void* workspace,
                               size_t workspace_bytes, void* stream);

/*
 * N2 - batched Lomb-Scargle initialisation (the step before the path).
 * pgm_lombscargle_f64 replaces  LombScargle(t, y, dy).power(freq)  of Lightcurve.fit_LS
 * (pgmuvi/lightcurve.py:4214-4611; astropy floating-mean periodogram, 'standard'
 * normalisation) on the regular grid  freq[k] = f0[b] + k * df[b], k < nf[b]  that
 * LombScargle.autofrequency(nyquist_factor) produces (host: pgmuvi_b200/lombscargle.py).
 *   t, y, dy  [B, n_max] (dy NULL = unit errors), n_valid [B] or NULL
 *   flags     PGM_LS_FIT_MEAN | PGM_LS_CENTER_DATA (astropy defaults: both)
 *   power     [B, nf_max] out (entries k >= nf[b] untouched)
 * pgm_ls_peaks_f64 replaces  find_peaks(power, distance=Nyquist_factor)  + sort by height
 * (lightcurve.py:4531-4532): peak_idx / peak_power [B, num_peaks], highest first, padded with
 * -1 / NaN; scratch = B * nf_max bytes.
 */
#define PGM_LS_FIT_MEAN 1
#define PGM_LS_CENTER_DATA 2
int pgm_lombscargle_f64(const double* t, const int32_t* n_valid, const double* y, const double* dy,
                        int B, int n_max, const double* f0, const double* df, const int32_t* nf,
                        int nf_max, int flags, double* power, void* stream);
int pgm_ls_peaks_f64(const double* power, const int32_t* nf, int B, int nf_max, int distance,
                     int num_peaks, int32_t* peak_idx, double* peak_power, void* scratch,
                     size_t scratch_bytes, void* stream);

/*
 * N4 (first stage) - PSD period summary for whole batches: the summed spectral-mixture PSD
 *   PSD(f) = sum_q w_q exp(-0.5 ((f - mu_q) / sigma_q)^2)   on   logspace(log10 fmin, log10 fmax, n_grid)
 * and its dominant peak = highest local maximum, else the arg-max (the first stage of
 * Lightcurve.get_period_summary, pgmuvi/lightcurve.py:6537-6578, 7474-7482, 7900-7940; the
 * grid expansion, basin-mass intervals and LSP flags that follow are host post-processing and
 * not part of this call).  freq / fscale / weight [B, Q] are the component frequencies, scales
 * and weights in raw data units (Lightcurve._extract_sm_params, :6397-6535).
 *   grid [B, n_grid] or NULL, psd [B, n_grid] (required), dom_idx / dom_freq / dom_height /
 *   n_peaks [B] outputs.
 */
int pgm_sm_psd_peak_f64(const double* freq, const double* fscale, const double* weight,
                        const double* fmin, const double* fmax, int B, int Q, int n_grid,
                        double* grid, double* psd, int32_t* dom_idx, double* dom_freq,
                        double* dom_height, int32_t* n_peaks, void* stream);

/*
 * Expected (Fisher) information of the exact Gaussian log-likelihood l = n * mll in the
 * CONSTRAINED parameters theta (the standard errors of a fit): fisher [B, P, P] with
 *   I_pq = 1/2 tr(K~^-1 dK~/dtheta_p K~^-1 dK~/dtheta_q)   (covariance slots p, q >= 1)
 *   I_00 = 1^T K~^-1 1   (constant mean),   I_0p = 0.
 * K~ includes the noise and the jitter rung its Cholesky needed (info, as the _staged entries:
 * 0..3 the rung, -1 NaN, -2 not positive definite); rows of a light curve with info < 0 are NaN.
 * Runs the P and T phases of the staged engine, then B_s = X dK_s X^T (X = L^-1) per used slot on
 * the FP64 tile engine and the Gram matrix <B_p, B_q> in a fixed order (deterministic); about
 * (P - 1) n^3 flops per light curve.  Same arguments as pgm_sm_mll_grad_staged_f64 (flags:
 * PGM_FLAG_LEARN_NOISE / PGM_FLAG_BOUNDS_PER_LC / PGM_FLAG_JITTER_F32; B <= 65535); workspace =
 * pgm_fisher_workspace_bytes(...) (0 for invalid arguments).  Blocking.
 */
size_t pgm_fisher_workspace_bytes(int n_max, int B, int d, int Q, int kernel_kind, int flags);
int pgm_sm_fisher_f64(const double* x, const int32_t* n_valid, const double* y,
                      const double* fixed_noise, const double* raw, const int32_t* con_kind,
                      const double* con_lb, const double* con_ub, int B, int n_max, int d, int Q,
                      int kernel_kind, int flags, double* fisher, int32_t* info, void* workspace,
                      size_t workspace_bytes, void* stream);

/* Device yardsticks used by bench.py for the self-measured FP64 roofline: runs `iters`
 * dependent-free FP64 DMMA (kind 0), FP64 DFMA (kind 1), FP32 FFMA (kind 2) or interleaved
 * DMMA+DFMA (kind 3, equal flops each) instructions per thread on every SM and returns the
 * achieved TFLOP/s in *tflops (host pointer).  kind 4: dense TF32 tcgen05.mma (M = N = 128, one
 * issuing thread per SM, operands resident in shared memory): the yardstick of the 3xTF32 path,
 * whose effective peak is a third of it. */
int pgm_peak_probe(int kind, int iters, double* tflops_host, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PGMUVI_B200_H */
