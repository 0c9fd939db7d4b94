/* libgprb200.so - C ABI of the B200-native GP-regression hot path of GPR.jl.
 *
 * Drop-in boundary (SURVEY.md section 8b): these entry points are what a Julia `ccall`
 * shim bound in place of the four GaussianProcesses.jl calls the reference makes
 * would hit.  Citations are relative to /root/reference.
 *
 *   SEArd(log.(l), log(sf)); GP(X, y, mean, kernel)        examples/maximal_coordinates/CPnoise.jl:38-40
 *       -> gprb_dataset_create (X, shared by the G GPs of a trial)
 *          gprb_batch_create   (y - m(X) per GP; m(.) stays on the host: src/mDynamics.jl:41-55)
 *   update_mll! / update_mll_and_dmll!  (objective inside optimize!, CPnoise.jl:41)
 *       -> gprb_eval           (value-only when grad == NULL)
 *   GaussianProcesses.optimize!(gp, LBFGS(linesearch=BackTracking(order=2)), Optim.Options(...))   CPnoise.jl:41
 *       -> gprb_optimize       (batched lock-step restatement, per-GP masks)
 *   predict_y(gp, Xstar)                                   examples/utils/predictdynamics.jl:13
 *       -> gprb_predict
 *   predict_f / predict_y(gp, Xstar; full_cov=true), rand(gp, Xstar, n)   (GaussianProcesses 0.12.4 GP.jl / GPE.jl)
 *       -> gprb_predict_cov, gprb_sample_posterior
 *   predict_LOO(gp), logp_CVLOO(gp), dlogpdtheta_CVLOO(gp)   (GaussianProcesses 0.12 crossvalidation.jl)
 *       -> gprb_eval_loo
 *   append!(gp, x, y)  (ElasticGPE, GaussianProcesses 0.12 GP.jl)   -> gprb_batch_append
 *   gp.cK / gp.alpha inspection (parity taps)              -> gprb_get_K / _chol / _alpha / _Kinv
 *
 * Conventions
 *   - All matrices are column-major doubles, exactly Julia's Array{Float64} memory.
 *     X is d x n (one CState sample per column, src/CState.jl:20), Xstar is d x m.
 *   - theta per GP has P = d + 2 entries in GaussianProcesses get_params order:
 *         [logNoise, ll_1 .. ll_d, lsigma]      (log std-dev noise, log length-scales, log signal std)
 *   - Every function returns an int status: 0 = OK, < 0 = error (message via gprb_last_error()).
 *     No exceptions cross the boundary.  Numerical status is per GP in info[b]:
 *         0        factorised first try
 *         1..10    succeeded after that many cumulative jitter additions of 1e-6*tr(K)/n (make_posdef!)
 *         -1       not positive definite after 10 jitters  => mll = -Inf (shim maps to objective +Inf)
 *         -2       non-finite theta / kernel matrix        => mll = -Inf
 *   - Caller owns every host buffer; handles own device memory.  Calls are synchronous on return.
 *   - One gprb_ctx per GPU.  Either one process per GPU (ranks launched by torchrun / Distributed.jl / MPI, joined by
 *     gprb_comm_unique_id + gprb_comm_init_rank) or one process driving several GPUs (gprb_init_multi, one host thread
 *     per context or sequential calls); handles of different contexts are independent.
 *   - A GP whose factorisation failed never poisons its batch: every entry point reports per GP and carries on with
 *     the others (the reference swallows a failed trial and continues, examples/parallel/core.jl:41-46).
 *   - There is NO CPU fallback: gprb_init fails when no sm_100 device is present.
 */
#ifndef GPRB200_H
#define GPRB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gprb_ctx gprb_ctx;
typedef struct gprb_dataset gprb_dataset;
typedef struct gprb_batch gprb_batch;

/* kernel_kind: SEArd is the only family the reference uses (18 call sites);
 * Mat12Ard/Mat32Ard/Mat52Ard are the north_star extension (same theta layout). */
enum { GPRB_KERNEL_SE_ARD = 0, GPRB_KERNEL_MAT12_ARD = 1, GPRB_KERNEL_MAT32_ARD = 2, GPRB_KERNEL_MAT52_ARD = 3 };

enum {
  GPRB_OK = 0,
  GPRB_ERR_ARG = -1,      /* API misuse (null pointer, bad size, mismatched handles) */
  GPRB_ERR_CUDA = -2,     /* CUDA runtime error */
  GPRB_ERR_NODEVICE = -3, /* no sm_100 GPU visible: there is no CPU fallback */
  GPRB_ERR_NOMEM = -4,    /* device allocation failed */
  GPRB_ERR_NCCL = -5      /* NCCL error, or libnccl.so.2 not loadable (only the multi-GPU gather needs it) */
};

int gprb_version(void);               /* major*10000 + minor*100 + patch */
const char* gprb_last_error(void);    /* thread-local, never NULL */

/* ---- context ------------------------------------------------------------------------ */
int gprb_init(gprb_ctx** ctx, int device);
int gprb_destroy(gprb_ctx* ctx);
/* One process, several GPUs (the shape of SURVEY.md section 8b's `gprb_init(ctx**, ngpus, devs)`): creates one context
 * per entry of devs (NULL = devices 0..ngpus-1) and joins them into one NCCL clique (ncclCommInitAll) for
 * gprb_gather_multi.  ctxs receives ngpus handles; destroy each with gprb_destroy. */
int gprb_init_multi(gprb_ctx** ctxs, int32_t ngpus, const int* devs);
/* Device facts for roofline reporting: out[0]=SM count, out[1]=sm clock kHz, out[2]=L2 bytes, out[3]=free HBM bytes */
int gprb_device_info(gprb_ctx* ctx, int64_t out[4]);

/* ---- dataset: X of one trial, uploaded once (CPnoise.jl:26 `reduce(hcat, ...)`) ------ */
int gprb_dataset_create(gprb_ctx* ctx, int64_t n, int32_t d, const double* X, int64_t ldx, gprb_dataset** out);
int gprb_dataset_update(gprb_dataset* ds, const double* X, int64_t ldx); /* same n, d; new samples */
/* Re-upload `count` datasets in one call: all copies are queued back to back (asynchronous when the host matrices are
 * page-locked) and the call returns after one synchronisation.  X[i] is d x n with leading dimension ldx. */
int gprb_datasets_update(gprb_ctx* ctx, int32_t count, gprb_dataset* const* ds, const double* const* X, int64_t ldx);
int gprb_dataset_destroy(gprb_dataset* ds);
/* All the trial datasets of a batch in ONE device allocation: `count` matrices of identical n, d.  When the host
 * matrices are one contiguous block (X[i+1] == X[i] + n*ldx, e.g. a 3-d array of trials) creation and every later
 * gprb_datasets_update is one host->device copy plus one transpose launch instead of `count` of each.
 * out receives `count` handles (each still destroyed individually; the allocation is freed with the last one). */
int gprb_datasets_create(gprb_ctx* ctx, int32_t count, int64_t n, int32_t d, const double* const* X, int64_t ldx,
                         gprb_dataset** out);

/* ---- batch: B independent GPs, GP b uses dataset ds[b] and targets ymm[:, b] ---------- */
/* ymm = y - m(X), n x B column-major.  All datasets must share n and d. */
int gprb_batch_create(gprb_ctx* ctx, int32_t B, gprb_dataset* const* ds, const double* ymm, int32_t kernel_kind,
                      gprb_batch** out);
int gprb_batch_set_targets(gprb_batch* batch, const double* ymm); /* n x B */
/* Fixed per-GP nugget: offset[b] is added to every diagonal entry of K_b (on top of exp(2 logNoise) + eps) in every
 * later evaluation; NULL resets it to 0.  It is part of the matrix make_posdef! sees (tr(K)/n includes it).  Negative
 * values are allowed - the parity tests use them to build matrices that need exactly k >= 2 jitter additions, which
 * positive-semidefinite kernels never produce by rounding alone. */
int gprb_batch_set_diag_offset(gprb_batch* batch, const double* offset /* B or NULL */);
int gprb_batch_destroy(gprb_batch* batch);
/* Append k samples to every dataset of the batch and condition every GP that has a resident state on them, at the theta
 * of that state (GaussianProcesses ElasticGPE append!).
 *   Xnew     one d x k block per distinct dataset of the batch, in order of first use by GP index, leading dimension ldx
 *   ymm_new  k x B    y - m(Xnew) per GP (the prior mean stays on the host, as everywhere)
 *   mll      B  out   (NULL allowed)
 *   info     B  out   (NULL allowed)
 * GPs without a resident state have their data grown, but their outputs are not written and they stay without a state.
 * Afterwards every GP that had a state is in the state gprb_eval(theta, grad = NULL) leaves on the enlarged data, bit for
 * bit (same info, mll, K, factor, alpha and predictions).  A state factorised without jitter keeps the block rows
 * < floor(n / 128) of its factor and refactorises only the rest; a state that carried jitter (1e-6 tr(K)/n depends on n),
 * one with n < 128, and one whose new diagonal blocks fail a pivot get an ordinary value-only evaluation with the
 * make_posdef! ladder.  A following gprb_eval at the same theta with a gradient runs only the inverse and the gradient.
 * Refused with GPRB_ERR_ARG, the batch unchanged: k < 1, a NULL pointer, a prediction in flight on either slot, a dataset
 * that another live batch also uses.  GPRB_ERR_NOMEM leaves the batch unchanged as well. */
int gprb_batch_append(gprb_batch* batch, int64_t k, const double* const* Xnew, int64_t ldx, const double* ymm_new,
                      double* mll, int32_t* info);

/* One objective evaluation per active GP (rows a5-a9 of SURVEY.md section 8a).
 *   theta  P x B    in
 *   active B        in, NULL = all; inactive GPs keep their previous state and outputs are untouched
 *   mll    B        out  log marginal likelihood
 *   grad   P x B    out  d mll / d theta, NULL => value-only (assembly + Cholesky + solve)
 *   info   B        out  see above
 * After return, the factor, alpha and theta of every evaluated GP stay resident for gprb_predict. */
int gprb_eval(gprb_batch* batch, const double* theta, const uint8_t* active, double* mll, double* grad, int32_t* info);

/* Mixed pass: mode[b] = 0 skip, 1 value only, 2 value + gradient.  One pipeline pass evaluates the value-only and the
 * value+gradient GPs together (factorisation for all, inverse + gradient for the mode-2 subset); this is what the
 * batched optimiser issues once per round (line-search trials of some GPs next to the gradient evaluations of the
 * GPs that just accepted a step).  grad may be NULL when no GP asks for mode 2; grad rows of other GPs are untouched. */
int gprb_eval_mixed(gprb_batch* batch, const double* theta, const uint8_t* mode, double* mll, double* grad, int32_t* info);

/* Same evaluation for ALL GPs with theta / outputs already in device memory: no payload crosses PCIe (only the
 * 4-byte per-GP status the make_posdef! retry loop needs).  Ordered after prior work on `stream` (a cudaStream_t);
 * complete on return.  grad_dev / info_dev may be NULL. */
int gprb_eval_device(gprb_batch* batch, const double* theta_dev, double* mll_dev, double* grad_dev, int32_t* info_dev,
                     void* stream);

/* ---- batched L-BFGS + BackTracking(order=2) (Optim 1.4.1 semantics, SURVEY.md A.4/A.5) -- */
typedef struct gprb_lbfgs_opts {
  int32_t m;             /* history, default 10 */
  int32_t iterations;    /* default 1000 */
  int32_t max_evals;     /* 0 = unlimited; per-GP cap on f_calls + fg_calls, checked once per iteration */
  int32_t ls_iterations; /* default 1000 */
  double g_abstol;       /* default 1e-8 on ||g||_inf */
  /* time_limit (seconds, <= 0 = none).  The reference gives EVERY GP its own 10 s of CPU wall clock
   * (Optim.Options(time_limit=10.), CPnoise.jl:41), checked once per iteration.  Two ways to express it:
   *   cost_value == cost_grad == 0 : wall clock of the whole lock-step batch (all GPs stop together);
   *   cost_value, cost_grad  > 0   : deterministic PER-GP virtual clock - a value-only evaluation advances a GP's clock
   *                                  by cost_value seconds and a value+gradient evaluation by cost_grad seconds (the cost of
   *                                  one evaluation on the machine being emulated, e.g. the reference CPU), and a GP stops
   *                                  at the first iteration boundary where its own clock exceeds time_limit - what
   *                                  "10 s per GP" means on the reference, reproducible and independent of GPU speed. */
  double time_limit;
  double c_1, rho_hi, rho_lo; /* 1e-4, 0.5, 0.1 */
  double cost_value, cost_grad; /* virtual seconds per evaluation, default 0 (see time_limit) */
} gprb_lbfgs_opts;

typedef struct gprb_opt_result {
  double mll;          /* final log marginal likelihood at theta_inout */
  double g_norm;       /* ||grad||_inf there */
  int32_t iterations;
  int32_t f_calls;     /* value-only evaluations */
  int32_t fg_calls;    /* value+gradient evaluations */
  int32_t converged;   /* 1 = g_abstol / stall criterion met */
  int32_t ls_failed;   /* 1 = LineSearchException equivalent */
  int32_t info;        /* info of the final evaluation */
} gprb_opt_result;

void gprb_lbfgs_default_opts(gprb_lbfgs_opts* o);
/* theta_inout P x B: start point in, minimiser of -mll out.  Final state is left evaluated at the minimiser
 * (mirrors optimize! writing the minimiser back and calling update_target!). */
int gprb_optimize(gprb_batch* batch, double* theta_inout, const gprb_lbfgs_opts* opts, gprb_opt_result* results);

/* Host-only self test of the batched optimiser state machine (no GPU needed): B copies of the P-dimensional
 * Rosenbrock function, +Inf outside |x_i| <= bound.  results[b].mll carries the final objective value.
 * Test hook for tests/test_lbfgs_cpu.py; not part of the reference-facing surface. */
int gprb_lbfgs_selftest(int32_t B, int32_t P, double* theta_inout, const gprb_lbfgs_opts* opts, double bound,
                        gprb_opt_result* results);

/* ---- prediction (predict_y) ------------------------------------------------------------ */
/* Xstar: d x m column-major.  xstar_stride = 0: the same d x m block is used by every GP; otherwise GP b reads
 * its own block at Xstar + b*xstar_stride doubles (xstar_stride >= d*m).
 *   mstar m x B  prior mean m(x*) evaluated on the host, NULL = zero mean
 *   mu    m x B  out
 *   var   m x B  out, NULL => mean only (the reference discards the variance: predictdynamics.jl:13) */
int gprb_predict(gprb_batch* batch, int64_t m, const double* Xstar, int64_t xstar_stride, const double* mstar,
                 double* mu, double* var);
/* A GP without an evaluated state (never evaluated, or its last evaluation ended with info < 0) does not block the call:
 * its rows of mu / var come back as NaN and every other GP is predicted normally.
 *
 * Asynchronous form for the rollout loop (examples/utils/predictdynamics.jl:11-19): the per-step sequence
 * "device predict -> D2H mu -> host projectv! -> H2D next states" of one group of trials overlaps the host projection of
 * another.  gprb_predict_async enqueues the prediction of the GPs gp0 .. gp1-1 (a contiguous range of the batch, e.g. the
 * G GPs x T/2 trials of one group) on pipeline `slot` (0 or 1; each slot has its own streams, staging and scratch) and
 * returns at once; Xstar / mstar are indexed relative to gp0: GP gp0+k reads the test block
 * Xstar + (k / gps_per_block)*xstar_stride - gps_per_block consecutive GPs (the G outputs of a trial, which all predict
 * from the trial's own states) share one block, so a step uploads each trial's states once, not G times - and the prior
 * means mstar + k*m.  Both are copied to pinned staging before the call returns, so the caller may overwrite them.  gprb_predict_wait blocks until
 * the slot's prediction is complete and writes mu / var ((gp1-gp0) x m each; var may be NULL when want_var was 0).
 * While a prediction is in flight it reads the batch's resident state and the datasets of its GPs on the slot's own
 * streams, which nothing orders with evaluations or uploads.  So until gprb_predict_wait, the calls that write that state
 * are refused with GPRB_ERR_ARG and leave everything unchanged: gprb_eval, gprb_eval_mixed, gprb_eval_device,
 * gprb_eval_loo, gprb_optimize, gprb_batch_set_targets, gprb_batch_set_diag_offset and gprb_batch_append while either
 * slot of the batch is pending, and gprb_dataset_update / gprb_datasets_update of a dataset that a pending prediction
 * of any batch reads. */
int gprb_predict_async(gprb_batch* batch, int32_t slot, int32_t gp0, int32_t gp1, int64_t m, const double* Xstar,
                       int64_t xstar_stride, int32_t gps_per_block, const double* mstar, int32_t want_var);
int gprb_predict_wait(gprb_batch* batch, int32_t slot, double* mu, double* var);
/* Device time (ms, CUDA events on the slot's stream) of the most recent completed prediction on `slot`. */
int gprb_last_predict_ms(gprb_batch* batch, int32_t slot, double* ms);

/* ---- full covariance and posterior draws (predict_f / predict_y with full_cov = true, rand) -------------------- */
/* Synchronous, on prediction slot 0 (refused while slot 0 has an asynchronous prediction in flight); 1 <= m <= 8192,
 * larger m is GPRB_ERR_ARG, a workspace that cannot be allocated GPRB_ERR_NOMEM.  Xstar / xstar_stride / mstar as for
 * gprb_predict.  gprb_last_predict_ms(batch, 0) reports the device time (without the copy of the m x m blocks).
 * With T = L^-1 K*, K** = K_f(X*, X*) (no noise, no eps):
 *   Sigma_f = K** - T'T (symmetric, not clamped),  Sigma_y = Sigma_f + exp(2 logNoise) I
 *   mu   m x B      out, as gprb_predict
 *   cov  m x m x B  out, both triangles; add_noise = 0: Sigma_f (predict_f), 1: Sigma_y (predict_y)
 * A GP without an evaluated state gets NaN mu / cov and blocks nobody. */
int gprb_predict_cov(gprb_batch* batch, int64_t m, const double* Xstar, int64_t xstar_stride, const double* mstar,
                     int32_t add_noise, double* mu, double* cov);
/* Posterior draws of the latent function (rand / rand!): out[:, s, b] = mu_b + L_b Z[:, s, b], L_b the lower Cholesky
 * factor of make_posdef!(Sigma_f) (cumulative Sigma_ii += 1e-6 tr(Sigma)/m, up to 10 times).  The standard normals come
 * from the caller's RNG.
 *   Z    m x ns x B  in
 *   out  m x ns x B  out
 *   info B           out: 0..10 jitter rung, -1 still indefinite after 10 jitters, -2 non-finite Sigma_f or no evaluated
 *                    state; a GP with info < 0 gets NaN draws and blocks nobody */
int gprb_sample_posterior(gprb_batch* batch, int64_t m, const double* Xstar, int64_t xstar_stride, const double* mstar,
                          int32_t ns, const double* Z, double* out, int32_t* info);

/* ---- leave-one-out cross-validation (predict_LOO, logp_CVLOO, dlogpdtheta_CVLOO) ---------------------------------- */
/* Evaluates like gprb_eval with a gradient (same make_posdef! ladder, info codes, active semantics and state reuse; the
 * resident state afterwards is what gprb_eval(theta, grad) leaves), then the leave-one-out terms of every GP with
 * info >= 0 (Rasmussen & Williams eqs. 5.10-5.13) on the K that was factorised - noise, eps, jitter and diagonal offset
 * included.  With d = diag(K^-1), alpha = K^-1 (y - m(X)):
 *   mll, grad  B, P x B  out, as gprb_eval with a gradient; either may be NULL
 *   logp_loo   B         out  sum_i 1/2 log d_i - 1/2 alpha_i^2 / d_i - 1/2 log 2pi
 *   grad_loo   P x B     out  d logp_loo / d theta; NULL = value only (no n^3 stage)
 *   mu_loo     n x B     out  y_i - m(x_i) - alpha_i / d_i (the caller adds m(X) back), or NULL
 *   var_loo    n x B     out  1 / d_i, or NULL
 *   info       B         out
 * A GP with info < 0 gets logp_loo = -Inf and NaN grad_loo / mu_loo / var_loo and blocks nobody; inactive GPs' outputs
 * are untouched.  The gradient stage works on groups of GPs with a bounded per-call workspace (about 2 n^2 doubles per
 * GP of a group, groups of at most 8 GiB, halved while the device cannot hold them). */
int gprb_eval_loo(gprb_batch* batch, const double* theta, const uint8_t* active, double* mll, double* grad,
                  double* logp_loo, double* grad_loo, double* mu_loo, double* var_loo, int32_t* info);

/* ---- predictive gradients: Jacobians of the posterior mean and variance with respect to the test inputs -------- */
/* Synchronous, on prediction slot 0 (refused while slot 0 has an asynchronous prediction in flight), any m >= 1.
 * Works on any state gprb_predict works on, value-only states included (it needs L, the inverted diagonal blocks and
 * alpha).  For stationary ARD kernels k = g(r2), dk(x*, x_i) / dx*_p = 2 g'(r2) w_p (x*_p - x_ip), and with
 * beta = K^-1 K* (K the resident matrix: noise, eps, jitter and diagonal offset included):
 *   dmu_j  / dx*_jp = dm(x*_j) / dx*_jp + sum_i alpha_i dk(x*_j, x_i) / dx*_jp
 *   dvar_j / dx*_jp = -2 sum_i beta_ij dk(x*_j, x_i) / dx*_jp
 * dvar is the gradient of the unclamped K** - T'T: the floor of the variance at 0 is not differentiated, and it is the
 * same for sigma^2_f and sigma^2_y.
 *   Xstar, xstar_stride, mstar   as for gprb_predict
 *   dmstar  d x m x B  in, the prior mean's Jacobian (added like mstar), or NULL for none
 *   mu, var m x B      out, bit-identical to gprb_predict's tiled path on the same state; var may be NULL
 *   dmu     d x m x B  out, dmu[p + d*(j + m*b)]
 *   dvar    d x m x B  out, or NULL: mean only, no triangular substitution runs at all
 * A GP without an evaluated state gets NaN rows and blocks nobody.  gprb_last_predict_ms(batch, 0) reports the device
 * time (without the copy of the Jacobians).  The workspace holds one 128-column chunk of right-hand sides per GP. */
int gprb_predict_grad(gprb_batch* batch, int64_t m, const double* Xstar, int64_t xstar_stride, const double* mstar,
                      const double* dmstar, double* mu, double* var, double* dmu, double* dvar);

/* ---- parity taps (state after the last gprb_eval of GP b) ------------------------------ */
int gprb_get_K(gprb_batch* batch, int32_t b, double* out /* n x n, symmetric, noise + jitter included */);
int gprb_get_chol(gprb_batch* batch, int32_t b, double* out /* n x n upper U with K = U'U, zeros below */);
int gprb_get_alpha(gprb_batch* batch, int32_t b, double* out /* n */);
int gprb_get_Kinv(gprb_batch* batch, int32_t b, double* out /* n x n symmetric; needs a value+grad eval */);

/* ---- multi-GPU: the final gather of per-trial results (examples/parallel/core.jl:47-56) ---------- */
/* The path shards by trial with no data-path collective; the only exchange is one NCCL all-gather of the small per-trial
 * result rows (theta*, mll, info, predictions) over NVLink at the end.
 *   multi-process (one rank per GPU): rank 0 calls gprb_comm_unique_id and hands the 128 bytes to the other ranks through
 *   whatever the host uses (a file, MPI, torch.distributed, Distributed.jl); every rank calls gprb_comm_init_rank. */
int gprb_comm_unique_id(void* id128);
int gprb_comm_init_rank(gprb_ctx* ctx, int32_t nranks, int32_t rank, const void* id128);
/* rows: count_local x width doubles (row-major), row_ids[k] in 0..n_rows-1 = global index (trial id) of local row k.
 * out: n_rows x width on every rank, rows never contributed are NaN.  count_local <= ceil(n_rows / nranks) (any
 * round-robin / block partition of the trials).  Without a communicator (single rank) it degenerates to the local scatter. */
int gprb_gather(gprb_ctx* ctx, int32_t n_rows, int32_t width, int32_t count_local, const int32_t* row_ids,
                const double* rows, double* out);
/* single-process form over the contexts of gprb_init_multi: counts[g], row_ids[g], rows[g] are rank g's arguments. */
int gprb_gather_multi(gprb_ctx* const* ctxs, int32_t ngpus, int32_t n_rows, int32_t width, const int32_t* counts,
                      const int32_t* const* row_ids, const double* const* rows, double* out);

/* ---- timing hooks for bench.py (CUDA events on the library's own streams) -------------- */
/* Per-stage device time of the most recent gprb_eval / gprb_eval_device, milliseconds:
 * out[0]=assembly out[1]=cholesky out[2]=solve+mll out[3]=inverse out[4]=gradient out[5]=total
 * out[6]=sum over the DMMA tile-GEMM launches alone, out[7]=number of those launches.
 * Valid only when profiling was enabled with gprb_set_profiling(batch, 1) (single stream, stages serialised). */
int gprb_set_profiling(gprb_batch* batch, int32_t on);
int gprb_last_stage_ms(gprb_batch* batch, double out[8]);
/* Device time of every tile-GEMM launch of the last profiled evaluation, in launch order (J x [CHOL_DIAG, CHOL_COL],
 * then TRTRI_ROW 1..J-1, then LAUUM).  Writes at most `cap` values, returns the number of launches (>= 0). */
int gprb_last_gemm_launch_ms(gprb_batch* batch, double* out, int32_t cap);
/* Number of kernel launches issued by the library since the context was created. */
int64_t gprb_launch_count(gprb_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* GPRB200_H */
