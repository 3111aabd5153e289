/*
 * mcmcgpu.h -- C ABI of libmcmcgpu.so, the B200 (sm_100a) many-chain engine for the MCMC.jl hot path.
 *
 * The reference (dingliumath/MCMC.jl) has no FFI layer: its extension surface is Julia multiple
 * dispatch.  Each entry point below states the reference interface (file:line under the reference
 * tree) it stands in for; the Julia-side `ccall` binding a maintainer would add is in
 * INTEGRATION.md and mcmc.jl_b200/julia/GPUMC.jl.
 *
 * Conventions
 *  - every function returns int32 status: 0 ok, <0 error (MCMCGPU_E_*); mcmcgpu_last_error() gives
 *    the message (library-owned, valid until the next call on the same thread).
 *  - the host owns every input and output buffer; the library copies inputs at *_create time and
 *    fills caller-allocated outputs.  Only opaque handles cross the boundary.
 *  - arrays are dense, column-major Float64 (Julia native); sizes int64; flags uint8.
 *  - calls are blocking; one host thread per context.  One context == one GPU (one process per GPU).
 *  - there is NO CPU fallback: without a CUDA device every compute entry point fails with
 *    MCMCGPU_E_CUDA.
 */
#ifndef MCMCGPU_H
#define MCMCGPU_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define MCMCGPU_ABI_VERSION 3   /* 2: mcmcgpu_run_info.comm_ms; 3: mcmcgpu_runner_cfg.stream_stats / stream_batchlen */
/* The version counts changes of the structs' layouts and of existing functions.  Functions that are only added (e.g.
 * mcmcgpu_run_set_metric) leave it as is: a binding written for version 3 keeps working, and the new symbols can be
 * looked up by name. */

/* status codes */
#define MCMCGPU_OK 0
#define MCMCGPU_E_ARG (-1)       /* bad argument (maps the reference's ctor assertions)              */
#define MCMCGPU_E_SUPPORT (-2)   /* "Initial values out of model support" RWM.jl:55 MALA.jl:85 HMC.jl:121 HMCDA.jl:88 likmodel.jl:54 */
#define MCMCGPU_E_NOGRAD (-3)    /* gradient sampler on a gradient-less model MALA.jl:72 HMC.jl:111 HMCDA.jl:79 */
#define MCMCGPU_E_CUDA (-4)      /* CUDA / device failure, or no device                               */
#define MCMCGPU_E_COMM (-5)      /* NCCL failure / not initialised                                    */
#define MCMCGPU_E_STATE (-6)     /* call out of order (e.g. fetch before execute)                     */

/* likelihood families: the GPU registry behind model() (src/modellers/mcmcmodels.jl:27-33,
 * src/modellers/likmodel.jl:100-143); formulas from README.md:60-72 and examples/ */
#define MCMCGPU_FAM_NORMAL_FN 0  /* README.md:60,63  v -> -dot(v,v), grad -2v                          */
#define MCMCGPU_FAM_NORMAL_DSL 1 /* README.md:67-72  v ~ Normal(mu, sigma)     hyper = {mu, sigma}     */
#define MCMCGPU_FAM_LINEAR 2     /* examples/linear_regression.jl:14-18        hyper = {prior_sd, noise_sd} */
#define MCMCGPU_FAM_LOGISTIC 3   /* examples/logistic_regression.jl:16-20      hyper = {prior_sd, sign}  (sign -1: exp(-X*b); +1: test/test_syntax.jl:18; any other value is MCMCGPU_E_ARG) */
#define MCMCGPU_FAM_PROBIT 4     /* examples/probit_regression.jl:18-41        hyper = {prior_sd}        */
#define MCMCGPU_FAM_OU 5         /* examples/ornstein.jl:19-27                 hyper = {tau_hi, sigma_hi, mu_hi}; y = series, d = 3 */
#define MCMCGPU_FAM_ABS_NORMAL 6 /* README.md:253-259  y = abs(x); y ~ Normal(mu, sigma)   hyper = {mu, sigma} (the SeqMC ladder) */

/* samplers: src/samplers/RWM.jl:24-36, MALA.jl:50-62, HMC.jl:53-74, HMCDA.jl:24-43 */
#define MCMCGPU_RWM 0
#define MCMCGPU_MALA 1
#define MCMCGPU_HMC 2
#define MCMCGPU_HMCDA 3
#define MCMCGPU_RAM 4          /* src/samplers/RAM.jl:24-36: scale, rate (robust adaptive Metropolis); d <= 8 fused, d <= 128 wave */
/* No-U-Turn sampler with dual averaging, with the identity, a diagonal or a dense mass matrix, fixed
 * (mcmcgpu_run_set_metric / _set_dense_metric) or adapted per chain in Stan's warm-up windows
 * (mcmcgpu_run_set_metric_adaptation), engine WAVE only (one leapfrog leaf per chain per wave).  Two transitions
 * (mcmcgpu_run_set_nuts_transition): slice NUTS (Hoffman & Gelman 2014, Algorithms 3 and 6; the default) and Stan's
 * multinomial NUTS (biased progressive sampling, U-turn checks across neighbouring sub-trees, divergences at
 * H - H0 > 1000).  It reads mcmcgpu_sampler_cfg as follows:
 *   nleaps = maxdoublings (1..10: at most 2^maxdoublings - 1 leapfrogs per step);
 *   rate, shrinkage, t0, step = the dual averaging, HMCDA's rules.  Its target statistic is, for slice NUTS, the mean
 *   of min(1, exp(H0 - H)) over the last doubling's leaves and, for multinomial NUTS, Stan's accept_stat: the same
 *   mean over every leaf of the step's trajectory.  scale, len and max_leaps are ignored, and so is the model scale
 *   passed to the run.
 * fetch_diag returns the step size and the leapfrog count of every kept step (ndoublings = floor(log2(leaps)) + 1);
 * set_state / get_state carry (step size, dual step size, dualH) as for HMCDA.  Not supported: engine FUSED, injected
 * draws, store_rb, a tuner, row-sharded models (MCMCGPU_E_ARG). */
#define MCMCGPU_NUTS 5
#define MCMCGPU_NUTS_SLICE 0         /* mcmcgpu_run_set_nuts_transition */
#define MCMCGPU_NUTS_MULTINOMIAL 1

/* engines */
#define MCMCGPU_ENGINE_AUTO 0
#define MCMCGPU_ENGINE_FUSED 1   /* whole chain in one per-chain kernel (closed-form families)       */
#define MCMCGPU_ENGINE_WAVE 2    /* one gradient evaluation for every chain per wave (K1 + transition) */

/* variance estimators src/stats/var.jl:137-166 */
#define MCMCGPU_VAR_IID 0
#define MCMCGPU_VAR_BM 1
#define MCMCGPU_VAR_IMSE 2
#define MCMCGPU_VAR_IPSE 3

typedef struct mcmcgpu_ctx mcmcgpu_ctx;
typedef struct mcmcgpu_model mcmcgpu_model;
typedef struct mcmcgpu_run mcmcgpu_run;

/* sampler parameters; mirrors the reference constructors' fields */
typedef struct {
  int32_t kind;        /* MCMCGPU_RWM | MALA | HMC | HMCDA                                           */
  int32_t nleaps;      /* HMC.nLeaps   (HMC.jl:54)                                                   */
  double scale;        /* RWM.scale (RWM.jl:25) | MALA.driftStep (MALA.jl:51) | HMC.leapStep (HMC.jl:55) | RAM.scale (RAM.jl:25) */
  double rate, len, shrinkage, t0, step; /* HMCDA fields HMCDA.jl:25-29; rate is also RAM.rate (RAM.jl:26) */
  int64_t max_leaps;   /* cap on HMCDA nLeaps = max(1, round(len/leapStep)) (HMCDA.jl:104); 0 = library default 1<<20 */
  int32_t tuner_on;    /* EmpMCTuner attached (samplers.jl:32-50); MALA/HMC only                     */
  int32_t adapt_step, max_step;
  double target_path, target_rate;
} mcmcgpu_sampler_cfg;

/* runner parameters: SerialMC's range (src/runners/SerialMC.jl:12-35) + the many-chain additions */
typedef struct {
  int64_t first, step, last; /* kept steps first:step:last; burnin = first-1, len = last            */
  int64_t nchains;           /* chains run by THIS context                                           */
  int64_t chain_offset;      /* global id of this context's first chain (Philox key; chain sharding) */
  uint64_t seed;
  int32_t init_per_chain;    /* 0: init is d (shared); 1: init is d x nchains                         */
  int32_t store_grad;        /* keep pgrads (SerialMC.jl:51-53)                                       */
  int32_t store_logtarget;   /* keep plogtarget of every kept sample                                   */
  int32_t engine;            /* MCMCGPU_ENGINE_*                                                       */
  int32_t store_rb;          /* HMC storeLeaps (HMC.jl:145-150): keep, per kept step, the Rao-Blackwell sum of
                                mean_rb_hmc (src/stats/mean.jl:11-35) accumulated over the leapfrog states on the fly
                                (the leap states themselves are not stored); fetched with mcmcgpu_run_fetch_rb */
  int32_t stream_stats;      /* engine FUSED only: do NOT store the draws; instead accumulate, in registers while sampling, what
                                src/stats needs for mean (mean.jl:6), mcvar_iid (var.jl:7-8), mcvar_bm (var.jl:20-26; batch
                                length stream_batchlen, 0 = 100), ess / actime of vtype :bm (ess.jl:6-19) and acceptance
                                (summary.jl:6-15).  mcmcgpu_run_stats(vtype IID or BM) then returns them; fetch is an error.
                                The mean is the two-pass code's sum bit for bit; the variances are one-pass (shifted by the
                                first kept draw) and agree with it to ~1e-12. */
  int32_t stream_batchlen;
} mcmcgpu_runner_cfg;

typedef struct {
  double gpu_ms;          /* device time of the sampling loop (CUDA events on the library stream)   */
  int64_t n_grad_evals;   /* log-target(+gradient) evaluations summed over chains                   */
  int64_t n_waves;        /* wave-engine iterations (0 for the fused engine)                        */
  int64_t n_launches;     /* kernels launched by the library during execute                         */
  double eval_ms;         /* device time spent in the likelihood kernel (wave engine, option time_eval) */
  double comm_ms;         /* device time between the likelihood kernel and the transition kernel: the fold of the
                             row-split partials and, for row-sharded models, the NCCL all-reduce (time_eval)  */
} mcmcgpu_run_info;

/* ---- context ---- */
int32_t mcmcgpu_abi_version(void);
const char* mcmcgpu_last_error(void);
/* one context per GPU / process. device_id < 0: current device. */
int32_t mcmcgpu_init(int32_t device_id, mcmcgpu_ctx** out);
int32_t mcmcgpu_destroy(mcmcgpu_ctx* ctx);
/* use a caller-owned CUDA stream (cudaStream_t as void*) for all launches and copies; NULL = library stream */
int32_t mcmcgpu_set_stream(mcmcgpu_ctx* ctx, void* cuda_stream);
/* engine options: "time_eval" (1: time every likelihood launch with CUDA events -> run_info.eval_ms),
 * "poll_every" (waves between completion polls for HMCDA / tuned HMC), "force_splits" (K1 row splits) */
int32_t mcmcgpu_set_option(mcmcgpu_ctx* ctx, const char* key, int64_t value);
/* row-sharded tall data (SURVEY 8e.2): NCCL communicator over the ranks holding the row shards.
 * unique_id is the 128-byte ncclUniqueId produced by mcmcgpu_comm_unique_id on rank 0. */
int32_t mcmcgpu_comm_unique_id(void* out128);
int32_t mcmcgpu_comm_init(mcmcgpu_ctx* ctx, int32_t rank, int32_t nranks, const void* unique_id128);

/* ---- model: stands in for model(...) -> MCMCLikelihoodModel (likmodel.jl:20-58,100-143) ----
 * X: N x d column-major (NULL for Normal/OU), y: N (NULL for Normal).  With a communicator and
 * row_sharded != 0, X/y are THIS rank's rows and the prior is added once after the all-reduce. */
int32_t mcmcgpu_model_create(mcmcgpu_ctx* ctx, int32_t family, int64_t N, int64_t d, const double* X,
                             const double* y, const double* hyper, int32_t nhyper, int32_t row_sharded,
                             mcmcgpu_model** out);
/* same, with X (N x d column-major) and y already resident on this context's device (tall data generated or
 * loaded shard by shard on the GPU); hyper stays a host pointer. */
int32_t mcmcgpu_model_create_device(mcmcgpu_ctx* ctx, int32_t family, int64_t N, int64_t d, const double* X_dev,
                                    const double* y_dev, const double* hyper, int32_t nhyper, int32_t row_sharded,
                                    mcmcgpu_model** out);
int32_t mcmcgpu_model_destroy(mcmcgpu_model* m);

/* model.eval / model.evalallg for C parameter vectors at once (likmodel.jl:21,25).
 * B: d x C; out_lt: C; out_grad: d x C or NULL (eval only). */
int32_t mcmcgpu_logtarget_grad(mcmcgpu_model* m, const double* B, int64_t C, double* out_lt, double* out_grad);

/* ---- run: stands in for run(model * sampler * runner) (runners.jl:7-32, SerialMC.jl:37-85) ----
 * init: d or d x nchains; scale: d (model.scale, likmodel.jl:30) or NULL = ones;
 * inj_normals: NULL (Philox) or d x (last+1) x nchains [column 0 = pre-loop draw, HMCDA.jl:90];
 * inj_uniforms: NULL or (last+1) x nchains.
 * outputs (NULL = not wanted): samples d x S x nchains, grads d x S x nchains (NaN for RWM,
 * SerialMC.jl:42), accept S x nchains, logtarget S x nchains, S = length(first:step:last). */
int32_t mcmcgpu_run_chains(mcmcgpu_model* m, const mcmcgpu_sampler_cfg* s, const mcmcgpu_runner_cfg* r,
                           const double* init, const double* scale, const double* inj_normals,
                           const double* inj_uniforms, double* out_samples, double* out_grads,
                           uint8_t* out_accept, double* out_logtarget, mcmcgpu_run_info* info);

/* split form: inputs resident in HBM after create; execute may be timed alone; results stay on the device */
int32_t mcmcgpu_run_create(mcmcgpu_model* m, const mcmcgpu_sampler_cfg* s, const mcmcgpu_runner_cfg* r,
                           const double* init, const double* scale, const double* inj_normals,
                           const double* inj_uniforms, mcmcgpu_run** out);
int32_t mcmcgpu_run_execute(mcmcgpu_run* run, mcmcgpu_run_info* info);
/* stepwise execution (engine WAVE): advance every chain by nsteps more MCMC steps and pause; a later
 * call continues exactly where the chains stopped (same Philox counters, same adaptation state). */
int32_t mcmcgpu_run_execute_steps(mcmcgpu_run* run, int64_t nsteps, mcmcgpu_run_info* info);
/* true resume (the reference's resume restarts from model.init, SerialMC.jl:93-97): before the first
 * execute, start the chains at step step0 + 1 (init = the saved positions) and, for HMCDA / NUTS, restore the
 * dual-averaging state (arrays of nchains, or all NULL for the reference's initial values). */
int32_t mcmcgpu_run_set_state(mcmcgpu_run* run, int64_t step0, const double* leapstep, const double* dual_leapstep,
                              const double* dualH);
/* current positions (d x nchains) and HMCDA / NUTS step-size state (nchains each); any pointer may be NULL */
int32_t mcmcgpu_run_get_state(mcmcgpu_run* run, double* pars, double* leapstep, double* dual_leapstep, double* dualH);
/* NUTS only, before the first execute: diagonal INVERSE metric, d (shared) or d x nchains (per_chain != 0); every entry
 * finite and > 0.  Without this call the metric is the identity (the run is bit-identical to one without the call when
 * all entries are 1).  With adaptation on it is the starting metric.  MCMCGPU_E_ARG for another sampler or a bad entry,
 * MCMCGPU_E_STATE after the first execute. */
int32_t mcmcgpu_run_set_metric(mcmcgpu_run* run, const double* inv_metric, int32_t per_chain);
/* NUTS only, before the first execute: adapt every chain's diagonal metric during warm-up in Stan's windows
 * (Stan's defaults: 75, 50, 25).  The warm-up is the W = first - 2 steps on which the step size adapts; with W < 20 the
 * metric is not updated, and when the buffers and the window do not fit they become 15 % / 10 % of W and the rest.
 * Each window's final samples give a Welford variance, regularised as Stan does (n / (n + 5) var + 1e-3 * 5 / (n + 5));
 * the dual averaging then restarts at mu = log(10 eps).  Stan's step-size search at a window end is not made.  Each chain
 * adapts alone (no pooling across chains).  Not with set_state step0 inside the warm-up (0 < step0 < first - 2).
 * MCMCGPU_E_ARG for another sampler, negative buffers or window < 1; MCMCGPU_E_STATE after the first execute. */
int32_t mcmcgpu_run_set_metric_adaptation(mcmcgpu_run* run, int64_t init_buffer, int64_t term_buffer, int64_t window);
/* the current inverse metric, d x nchains (after execute / execute_steps; before, the starting metric).  MCMCGPU_E_ARG on
 * a run with a dense metric. */
int32_t mcmcgpu_run_get_metric(mcmcgpu_run* run, double* out_inv_metric);
/* NUTS only, before the first execute: a dense INVERSE metric M^-1 (Stan's dense_e), d x d shared by every chain, or
 * d x d x nchains (per_chain != 0), column-major: element (i, j) of chain c at (c*d + j)*d + i.  NULL: the identity.  Every
 * matrix must be finite, exactly symmetric and positive definite (the Cholesky factorisation the kernel uses succeeds).
 * Arithmetic (DESIGN.md, NUTS): p = L^-T z with A = L L^T; K = 0.5 m . (A m); theta += e (A m); U-turn dots delta . (A p).
 * A diagonal A gives the bits of mcmcgpu_run_set_metric with its diagonal, the identity those of a run without a metric.
 * A following mcmcgpu_run_set_metric_adaptation adapts the dense metric per chain in Stan's windows from a Welford
 * covariance: A = (n / (n + 5)) cov + 1e-3 (5 / (n + 5)) I; a chain whose new A fails the Cholesky keeps its previous A.
 * MCMCGPU_E_ARG for another sampler, a bad matrix, a run that has a diagonal metric or already adapts one;
 * MCMCGPU_E_STATE after the first execute.  Memory: A and L (d*d doubles each) per chain, or once when shared and fixed;
 * with adaptation also the d*d Welford sums per chain. */
int32_t mcmcgpu_run_set_dense_metric(mcmcgpu_run* run, const double* inv_metric, int32_t per_chain);
/* the current dense inverse metric, d x d x nchains column-major as above (before execute: the starting one).  An adapted
 * metric is Stan's unsymmetrised covariance estimate, so it need not be exactly symmetric.  MCMCGPU_E_ARG on a run
 * without a dense metric. */
int32_t mcmcgpu_run_get_dense_metric(mcmcgpu_run* run, double* out);
/* NUTS only, before the first execute: the transition, MCMCGPU_NUTS_SLICE (the default: a run with this call gives the
 * bits of one without it) or MCMCGPU_NUTS_MULTINOMIAL (Stan's base_nuts transition, pinned in DESIGN.md, NUTS).  A
 * multinomial run keeps per kept step Stan's accept_stat, the energy H of the sample and the divergence flag
 * (mcmcgpu_run_fetch_nuts_stats); its tree state is (5 maxdoublings + 2) d + 3 maxdoublings + 2 doubles per chain, and
 * (7 maxdoublings + 3) d + 3 maxdoublings + 2 with a dense metric.  MCMCGPU_E_ARG for another sampler or an unknown
 * value, MCMCGPU_E_STATE after the first execute. */
int32_t mcmcgpu_run_set_nuts_transition(mcmcgpu_run* run, int32_t transition);
/* multinomial NUTS: per kept step (S x nchains each; any pointer may be NULL) the accept_stat (sum over the trajectory's
 * leaves of min(1, exp(H0 - H)), over the leapfrog count), the energy H of the step's sample, and divergent = 1 when the
 * step's last subtree stopped at a leaf with H - H0 > 1000.  MCMCGPU_E_ARG for a run that is not multinomial NUTS,
 * MCMCGPU_E_STATE before the first execute. */
int32_t mcmcgpu_run_fetch_nuts_stats(mcmcgpu_run* run, double* accept_stat, double* energy, uint8_t* divergent);
int32_t mcmcgpu_run_fetch(mcmcgpu_run* run, double* out_samples, double* out_grads, uint8_t* out_accept,
                          double* out_logtarget);
/* Rao-Blackwellised draws (store_rb): out_rb d x S x nchains; their column means are mean_rb(chain) (mean.jl:37-41) */
int32_t mcmcgpu_run_fetch_rb(mcmcgpu_run* run, double* out_rb);
/* per-chain diagnostics: final leap step (HMCDA/NUTS/tuned), kept-step leap steps (S x nchains) and leap counts */
int32_t mcmcgpu_run_fetch_diag(mcmcgpu_run* run, double* out_eps, int64_t* out_nleaps);
/* src/stats on the device-resident draws: outputs d x nchains each (NULL = skip).
 * mean (mean.jl:6), var_iid (var.jl:7-8), var (vtype: var.jl:137-166), ess / actime (ess.jl:6-19),
 * accept_rate nchains in percent (summary.jl:6-15).  maxlag < 0: S-1; batchlen <= 0: 100. */
int32_t mcmcgpu_run_stats(mcmcgpu_run* run, int32_t vtype, int64_t maxlag, int64_t batchlen, double* out_mean,
                          double* out_var_iid, double* out_var, double* out_ess, double* out_actime,
                          double* out_accept_rate);
/* zero-variance control variates on the device-resident draws and gradients (needs store_grad):
 * linearZv (order 1) / quadraticZv (order 2) of src/stats/zv.jl:8-66 for every chain.
 * out_zv d x S x nchains (may be NULL), out_a k x d x nchains with k = d (order 1) or d(d+3)/2 (order 2),
 * element (p, i, c) at out_a[(c*k + p)*d + i]  (row-major k x d per chain, as the reference's `a`). */
int32_t mcmcgpu_run_zv(mcmcgpu_run* run, int32_t order, double* out_zv, double* out_a);
int32_t mcmcgpu_run_destroy(mcmcgpu_run* run);

/* src/stats from host draws: samples d x S x C (the layout mcmcgpu_run_chains fills) */
int32_t mcmcgpu_stats(mcmcgpu_ctx* ctx, const double* samples, int64_t S, int64_t d, int64_t C, int32_t vtype,
                      int64_t maxlag, int64_t batchlen, double* out_mean, double* out_var_iid, double* out_var,
                      double* out_ess, double* out_actime);

/* ---- population runners (SURVEY.md 8f.1; closed-form families NORMAL_FN / NORMAL_DSL / ABS_NORMAL, d <= 8) ----
 * nt tasks share family and size; task t has hypers[4*t .. 4*t+3] and samplers[t] (RWM / MALA / HMC, no tuner).
 *
 * mcmcgpu_run_seqmc stands in for run(targets::Array{MCMCTask}; particles=...) with SeqMC runners
 * (src/runners/SeqMC.jl:39-122): one thread mutates one particle per target; weights, the variance trigger, the
 * cumulative sum and the multinomial resampling (prefix sum + binary search) stay on the device.
 * particles d x npart; injected draws (all NULL for Philox): normals d x npart x nt x steps, uniforms and
 * res_uniforms npart x nt x steps.  out_samples d x ((steps-burnin)*npart), out_weights (steps-burnin)*npart.
 * With a communicator (mcmcgpu_comm_init) the population is sharded: npart is THIS rank's share (equal on every
 * rank, global particle g = rank*npart + n), the ranks exchange (pars, logtarget, logW) with one ncclAllGather per
 * target and resample their own slots from the global weights; injected draws are then the GLOBAL arrays
 * (npart*nranks particles) and the outputs hold this rank's particles only.
 *
 * mcmcgpu_run_serialtemp stands in for run(tasks) with SerialTempMC runners (src/runners/SerialTempMC.jl:31-85)
 * for nrep independent replicas at once.  inits d x nt; injected draws (all NULL for Philox): normals
 * d x (steps+2) x nrep, uniforms (steps+2) x nrep, pick and swap (steps+1) x nrep.
 * out_samples d x (steps-burnin) x nrep, out_at (steps-burnin) x nrep (0-based task index, may be NULL). */
int32_t mcmcgpu_run_seqmc(mcmcgpu_ctx* ctx, int32_t family, int64_t d, int32_t nt, const double* hypers,
                          const mcmcgpu_sampler_cfg* samplers, int64_t steps, int64_t burnin, double trigger,
                          int64_t npart, const double* particles, uint64_t seed, const double* inj_normals,
                          const double* inj_uniforms, const double* inj_res_uniforms, double* out_samples,
                          double* out_weights, int64_t* out_nresamples, mcmcgpu_run_info* info);
/* SeqMC over arbitrary models of this context (any family, any d; the regression families evaluate all particles at once
 * through the likelihood kernel): task t = (models[t], samplers[t]); everything else as mcmcgpu_run_seqmc. */
int32_t mcmcgpu_run_seqmc_models(mcmcgpu_ctx* ctx, int32_t nt, mcmcgpu_model* const* models, const mcmcgpu_sampler_cfg* samplers,
                                 int64_t steps, int64_t burnin, double trigger, int64_t npart, const double* particles,
                                 uint64_t seed, const double* inj_normals, const double* inj_uniforms,
                                 const double* inj_res_uniforms, double* out_samples, double* out_weights,
                                 int64_t* out_nresamples, mcmcgpu_run_info* info);
/* SerialTempMC over arbitrary models of this context (any family, any d): nrep independent replicas, regrouped at every
 * iteration by the task they consume; rep_offset = global id of this context's first replica (Philox key: replicas shard
 * over GPUs with no communication -- serial tempering moves ONE chain between tasks, SerialTempMC.jl:57-66, it never
 * exchanges states between chains).  Everything else as mcmcgpu_run_serialtemp. */
int32_t mcmcgpu_run_serialtemp_models(mcmcgpu_ctx* ctx, int32_t nt, mcmcgpu_model* const* models, const mcmcgpu_sampler_cfg* samplers,
                                      int64_t steps, int64_t burnin, int64_t swap_period, int64_t nrep, int64_t rep_offset,
                                      const double* inits, uint64_t seed, const double* inj_normals, const double* inj_uniforms,
                                      const double* inj_pick, const double* inj_swap, double* out_samples, int32_t* out_at,
                                      mcmcgpu_run_info* info);
int32_t mcmcgpu_run_serialtemp(mcmcgpu_ctx* ctx, int32_t family, int64_t d, int32_t nt, const double* hypers,
                               const mcmcgpu_sampler_cfg* samplers, int64_t steps, int64_t burnin, int64_t swap_period,
                               int64_t nrep, const double* inits, uint64_t seed, const double* inj_normals,
                               const double* inj_uniforms, const double* inj_pick, const double* inj_swap,
                               double* out_samples, int32_t* out_at, mcmcgpu_run_info* info);

/* zero-variance control variates from host draws / gradients (layouts as mcmcgpu_run_chains fills them) */
int32_t mcmcgpu_zv(mcmcgpu_ctx* ctx, const double* samples, const double* grads, int64_t S, int64_t d, int64_t C,
                   int32_t order, double* out_zv, double* out_a);

/* the engine's own draws, for draw-matched replay through another implementation:
 * normals d x (last+1) x nchains and uniforms (last+1) x nchains exactly as the samplers consume them */
int32_t mcmcgpu_philox_draws(mcmcgpu_ctx* ctx, uint64_t seed, int64_t chain_offset, int64_t nchains, int64_t d,
                             int64_t last, double* out_normals, double* out_uniforms);

#ifdef __cplusplus
}
#endif
#endif
