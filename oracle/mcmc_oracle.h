/*
 * mcmc_oracle.h -- CPU restatement (plain C99, FP64, scalar, single thread) of the MCMC.jl hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under oracle/ is part of the product: only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may build, load or
 * call it, and there only as the checker / the timed CPU baseline.  The product (libmcmcgpu.so)
 * never links or calls it.
 *
 * PARITY STATUS: "parity unpinned".  The reference (dingliumath/MCMC.jl, Julia 0.2) cannot be run
 * here (no julia; src/dsl/modelparser.jl:13 includes a file from the author's home directory) and
 * its own tests hold no numeric golden vectors for this path (SURVEY.md section 8c).  The oracle is
 * therefore anchored on (i) line-by-line restatement, each function citing the reference file:line,
 * (ii) independent numpy/scipy re-derivations and finite differences in tests/, (iii) the soft
 * statistical bands of README.md:121-204 and (iv) Random123 known-answer vectors for Philox.
 *
 * All matrices are dense column-major double (Julia native layout).
 */
#ifndef MCMC_ORACLE_H
#define MCMC_ORACLE_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

/* Likelihood families (SURVEY.md 8a rows M1..M5). */
enum {
  ORC_FAM_NORMAL_FN = 0, /* README.md:60,63  v -> -dot(v,v), grad v -> -2v                         */
  ORC_FAM_NORMAL_DSL = 1,/* README.md:67-72  v ~ Normal(mu, sigma)         hyper = {mu, sigma}      */
  ORC_FAM_LINEAR = 2,    /* examples/linear_regression.jl:14-18            hyper = {prior_sd, noise_sd} */
  ORC_FAM_LOGISTIC = 3,  /* examples/logistic_regression.jl:16-20          hyper = {prior_sd, sign} sign=-1: exp(-X*b) (example); +1: test/test_syntax.jl:18 */
  ORC_FAM_PROBIT = 4,    /* examples/probit_regression.jl:18-41            hyper = {prior_sd}        */
  ORC_FAM_OU = 5,        /* examples/ornstein.jl:19-27                     hyper = {tau_hi, sigma_hi, mu_hi}; y = series x[0..N-1], d = 3 (tau, sigma, mu) */
  ORC_FAM_ABS_NORMAL = 6 /* README.md:253-259  y = abs(x); y ~ Normal(mu, sigma)   hyper = {mu, sigma}  (the SeqMC ladder) */
};

typedef struct {
  int32_t family;
  int64_t N;       /* observations (rows of X / length of series); 0 for the Normal families */
  int64_t d;       /* parameter count */
  const double* X; /* N x d column-major, or NULL */
  const double* y; /* N, or NULL */
  double hyper[4];
} orc_model;

/* Samplers (SURVEY.md 8a rows S1..S4). */
enum { ORC_RWM = 0, ORC_MALA = 1, ORC_HMC = 2, ORC_HMCDA = 3, ORC_RAM = 4 /* src/samplers/RAM.jl: scale, rate */ };

typedef struct {
  int32_t kind;
  double scale;      /* RWM scale (RWM.jl:24-36) | MALA driftStep (MALA.jl:50-62) | HMC leapStep (HMC.jl:53-74) */
  int32_t nleaps;    /* HMC nLeaps */
  /* HMCDA (HMCDA.jl:24-43) */
  double rate, len, shrinkage, t0, step;
  int64_t max_leaps; /* safety cap on HMCDA nLeaps (documented deviation; 0 = uncapped) */
  /* EmpMCTuner (samplers.jl:32-50) for MALA / HMC; enabled when tuner_on != 0 */
  int32_t tuner_on;
  int32_t adapt_step, max_step;
  double target_path, target_rate;
  /* test aid (not in the reference): HMCDA adaptation is a chaotic map once the step size crosses the
   * integrator's stability limit, so last-bit differences between libm implementations grow without
   * bound over a burn-in.  When force_eps != NULL (length last+1) the trajectory of step i uses
   * force_eps[i] while diag_eps still reports the oracle's own adapted value: a one-step-ahead check. */
  const double* force_eps;
  /* HMC / HMCDA storeLeaps (HMC.jl:145-150): when rb_out != NULL (S x d) the leap states are kept for the step and the
   * Rao-Blackwell sums of mean_rb_hmc (src/stats/mean.jl:11-35) are written per kept step; the sample they start from
   * is the one the sampler's own acceptance test keeps (HMCDA: u < min(1, e)). */
  double* rb_out;
  /* test aid (not in the reference, whose resume restarts from model.init, SerialMC.jl:93-97): the chain starts at
   * step start_step + 1 from `init` (draw columns keep their absolute step index), and, for HMCDA, da_state != NULL
   * restores {leapStep, dualLeapStep, dualH} -- the counterpart of the engine's mcmcgpu_run_set_state. */
  int64_t start_step;
  const double* da_state;
} orc_sampler;

typedef struct {
  int64_t first, step, last; /* SerialMC range first:step:last (SerialMC.jl:12-35); burnin = first-1 */
} orc_range;

/* ---- models ---- */
double orc_eval(const orc_model* m, const double* beta);                  /* model.eval     */
double orc_evalallg(const orc_model* m, const double* beta, double* grad); /* model.evalallg */
double orc_log_ndtr(double x); /* log Phi(x) */
/* CPU-baseline shape of the logistic evaluation (row-blocked, X read once, 4 partial sums per dot product); process-wide
 * switch, used by bench.py's timed CPU legs only -- parity tests run with it off */
void orc_set_fast_baseline(int on);

/* ---- one chain, injected draws (SerialMC.jl:37-85 around the sampler loop bodies) ----
 * normals : d x (last+1) column-major; column 0 is the pre-loop draw (used by HMCDA only,
 *           HMCDA.jl:90), column i (1-based step index) feeds step i.
 * uniforms: last+1; entry i feeds the MH test of step i (entry 0 unused).
 * outputs (any may be NULL): samples d x S, grads d x S (NaN-filled for RWM), accept S,
 * logtarget S (plogtarget of the produced MCMCSample), diag_eps S (HMCDA leapStep used at the
 * kept step), diag_nleaps S.  S = number of kept steps = length(first:step:last).
 * returns 0, or -1 "Initial values out of model support", -2 bad arguments.
 */
int32_t orc_run_chain(const orc_model* m, const orc_sampler* s, const orc_range* r,
                      const double* init, const double* scale,
                      const double* normals, const double* uniforms,
                      double* samples, double* grads, uint8_t* accept, double* logtarget,
                      double* diag_eps, int64_t* diag_nleaps, int64_t* n_grad_evals);
int64_t orc_range_length(const orc_range* r);

/* ---- population runners (SURVEY.md 8f.1) --------------------------------------------------------------
 * Targets/tasks t = 0..nt-1 share family and size; models[t], samplers[t] (RWM / MALA / HMC without tuner).
 *
 * SeqMC (src/runners/SeqMC.jl:39-122): particles npart x d (column-major d x npart).  Draw layout, all indexed by
 * k = ((i-1)*nt + t)*npart + n for iteration i (1-based), target t, particle n:
 *   normals d x K, uniforms K (MH test), res_uniforms K (multinomial resampling, used only when it triggers).
 * Outputs: samples d x ((steps-burnin)*npart), weights (steps-burnin)*npart, n_resamples.
 *
 * SerialTempMC (src/runners/SerialTempMC.jl:31-85), one replica: inits d x nt (model.init of every task),
 * normals d x (steps+2) and uniforms steps+2 (MH tests): column 0 = the first consume of task 1 (:44), column 1 = the
 * consume before the loop (:51), column i+1 = iteration i; u_pick steps+1 (at2 = floor(u*(nt-1)) shifted past `at`,
 * :59-60) and u_swap steps+1 (:64), both indexed by iteration i (entry 0 unused).
 * Outputs: samples d x (steps-burnin) (ppars, :73-75), at (steps-burnin) the task the replica is on. */
int32_t orc_run_seqmc(const orc_model* models, const orc_sampler* samplers, int32_t nt, int64_t steps, int64_t burnin,
                      double trigger, int64_t npart, const double* particles, const double* normals,
                      const double* uniforms, const double* res_uniforms, double* samples, double* weights,
                      int64_t* n_resamples);
int32_t orc_run_serialtemp(const orc_model* models, const orc_sampler* samplers, int32_t nt, int64_t steps, int64_t burnin,
                           int64_t swap_period, const double* inits, const double* normals, const double* uniforms,
                           const double* u_pick, const double* u_swap, double* samples, int32_t* at_out);

/* ---- stats over one stored series x[0..n-1] (src/stats) ---- */
double orc_mean(const double* x, int64_t n);                     /* mean.jl:6         */
double orc_mcvar_iid(const double* x, int64_t n);                /* var.jl:7-8        */
double orc_mcvar_bm(const double* x, int64_t n, int64_t batchlen); /* var.jl:20-26    */
double orc_mcvar_imse(const double* x, int64_t n, int64_t maxlag); /* var.jl:45-75    */
double orc_mcvar_ipse(const double* x, int64_t n, int64_t maxlag); /* var.jl:95-116   */
void orc_acov(const double* x, int64_t n, int64_t maxlag, double* acv); /* StatsBase.acf(x, 0:maxlag, correlation=false) */

/* ---- zero-variance control variates (src/stats/zv.jl:8-66; Mira, Solgi, Imparato 2013) ----
 * x, grad: S x d row-major (one chain).  order 1: linearZv (k = d features z = -grad/2); order 2: quadraticZv
 * (k = d(d+3)/2 features: z, 2 z.*x - 1, x_i z_j + x_j z_i for i < j).  Outputs: zv S x d, a k x d (row-major).
 * a[:, i] = -inv(cov(features)) * cov(features, x_i), computed as the Gauss-Jordan solution of [C | Sigma]
 * with partial pivoting (the reference calls LAPACK inv; same value up to conditioning).  returns 0, -2 bad args,
 * -3 singular covariance. */
int32_t orc_zv(const double* x, const double* grad, int64_t S, int64_t d, int32_t order, double* zv, double* a);

/* ---- Philox4x32-10 (Random123; Salmon et al. SC'11) and the draw conventions of the engine ---- */
void orc_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);
/* engine conventions: key = (seed lo, seed hi); ctr = (chain lo, chain hi, step, block);
 * normals block b -> normals 2b, 2b+1 (Box-Muller); uniform for the MH test uses block 0xFFFFFFFF. */
void orc_draw_normals(uint64_t seed, uint64_t chain, uint32_t step, int64_t d, double* z);
double orc_draw_uniform(uint64_t seed, uint64_t chain, uint32_t step);

#ifdef __cplusplus
}
#endif
#endif
