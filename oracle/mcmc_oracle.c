/*
 * mcmc_oracle.c -- CPU restatement of the MCMC.jl hot path.  See mcmc_oracle.h for the contract
 * ("TEST INFRASTRUCTURE ONLY", "parity unpinned").  Citations are file:line into the reference
 * tree (dingliumath/MCMC.jl).  Build: gcc -O2 -std=c99 -ffp-contract=off -fPIC -shared (no
 * -ffast-math; contraction off so every rounding is the one written here).
 */
#include "mcmc_oracle.h"
#include <math.h>
#include <stdlib.h>
#include <string.h>

#define LOG2PI 1.8378770664093453        /* log(2*pi) */
#define LN_SQRT_2PI 0.91893853320467274178 /* Rmath M_LN_SQRT_2PI */
#define TWO_PI 6.283185307179586          /* Julia: 2*pi -> Float64 */

/* ------------------------------------------------------------------------------------------ */
/* scalar log-densities, restating Distributions.jl (2013: Rmath dnorm4 / dunif / pnorm)       */
/* ------------------------------------------------------------------------------------------ */

/* logpdf(Normal(mu,sigma), x): Rmath dnorm4(x, mu, sigma, give_log=TRUE) */
static double logpdf_normal(double x, double mu, double sigma) {
  double z = (x - mu) / sigma;
  return -(LN_SQRT_2PI + 0.5 * z * z + log(sigma));
}

/* logpdf(Uniform(a,b), x): -log(b-a) inside [a,b], -Inf outside (Rmath dunif, give_log) */
static double logpdf_uniform(double x, double a, double b) {
  if (a <= x && x <= b) return -log(b - a);
  return -INFINITY;
}

/* log Phi(x) = logcdf(Normal(), x) (examples/probit_regression.jl:29).  The 2013 Distributions.jl
 * delegated to Rmath pnorm(log.p=TRUE); restated here through erfc with the standard asymptotic
 * series in the far lower tail; tests/ check it against scipy.special.log_ndtr. */
double orc_log_ndtr(double x) {
  if (x > 0.0) {
    return log1p(-0.5 * erfc(x * 0.70710678118654752440)); /* upper half: 1 - upper tail, as pnorm does */
  } else if (x > -37.0) {
    return log(0.5 * erfc(-x * 0.70710678118654752440));
  } else {
    /* Phi(x) ~ phi(x)/|x| * (1 - 1/x^2 + 3/x^4 - 15/x^6 + 105/x^8 - 945/x^10) */
    double x2 = x * x, r = 1.0 / x2;
    double s = 1.0 - r * (1.0 - 3.0 * r * (1.0 - 5.0 * r * (1.0 - 7.0 * r * (1.0 - 9.0 * r))));
    return -0.5 * x2 - LN_SQRT_2PI - log(-x) + log(s);
  }
}

/* ------------------------------------------------------------------------------------------ */
/* models                                                                                      */
/* ------------------------------------------------------------------------------------------ */

/* eta = X*beta (examples/logistic_regression.jl:18 `X * vars`): dgemv 'N', accumulated per row in
 * column order. */
static void x_times_beta(const orc_model* m, const double* beta, double* eta) {
  int64_t N = m->N, d = m->d;
  for (int64_t i = 0; i < N; i++) eta[i] = 0.0;
  for (int64_t j = 0; j < d; j++) {
    const double* col = m->X + j * N;
    double b = beta[j];
    for (int64_t i = 0; i < N; i++) eta[i] += col[i] * b;
  }
}
/* g = X'*r : dgemv 'T' (reverse rule of X*vars; probit_regression.jl:39 `X'*(...)`) */
static void xt_times_r(const orc_model* m, const double* r, double* g) {
  int64_t N = m->N, d = m->d;
  for (int64_t j = 0; j < d; j++) {
    const double* col = m->X + j * N;
    double s = 0.0;
    for (int64_t i = 0; i < N; i++) s += col[i] * r[i];
    g[j] = s;
  }
}

/* LLAcc semantics (src/dsl/definitions/AccumulatorDerivRules.jl:10-20, src/dsl/modelparser.jl:64-92):
 * after every `~` statement the accumulator must be finite, else the generated function returns
 * -Inf (and a zero gradient). */
#define OOS_RETURN(grad, d) do { if (grad) memset(grad, 0, sizeof(double) * (size_t)(d)); return -INFINITY; } while (0)

static double eval_normal_fn(const orc_model* m, const double* v, double* grad) {
  /* README.md:60,63: v -> -dot(v,v), grad v -> -2v */
  double s = 0.0;
  for (int64_t j = 0; j < m->d; j++) s += v[j] * v[j];
  if (grad) for (int64_t j = 0; j < m->d; j++) grad[j] = -2.0 * v[j];
  return -s;
}

static double eval_normal_dsl(const orc_model* m, const double* v, double* grad) {
  /* README.md:67-72 `v ~ Normal(0, 1)`; grad rule MCMCDerivRules.jl:57 dx += (mu - x)/(sigma*sigma)*ds */
  double mu = m->hyper[0], sigma = m->hyper[1];
  double s = 0.0;
  for (int64_t j = 0; j < m->d; j++) s += logpdf_normal(v[j], mu, sigma);
  double acc = 0.0 + s;
  if (!isfinite(acc)) OOS_RETURN(grad, m->d);
  if (grad) for (int64_t j = 0; j < m->d; j++) grad[j] = (mu - v[j]) / (sigma * sigma);
  return acc;
}

static double eval_linear(const orc_model* m, const double* b, double* grad) {
  /* examples/linear_regression.jl:14-18:
   *   vars ~ Normal(0, 1.0); resid = Y - X * vars; resid ~ Normal(0, 1.0) */
  int64_t N = m->N, d = m->d;
  double psd = m->hyper[0], nsd = m->hyper[1];
  double s = 0.0;
  for (int64_t j = 0; j < d; j++) s += logpdf_normal(b[j], 0.0, psd);
  double acc = 0.0 + s;
  if (!isfinite(acc)) OOS_RETURN(grad, d);
  double* eta = (double*)malloc(sizeof(double) * (size_t)N);
  x_times_beta(m, b, eta);
  double s2 = 0.0;
  for (int64_t i = 0; i < N; i++) { eta[i] = m->y[i] - eta[i]; s2 += logpdf_normal(eta[i], 0.0, nsd); }
  acc = acc + s2;
  if (!isfinite(acc)) { free(eta); OOS_RETURN(grad, d); }
  if (grad) {
    /* dresid = (0 - resid)/(sd*sd) (MCMCDerivRules.jl:57); resid = Y - X*vars => dvars = -X' dresid */
    for (int64_t i = 0; i < N; i++) eta[i] = -((0.0 - eta[i]) / (nsd * nsd));
    xt_times_r(m, eta, grad);
    for (int64_t j = 0; j < d; j++) grad[j] += (0.0 - b[j]) / (psd * psd);
  }
  free(eta);
  return acc;
}

/* ---- CPU-baseline variant of the logistic evaluation (bench.py's cpu_baseline / --impl reference only) --------------------
 * The plain restatement below makes two passes over X (dgemv 'N', then dgemv 'T') with one serial accumulator each, which
 * is what the reference's expression graph does but undersells a CPU: an optimised BLAS blocks the rows so that X is read
 * from DRAM once per evaluation and keeps several accumulators in flight.  orc_set_fast_baseline(1) switches eval_logistic
 * to that shape (256-row blocks that stay in L2 between X*beta and X'r, 4 partial sums per dot product; same elementwise
 * arithmetic).  Parity tests never enable it: its sums are reassociated (agreement ~1e-13, checked in tests/test_oracle.py). */
static int g_fast_baseline = 0;
void orc_set_fast_baseline(int on) { g_fast_baseline = on; }

/* cloned for AVX2 / AVX-512 hosts and dispatched at load time (the library is built on one machine and timed on another) */
__attribute__((target_clones("avx512f", "avx2", "default")))
static double eval_logistic_blocked(const orc_model* m, const double* b, double* grad) {
  enum { RB = 256 };
  int64_t N = m->N, d = m->d;
  double psd = m->hyper[0], sgn = m->hyper[1];
  double s = 0.0;
  for (int64_t j = 0; j < d; j++) s += logpdf_normal(b[j], 0.0, psd);
  double acc = 0.0 + s;
  if (!isfinite(acc)) OOS_RETURN(grad, d);
  double eta[RB];
  double ll0 = 0.0, ll1 = 0.0;
  if (grad) for (int64_t j = 0; j < d; j++) grad[j] = 0.0;
  for (int64_t i0 = 0; i0 < N; i0 += RB) {
    int64_t nb = (N - i0 < RB) ? N - i0 : RB;
    for (int64_t i = 0; i < nb; i++) eta[i] = 0.0;
    for (int64_t j = 0; j < d; j++) {
      const double* col = m->X + j * N + i0;
      double bj = b[j];
      for (int64_t i = 0; i < nb; i++) eta[i] += col[i] * bj;
    }
    for (int64_t i = 0; i < nb; i++) {
      double e = exp(sgn * eta[i]);
      double den = 1.0 + e;
      double p = 1.0 / den;
      double yi = m->y[i0 + i];
      double ll = (yi != 0.0) ? log(p) : log(1.0 - p);
      if (i & 1) ll1 += ll; else ll0 += ll;
      double dprob = 1.0 / (p - 1.0 + yi);
      double dden = -(dprob / (den * den));
      eta[i] = sgn * (e * dden);
    }
    if (grad) {
      for (int64_t j = 0; j < d; j++) {
        const double* col = m->X + j * N + i0;
        double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
        int64_t i = 0;
        for (; i + 4 <= nb; i += 4) { s0 += col[i] * eta[i]; s1 += col[i + 1] * eta[i + 1]; s2 += col[i + 2] * eta[i + 2]; s3 += col[i + 3] * eta[i + 3]; }
        for (; i < nb; i++) s0 += col[i] * eta[i];
        grad[j] += (s0 + s1) + (s2 + s3);
      }
    }
  }
  acc = acc + (ll0 + ll1);
  if (!isfinite(acc)) OOS_RETURN(grad, d);
  if (grad) for (int64_t j = 0; j < d; j++) grad[j] += (0.0 - b[j]) / (psd * psd);
  return acc;
}

static double eval_logistic(const orc_model* m, const double* b, double* grad) {
  if (g_fast_baseline) return eval_logistic_blocked(m, b, grad);
  /* examples/logistic_regression.jl:16-20:
   *   vars ~ Normal(0, 1.0); prob = 1 / (1. + exp(- X * vars)); Y ~ Bernoulli(prob)
   * Bernoulli logpdf: x==1 ? log(p1) : log(p0), p0 = 1 - p1 (Distributions.jl Bernoulli);
   * gradient rule MCMCDerivRules.jl:111: dd1 += 1/(p1 - 1 + x)*ds, chained through `/`, `+`,
   * `exp`, unary minus and X*vars. hyper[1] = sign inside exp (-1 example, +1 test/test_syntax.jl:18). */
  int64_t N = m->N, d = m->d;
  double psd = m->hyper[0], sgn = m->hyper[1];
  double s = 0.0;
  for (int64_t j = 0; j < d; j++) s += logpdf_normal(b[j], 0.0, psd);
  double acc = 0.0 + s;
  if (!isfinite(acc)) OOS_RETURN(grad, d);
  double* eta = (double*)malloc(sizeof(double) * (size_t)N);
  x_times_beta(m, b, eta);
  double s2 = 0.0;
  for (int64_t i = 0; i < N; i++) {
    double e = exp(sgn * eta[i]);
    double den = 1.0 + e;
    double p = 1.0 / den;
    double yi = m->y[i];
    double ll = (yi != 0.0) ? log(p) : log(1.0 - p);
    s2 += ll;
    /* reverse sweep for this row: dprob = 1/(p-1+y); dden = -dprob/(den*den); de = dden;
     * d(sgn*eta) = e*de; deta = sgn * that */
    double dprob = 1.0 / (p - 1.0 + yi);
    double dden = -(dprob / (den * den));
    eta[i] = sgn * (e * dden);
  }
  acc = acc + s2;
  if (!isfinite(acc)) { free(eta); OOS_RETURN(grad, d); }
  if (grad) {
    xt_times_r(m, eta, grad);
    for (int64_t j = 0; j < d; j++) grad[j] += (0.0 - b[j]) / (psd * psd);
  }
  free(eta);
  return acc;
}

static double eval_probit(const orc_model* m, const double* b, double* grad) {
  /* examples/probit_regression.jl:18-41 (plain user functions: no LLAcc, NaN/Inf propagate):
   *   logprior = logpdf(MvNormal(0, priorvar*I), pars)
   *   loglik   = dot(logcdf(normal, XPars), y) + dot(logcdf(normal, -XPars), 1-y)
   *   grad     = X'*( y.*exp(-(XPars.^2+log(2*pi))/2 - logcdf(normal, XPars))
   *                  -(1-y).*exp(-(XPars.^2+log(2*pi))/2 - logcdf(normal, -XPars)) ) - pars/priorvar */
  int64_t N = m->N, d = m->d;
  double psd = m->hyper[0], pvar = psd * psd;
  double q = 0.0;
  for (int64_t j = 0; j < d; j++) q += b[j] * b[j];
  double logprior = -0.5 * ((double)d * LOG2PI + (double)d * log(pvar)) - 0.5 * (q / pvar);
  double* eta = (double*)malloc(sizeof(double) * (size_t)N);
  x_times_beta(m, b, eta);
  double d1 = 0.0, d2 = 0.0;
  for (int64_t i = 0; i < N; i++) {
    double xi = eta[i], yi = m->y[i];
    double lp = orc_log_ndtr(xi), lm = orc_log_ndtr(-xi);
    d1 += lp * yi;
    d2 += lm * (1.0 - yi);
    double base = -(xi * xi + LOG2PI) / 2.0;
    eta[i] = yi * exp(base - lp) - (1.0 - yi) * exp(base - lm);
  }
  double loglik = d1 + d2;
  if (grad) {
    xt_times_r(m, eta, grad);
    for (int64_t j = 0; j < d; j++) grad[j] = grad[j] - b[j] / pvar;
  }
  free(eta);
  return logprior + loglik;
}

static double eval_ou(const orc_model* m, const double* v, double* grad) {
  /* examples/ornstein.jl:19-27:
   *   tau ~ Uniform(0,100); sigma ~ Uniform(0,2); mu ~ Uniform(0,20)
   *   fac = exp(- 1. / tau); resid = x[2:end] - x[1:end-1]*fac - mu*(1.-fac); resid ~ Normal(0, sigma)
   * parameter vector = (tau, sigma, mu) (keyword order ornstein.jl:29).  Rules MCMCDerivRules.jl:57-64. */
  int64_t T = m->N;
  const double* x = m->y;
  double tau = v[0], sigma = v[1], mu = v[2];
  double acc = 0.0;
  acc = acc + logpdf_uniform(tau, 0.0, m->hyper[0]);   if (!isfinite(acc)) OOS_RETURN(grad, 3);
  acc = acc + logpdf_uniform(sigma, 0.0, m->hyper[1]); if (!isfinite(acc)) OOS_RETURN(grad, 3);
  acc = acc + logpdf_uniform(mu, 0.0, m->hyper[2]);    if (!isfinite(acc)) OOS_RETURN(grad, 3);
  double fac = exp(-1.0 / tau);
  double omf = 1.0 - fac;
  double s = 0.0, dfac = 0.0, dsigma = 0.0, dmu = 0.0;
  for (int64_t t = 0; t + 1 < T; t++) {
    double resid = x[t + 1] - x[t] * fac - mu * omf;
    s += logpdf_normal(resid, 0.0, sigma);
    double dres = (0.0 - resid) / (sigma * sigma);               /* MCMCDerivRules.jl:57 */
    dsigma += ((resid - 0.0) * (resid - 0.0) / (sigma * sigma) - 1.0) / sigma; /* :59 */
    dfac += dres * (mu - x[t]);   /* d resid / d fac = -x[t] + mu */
    dmu += dres * (-omf);
  }
  acc = acc + s;
  if (!isfinite(acc)) OOS_RETURN(grad, 3);
  if (grad) {
    grad[0] = dfac * fac * (1.0 / (tau * tau)); /* fac = exp(-1/tau): dfac/dtau = fac/tau^2; Uniform dx += 0 (:62) */
    grad[1] = dsigma;
    grad[2] = dmu;
  }
  return acc;
}

static double eval_abs_normal(const orc_model* m, const double* v, double* grad) {
  /* README.md:253-259: y = abs(x); y ~ Normal(mu, sigma).  abs rule: dx += sign(x) * ds; Normal rule MCMCDerivRules.jl:57 */
  double mu = m->hyper[0], sigma = m->hyper[1];
  double s = 0.0;
  for (int64_t j = 0; j < m->d; j++) s += logpdf_normal(fabs(v[j]), mu, sigma);
  double acc = 0.0 + s;
  if (!isfinite(acc)) OOS_RETURN(grad, m->d);
  if (grad) for (int64_t j = 0; j < m->d; j++) {
    double sg = (v[j] > 0.0) ? 1.0 : ((v[j] < 0.0) ? -1.0 : 0.0);
    grad[j] = sg * ((mu - fabs(v[j])) / (sigma * sigma));
  }
  return acc;
}

static double eval_any(const orc_model* m, const double* beta, double* grad) {
  switch (m->family) {
    case ORC_FAM_ABS_NORMAL: return eval_abs_normal(m, beta, grad);
    case ORC_FAM_NORMAL_FN: return eval_normal_fn(m, beta, grad);
    case ORC_FAM_NORMAL_DSL: return eval_normal_dsl(m, beta, grad);
    case ORC_FAM_LINEAR: return eval_linear(m, beta, grad);
    case ORC_FAM_LOGISTIC: return eval_logistic(m, beta, grad);
    case ORC_FAM_PROBIT: return eval_probit(m, beta, grad);
    case ORC_FAM_OU: return eval_ou(m, beta, grad);
  }
  return NAN;
}
double orc_eval(const orc_model* m, const double* beta) { return eval_any(m, beta, NULL); }
double orc_evalallg(const orc_model* m, const double* beta, double* grad) { return eval_any(m, beta, grad); }

/* ------------------------------------------------------------------------------------------ */
/* runner + samplers                                                                           */
/* ------------------------------------------------------------------------------------------ */

int64_t orc_range_length(const orc_range* r) {
  if (r->step < 1 || r->last < r->first) return 0;
  return (r->last - r->first) / r->step + 1;
}
/* in(i, r) for r = first:step:last (SerialMC.jl:49) */
static int in_range(int64_t i, const orc_range* r) {
  return i >= r->first && i <= r->last && ((i - r->first) % r->step) == 0;
}

typedef struct { /* HMCSample, HMC.jl:81-88 */
  double *pars, *grad, *m;
  double logTarget, H;
} hmc_state;

static double dotp(const double* a, const double* b, int64_t d) {
  double s = 0.0;
  for (int64_t j = 0; j < d; j++) s += a[j] * b[j];
  return s;
}
static void hs_alloc(hmc_state* s, int64_t d) {
  s->pars = (double*)calloc((size_t)d, sizeof(double));
  s->grad = (double*)calloc((size_t)d, sizeof(double));
  s->m = (double*)calloc((size_t)d, sizeof(double));
  s->logTarget = NAN; s->H = NAN;
}
static void hs_free(hmc_state* s) { free(s->pars); free(s->grad); free(s->m); }
static void hs_copy(hmc_state* dst, const hmc_state* src, int64_t d) { /* deepcopy */
  memcpy(dst->pars, src->pars, sizeof(double) * (size_t)d);
  memcpy(dst->grad, src->grad, sizeof(double) * (size_t)d);
  memcpy(dst->m, src->m, sizeof(double) * (size_t)d);
  dst->logTarget = src->logTarget; dst->H = src->H;
}
/* calc! HMC.jl:90 ; update! HMC.jl:91 */
static void hs_calc(hmc_state* s, const orc_model* m, int64_t* nev) { s->logTarget = orc_evalallg(m, s->pars, s->grad); if (nev) (*nev)++; }
static void hs_update(hmc_state* s, int64_t d) { s->H = -s->logTarget + 0.5 * dotp(s->m, s->m, d); }
/* leapfrog HMC.jl:93-102, in place on a copy held by the caller */
static void hs_leapfrog(hmc_state* n, double ve, const orc_model* m, int64_t* nev) {
  int64_t d = m->d;
  for (int64_t j = 0; j < d; j++) n->m[j] += (0.5 * n->grad[j]) * ve;
  for (int64_t j = 0; j < d; j++) n->pars[j] += ve * n->m[j];
  hs_calc(n, m, nev);
  for (int64_t j = 0; j < d; j++) n->m[j] += (0.5 * n->grad[j]) * ve;
  hs_update(n, d);
}

/* SerialMC.jl:49-66: store the produced MCMCSample at a kept step */
static void store_kept(int64_t d, int64_t kept, const double* pp, double plt, const double* pg, int acc,
                       double eps, int64_t nl, double* samples, double* grads, uint8_t* accept,
                       double* logtarget, double* diag_eps, int64_t* diag_nleaps) {
  if (samples) memcpy(samples + kept * d, pp, sizeof(double) * (size_t)d);
  if (grads) {
    if (pg) memcpy(grads + kept * d, pg, sizeof(double) * (size_t)d);
    else for (int64_t jj = 0; jj < d; jj++) grads[kept * d + jj] = NAN; /* SerialMC.jl:42 */
  }
  if (accept) accept[kept] = (uint8_t)acc;
  if (logtarget) logtarget[kept] = plt;
  if (diag_eps) diag_eps[kept] = eps;
  if (diag_nleaps) diag_nleaps[kept] = nl;
}

/* mean_rb_hmc, src/stats/mean.jl:17-31: (sample + sum_k exp(H0 - H_k) pars_k) / (nLeaps + 1) over the recorded leap
 * states of one trajectory, written to rb_out[kept] */
static void store_rb(double* rb_out, int64_t kept, int64_t d, const double* smp, double H0, const double* leapP,
                     const double* leapH, int64_t nLeaps) {
  for (int64_t jj = 0; jj < d; jj++) {
    double sm = smp[jj];
    for (int64_t k = 0; k < nLeaps; k++) sm += exp(H0 - leapH[k]) * leapP[k * d + jj];
    rb_out[kept * d + jj] = sm / (double)(nLeaps + 1);
  }
}

/* round() of Julia 0.2 == C round (half away from zero) (HMCDA.jl:104) */

int32_t orc_run_chain(const orc_model* m, const orc_sampler* s, const orc_range* r,
                      const double* init, const double* scale,
                      const double* normals, const double* uniforms,
                      double* samples, double* grads, uint8_t* accept, double* logtarget,
                      double* diag_eps, int64_t* diag_nleaps, int64_t* n_grad_evals) {
  int64_t d = m->d;
  int64_t burnin = r->first - 1, len = r->last;
  /* SerialMC.jl:25-27 */
  if (burnin < 0 || len <= burnin || r->step < 1) return -2;
  int64_t nev = 0;
  int64_t kept = 0;
  int32_t rc = 0;

#define STORE(PP, PLT, PG, ACC, EPS, NL)                                                   \
  do {                                                                                     \
    if (in_range(i, r)) {                                                                  \
      store_kept(d, kept, (PP), (PLT), (PG), (ACC), (EPS), (NL), samples, grads, accept,   \
                 logtarget, diag_eps, diag_nleaps);                                        \
      kept++;                                                                              \
    }                                                                                      \
  } while (0)

  if (s->kind == ORC_RWM) {
    /* RWM.jl:43-72 */
    double* sc = (double*)malloc(sizeof(double) * (size_t)d);
    double* pars = (double*)malloc(sizeof(double) * (size_t)d);
    double* prop = (double*)malloc(sizeof(double) * (size_t)d);
    for (int64_t j = 0; j < d; j++) sc[j] = scale[j] * s->scale;  /* :52 */
    memcpy(pars, init, sizeof(double) * (size_t)d);
    double lt = orc_eval(m, pars);
    if (!isfinite(lt)) rc = -1;
    for (int64_t i = s->start_step + 1; rc == 0 && i <= len; i++) {
      const double* z = normals + i * d;
      for (int64_t j = 0; j < d; j++) prop[j] = pars[j] + z[j] * sc[j]; /* :59 */
      double plt = orc_eval(m, prop);                                    /* :60 */
      double ratio = plt - lt;                                           /* :62 */
      if (ratio > 0 || ratio > log(uniforms[i])) {                       /* :63 */
        STORE(prop, plt, (const double*)NULL, 1, NAN, 0);
        memcpy(pars, prop, sizeof(double) * (size_t)d); lt = plt;
      } else {
        STORE(pars, lt, (const double*)NULL, 0, NAN, 0);
      }
    }
    free(sc); free(pars); free(prop);
  } else if (s->kind == ORC_MALA) {
    /* MALA.jl:65-126 */
    double* pars = (double*)malloc(sizeof(double) * (size_t)d);
    double* grad = (double*)malloc(sizeof(double) * (size_t)d);
    double* mean = (double*)malloc(sizeof(double) * (size_t)d);
    double* prop = (double*)malloc(sizeof(double) * (size_t)d);
    double* pgrad = (double*)malloc(sizeof(double) * (size_t)d);
    memcpy(pars, init, sizeof(double) * (size_t)d);
    double lt = orc_evalallg(m, pars, grad); nev++;
    if (!isfinite(lt)) rc = -1;
    double tune_step = s->scale; int64_t accepted = 0, proposed = 0; /* EmpiricalMALATune :19-43 */
    for (int64_t i = s->start_step + 1; rc == 0 && i <= len; i++) {
      double h;
      if (s->tuner_on) { proposed += 1; h = tune_step; } else h = s->scale; /* :91-96 */
      const double* z = normals + i * d;
      double sq = sqrt(h);
      for (int64_t j = 0; j < d; j++) mean[j] = pars[j] + (h / 2.0) * grad[j];   /* :98 */
      for (int64_t j = 0; j < d; j++) prop[j] = mean[j] + sq * z[j];             /* :100 */
      double plt = orc_evalallg(m, prop, pgrad); nev++;                          /* :101 */
      double lc = log(TWO_PI * h) / 2.0;
      double qno = 0.0;                                                          /* :103 */
      for (int64_t j = 0; j < d; j++) { double t = mean[j] - prop[j]; qno += -(t * t) / (2.0 * h) - lc; }
      for (int64_t j = 0; j < d; j++) mean[j] = prop[j] + (h / 2.0) * pgrad[j];  /* :104 */
      double qon = 0.0;                                                          /* :105 */
      for (int64_t j = 0; j < d; j++) { double t = mean[j] - pars[j]; qon += -(t * t) / (2.0 * h) - lc; }
      double ratio = plt + qon - lt - qno;                                       /* :107 */
      if (ratio > 0 || ratio > log(uniforms[i])) {                               /* :108 */
        STORE(prop, plt, pgrad, 1, h, 0);
        memcpy(pars, prop, sizeof(double) * (size_t)d); lt = plt;
        memcpy(grad, pgrad, sizeof(double) * (size_t)d);
        if (s->tuner_on) accepted += 1;
      } else {
        STORE(pars, lt, grad, 0, h, 0);
      }
      if (s->tuner_on && i <= burnin && (i % s->adapt_step) == 0) {              /* :116-118, adapt! :36-39 */
        double rate = (double)accepted / (double)proposed;
        tune_step *= (1.0 / (1.0 + exp(-11.0 * (rate - s->target_rate))) + 0.5);
        accepted = 0; proposed = 0;
      }
    }
    free(pars); free(grad); free(mean); free(prop); free(pgrad);
  } else if (s->kind == ORC_HMC) {
    /* HMC.jl:106-175 */
    hmc_state st0, st; hs_alloc(&st0, d); hs_alloc(&st, d);
    memcpy(st0.pars, init, sizeof(double) * (size_t)d);
    hs_calc(&st0, m, &nev);                                       /* :119-120 */
    if (!isfinite(st0.logTarget)) rc = -1;                        /* :121 */
    int64_t t_nleaps = s->nleaps; double t_step = s->scale; int64_t accepted = 0, proposed = 0; /* :20-47 */
    for (int64_t i = s->start_step + 1; rc == 0 && i <= len; i++) {
      int64_t nLeaps; double leapStep;
      if (s->tuner_on) { proposed += 1; nLeaps = t_nleaps; leapStep = t_step; }
      else { nLeaps = s->nleaps; leapStep = s->scale; }           /* :129-134 */
      memcpy(st0.m, normals + i * d, sizeof(double) * (size_t)d); /* :136 */
      hs_update(&st0, d);                                         /* :137 */
      hs_copy(&st, &st0, d);                                      /* :138 */
      double* leapP = NULL; double* leapH = NULL;                 /* leapStates[2..nLeaps+1] (:145-150) */
      if (s->rb_out) { leapP = (double*)malloc(sizeof(double) * (size_t)(nLeaps * d)); leapH = (double*)malloc(sizeof(double) * (size_t)nLeaps); }
      for (int64_t j = 0; j < nLeaps; j++) {                      /* :141-143 */
        hs_leapfrog(&st, leapStep, m, &nev);
        if (s->rb_out) { memcpy(leapP + j * d, st.pars, sizeof(double) * (size_t)d); leapH[j] = st.H; }
      }
      if (s->rb_out && in_range(i, r)) {                          /* mean_rb_hmc, src/stats/mean.jl:17-31 */
        int accn = uniforms[i] < exp(st0.H - st.H);
        store_rb(s->rb_out, kept, d, accn ? st.pars : st0.pars, st0.H, leapP, leapH, nLeaps);   /* c.samples[i, :] */
      }
      if (leapP) { free(leapP); free(leapH); }
      if (uniforms[i] < exp(st0.H - st.H)) {                      /* :154 */
        STORE(st.pars, st.logTarget, st.grad, 1, leapStep, nLeaps);
        hs_copy(&st0, &st, d);                                    /* :158 */
        if (s->tuner_on) accepted += 1;
      } else {
        STORE(st0.pars, st0.logTarget, st0.grad, 0, leapStep, nLeaps);
      }
      if (s->tuner_on && i <= burnin && (i % s->adapt_step) == 0) { /* :167-169, adapt! :39-43 */
        double rate = (double)accepted / (double)proposed;
        t_step *= (1.0 / (1.0 + exp(-11.0 * (rate - s->target_rate))) + 0.5);
        double c = ceil(s->target_path / t_step);
        t_nleaps = (c < (double)s->max_step) ? (int64_t)c : (int64_t)s->max_step;
        accepted = 0; proposed = 0;
      }
    }
    hs_free(&st0); hs_free(&st);
  } else if (s->kind == ORC_HMCDA) {
    /* HMCDA.jl:72-143 */
    hmc_state st0, st; hs_alloc(&st0, d); hs_alloc(&st, d);
    memcpy(st0.pars, init, sizeof(double) * (size_t)d);
    hs_calc(&st0, m, &nev);                                       /* :86-87 */
    if (!isfinite(st0.logTarget)) rc = -1;                        /* :88 */
    double leapStep = 1.0, mu = 0.0, dualLeapStep = 1.0, dualH = 0.0;
    if (rc == 0) {
      memcpy(st0.m, normals + 0 * d, sizeof(double) * (size_t)d); /* :90 pre-loop randn */
      /* initializeHMCDAStep HMCDA.jl:51-69, restated literally.  st0.H is still NaN here
       * (HMC.jl:88: new HMCSample has H = NaN; update! has not been called), so p is NaN, a = -1,
       * the while test is false and the function returns 1.0 after one leapfrog. */
      {
        double ls = 1.0;
        hs_copy(&st, &st0, d); hs_leapfrog(&st, ls, m, &nev);     /* :55-56 */
        double p = exp(st.H - st0.H);                             /* :57 */
        int a = 2 * (p > 0.5) - 1;                                /* :58 */
        while (pow(p, (double)a) > pow(2.0, (double)(-a))) {      /* :61 */
          ls = ls * pow(2.0, (double)a);
          hs_copy(&st, &st0, d); hs_leapfrog(&st, ls, m, &nev);
          p = exp(st.H - st0.H);
        }
        leapStep = ls;
      }
      mu = log(10.0 * leapStep);                                  /* :92 */
      /* test aid (true resume, the engine's mcmcgpu_run_set_state): continue from a saved dual-averaging state.
       * mu keeps the reference's value log(10 * 1.0): the initial search always returns 1.0 (see above). */
      if (s->da_state) { leapStep = s->da_state[0]; dualLeapStep = s->da_state[1]; dualH = s->da_state[2]; }
    }
    for (int64_t i = s->start_step + 1; rc == 0 && i <= len; i++) {
      memcpy(st0.m, normals + i * d, sizeof(double) * (size_t)d); /* :100 */
      hs_update(&st0, d);                                         /* :101 */
      hs_copy(&st, &st0, d);                                      /* :102 */
      const double own_eps = leapStep;
      if (s->force_eps) leapStep = s->force_eps[i];               /* teacher forcing (test aid, see header) */
      double nl = round(s->len / leapStep);                       /* :104 */
      if (!(nl >= 1.0)) nl = 1.0;                                 /* max(1, .) */
      if (s->max_leaps > 0 && nl > (double)s->max_leaps) nl = (double)s->max_leaps; /* documented cap */
      int64_t nLeaps = (int64_t)nl;
      double* leapP = NULL; double* leapH = NULL;                 /* storeLeaps, as in the HMC branch */
      if (s->rb_out) { leapP = (double*)malloc(sizeof(double) * (size_t)(nLeaps * d)); leapH = (double*)malloc(sizeof(double) * (size_t)nLeaps); }
      for (int64_t j = 0; j < nLeaps; j++) {                      /* :107-109 */
        hs_leapfrog(&st, leapStep, m, &nev);
        if (s->rb_out) { memcpy(leapP + j * d, st.pars, sizeof(double) * (size_t)d); leapH[j] = st.H; }
      }
      double e = exp(st0.H - st.H);
      /* p = min(1, exp(H0-H)) (:120).  Documented deviation: a NaN ratio is treated as p = 0
       * (reject, adapt with 0) instead of poisoning dualH/leapStep for the rest of the run. */
      double p = isnan(e) ? 0.0 : (e < 1.0 ? e : 1.0);
      if (s->rb_out && in_range(i, r)) store_rb(s->rb_out, kept, d, uniforms[i] < p ? st.pars : st0.pars, st0.H, leapP, leapH, nLeaps);
      if (leapP) { free(leapP); free(leapH); }
      double eps_used = own_eps;
      if (uniforms[i] < p) {                                      /* :121 */
        STORE(st.pars, st.logTarget, st.grad, 1, eps_used, nLeaps);
        hs_copy(&st0, &st, d);                                    /* :125 */
      } else {
        STORE(st0.pars, st0.logTarget, st0.grad, 0, eps_used, nLeaps);
      }
      if (i < burnin) {                                           /* :133 */
        double fi = (double)i;
        double eta = 1.0 / (fi + s->t0);                          /* :134 */
        dualH = (1.0 - eta) * dualH + eta * (s->rate - p);        /* :135 */
        leapStep = exp(mu - sqrt(fi) * dualH / s->shrinkage);     /* :136 */
        eta = pow(fi, -s->step);                                  /* :137 */
        dualLeapStep = exp((1.0 - eta) * log(dualLeapStep) + eta * log(leapStep)); /* :138 */
      } else {
        leapStep = dualLeapStep;                                  /* :140 */
      }
    }
    hs_free(&st0); hs_free(&st);
  } else if (s->kind == ORC_RAM) {
    /* RAM.jl:41-80 (Vihola 2012).  diag_eps carries the "scale" diagnostic trace(S) of the kept step (:65,69). */
    double* pars = (double*)malloc(sizeof(double) * (size_t)d);
    double* prop = (double*)malloc(sizeof(double) * (size_t)d);
    double* S = (double*)calloc((size_t)(d * d), sizeof(double));     /* row-major S[a*d+b] */
    double* A = (double*)malloc(sizeof(double) * (size_t)(d * d));
    double* Bm = (double*)malloc(sizeof(double) * (size_t)(d * d));
    for (int64_t j = 0; j < d; j++) S[j * d + j] = scale[j] * s->scale;       /* :50,55 */
    memcpy(pars, init, sizeof(double) * (size_t)d);
    double lt = orc_eval(m, pars);
    if (!isfinite(lt)) rc = -1;                                               /* :53 */
    for (int64_t i = s->start_step + 1; rc == 0 && i <= len; i++) {
      const double* z = normals + i * d;                                      /* :59 rvec */
      for (int64_t a = 0; a < d; a++) {                                       /* :60 pars + S * rvec */
        double acc = 0.0;
        for (int64_t b = 0; b < d; b++) acc += S[a * d + b] * z[b];
        prop[a] = pars[a] + acc;
      }
      double plt = orc_eval(m, prop);                                         /* :61 */
      double ratio = plt - lt;                                                /* :63 */
      double tr = 0.0;
      for (int64_t j = 0; j < d; j++) tr += S[j * d + j];                     /* trace(S) */
      if (ratio > 0 || ratio > log(uniforms[i])) {                            /* :64 */
        STORE(prop, plt, (const double*)NULL, 1, tr, 0);
        memcpy(pars, prop, sizeof(double) * (size_t)d); lt = plt;
      } else {
        STORE(pars, lt, (const double*)NULL, 0, tr, 0);
      }
      /* scale tuning :73-78 */
      double eta = (double)d * pow((double)i, -2.0 / 3.0);
      if (!(eta < 1.0)) eta = 1.0;                                            /* min(1, .) */
      double er = exp(ratio);
      double al = isnan(er) ? 0.0 : (er < 1.0 ? er : 1.0);                    /* min(1, exp(ratio)); NaN => 0 (documented) */
      double zz = dotp(z, z, d);
      for (int64_t a = 0; a < d; a++)                                         /* I + (r r')/dot(r,r) * eta * (al - rate) */
        for (int64_t b = 0; b < d; b++)
          A[a * d + b] = ((a == b) ? 1.0 : 0.0) + (z[a] * z[b]) / zz * eta * (al - s->rate);
      for (int64_t a = 0; a < d; a++)                                         /* Bm = S * A */
        for (int64_t b = 0; b < d; b++) {
          double acc = 0.0;
          for (int64_t k = 0; k < d; k++) acc += S[a * d + k] * A[k * d + b];
          Bm[a * d + b] = acc;
        }
      for (int64_t a = 0; a < d; a++)                                         /* A = Bm * S' */
        for (int64_t b = 0; b < d; b++) {
          double acc = 0.0;
          for (int64_t k = 0; k < d; k++) acc += Bm[a * d + k] * S[b * d + k];
          A[a * d + b] = acc;
        }
      /* S = chol(SS)' : lower Cholesky factor, row by row (Cholesky-Banachiewicz) */
      for (int64_t a = 0; a < d; a++)
        for (int64_t b = 0; b < d; b++) {
          if (b > a) { S[a * d + b] = 0.0; continue; }
          double acc = A[a * d + b];
          for (int64_t k = 0; k < b; k++) acc -= S[a * d + k] * S[b * d + k];
          S[a * d + b] = (a == b) ? sqrt(acc) : acc / S[b * d + b];
        }
    }
    free(pars); free(prop); free(S); free(A); free(Bm);
  } else {
    rc = -2;
  }
  if (n_grad_evals) *n_grad_evals = nev;
  return rc;
}


/* ------------------------------------------------------------------------------------------ */
/* population runners                                                                          */
/* ------------------------------------------------------------------------------------------ */

static double sample_var(const double* x, int64_t n);

/* reset(t, pars) followed by one consume(t.task): the sampler's reset hook re-evaluates the log-target
 * (and gradient) at pars (RWM.jl:49, MALA.jl:75-78, HMC.jl:114-116), then one loop body runs.
 * In: pars.  Out: ppars (post-decision state), *plt (its log-target), *lt0 (log-target at pars before the step). */
static void reset_and_step(const orc_model* m, const orc_sampler* s, const double* pars, const double* z, double u,
                           double* ppars, double* plt, double* lt0) {
  int64_t d = m->d;
  double* prop = (double*)malloc(sizeof(double) * (size_t)d);
  double* grad = (double*)malloc(sizeof(double) * (size_t)d);
  double* pg = (double*)malloc(sizeof(double) * (size_t)d);
  double* mom = (double*)malloc(sizeof(double) * (size_t)d);
  int acc = 0;
  double lt, l2 = NAN;
  if (s->kind == ORC_RWM) {
    lt = orc_eval(m, pars);
    for (int64_t j = 0; j < d; j++) prop[j] = pars[j] + z[j] * (1.0 * s->scale);   /* model.scale = ones (RWM.jl:52,59) */
    l2 = orc_eval(m, prop);
    double ratio = l2 - lt;
    acc = ratio > 0 || ratio > log(u);                                             /* RWM.jl:63 */
  } else if (s->kind == ORC_MALA) {
    double h = s->scale, sq = sqrt(h), lc = log(TWO_PI * h) / 2.0, qno = 0.0, qon = 0.0;
    lt = orc_evalallg(m, pars, grad);
    for (int64_t j = 0; j < d; j++) { mom[j] = pars[j] + (h / 2.0) * grad[j]; prop[j] = mom[j] + sq * z[j]; }  /* MALA.jl:98-100 */
    l2 = orc_evalallg(m, prop, pg);
    for (int64_t j = 0; j < d; j++) { double t = mom[j] - prop[j]; qno += -(t * t) / (2.0 * h) - lc; }
    for (int64_t j = 0; j < d; j++) { double m2 = prop[j] + (h / 2.0) * pg[j]; double t = m2 - pars[j]; qon += -(t * t) / (2.0 * h) - lc; }
    double ratio = l2 + qon - lt - qno;
    acc = ratio > 0 || ratio > log(u);                                             /* MALA.jl:107-108 */
  } else {  /* HMC, fixed nLeaps (HMC.jl:136-158) */
    double eps = s->scale;
    lt = orc_evalallg(m, pars, grad);
    double H0 = -lt + 0.5 * dotp(z, z, d);
    for (int64_t j = 0; j < d; j++) { mom[j] = z[j]; prop[j] = pars[j]; pg[j] = grad[j]; }
    l2 = lt;
    for (int l = 0; l < s->nleaps; l++) {
      for (int64_t j = 0; j < d; j++) mom[j] += (0.5 * pg[j]) * eps;
      for (int64_t j = 0; j < d; j++) prop[j] += eps * mom[j];
      l2 = orc_evalallg(m, prop, pg);
      for (int64_t j = 0; j < d; j++) mom[j] += (0.5 * pg[j]) * eps;
    }
    double H = -l2 + 0.5 * dotp(mom, mom, d);
    acc = u < exp(H0 - H);
  }
  if (acc) { memcpy(ppars, prop, sizeof(double) * (size_t)d); *plt = l2; }
  else { memcpy(ppars, pars, sizeof(double) * (size_t)d); *plt = lt; }
  *lt0 = lt;
  free(prop); free(grad); free(pg); free(mom);
}

int32_t orc_run_seqmc(const orc_model* models, const orc_sampler* samplers, int32_t nt, int64_t steps, int64_t burnin,
                      double trigger, int64_t npart, const double* particles, const double* normals,
                      const double* uniforms, const double* res_uniforms, double* samples, double* weights,
                      int64_t* n_resamples) {
  /* SeqMC.jl:39-122 */
  if (burnin < 0 || steps <= burnin || nt < 1 || npart < 2) return -2;        /* :29-30 */
  int64_t d = models[0].d;
  for (int t = 0; t < nt; t++) if (models[t].d != d) return -2;               /* :47 */
  double* pars = (double*)malloc(sizeof(double) * (size_t)(d * npart));
  double* tmp = (double*)malloc(sizeof(double) * (size_t)(d * npart));
  double* logW = (double*)calloc((size_t)npart, sizeof(double));
  double* logtarget = (double*)calloc((size_t)npart, sizeof(double));
  double* W = (double*)malloc(sizeof(double) * (size_t)npart);
  double* cp = (double*)malloc(sizeof(double) * (size_t)npart);
  double* lt2 = (double*)malloc(sizeof(double) * (size_t)npart);
  int64_t* rs = (int64_t*)malloc(sizeof(int64_t) * (size_t)npart);
  double* pp = (double*)malloc(sizeof(double) * (size_t)d);
  memcpy(pars, particles, sizeof(double) * (size_t)(d * npart));               /* :58 */
  int64_t nres = 0;
  for (int64_t i = 1; i <= steps; i++) {
    for (int t = 0; t < nt; t++) {
      for (int64_t n = 0; n < npart; n++) {                                    /* :66-72 mutate each particle with task t */
        int64_t k = ((i - 1) * nt + t) * npart + n;
        double plt, ll0;
        reset_and_step(&models[t], &samplers[t], pars + n * d, normals + k * d, uniforms[k], pp, &plt, &ll0);
        memcpy(pars + n * d, pp, sizeof(double) * (size_t)d);
        logW[n] += ll0 - logtarget[n];
        logtarget[n] = plt;
      }
      for (int64_t n = 0; n < npart; n++) W[n] = exp(logW[n]);                 /* :76 */
      if (sample_var(W, npart) < trigger) {                                    /* :77 */
        double c = 0.0, tot = 0.0;
        for (int64_t n = 0; n < npart; n++) tot += W[n];
        for (int64_t n = 0; n < npart; n++) { c += W[n]; cp[n] = c / tot; }     /* :78 cumsum(W) / sum(W) */
        for (int64_t n = 0; n < npart; n++) {                                  /* :80-83 */
          double l = res_uniforms[((i - 1) * nt + t) * npart + n];
          int64_t f = npart - 1;
          for (int64_t q = 0; q < npart; q++) if (cp[q] >= l) { f = q; break; }
          rs[n] = f;
        }
        for (int64_t n = 0; n < npart; n++) { memcpy(tmp + n * d, pars + rs[n] * d, sizeof(double) * (size_t)d); lt2[n] = logtarget[rs[n]]; }
        memcpy(pars, tmp, sizeof(double) * (size_t)(d * npart));               /* :84 */
        memcpy(logtarget, lt2, sizeof(double) * (size_t)npart);                /* :86 */
        for (int64_t n = 0; n < npart; n++) logW[n] = 0.0;                     /* :85 */
        nres++;
      }
    }
    for (int64_t n = 0; n < npart; n++) logtarget[n] = 0.0;                    /* :92 */
    if (i > burnin) {                                                          /* :94-100 */
      int64_t pos = (i - burnin - 1) * npart;
      for (int64_t n = 0; n < npart; n++) {
        memcpy(samples + (pos + n) * d, pars + n * d, sizeof(double) * (size_t)d);
        weights[pos + n] = exp(logW[n]);
      }
    }
  }
  if (n_resamples) *n_resamples = nres;
  free(pars); free(tmp); free(logW); free(logtarget); free(W); free(cp); free(lt2); free(rs); free(pp);
  return 0;
}

int32_t orc_run_serialtemp(const orc_model* models, const orc_sampler* samplers, int32_t nt, int64_t steps, int64_t burnin,
                           int64_t swap_period, const double* inits, const double* normals, const double* uniforms,
                           const double* u_pick, const double* u_swap, double* samples, int32_t* at_out) {
  /* SerialTempMC.jl:31-85.  Only the active task's sampler state matters: any other task is reset (:62) before it is
   * consumed.  s = (ppars, logtarget, pars) is the last accepted-as-current MCMCSample (:53,71). */
  if (burnin < 0 || steps <= burnin || nt < 2 || swap_period < 1) return -2;   /* :22-23 */
  int64_t d = models[0].d;
  for (int t = 0; t < nt; t++) {
    if (models[t].d != d) return -2;                                           /* :39 */
    if (!isfinite(orc_eval(&models[t], inits + t * d))) return -1;             /* every task is started (:44) */
  }
  double* state = (double*)malloc(sizeof(double) * (size_t)d);  /* internal pars of the active task (post-decision) */
  double* ppars = (double*)malloc(sizeof(double) * (size_t)d);  /* s.ppars */
  double* pars = (double*)malloc(sizeof(double) * (size_t)d);   /* s.pars: the state BEFORE the step that produced s */
  double* pp2 = (double*)malloc(sizeof(double) * (size_t)d);
  int at = 0;
  double plt, lt0, logtarget;
  /* :44 map(t -> consume(t.task), tasks): first step of every task from its model.init; only task 1's persists */
  reset_and_step(&models[0], &samplers[0], inits, normals + 0 * d, uniforms[0], state, &plt, &lt0);
  /* :51 s = consume(tasks[at].task): task 1's second step, from its own state (draw column 1) */
  memcpy(pars, state, sizeof(double) * (size_t)d);
  reset_and_step(&models[0], &samplers[0], pars, normals + 1 * d, uniforms[1], ppars, &plt, &lt0);
  memcpy(state, ppars, sizeof(double) * (size_t)d);
  logtarget = lt0;                                                             /* s.logtarget (:53) */
  for (int64_t i = 1; i <= steps; i++) {
    const double* z = normals + (i + 1) * d;
    const double u = uniforms[i + 1];
    if (i % swap_period == 0) {                                                /* :57 attempt a task switch */
      int at2 = (int)floor(u_pick[i] * (double)(nt - 1));                      /* :59 rand(1:(nmods-1)), 0-based here */
      if (at2 > nt - 2) at2 = nt - 2;
      if (at2 >= at) at2 += 1;                                                 /* :60 */
      double plt2, lt02;
      reset_and_step(&models[at2], &samplers[at2], pars, z, u, pp2, &plt2, &lt02);   /* :62-63 reset to s.pars, consume */
      if (u_swap[i] < exp(logtarget - lt02 + 0.0 - 0.0)) {                     /* :64; logW stays 0 (:48,:70) */
        at = at2;                                                              /* :65 at, s = at2, s2 */
        memcpy(ppars, pp2, sizeof(double) * (size_t)d);
        memcpy(state, pp2, sizeof(double) * (size_t)d);
        logtarget = lt02;                                                      /* s2.pars == pars already */
      }
    } else {                                                                   /* :68 */
      memcpy(pars, state, sizeof(double) * (size_t)d);
      reset_and_step(&models[at], &samplers[at], pars, z, u, ppars, &plt, &lt0);
      memcpy(state, ppars, sizeof(double) * (size_t)d);
      logtarget = lt0;
    }
    if (i > burnin) {                                                          /* :73-76 */
      memcpy(samples + (i - burnin - 1) * d, ppars, sizeof(double) * (size_t)d);
      if (at_out) at_out[i - burnin - 1] = at;
    }
  }
  free(state); free(ppars); free(pars); free(pp2);
  return 0;
}

/* ------------------------------------------------------------------------------------------ */
/* stats                                                                                       */
/* ------------------------------------------------------------------------------------------ */
double orc_mean(const double* x, int64_t n) { /* mean.jl:6 */
  double s = 0.0;
  for (int64_t i = 0; i < n; i++) s += x[i];
  return s / (double)n;
}
static double sample_var(const double* x, int64_t n) { /* Base.var: two-pass, n-1 */
  double mu = orc_mean(x, n), s = 0.0;
  for (int64_t i = 0; i < n; i++) { double t = x[i] - mu; s += t * t; }
  return s / (double)(n - 1);
}
double orc_mcvar_iid(const double* x, int64_t n) { return sample_var(x, n) / (double)n; } /* var.jl:7-8 */

double orc_mcvar_bm(const double* x, int64_t n, int64_t batchlen) { /* var.jl:20-26 */
  int64_t nb = n / batchlen;
  if (nb <= 1) return NAN;
  int64_t nbs = nb * batchlen;
  double* bm = (double*)malloc(sizeof(double) * (size_t)nb);
  for (int64_t j = 0; j < nb; j++) bm[j] = orc_mean(x + j * batchlen, batchlen);
  double v = (double)batchlen * sample_var(bm, nb) / (double)nbs;
  free(bm);
  return v;
}

/* StatsBase.acf(x, 0:maxlag, correlation=false): demeaned autocovariance divided by n
 * (unpinned dependency; Geyer 1992 convention -- SURVEY.md 8c). */
void orc_acov(const double* x, int64_t n, int64_t maxlag, double* acv) {
  double mu = orc_mean(x, n);
  for (int64_t k = 0; k <= maxlag; k++) {
    double s = 0.0;
    for (int64_t t = 0; t + k < n; t++) s += (x[t] - mu) * (x[t + k] - mu);
    acv[k] = s / (double)n;
  }
}

static double geyer(const double* x, int64_t n, int64_t maxlag, int monotone) {
  /* var.jl:45-75 (imse) / :95-116 (ipse) */
  int64_t k = (int64_t)floor(((double)maxlag - 1.0) / 2.0);
  int64_t mm = k + 1;
  if (k < 0) return NAN;
  double* g = (double*)malloc(sizeof(double) * (size_t)(k + 1));
  double* acv = (double*)malloc(sizeof(double) * (size_t)(maxlag + 1));
  orc_acov(x, n, maxlag, acv);
  for (int64_t j = 0; j <= k; j++) {
    g[j] = acv[2 * j] + acv[2 * j + 1];
    if (g[j] <= 0) { mm = j; break; }
  }
  if (monotone && mm > 1)
    for (int64_t j = 1; j < mm; j++) if (g[j] > g[j - 1]) g[j] = g[j - 1];
  double s = 0.0;
  for (int64_t j = 0; j < mm; j++) s += g[j];
  double v = (-acv[0] + 2.0 * s) / (double)n;
  free(g); free(acv);
  return v;
}
double orc_mcvar_imse(const double* x, int64_t n, int64_t maxlag) { return geyer(x, n, maxlag, 1); }
double orc_mcvar_ipse(const double* x, int64_t n, int64_t maxlag) { return geyer(x, n, maxlag, 0); }


/* ------------------------------------------------------------------------------------------ */
/* zero-variance control variates (src/stats/zv.jl)                                            */
/* ------------------------------------------------------------------------------------------ */
static double zv_feature(int64_t p, int64_t d, const double* x, const double* g) {
  /* zv.jl:16,48-56: z = -grad/2; zQuadratic = [z, 2*z.*x - 1, x_i*z_j + x_j*z_i (i<j)] */
  if (p < d) return (-g[p]) / 2.0;
  if (p < 2 * d) { int64_t j = p - d; return (2.0 * ((-g[j]) / 2.0)) * x[j] - 1.0; }
  int64_t l = p - 2 * d, i = 0;
  while (l >= d - 1 - i) { l -= d - 1 - i; i++; }
  int64_t j = i + 1 + l;
  return x[i] * ((-g[j]) / 2.0) + x[j] * ((-g[i]) / 2.0);
}

int32_t orc_zv(const double* x, const double* grad, int64_t S, int64_t d, int32_t order, double* zv, double* a) {
  if (S < 2 || d < 1 || (order != 1 && order != 2)) return -2;
  const int64_t k = (order == 1) ? d : d * (d + 3) / 2, w = k + d;
  double* mean = (double*)calloc((size_t)w, sizeof(double));
  double* M = (double*)calloc((size_t)(k * w), sizeof(double));
  /* column means of [features x] */
  for (int64_t p = 0; p < w; p++) {
    double s = 0.0;
    for (int64_t t = 0; t < S; t++) s += (p < k) ? zv_feature(p, d, x + t * d, grad + t * d) : x[t * d + (p - k)];
    mean[p] = s / (double)S;
  }
  /* cov([features x_i]) (zv.jl:19,58): rows = features, columns = features then the d parameters */
  for (int64_t p = 0; p < k; p++)
    for (int64_t q = 0; q < w; q++) {
      double s = 0.0;
      for (int64_t t = 0; t < S; t++) {
        double fp = zv_feature(p, d, x + t * d, grad + t * d) - mean[p];
        double fq = ((q < k) ? zv_feature(q, d, x + t * d, grad + t * d) : x[t * d + (q - k)]) - mean[q];
        s += fp * fq;
      }
      M[p * w + q] = s / (double)(S - 1);
    }
  /* Gauss-Jordan with partial pivoting on [C | Sigma] -> [I | inv(C) Sigma] (zv.jl:20-22,59-61) */
  int32_t rc = 0;
  for (int64_t c = 0; c < k && rc == 0; c++) {
    int64_t piv = c; double best = fabs(M[c * w + c]);
    for (int64_t r = c + 1; r < k; r++) if (fabs(M[r * w + c]) > best) { best = fabs(M[r * w + c]); piv = r; }
    if (!(best > 0.0)) { rc = -3; break; }
    if (piv != c) for (int64_t q = 0; q < w; q++) { double tmp = M[c * w + q]; M[c * w + q] = M[piv * w + q]; M[piv * w + q] = tmp; }
    double pv = M[c * w + c];
    for (int64_t q = 0; q < w; q++) M[c * w + q] = M[c * w + q] / pv;
    for (int64_t r = 0; r < k; r++) {
      if (r == c) continue;
      double f = M[r * w + c];
      for (int64_t q = 0; q < w; q++) M[r * w + q] = M[r * w + q] - f * M[c * w + q];
    }
  }
  if (rc == 0) {
    for (int64_t p = 0; p < k; p++) for (int64_t i = 0; i < d; i++) a[p * d + i] = -M[p * w + k + i];   /* a = -precision*sigma */
    if (zv)                                                                                              /* zv.jl:25,63 */
      for (int64_t t = 0; t < S; t++)
        for (int64_t i = 0; i < d; i++) {
          double s = 0.0;
          for (int64_t p = 0; p < k; p++) s += zv_feature(p, d, x + t * d, grad + t * d) * a[p * d + i];
          zv[t * d + i] = x[t * d + i] + s;
        }
  }
  free(mean); free(M);
  return rc;
}

/* ------------------------------------------------------------------------------------------ */
/* Philox4x32-10 (Salmon, Moraes, Dror, Shaw: "Parallel random numbers: as easy as 1, 2, 3")    */
/* ------------------------------------------------------------------------------------------ */
void orc_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
  uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3], k0 = key[0], k1 = key[1];
  for (int r = 0; r < 10; r++) {
    uint64_t p0 = (uint64_t)M0 * c0, p1 = (uint64_t)M1 * c2;
    uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0, hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
    uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += W0; k1 += W1;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
/* uniform from 53 random bits: (b + 0.5) * 2^-53 in (0, 1]; b + 0.5 rounds to even for b >= 2^52, so 1.0 occurs with probability 2^-54 (the engine does the same) */
static double u01(uint32_t hi, uint32_t lo) {
  uint64_t b = (((uint64_t)hi << 21) ^ ((uint64_t)lo >> 11)) & ((1ull << 53) - 1);
  return ((double)b + 0.5) * (1.0 / 9007199254740992.0);
}
void orc_draw_normals(uint64_t seed, uint64_t chain, uint32_t step, int64_t d, double* z) {
  uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
  for (int64_t b = 0; 2 * b < d; b++) {
    uint32_t ctr[4] = {(uint32_t)chain, (uint32_t)(chain >> 32), step, (uint32_t)b}, o[4];
    orc_philox4x32_10(ctr, key, o);
    double u1 = u01(o[0], o[1]), u2 = u01(o[2], o[3]);
    double rr = sqrt(-2.0 * log(u1));
    double th = TWO_PI * u2;
    z[2 * b] = rr * cos(th);
    if (2 * b + 1 < d) z[2 * b + 1] = rr * sin(th);
  }
}
double orc_draw_uniform(uint64_t seed, uint64_t chain, uint32_t step) {
  uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
  uint32_t ctr[4] = {(uint32_t)chain, (uint32_t)(chain >> 32), step, 0xFFFFFFFFu}, o[4];
  orc_philox4x32_10(ctr, key, o);
  return u01(o[0], o[1]);
}
