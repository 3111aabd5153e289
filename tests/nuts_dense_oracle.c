/*
 * nuts_dense_oracle.c -- CPU restatement (plain C99, FP64, scalar, single thread) of the engine's No-U-Turn sampler with
 * a dense inverse metric A = M^-1 (Stan's dense_e), fixed or adapted in Stan's warm-up windows from a Welford covariance
 * (covar_adaptation.hpp, welford_covar_estimator.hpp and the step-size restart of adapt_dense_e_nuts.hpp), restated from
 * Stan's rules in the order DESIGN.md pins.
 *
 * TEST INFRASTRUCTURE ONLY: tests/test_nuts_dense.py compiles it together with tests/nuts_oracle.c (whose Philox slot
 * uniforms it uses), tests/nuts_metric_oracle.c (whose window schedule it uses) and oracle/mcmc_oracle.c into a temporary
 * library.  It is written apart from orc_run_nuts and orc_run_nuts_metric, so that A = diag(minv) reproducing
 * orc_run_nuts_metric and A = I reproducing orc_run_nuts bit for bit check the dense arithmetic against independent
 * restatements.  Matrices are row-major here: element (j, k) at j*d + k.  U-turn checks are made against the stored
 * leaves of the subtree, with their stored v = A p.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include "../oracle/mcmc_oracle.h"

/* tests/nuts_oracle.c, tests/nuts_metric_oracle.c */
double orc_nuts_slot_uniform(uint64_t seed, uint64_t chain, uint32_t step, uint32_t block);
int32_t orc_nuts_windows(int64_t W, int64_t init, int64_t term, int64_t window, int64_t* ends, int64_t* lo, int64_t* hi);

/* lower Cholesky factor l of the matrix whose lower triangle a holds; 0, or -1 when a pivot is not finite and > 0 */
int32_t orc_dense_cholesky(const double* a, double* l, int64_t d) {
  for (int64_t j = 0; j < d; j++) {
    double s = a[j * d + j];
    for (int64_t k = 0; k < j; k++) s -= l[j * d + k] * l[j * d + k];
    if (!(s > 0.0 && isfinite(s))) return -1;
    l[j * d + j] = sqrt(s);
    for (int64_t i = j + 1; i < d; i++) {
      double t = a[i * d + j];
      for (int64_t k = 0; k < j; k++) t -= l[i * d + k] * l[j * d + k];
      l[i * d + j] = t / l[j * d + j];
    }
  }
  return 0;
}

/* p = L^-T z (Stan's llt().matrixU().solve(z)): back substitution from j = d - 1 */
void orc_dense_backsub(const double* l, const double* z, double* p, int64_t d) {
  for (int64_t j = d - 1; j >= 0; j--) {
    double s = z[j];
    for (int64_t k = j + 1; k < d; k++) s -= l[k * d + j] * p[k];
    p[j] = s / l[j * d + j];
  }
}

/* Welford sums over n samples x (n x d) from zero: mean (d) and the unsymmetrised cross products m2 (d x d) */
void orc_welford_covar(const double* x, int64_t n, int64_t d, double* mean, double* m2) {
  double* delta = (double*)malloc(sizeof(double) * (size_t)d);
  memset(mean, 0, sizeof(double) * (size_t)d);
  memset(m2, 0, sizeof(double) * (size_t)(d * d));
  for (int64_t t = 0; t < n; t++) {
    const double* xt = x + t * d;
    for (int64_t j = 0; j < d; j++) { delta[j] = xt[j] - mean[j]; mean[j] += delta[j] / (double)(t + 1); }
    for (int64_t a = 0; a < d; a++)
      for (int64_t b = 0; b < d; b++) m2[a * d + b] += (xt[a] - mean[a]) * delta[b];
  }
  free(delta);
}

/* v = A x, each v_j summed from 0.0 with k ascending */
static void matvec(const double* a, const double* x, double* v, int64_t d) {
  for (int64_t j = 0; j < d; j++) {
    double s = 0.0;
    for (int64_t k = 0; k < d; k++) s += a[j * d + k] * x[k];
    v[j] = s;
  }
}

static double dot(const double* x, const double* y, int64_t d) {
  double s = 0.0;
  for (int64_t j = 0; j < d; j++) s += x[j] * y[j];
  return s;
}

/* no U-turn between a later point (th_m, v_m) and an earlier one (th_s, v_s) of direction dir: both dots >= 0 */
static int no_uturn(const double* th_m, const double* v_m, const double* th_s, const double* v_s, double dir, int64_t d) {
  double ds = 0.0, dm = 0.0;
  for (int64_t j = 0; j < d; j++) {
    const double delta = dir * (th_m[j] - th_s[j]);
    ds += delta * v_s[j];
    dm += delta * v_m[j];
  }
  return ds >= 0.0 && dm >= 0.0;
}

#define CPY(dst, src, n) memcpy((dst), (src), sizeof(double) * (size_t)(n))

/* s->nleaps = maxdoublings; s->rate, shrinkage, t0, step = dual averaging; s->force_eps, start_step, da_state as for
 * orc_run_chain's HMCDA.  inv_metric (d x d) the starting dense inverse metric, NULL = the identity.  adapt (3:
 * init_buffer, term_buffer, window) or NULL: adapt it in Stan's windows over the W = first - 2 warm-up steps.  force_A
 * ((last+1) x d x d) or NULL: the trajectory of step i uses matrix i and its factor (teacher forcing) while the oracle's own
 * metric goes on adapting.  Outputs (any may be NULL) per kept step: samples / grads d x S, accept, logtarget, the step size
 * (the oracle's own, also under force_eps), leapfrog count, alpha / n_alpha of the last doubling, doubling count; win_A
 * (64 x d x d) the metric after each window end and n_win their number; final_A (d x d) the metric at the end.  Returns 0,
 * -1 "Initial values out of model support", -2 bad arguments, -3 a starting or forced metric that is not positive
 * definite. */
int32_t orc_run_nuts_dense(const orc_model* m, const orc_sampler* s, const orc_range* r, const double* init, uint64_t seed,
                           uint64_t chain, const double* normals, const double* inv_metric, const int64_t* adapt,
                           const double* force_A, double* samples, double* grads, uint8_t* accept, double* logtarget,
                           double* diag_eps, int64_t* diag_leaps, double* diag_alpha, int64_t* diag_ndoublings,
                           int64_t* n_grad_evals, double* win_A, int64_t* n_win, double* final_A) {
  const int64_t d = m->d, dd = d * d, burnin = r->first - 1, len = r->last;
  const int maxd = s->nleaps;
  if (burnin < 0 || len <= burnin || r->step < 1 || maxd < 1 || maxd > 10) return -2;
  if (adapt && (adapt[0] < 0 || adapt[1] < 0 || adapt[2] < 1)) return -2;
  const int64_t nleaf = (int64_t)1 << (maxd - 1);
  double* mats = (double*)calloc((size_t)(5 * dd), sizeof(double));
  double *ownA = mats, *ownL = mats + dd, *fL = mats + 2 * dd, *wm2 = mats + 3 * dd, *cand = mats + 4 * dd;
  double* buf = (double*)calloc((size_t)(d * (20 + 3 * nleaf)), sizeof(double));
  double *pars = buf, *grad = buf + d, *z = buf + 2 * d, *tmp = buf + 3 * d;
  double *thm = buf + 4 * d, *pm = buf + 5 * d, *gm = buf + 6 * d, *vm = buf + 7 * d;
  double *thp = buf + 8 * d, *pp = buf + 9 * d, *gp = buf + 10 * d, *vp = buf + 11 * d;
  double *th = buf + 12 * d, *p = buf + 13 * d, *g = buf + 14 * d, *v = buf + 15 * d;
  double *sth = buf + 16 * d, *sg = buf + 17 * d, *wmean = buf + 18 * d, *delta = buf + 19 * d;
  double *Lth = buf + 20 * d, *Lv = Lth + nleaf * d;
  int64_t nev = 0, kept = 0, wn = 0, nw = 0, ends[64], lo = 1, hi = 0;
  int32_t rc = 0, nends = 0;
  if (inv_metric) CPY(ownA, inv_metric, dd);
  else for (int64_t j = 0; j < d; j++) ownA[j * d + j] = 1.0;
  if (orc_dense_cholesky(ownA, ownL, d)) rc = -3;
  if (adapt) nends = orc_nuts_windows(r->first - 2, adapt[0], adapt[1], adapt[2], ends, &lo, &hi);
  CPY(pars, init, d);
  double lt = orc_evalallg(m, pars, grad); nev++;
  if (rc == 0 && !isfinite(lt)) rc = -1;
  double leapStep = 1.0, dualLeapStep = 1.0, dualH = 0.0;
  double mu = log(10.0 * 1.0);
  int64_t i0 = 0;
  if (s->da_state) { leapStep = s->da_state[0]; dualLeapStep = s->da_state[1]; dualH = s->da_state[2]; }
  for (int64_t i = s->start_step + 1; rc == 0 && i <= len; i++) {
    const double own_eps = leapStep;
    const double eps = s->force_eps ? s->force_eps[i] : leapStep;
    const double *A = ownA, *L = ownL;
    if (force_A) {
      A = force_A + i * dd;
      if (orc_dense_cholesky(A, fL, d)) { rc = -3; break; }
      L = fL;
    }
    if (normals) CPY(z, normals + i * d, d); else orc_draw_normals(seed, chain, (uint32_t)i, d, z);
    orc_dense_backsub(L, z, pp, d);                                     /* p = L^-T z */
    matvec(A, pp, vp, d);
    const double H0 = -lt + 0.5 * dot(vp, pp, d);
    const double lu0 = log(orc_draw_uniform(seed, chain, (uint32_t)i));
    CPY(thm, pars, d); CPY(thp, pars, d); CPY(pm, pp, d); CPY(vm, vp, d); CPY(gm, grad, d); CPY(gp, grad, d);
    int64_t n = 1, leaps = 0, ndbl = 0, nalpha = 0;
    int moved = 0;
    double alpha = 0.0, slt = 0.0;
    for (int j = 0; j < maxd; j++) {
      ndbl = j + 1;
      const double dir = orc_nuts_slot_uniform(seed, chain, (uint32_t)i, 0x80000000u + 2u * (uint32_t)j) >= 0.5 ? 1.0 : -1.0;
      const double e = dir * eps;
      double *eth = dir > 0 ? thp : thm, *ep = dir > 0 ? pp : pm, *eg = dir > 0 ? gp : gm, *ev = dir > 0 ? vp : vm;
      CPY(th, eth, d); CPY(p, ep, d); CPY(g, eg, d);
      alpha = 0.0; nalpha = 0;
      int64_t nsub = 0;
      int ok = 1;
      for (int64_t leaf = 1; leaf <= ((int64_t)1 << j); leaf++) {
        for (int64_t q = 0; q < d; q++) p[q] += (0.5 * g[q]) * e;       /* HMC.jl:95 */
        matvec(A, p, tmp, d);
        for (int64_t q = 0; q < d; q++) th[q] += e * tmp[q];            /* HMC.jl:96 with v = A p */
        const double llt = orc_evalallg(m, th, g); nev++;
        for (int64_t q = 0; q < d; q++) p[q] += (0.5 * g[q]) * e;       /* HMC.jl:98 */
        matvec(A, p, v, d);
        const double H = -llt + 0.5 * dot(v, p, d);
        const int64_t k = leaps++;
        const double ea = exp(H0 - H);
        alpha += isnan(ea) ? 0.0 : (ea < 1.0 ? ea : 1.0);
        nalpha++;
        CPY(eth, th, d); CPY(ep, p, d); CPY(eg, g, d); CPY(ev, v, d);
        CPY(Lth + (leaf - 1) * d, th, d); CPY(Lv + (leaf - 1) * d, v, d);
        if (lu0 <= H0 - H) {
          nsub++;
          if (nsub == 1 || orc_nuts_slot_uniform(seed, chain, (uint32_t)i, 0x40000000u + (uint32_t)k) * (double)nsub < 1.0) {
            CPY(sth, th, d); CPY(sg, g, d); slt = llt;
          }
        }
        if (!(H - H0 < 1000.0 - lu0)) { ok = 0; break; }
        for (int rr = 1; rr <= j && leaf % ((int64_t)1 << rr) == 0; rr++) {
          const int64_t first = leaf - ((int64_t)1 << rr) + 1;
          if (!no_uturn(Lth + (leaf - 1) * d, Lv + (leaf - 1) * d, Lth + (first - 1) * d, Lv + (first - 1) * d, dir, d)) { ok = 0; break; }
        }
        if (!ok) break;
      }
      if (!ok) break;
      if (orc_nuts_slot_uniform(seed, chain, (uint32_t)i, 0x80000000u + 2u * (uint32_t)j + 1u) * (double)n < (double)nsub) {
        CPY(pars, sth, d); CPY(grad, sg, d); lt = slt; moved = 1;
      }
      n += nsub;
      if (!no_uturn(thp, vp, thm, vm, 1.0, d)) break;
    }
    const double pacc = alpha / (double)nalpha;
    if (i >= r->first && i <= r->last && (i - r->first) % r->step == 0) {   /* SerialMC.jl:49-66 */
      if (samples) CPY(samples + kept * d, pars, d);
      if (grads) CPY(grads + kept * d, grad, d);
      if (accept) accept[kept] = (uint8_t)moved;
      if (logtarget) logtarget[kept] = lt;
      if (diag_eps) diag_eps[kept] = own_eps;
      if (diag_leaps) diag_leaps[kept] = leaps;
      if (diag_alpha) diag_alpha[kept] = pacc;
      if (diag_ndoublings) diag_ndoublings[kept] = ndbl;
      kept++;
    }
    if (i < burnin) {                                                   /* HMCDA.jl:133-138 with pacc = alpha / n_alpha */
      const double fi = (double)(i - i0);
      double eta = 1.0 / (fi + s->t0);
      dualH = (1.0 - eta) * dualH + eta * (s->rate - pacc);
      leapStep = exp(mu - sqrt(fi) * dualH / s->shrinkage);
      eta = pow(fi, -s->step);
      dualLeapStep = exp((1.0 - eta) * log(dualLeapStep) + eta * log(leapStep));
      if (adapt && i >= lo && i <= hi) {                                /* welford_covar_estimator::add_sample */
        wn++;
        for (int64_t j = 0; j < d; j++) { delta[j] = pars[j] - wmean[j]; wmean[j] += delta[j] / (double)wn; }
        for (int64_t a = 0; a < d; a++)
          for (int64_t b = 0; b < d; b++) wm2[a * d + b] += (pars[a] - wmean[a]) * delta[b];
      }
      int end = 0;
      for (int32_t w = 0; w < nends; w++) end |= ends[w] == i;
      if (end) {                                                        /* covar_adaptation::learn_covariance */
        const double nn = (double)wn;
        for (int64_t a = 0; a < d; a++)
          for (int64_t b = 0; b < d; b++) {
            const double cov = wn > 1 ? wm2[a * d + b] / (nn - 1.0) : ownA[a * d + b];
            cand[a * d + b] = (nn / (nn + 5.0)) * cov;
            if (a == b) cand[a * d + b] = cand[a * d + b] + 1e-3 * (5.0 / (nn + 5.0));
          }
        if (orc_dense_cholesky(cand, fL, d) == 0) { CPY(ownA, cand, dd); CPY(ownL, fL, dd); }   /* else: keep A and L */
        memset(wm2, 0, sizeof(double) * (size_t)dd);
        memset(wmean, 0, sizeof(double) * (size_t)d);
        wn = 0;
        if (win_A && nw < 64) CPY(win_A + nw * dd, ownA, dd);
        nw++;
        mu = log(10.0 * leapStep); dualLeapStep = 1.0; dualH = 0.0; i0 = i;   /* stepsize_adaptation restart */
      }
    } else {
      leapStep = dualLeapStep;                                          /* HMCDA.jl:140 */
    }
  }
  if (n_grad_evals) *n_grad_evals = nev;
  if (n_win) *n_win = nw;
  if (final_A) CPY(final_A, ownA, dd);
  free(buf); free(mats);
  return rc;
}
