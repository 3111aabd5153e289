/*
 * nuts_metric_oracle.c -- CPU restatement (plain C99, FP64, scalar, single thread) of the engine's No-U-Turn sampler with
 * a diagonal inverse metric minv = M^-1, fixed or adapted in Stan's warm-up windows (windowed_adaptation.hpp,
 * var_adaptation.hpp, welford_var_estimator.hpp and the step-size restart of adapt_diag_e_nuts.hpp), restated from
 * Stan's rules in the order DESIGN.md pins.
 *
 * TEST INFRASTRUCTURE ONLY: tests/test_nuts_metric.py compiles it together with tests/nuts_oracle.c (the identity-metric
 * restatement, whose Philox slot uniforms it uses) and oracle/mcmc_oracle.c into a temporary library.  It is written
 * apart from orc_run_nuts, so that an all-ones metric reproducing orc_run_nuts bit for bit checks the metric arithmetic
 * against an independent restatement.  Draws, tree and U-turn bookkeeping are those of tests/nuts_oracle.c: the U-turn
 * checks are made against the stored leaves of the subtree.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include "../oracle/mcmc_oracle.h"

/* tests/nuts_oracle.c */
double orc_nuts_slot_uniform(uint64_t seed, uint64_t chain, uint32_t step, uint32_t block);

/* minv_j * x, or x without a metric */
static double mv(const double* minv, int64_t j, double x) { return minv ? minv[j] * x : x; }

/* no U-turn between a later point (th_m, p_m) and an earlier one (th_s, p_s) of direction v: both dots >= 0 */
static int no_uturn(const double* th_m, const double* p_m, const double* th_s, const double* p_s, double v,
                    const double* minv, int64_t d) {
  double ds = 0.0, dm = 0.0;
  for (int64_t j = 0; j < d; j++) {
    const double delta = v * (th_m[j] - th_s[j]);
    ds += delta * mv(minv, j, p_s[j]);
    dm += delta * mv(minv, j, p_m[j]);
  }
  return ds >= 0.0 && dm >= 0.0;
}

/* sum_j (minv_j p_j) p_j */
static double kin(const double* p, const double* minv, int64_t d) {
  double s = 0.0;
  for (int64_t j = 0; j < d; j++) s += mv(minv, j, p[j]) * p[j];
  return s;
}

/* Stan's adaptation windows over W warm-up steps (window counter k = step - 1): writes the window-end STEPS to ends
 * (at most 64) and the steps lo..hi whose samples enter the estimate; returns the number of windows (0 when W < 20). */
int32_t orc_nuts_windows(int64_t W, int64_t init, int64_t term, int64_t window, int64_t* ends, int64_t* lo, int64_t* hi) {
  *lo = 1; *hi = 0;
  if (W < 20) return 0;
  if (init + window + term > W) {
    init = (int64_t)(0.15 * (double)W);
    term = (int64_t)(0.1 * (double)W);
    window = W - (init + term);
  }
  int64_t size = window, next = init + window - 1;
  int32_t n = 0;
  for (int64_t k = 0; k < W && n < 64; k++) {           /* windowed_adaptation::end_adaptation_window */
    if (k != next) continue;
    ends[n++] = k + 1;
    if (next == W - term - 1) break;                     /* compute_next_window */
    size *= 2;
    next = k + size;
    if (next != W - term - 1 && next + 2 * size >= W - term) next = W - term - 1;
  }
  *lo = init + 1; *hi = W - term;
  return n;
}

#define CPY(dst, src) memcpy((dst), (src), sizeof(double) * (size_t)d)

/* s->nleaps = maxdoublings; s->rate, shrinkage, t0, step = dual averaging; s->force_eps, start_step, da_state as for
 * orc_run_chain's HMCDA.  inv_metric (d): the starting diagonal inverse metric, NULL = the identity.  adapt (3:
 * init_buffer, term_buffer, window) or NULL: adapt the metric in Stan's windows over the W = first - 2 warm-up steps
 * (a NULL inv_metric then starts at ones).  force_minv ((last+1) x d) or NULL: the trajectory of step i uses row i as
 * its metric (teacher forcing) while the oracle's own metric goes on adapting.  Outputs (any may be NULL) per kept step:
 * samples / grads d x S, accept, logtarget, the step size (the oracle's own, also under force_eps), leapfrog count,
 * alpha / n_alpha of the last doubling and the doubling count; win_minv (64 x d) the metric after each window end and
 * n_win their number; final_minv (d) the metric at the end.  returns 0, -1 "Initial values out of model support",
 * -2 bad arguments. */
int32_t orc_run_nuts_metric(const orc_model* m, const orc_sampler* s, const orc_range* r, const double* init, uint64_t seed,
                            uint64_t chain, const double* normals, const double* inv_metric, const int64_t* adapt,
                            const double* force_minv, double* samples, double* grads, uint8_t* accept, double* logtarget,
                            double* diag_eps, int64_t* diag_leaps, double* diag_alpha, int64_t* diag_ndoublings,
                            int64_t* n_grad_evals, double* win_minv, int64_t* n_win, double* final_minv) {
  const int64_t d = m->d, burnin = r->first - 1, len = r->last;
  const int maxd = s->nleaps;
  if (burnin < 0 || len <= burnin || r->step < 1 || maxd < 1 || maxd > 10) return -2;
  if (adapt && (adapt[0] < 0 || adapt[1] < 0 || adapt[2] < 1)) return -2;
  const int64_t nleaf = (int64_t)1 << (maxd - 1);
  double* buf = (double*)calloc((size_t)(d * (17 + 2 * nleaf)), sizeof(double));
  double *pars = buf, *grad = buf + d, *z = buf + 2 * d;
  double *thm = buf + 3 * d, *pm = buf + 4 * d, *gm = buf + 5 * d, *thp = buf + 6 * d, *pp = buf + 7 * d, *gp = buf + 8 * d;
  double *th = buf + 9 * d, *p = buf + 10 * d, *g = buf + 11 * d, *sth = buf + 12 * d, *sg = buf + 13 * d;
  double *own = buf + 14 * d, *wmean = buf + 15 * d, *wm2 = buf + 16 * d;
  double *Lth = buf + 17 * d, *Lp = Lth + nleaf * d;
  int64_t nev = 0, kept = 0, wn = 0, nw = 0, ends[64], lo = 1, hi = 0;
  int32_t rc = 0, nends = 0;
  /* the metric of the trajectories: NULL (identity), the oracle's own (own), or the forced row of the step */
  const int metric = inv_metric || adapt;
  if (metric) for (int64_t j = 0; j < d; j++) own[j] = inv_metric ? inv_metric[j] : 1.0;
  if (adapt) nends = orc_nuts_windows(r->first - 2, adapt[0], adapt[1], adapt[2], ends, &lo, &hi);
  CPY(pars, init);
  double lt = orc_evalallg(m, pars, grad); nev++;
  if (!isfinite(lt)) rc = -1;
  double leapStep = 1.0, dualLeapStep = 1.0, dualH = 0.0;
  double mu = log(10.0 * 1.0);
  int64_t i0 = 0;
  if (s->da_state) { leapStep = s->da_state[0]; dualLeapStep = s->da_state[1]; dualH = s->da_state[2]; }
  for (int64_t i = s->start_step + 1; rc == 0 && i <= len; i++) {
    const double own_eps = leapStep;
    const double eps = s->force_eps ? s->force_eps[i] : leapStep;
    const double* minv = force_minv ? force_minv + i * d : (metric ? own : NULL);
    if (normals) CPY(z, normals + i * d); else orc_draw_normals(seed, chain, (uint32_t)i, d, z);
    if (minv) for (int64_t j = 0; j < d; j++) z[j] = z[j] / sqrt(minv[j]);          /* p = z / sqrt(minv) */
    const double H0 = -lt + 0.5 * kin(z, minv, d);
    const double lu0 = log(orc_draw_uniform(seed, chain, (uint32_t)i));
    CPY(thm, pars); CPY(thp, pars); CPY(pm, z); CPY(pp, z); CPY(gm, grad); CPY(gp, grad);
    int64_t n = 1, leaps = 0, ndbl = 0, nalpha = 0;
    int moved = 0;
    double alpha = 0.0, slt = 0.0;
    for (int j = 0; j < maxd; j++) {
      ndbl = j + 1;
      const double v = orc_nuts_slot_uniform(seed, chain, (uint32_t)i, 0x80000000u + 2u * (uint32_t)j) >= 0.5 ? 1.0 : -1.0;
      const double e = v * eps;
      double *eth = v > 0 ? thp : thm, *ep = v > 0 ? pp : pm, *eg = v > 0 ? gp : gm;
      CPY(th, eth); CPY(p, ep); CPY(g, eg);
      alpha = 0.0; nalpha = 0;
      int64_t nsub = 0;
      int ok = 1;
      for (int64_t leaf = 1; leaf <= ((int64_t)1 << j); leaf++) {
        for (int64_t q = 0; q < d; q++) p[q] += (0.5 * g[q]) * e;       /* HMC.jl:95 */
        for (int64_t q = 0; q < d; q++) th[q] += e * mv(minv, q, p[q]);  /* HMC.jl:96 */
        const double llt = orc_evalallg(m, th, g); nev++;
        for (int64_t q = 0; q < d; q++) p[q] += (0.5 * g[q]) * e;       /* HMC.jl:98 */
        const double H = -llt + 0.5 * kin(p, minv, d);
        const int64_t k = leaps++;
        const double ea = exp(H0 - H);
        alpha += isnan(ea) ? 0.0 : (ea < 1.0 ? ea : 1.0);
        nalpha++;
        CPY(eth, th); CPY(ep, p); CPY(eg, g);
        CPY(Lth + (leaf - 1) * d, th); CPY(Lp + (leaf - 1) * d, p);
        if (lu0 <= H0 - H) {
          nsub++;
          if (nsub == 1 || orc_nuts_slot_uniform(seed, chain, (uint32_t)i, 0x40000000u + (uint32_t)k) * (double)nsub < 1.0) {
            CPY(sth, th); CPY(sg, g); slt = llt;
          }
        }
        if (!(H - H0 < 1000.0 - lu0)) { ok = 0; break; }
        for (int rr = 1; rr <= j && leaf % ((int64_t)1 << rr) == 0; rr++) {
          const int64_t first = leaf - ((int64_t)1 << rr) + 1;
          if (!no_uturn(Lth + (leaf - 1) * d, Lp + (leaf - 1) * d, Lth + (first - 1) * d, Lp + (first - 1) * d, v, minv, d)) { ok = 0; break; }
        }
        if (!ok) break;
      }
      if (!ok) break;
      if (orc_nuts_slot_uniform(seed, chain, (uint32_t)i, 0x80000000u + 2u * (uint32_t)j + 1u) * (double)n < (double)nsub) {
        CPY(pars, sth); CPY(grad, sg); lt = slt; moved = 1;
      }
      n += nsub;
      if (!no_uturn(thp, pp, thm, pm, 1.0, minv, d)) break;
    }
    const double pacc = alpha / (double)nalpha;
    if (i >= r->first && i <= r->last && (i - r->first) % r->step == 0) {   /* SerialMC.jl:49-66 */
      if (samples) CPY(samples + kept * d, pars);
      if (grads) CPY(grads + kept * d, grad);
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
      if (adapt && i >= lo && i <= hi) {                                /* welford_var_estimator::add_sample */
        wn++;
        for (int64_t j = 0; j < d; j++) {
          const double delta = pars[j] - wmean[j];
          wmean[j] += delta / (double)wn;
          wm2[j] += delta * (pars[j] - wmean[j]);
        }
      }
      int end = 0;
      for (int32_t w = 0; w < nends; w++) end |= ends[w] == i;
      if (end) {                                                        /* var_adaptation::learn_variance */
        const double n = (double)wn;
        for (int64_t j = 0; j < d; j++) {
          const double var = wn > 1 ? wm2[j] / (n - 1.0) : own[j];
          own[j] = (n / (n + 5.0)) * var + 1e-3 * (5.0 / (n + 5.0));
          wmean[j] = 0.0; wm2[j] = 0.0;
        }
        wn = 0;
        if (win_minv && nw < 64) CPY(win_minv + nw * d, own);
        nw++;
        mu = log(10.0 * leapStep); dualLeapStep = 1.0; dualH = 0.0; i0 = i;   /* stepsize_adaptation restart */
      }
    } else {
      leapStep = dualLeapStep;                                          /* HMCDA.jl:140 */
    }
  }
  if (n_grad_evals) *n_grad_evals = nev;
  if (n_win) *n_win = nw;
  if (final_minv) for (int64_t j = 0; j < d; j++) final_minv[j] = metric ? own[j] : 1.0;
  free(buf);
  return rc;
}
