/*
 * nuts_oracle.c -- CPU restatement (plain C99, FP64, scalar, single thread) of the engine's No-U-Turn sampler: slice NUTS
 * with dual averaging (Hoffman & Gelman 2014, Algorithms 3 and 6), written iteratively in the order DESIGN.md pins.
 *
 * TEST INFRASTRUCTURE ONLY: tests/test_nuts.py compiles it together with oracle/mcmc_oracle.c into a temporary
 * library.  It reuses the oracle's model evaluations and Philox4x32-10, and nothing of the engine.  The U-turn checks are
 * made here against the stored leaves of the subtree (leaf m against leaf m - 2^r + 1), not through the kernel's
 * checkpoint slots, so the slot bookkeeping is checked rather than restated.
 *
 * Step i of a chain draws: the momentum from the normal blocks (or `normals`, d x (last+1), when given: the engine's
 * own Box-Muller values differ from orc_draw_normals in the last bits), the slice uniform u0 from block 0xFFFFFFFF, the
 * direction of doubling j from block 0x80000000 + 2j, its merge from 0x80000000 + 2j + 1 and the candidate choice of
 * the step's leaf k (0-based) from 0x40000000 + k.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include "../oracle/mcmc_oracle.h"

double orc_nuts_slot_uniform(uint64_t seed, uint64_t chain, uint32_t step, uint32_t block) {
  uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
  uint32_t ctr[4] = {(uint32_t)chain, (uint32_t)(chain >> 32), step, block}, o[4];
  orc_philox4x32_10(ctr, key, o);
  uint64_t b = (((uint64_t)o[0] << 21) ^ ((uint64_t)o[1] >> 11)) & ((1ull << 53) - 1);
  return ((double)b + 0.5) * (1.0 / 9007199254740992.0);
}

/* no U-turn between a later point (th_m, p_m) and an earlier one (th_s, p_s) of direction v: both dots >= 0 */
static int no_uturn(const double* th_m, const double* p_m, const double* th_s, const double* p_s, double v, int64_t d) {
  double ds = 0.0, dm = 0.0;
  for (int64_t j = 0; j < d; j++) {
    const double delta = v * (th_m[j] - th_s[j]);
    ds += delta * p_s[j];
    dm += delta * p_m[j];
  }
  return ds >= 0.0 && dm >= 0.0;
}

static double dotp(const double* a, const double* b, int64_t d) {
  double s = 0.0;
  for (int64_t j = 0; j < d; j++) s += a[j] * b[j];
  return s;
}

#define CPY(dst, src) memcpy((dst), (src), sizeof(double) * (size_t)d)

/* s->nleaps = maxdoublings; s->rate, shrinkage, t0, step = dual averaging; s->force_eps, start_step, da_state as for
 * orc_run_chain's HMCDA.  Outputs (any may be NULL) per kept step: samples / grads d x S, accept, logtarget, the step
 * size (the oracle's own, also under force_eps), leapfrog count, alpha / n_alpha of the last doubling and the doubling
 * count.  returns 0, -1 "Initial values out of model support", -2 bad arguments. */
int32_t orc_run_nuts(const orc_model* m, const orc_sampler* s, const orc_range* r, const double* init, uint64_t seed,
                     uint64_t chain, const double* normals, double* samples, double* grads, uint8_t* accept,
                     double* logtarget, double* diag_eps, int64_t* diag_leaps, double* diag_alpha,
                     int64_t* diag_ndoublings, int64_t* n_grad_evals) {
  const int64_t d = m->d, burnin = r->first - 1, len = r->last;
  const int maxd = s->nleaps;
  if (burnin < 0 || len <= burnin || r->step < 1 || maxd < 1 || maxd > 10) return -2;
  const int64_t nleaf = (int64_t)1 << (maxd - 1);
  double* buf = (double*)calloc((size_t)(d * (14 + 2 * nleaf)), sizeof(double));
  double *pars = buf, *grad = buf + d, *z = buf + 2 * d;
  double *thm = buf + 3 * d, *pm = buf + 4 * d, *gm = buf + 5 * d, *thp = buf + 6 * d, *pp = buf + 7 * d, *gp = buf + 8 * d;
  double *th = buf + 9 * d, *p = buf + 10 * d, *g = buf + 11 * d, *sth = buf + 12 * d, *sg = buf + 13 * d;
  double *Lth = buf + 14 * d, *Lp = Lth + nleaf * d;
  int64_t nev = 0, kept = 0;
  int32_t rc = 0;
  CPY(pars, init);
  double lt = orc_evalallg(m, pars, grad); nev++;
  if (!isfinite(lt)) rc = -1;
  double leapStep = 1.0, dualLeapStep = 1.0, dualH = 0.0;
  const double mu = log(10.0 * 1.0);
  if (s->da_state) { leapStep = s->da_state[0]; dualLeapStep = s->da_state[1]; dualH = s->da_state[2]; }
  for (int64_t i = s->start_step + 1; rc == 0 && i <= len; i++) {
    const double own_eps = leapStep;
    const double eps = s->force_eps ? s->force_eps[i] : leapStep;
    if (normals) CPY(z, normals + i * d); else orc_draw_normals(seed, chain, (uint32_t)i, d, z);
    const double H0 = -lt + 0.5 * dotp(z, z, d);
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
        for (int64_t q = 0; q < d; q++) th[q] += e * p[q];              /* HMC.jl:96 */
        const double llt = orc_evalallg(m, th, g); nev++;
        for (int64_t q = 0; q < d; q++) p[q] += (0.5 * g[q]) * e;       /* HMC.jl:98 */
        const double H = -llt + 0.5 * dotp(p, p, d);
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
          if (!no_uturn(Lth + (leaf - 1) * d, Lp + (leaf - 1) * d, Lth + (first - 1) * d, Lp + (first - 1) * d, v, d)) { ok = 0; break; }
        }
        if (!ok) break;
      }
      if (!ok) break;
      if (orc_nuts_slot_uniform(seed, chain, (uint32_t)i, 0x80000000u + 2u * (uint32_t)j + 1u) * (double)n < (double)nsub) {
        CPY(pars, sth); CPY(grad, sg); lt = slt; moved = 1;
      }
      n += nsub;
      if (!no_uturn(thp, pp, thm, pm, 1.0, d)) break;
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
      const double fi = (double)i;
      double eta = 1.0 / (fi + s->t0);
      dualH = (1.0 - eta) * dualH + eta * (s->rate - pacc);
      leapStep = exp(mu - sqrt(fi) * dualH / s->shrinkage);
      eta = pow(fi, -s->step);
      dualLeapStep = exp((1.0 - eta) * log(dualLeapStep) + eta * log(leapStep));
    } else {
      leapStep = dualLeapStep;                                          /* HMCDA.jl:140 */
    }
  }
  if (n_grad_evals) *n_grad_evals = nev;
  free(buf);
  return rc;
}
