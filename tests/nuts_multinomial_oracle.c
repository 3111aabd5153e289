/*
 * nuts_multinomial_oracle.c -- CPU restatement (plain C99, FP64, scalar, single thread) of the engine's multinomial NUTS
 * transition (Stan's base_nuts::transition and build_tree, as DESIGN.md pins them) with dual averaging, for the identity,
 * a diagonal or a dense inverse metric.
 *
 * TEST INFRASTRUCTURE ONLY: tests/test_nuts_multinomial.py compiles it together with tests/nuts_oracle.c (whose Philox slot
 * uniforms it uses), tests/nuts_dense_oracle.c (Cholesky factor and back substitution), tests/nuts_metric_oracle.c and
 * oracle/mcmc_oracle.c into a temporary library.  build_tree recurses as Stan's does, so the kernel's record stack (which
 * record holds which open block, and when a leaf closes which internal nodes) is checked here rather than restated.
 *
 * Draws of step i: the momentum from the normal blocks (or `normals`, (last+1) x d), the direction of doubling j from
 * block 0x80000000 + 2j and the tree-level choice of its subtree from 0x80000000 + 2j + 1, the choice at the internal node
 * whose left half ends with the step's leaf k (0-based) from 0x40000000 + k.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include "../oracle/mcmc_oracle.h"

/* tests/nuts_oracle.c, tests/nuts_dense_oracle.c */
double orc_nuts_slot_uniform(uint64_t seed, uint64_t chain, uint32_t step, uint32_t block);
int32_t orc_dense_cholesky(const double* a, double* l, int64_t d);
void orc_dense_backsub(const double* l, const double* z, double* p, int64_t d);

#define CPY(dst, src) memcpy((dst), (src), sizeof(double) * (size_t)x->d)

static double log1p_exp(double a) { return a > 0.0 ? a + log1p(exp(-a)) : log1p(exp(a)); }
/* Stan Math's log_sum_exp(a, b) */
double orc_log_sum_exp(double a, double b) {
  if (a == -INFINITY) return b;
  if (a == INFINITY && b == INFINITY) return INFINITY;
  return a > b ? a + log1p_exp(b - a) : b + log1p_exp(a - b);
}

typedef struct {
  const orc_model* m;
  int64_t d;
  int32_t metric;            /* 0 identity, 1 diagonal (minv), 2 dense (A) */
  const double *minv, *A;
  double H0, e;              /* e: the signed step size of the subtree being built */
  uint64_t seed, chain;
  uint32_t step;
  double *th, *p, *g, lt;    /* the trajectory's current end */
  double *tmp;
  int64_t n_leap, nev;
  double sum_metro;
  int divergent;
} traj;

/* one block of the tree: what build_tree returns to its caller */
typedef struct {
  double *rho, *pb, *sb, *pe, *se, *th, *g;   /* sum of momenta; p and p# of the first- and last-built leaves; proposal */
  double lt, h, lsw;
} block;

static void block_alloc(block* b, int64_t d) {
  double* m = (double*)calloc((size_t)(7 * d), sizeof(double));
  b->rho = m; b->pb = m + d; b->sb = m + 2 * d; b->pe = m + 3 * d; b->se = m + 4 * d; b->th = m + 5 * d; b->g = m + 6 * d;
}
static void block_free(block* b) { free(b->rho); }

/* p# = M^-1 p: p, minv p, or A p with each entry summed k ascending from 0.0 */
static void sharp(const traj* x, const double* p, double* s) {
  for (int64_t j = 0; j < x->d; j++) {
    if (x->metric == 0) s[j] = p[j];
    else if (x->metric == 1) s[j] = x->minv[j] * p[j];
    else {
      double t = 0.0;
      for (int64_t k = 0; k < x->d; k++) t += x->A[j * x->d + k] * p[k];
      s[j] = t;
    }
  }
}

static double dot(const double* a, const double* b, int64_t d) {
  double s = 0.0;
  for (int64_t j = 0; j < d; j++) s += a[j] * b[j];
  return s;
}

/* Stan's compute_criterion: p#- . rho > 0 and p#+ . rho > 0 */
static int crit(const double* sm, const double* sp, const double* rho, int64_t d) { return dot(sm, rho, d) > 0.0 && dot(sp, rho, d) > 0.0; }

/* H at the trajectory's end after one leapfrog of step e from it */
static double leapfrog(traj* x) {
  const int64_t d = x->d;
  for (int64_t q = 0; q < d; q++) x->p[q] += (0.5 * x->g[q]) * x->e;  /* HMC.jl:95 */
  sharp(x, x->p, x->tmp);
  for (int64_t q = 0; q < d; q++) x->th[q] += x->e * x->tmp[q];       /* HMC.jl:96 */
  x->lt = orc_evalallg(x->m, x->th, x->g); x->nev++;
  for (int64_t q = 0; q < d; q++) x->p[q] += (0.5 * x->g[q]) * x->e;  /* HMC.jl:98 */
  sharp(x, x->p, x->tmp);
  return -x->lt + 0.5 * dot(x->tmp, x->p, d);
}

/* Stan's build_tree: a block of 2^depth leaves from the trajectory's end; 0 when it is invalid */
static int build_tree(traj* x, int depth, block* out) {
  const int64_t d = x->d;
  if (depth == 0) {
    double h = leapfrog(x);
    x->n_leap++;
    if (isnan(h)) h = INFINITY;
    if (h - x->H0 > 1000.0) x->divergent = 1;
    x->sum_metro += x->H0 - h > 0.0 ? 1.0 : exp(x->H0 - h);
    out->lsw = x->H0 - h;
    CPY(out->th, x->th); CPY(out->g, x->g); out->lt = x->lt; out->h = h;
    CPY(out->rho, x->p); CPY(out->pb, x->p); CPY(out->pe, x->p);
    sharp(x, x->p, out->sb); CPY(out->se, out->sb);
    return !x->divergent;
  }
  block L, R;
  block_alloc(&L, d); block_alloc(&R, d);
  double* ext = (double*)malloc(sizeof(double) * (size_t)d);
  int ok = build_tree(x, depth - 1, &L);
  const int64_t kL = x->n_leap - 1;                                     /* the step's index of L's last leaf */
  if (ok) ok = build_tree(x, depth - 1, &R);
  if (ok) {
    const double lsw = orc_log_sum_exp(L.lsw, R.lsw);
    const block* prop = &L;
    if (R.lsw > lsw) prop = &R;
    else if (orc_nuts_slot_uniform(x->seed, x->chain, x->step, 0x40000000u + (uint32_t)kL) < exp(R.lsw - lsw)) prop = &R;
    CPY(out->th, prop->th); CPY(out->g, prop->g); out->lt = prop->lt; out->h = prop->h;
    out->lsw = lsw;
    for (int64_t j = 0; j < d; j++) out->rho[j] = L.rho[j] + R.rho[j];
    ok = crit(L.sb, R.se, out->rho, d);
    for (int64_t j = 0; j < d; j++) ext[j] = L.rho[j] + R.pb[j];
    ok = ok && crit(L.sb, R.sb, ext, d);
    for (int64_t j = 0; j < d; j++) ext[j] = R.rho[j] + L.pe[j];
    ok = ok && crit(L.se, R.se, ext, d);
    CPY(out->pb, L.pb); CPY(out->sb, L.sb); CPY(out->pe, R.pe); CPY(out->se, R.se);
  }
  free(ext); block_free(&L); block_free(&R);
  return ok;
}

/* metric = 0 (identity), 1 (diagonal: inv_metric d) or 2 (dense: inv_metric d x d row-major); force_metric ((last+1) x d
 * or (last+1) x d x d) or NULL: step i uses entry i instead.  s->nleaps = maxdoublings; s->rate, shrinkage, t0, step = dual
 * averaging on accept_stat; s->force_eps, start_step, da_state as for orc_run_chain's HMCDA.  Outputs (any may be NULL)
 * per kept step: samples / grads d x S, accept (the sample moved), logtarget, the step size (the oracle's own), leapfrog
 * count, accept_stat, energy, divergent.  Returns 0, -1 "Initial values out of model support", -2 bad arguments, -3 a
 * dense metric that is not positive definite. */
int32_t orc_run_nuts_multinomial(const orc_model* m, const orc_sampler* s, const orc_range* r, const double* init,
                                 uint64_t seed, uint64_t chain, const double* normals, int32_t metric, const double* inv_metric,
                                 const double* force_metric, double* samples, double* grads, uint8_t* accept, double* logtarget,
                                 double* diag_eps, int64_t* diag_leaps, double* accept_stat, double* energy, uint8_t* divergent,
                                 int64_t* n_grad_evals) {
  const int64_t d = m->d, burnin = r->first - 1, len = r->last;
  const int64_t msz = metric == 2 ? d * d : d;
  const int maxd = s->nleaps;
  if (burnin < 0 || len <= burnin || r->step < 1 || maxd < 1 || maxd > 10 || metric < 0 || metric > 2) return -2;
  if (metric && !inv_metric && !force_metric) return -2;
  traj X, *x = &X;
  memset(x, 0, sizeof(X));
  x->m = m; x->d = d; x->metric = metric; x->seed = seed; x->chain = chain;
  double* buf = (double*)calloc((size_t)(d * 20), sizeof(double));
  double *pars = buf, *grad = buf + d, *z = buf + 2 * d, *p0 = buf + 3 * d, *s0 = buf + 4 * d, *ext = buf + 5 * d;
  double *thf = buf + 6 * d, *pf = buf + 7 * d, *gf = buf + 8 * d, *thb = buf + 9 * d, *pb = buf + 10 * d, *gb = buf + 11 * d;
  double *rho = buf + 12 * d, *rho_b = buf + 13 * d, *rho_f = buf + 14 * d;
  double *p_bb = buf + 15 * d, *s_bb = buf + 16 * d, *p_bf = buf + 17 * d, *s_bf = buf + 18 * d, *p_fb = buf + 19 * d;
  double* more = (double*)calloc((size_t)(3 * d + 2 * d * d), sizeof(double));
  double *s_fb = more, *p_ff = more + d, *s_ff = more + 2 * d, *Lf = more + 3 * d, *minv = more + 3 * d + d * d;
  x->tmp = (double*)calloc((size_t)d, sizeof(double));
  block sub;
  block_alloc(&sub, d);
  int64_t kept = 0;
  int32_t rc = 0;
  CPY(pars, init);
  double lt = orc_evalallg(m, pars, grad); x->nev++;
  if (!isfinite(lt)) rc = -1;
  double leapStep = 1.0, dualLeapStep = 1.0, dualH = 0.0;
  const double mu = log(10.0 * 1.0);
  if (s->da_state) { leapStep = s->da_state[0]; dualLeapStep = s->da_state[1]; dualH = s->da_state[2]; }
  for (int64_t i = s->start_step + 1; rc == 0 && i <= len; i++) {
    const double own_eps = leapStep;
    const double eps = s->force_eps ? s->force_eps[i] : leapStep;
    const double* met = force_metric ? force_metric + i * msz : inv_metric;
    if (metric == 1) { memcpy(minv, met, sizeof(double) * (size_t)d); x->minv = minv; }
    if (metric == 2) {
      x->A = met;
      if (orc_dense_cholesky(met, Lf, d)) { rc = -3; break; }
    }
    if (normals) CPY(z, normals + i * d); else orc_draw_normals(seed, chain, (uint32_t)i, d, z);
    if (metric == 0) CPY(p0, z);
    else if (metric == 1) for (int64_t j = 0; j < d; j++) p0[j] = z[j] / sqrt(minv[j]);
    else orc_dense_backsub(Lf, z, p0, d);                              /* p = L^-T z */
    sharp(x, p0, s0);
    const double H0 = -lt + 0.5 * dot(s0, p0, d);
    x->H0 = H0; x->step = (uint32_t)i; x->n_leap = 0; x->sum_metro = 0.0; x->divergent = 0;
    /* the one-point tree: B = F = the current point, rho = p, log-weight 0; the sample is the current point */
    CPY(thf, pars); CPY(pf, p0); CPY(gf, grad); CPY(thb, pars); CPY(pb, p0); CPY(gb, grad);
    CPY(rho, p0); CPY(p_bb, p0); CPY(p_bf, p0); CPY(p_fb, p0); CPY(p_ff, p0);
    CPY(s_bb, s0); CPY(s_bf, s0); CPY(s_fb, s0); CPY(s_ff, s0);
    double lsw = 0.0, sample_h = H0;
    int moved = 0;
    for (int j = 0; j < maxd; j++) {
      const int fwd = orc_nuts_slot_uniform(seed, chain, (uint32_t)i, 0x80000000u + 2u * (uint32_t)j) >= 0.5;
      x->e = fwd ? eps : -eps;
      x->th = fwd ? thf : thb; x->p = fwd ? pf : pb; x->g = fwd ? gf : gb;
      int valid;
      if (fwd) {                                                        /* B = the old tree, F = the new subtree */
        CPY(rho_b, rho); CPY(p_bf, p_ff); CPY(s_bf, s_ff);
        valid = build_tree(x, j, &sub);
        CPY(rho_f, sub.rho); CPY(p_fb, sub.pb); CPY(s_fb, sub.sb); CPY(p_ff, sub.pe); CPY(s_ff, sub.se);
      } else {                                                          /* B = the new subtree, F = the old tree */
        CPY(rho_f, rho); CPY(p_fb, p_bb); CPY(s_fb, s_bb);
        valid = build_tree(x, j, &sub);
        CPY(rho_b, sub.rho); CPY(p_bf, sub.pb); CPY(s_bf, sub.sb); CPY(p_bb, sub.pe); CPY(s_bb, sub.se);
      }
      if (!valid) break;
      if (sub.lsw > lsw || orc_nuts_slot_uniform(seed, chain, (uint32_t)i, 0x80000000u + 2u * (uint32_t)j + 1u) < exp(sub.lsw - lsw)) {
        CPY(pars, sub.th); CPY(grad, sub.g); lt = sub.lt; sample_h = sub.h; moved = 1;
      }
      lsw = orc_log_sum_exp(lsw, sub.lsw);
      for (int64_t q = 0; q < d; q++) rho[q] = rho_b[q] + rho_f[q];
      int go = crit(s_bb, s_ff, rho, d);
      for (int64_t q = 0; q < d; q++) ext[q] = rho_b[q] + p_fb[q];
      go = go && crit(s_bb, s_fb, ext, d);
      for (int64_t q = 0; q < d; q++) ext[q] = rho_f[q] + p_bf[q];
      go = go && crit(s_bf, s_ff, ext, d);
      if (!go) break;
    }
    const double astat = x->sum_metro / (double)x->n_leap;
    if (i >= r->first && i <= r->last && (i - r->first) % r->step == 0) {   /* SerialMC.jl:49-66 */
      if (samples) CPY(samples + kept * d, pars);
      if (grads) CPY(grads + kept * d, grad);
      if (accept) accept[kept] = (uint8_t)moved;
      if (logtarget) logtarget[kept] = lt;
      if (diag_eps) diag_eps[kept] = own_eps;
      if (diag_leaps) diag_leaps[kept] = x->n_leap;
      if (accept_stat) accept_stat[kept] = astat;
      if (energy) energy[kept] = sample_h;
      if (divergent) divergent[kept] = (uint8_t)x->divergent;
      kept++;
    }
    if (i < burnin) {                                                   /* HMCDA.jl:133-138 with pacc = accept_stat */
      const double fi = (double)i;
      double eta = 1.0 / (fi + s->t0);
      dualH = (1.0 - eta) * dualH + eta * (s->rate - astat);
      leapStep = exp(mu - sqrt(fi) * dualH / s->shrinkage);
      eta = pow(fi, -s->step);
      dualLeapStep = exp((1.0 - eta) * log(dualLeapStep) + eta * log(leapStep));
    } else {
      leapStep = dualLeapStep;                                          /* HMCDA.jl:140 */
    }
  }
  if (n_grad_evals) *n_grad_evals = x->nev;
  block_free(&sub); free(x->tmp); free(more); free(buf);
  return rc;
}
