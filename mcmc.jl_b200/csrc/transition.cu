// transition.cu -- the per-chain state machine of engine "WAVE", plus small layout / utility kernels.
//
// A wave is: one likelihood+gradient evaluation for every chain at its pending point q (K1 for the
// regression families, eval_closed_kernel otherwise), then transition_kernel, which consumes the
// evaluation and advances each chain by exactly one evaluation's worth of sampler logic: finish the
// leapfrog / take the Metropolis decision / adapt / store the kept draw / draw the next momentum or
// proposal and write the next pending point.  Chains are independent, so HMCDA chains with different
// trajectory lengths simply sit at different phases of the same wave ("leapfrog waves").
//
// Sampler arithmetic restates src/samplers/RWM.jl:43-72, MALA.jl:65-126, HMC.jl:81-175,
// HMCDA.jl:51-143 in the reference's operation order; keep/thin logic src/runners/SerialMC.jl:37-85.
// Compiled with -fmad=false.
#include "transition.h"
#include "families.cuh"

namespace mg {

__device__ __forceinline__ double sum_part(const double* part, int nsplit, int64_t row, int64_t d, int64_t Cp, int64_t c) {
  double s = part[row * Cp + c];
  for (int sp = 1; sp < nsplit; sp++) s += part[((int64_t)sp * (d + 2) + row) * Cp + c];
  return s;
}

// The model-side finish of an evaluation: prior terms, LLAcc support semantics (M6), gradient of the prior.
struct EvalFin {
  double lt;     // log-target at q (NaN when not requested)
  bool oos;      // DSL families: out of support => (-Inf, zeros)  (modelparser.jl:64-92)
  double ginv;   // gradient of the prior is (0 - q_j) * ginv  (or -q_j * ginv for probit)
  int fam;
};
// x / v for the prior gradient: when v is a power of two (prior sd 1, the examples' value: v = 1) the division is a
// multiplication by the exact reciprocal -- the same double for every x whose quotient is a normal number -- instead of the
// ~20-instruction IEEE division sequence
__device__ __forceinline__ double div_by_var(double x, double v) {
  // the test on v and the reciprocal are loop invariants of every caller (v is a model constant); the test on x is integer
  // work on its exponent: 2^-498 < |x| < 2^499, or x == 0
  const bool vpow2 = ((__double_as_longlong(v) & 0x000FFFFFFFFFFFFFll) == 0) && v > 1e-150 && v < 1e150;
  const int ex = (__double2hiint(x) >> 20) & 0x7ff;
  if (vpow2 && ((ex > 0x20d && ex < 0x5f2) || (__double_as_longlong(x) << 1) == 0)) return x * (1.0 / v);
  return x / v;
}

__device__ __forceinline__ EvalFin finalize_eval(const ModelDev& M, const double* q, const double* part, int nsplit,
                                                 int64_t Cp, int64_t c, bool want_lt) {
  EvalFin f; f.fam = M.family; f.oos = false; f.ginv = 0.0; f.lt = CUDART_NAN;
  const int64_t d = M.d;
  if (M.family == MCMCGPU_FAM_LINEAR || M.family == MCMCGPU_FAM_LOGISTIC) {
    const double psd = M.hyper[0];
    double bad = sum_part(part, nsplit, d + 1, d, Cp, c);
    f.oos = bad > 0.0;
    double acc = 0.0;
    if (want_lt) {
      // vars ~ Normal(0, prior_sd).  On interior leapfrogs the prior value is not needed and its only other role -- a
      // non-finite prior puts the point out of support -- is covered by the likelihood's support count: a non-finite
      // beta makes every eta NaN.  (A finite |beta_j| > 1e154, whose square overflows, is the one case left to the
      // trajectory's last evaluation.)
      const double lsd = log(psd);
      double s = 0.0;
#pragma unroll 4
      for (int64_t j = 0; j < d; j++) {
        double z = div_by_var(q[j * Cp + c] - 0.0, psd);
        s += -(MG_LN_SQRT_2PI + 0.5 * z * z + lsd);
      }
      acc = 0.0 + s;
      if (!isfinite(acc)) f.oos = true;
    }
    if (want_lt) {
      double ll = sum_part(part, nsplit, d, d, Cp, c);
      double acc2 = acc + ll;
      if (!isfinite(acc2)) f.oos = true;
      f.lt = f.oos ? -CUDART_INF : acc2;
    }
    f.ginv = 1.0 / (psd * psd);
  } else if (M.family == MCMCGPU_FAM_PROBIT) {
    const double psd = M.hyper[0], pvar = psd * psd;
    if (want_lt) {
      double qq = 0.0;
      for (int64_t j = 0; j < d; j++) { double v = q[j * Cp + c]; qq += v * v; }
      double logprior = -0.5 * ((double)d * MG_LOG2PI + (double)d * log(pvar)) - 0.5 * (qq / pvar);
      f.lt = logprior + sum_part(part, nsplit, d, d, Cp, c);
    }
    f.ginv = pvar;
  } else {
    f.lt = part[d * Cp + c];   // closed-form families: eval_closed_kernel wrote final values
  }
  return f;
}
__device__ __forceinline__ double fin_grad(const EvalFin& f, const ModelDev& M, const double* q, const double* part,
                                           int nsplit, int64_t Cp, int64_t c, int64_t j) {
  if (f.fam == MCMCGPU_FAM_LINEAR || f.fam == MCMCGPU_FAM_LOGISTIC) {
    if (f.oos) return 0.0;
    double psd = M.hyper[0];
    return sum_part(part, nsplit, j, M.d, Cp, c) + div_by_var(0.0 - q[j * Cp + c], psd * psd);
  } else if (f.fam == MCMCGPU_FAM_PROBIT) {
    return sum_part(part, nsplit, j, M.d, Cp, c) - div_by_var(q[j * Cp + c], f.ginv);
  }
  return part[j * Cp + c];
}

// Keeps chain c's current state as the draw of step `step` when the step is in first:step:last.
__device__ __forceinline__ void store_kept(const WaveArgs& W, const int64_t c, int64_t step, bool has_grad, bool acc, double eps, int nl) {
  const RunnerDev& R = W.R;
  const int64_t d = W.M.d, Cp = R.Cp;
  // SerialMC.jl:49-66: the post-decision state (ppars / plogtarget / pgrads) is what is kept
  if (!in_range(step, R.first, R.step, R.last)) return;
  int64_t k = W.kept[c];
  for (int64_t j = 0; j < d; j++) W.samples[(k * d + j) * Cp + c] = W.cur_pars[j * Cp + c];
  if (W.grads) for (int64_t j = 0; j < d; j++) W.grads[(k * d + j) * Cp + c] = has_grad ? W.cur_grad[j * Cp + c] : CUDART_NAN;
  W.accept[k * Cp + c] = acc ? 1 : 0;
  if (W.logtarget) W.logtarget[k * Cp + c] = W.cur_lt[c];
  if (W.eps) W.eps[k * Cp + c] = eps;
  if (W.nleaps) W.nleaps[k * Cp + c] = nl;
  W.kept[c] = k + 1;
}

// The dual-averaging update of step i < burnin (HMCDA.jl:133-138), shared by HMCDA (pacc = its acceptance probability)
// and NUTS (pacc = the mean acceptance statistic of the step's last doubling, or Stan's accept_stat over the whole trajectory).  The averaging counts steps from i0 and
// shrinks towards mu = log(ten_eps0): HMCDA passes 10 * leapStep0 (leapStep0 = 1) and i0 = 0; NUTS with metric adaptation
// restarts it at every window end (i0 = that step, ten_eps0 = 10 eps).  The log is taken here, where HMCDA always took it,
// so that the HMCDA kernels compile to the same instructions.
struct DaStep { double leapstep, dual, dualH; };
__device__ __forceinline__ DaStep da_adapt(const SamplerDev& S, int64_t i, double pacc, double dual, double dualH,
                                           double ten_eps0, int64_t i0) {
  const double fi = (double)(i - i0);
  double eta = 1.0 / (fi + S.t0);
  DaStep r;
  r.dualH = (1.0 - eta) * dualH + eta * (S.rate - pacc);
  r.leapstep = exp(log(ten_eps0) - sqrt(fi) * r.dualH / S.shrinkage);
  eta = pow(fi, -S.step);
  r.dual = exp((1.0 - eta) * log(dual) + eta * log(r.leapstep));
  return r;
}

// One chain's share of a wave.  Returns the number of evaluations it consumed (0 or 1).  `interior_done`: the chain is in the
// middle of a trajectory and its momentum / position update has already been made element-parallel by the caller
// (transition_kernel, stage A); only the per-chain counters are left.
__device__ int transition_chain(const WaveArgs& W, const int64_t c, const bool interior_done) {
  const RunnerDev& R = W.R;
  const SamplerDev& S = W.S;
  const ModelDev& M = W.M;
  const int ph = W.phase[c];
  if (ph == PH_DONE) return 0;
  if (W.resume) {
    if (ph != PH_PAUSE) return 0;
    atomicAdd(W.remaining, 1);
  } else if (ph == PH_PAUSE) return 0;
  const int64_t d = M.d, Cp = R.Cp;
  const uint64_t gchain = W.chain_ids ? (uint64_t)W.chain_ids[c] : (uint64_t)(R.chain_offset + c);
  const int64_t burnin = R.first - 1;
  const int kind = S.kind;
  const bool hmc_like = (kind == MCMCGPU_HMC || kind == MCMCGPU_HMCDA);
  double* q = W.q;
  const double* part = W.part;
  const int ns = W.nsplit;

  int64_t i = W.istep[c];
  int leap = hmc_like ? W.leap[c] : 0;
  int nl_cur = hmc_like ? W.nleaps_cur[c] : 0;
  const bool interior = (ph == PH_LEAP) && (leap + 1 < nl_cur) && (W.rb == nullptr);   // storeLeaps needs H at every leap
  EvalFin F; F.lt = CUDART_NAN; F.oos = false; F.ginv = 0.0; F.fam = M.family;
  if (ph != PH_PAUSE && !interior_done) F = finalize_eval(M, q, part, ns, Cp, c, !interior);
  const double lt_q = F.lt;
  const int nev = (ph != PH_PAUSE) ? 1 : 0;
  bool begin = false;

  auto uniform = [&](int64_t step) -> double {
    return W.inj_uniforms ? W.inj_uniforms[step * Cp + c] : philox_uniform(R.seed, gchain, (uint32_t)step);
  };
  auto store = [&](int64_t step, bool has_grad, bool acc, double eps, int nl) { store_kept(W, c, step, has_grad, acc, eps, nl); };

  if (ph == PH_PAUSE) {
    begin = true;
  } else if (ph == PH_INIT) {
    if (!isfinite(lt_q)) {   // "Initial values out of model support" RWM.jl:55 MALA.jl:85 HMC.jl:121 HMCDA.jl:88
      W.status[c] = 1; W.phase[c] = PH_DONE; atomicSub(W.remaining, 1);
      return nev;
    }
    W.status[c] = 0;
    W.cur_lt[c] = lt_q;
    if (W.init_lt) W.init_lt[c] = lt_q;
    for (int64_t j = 0; j < d; j++) {
      W.cur_pars[j * Cp + c] = q[j * Cp + c];
      if (kind != MCMCGPU_RWM && kind != MCMCGPU_RAM) W.cur_grad[j * Cp + c] = fin_grad(F, M, q, part, ns, Cp, c, j);
    }
    if (kind == MCMCGPU_HMCDA && !W.restore_da) {
      // HMCDA.jl:90-94; initializeHMCDAStep (HMCDA.jl:51-69) always returns 1.0 (state0.H is NaN, HMC.jl:88)
      W.da_leapstep[c] = 1.0; W.da_dual[c] = 1.0; W.da_dualH[c] = 0.0;
    }
    if (S.tuner_on) { W.tn_step[c] = S.scale; W.tn_nleaps[c] = S.nleaps; W.tn_acc[c] = 0; W.tn_prop[c] = 0; }
    i = W.step0 + 1;
    begin = true;
  } else if (ph == PH_RWM) {
    // RWM.jl:62-70 (and RAM.jl:63-71, the same Metropolis test)
    double ratio = lt_q - W.cur_lt[c];
    bool acc = ratio > 0 || ratio > log_lean_normal(uniform(i));
    if (acc) {
      for (int64_t j = 0; j < d; j++) W.cur_pars[j * Cp + c] = q[j * Cp + c];
      W.cur_lt[c] = lt_q;
    }
    double diag = CUDART_NAN;
    if (kind == MCMCGPU_RAM) {
      diag = 0.0;
      if (W.ram_Sb) { for (int64_t j = 0; j < d; j++) diag += W.ram_Sb[(c * d + j) * d + j]; }
      else for (int64_t j = 0; j < d; j++) diag += W.ram_S[(j * d + j) * Cp + c];     // "scale" => trace(S) (RAM.jl:65,69)
      const double er = exp(ratio);
      W.ram_al[c] = isnan(er) ? 0.0 : (er < 1.0 ? er : 1.0);                     // min(1, exp(ratio)) (RAM.jl:76); NaN => 0
      W.ram_pending[c] = 1;
    }
    store(i, false, acc, diag, 0);
    i++; begin = true;
  } else if (ph == PH_MALA) {
    // MALA.jl:103-113
    const double h = W.eps_cur[c];
    const double lc = log(MG_TWO_PI * h) / 2.0;
    double qno = 0.0, qon = 0.0;
    for (int64_t j = 0; j < d; j++) {
      double pj = W.cur_pars[j * Cp + c], gj = W.cur_grad[j * Cp + c], prop = q[j * Cp + c];
      double mean = pj + (h / 2.0) * gj;                              // :98 (recomputed, same roundings)
      double t1 = mean - prop;  qno += -(t1 * t1) / (2.0 * h) - lc;   // :103
      double mean2 = prop + (h / 2.0) * fin_grad(F, M, q, part, ns, Cp, c, j);  // :104
      double t2 = mean2 - pj;   qon += -(t2 * t2) / (2.0 * h) - lc;   // :105
    }
    double ratio = lt_q + qon - W.cur_lt[c] - qno;                    // :107
    bool acc = ratio > 0 || ratio > log_lean_normal(uniform(i));                  // :108
    if (acc) {
      for (int64_t j = 0; j < d; j++) {
        W.cur_pars[j * Cp + c] = q[j * Cp + c];
        W.cur_grad[j * Cp + c] = fin_grad(F, M, q, part, ns, Cp, c, j);
      }
      W.cur_lt[c] = lt_q;
      if (S.tuner_on) W.tn_acc[c] += 1;
    }
    store(i, true, acc, h, 0);
    if (S.tuner_on && i <= burnin && (i % S.adapt_step) == 0) {       // :116-118, adapt! :36-39
      double rate = (double)W.tn_acc[c] / (double)W.tn_prop[c];
      W.tn_step[c] *= (1.0 / (1.0 + exp(-11.0 * (rate - S.target_rate))) + 0.5);
      W.tn_acc[c] = 0; W.tn_prop[c] = 0;
    }
    i++; begin = true;
  } else {  // PH_LEAP: HMC.jl:93-102 second half, then either the next leapfrog or the decision
    const double eps = W.eps_cur[c];
    leap += 1;
    if (W.rb) {   // storeLeaps: weight of this leap state exp(H0 - H) and its contribution (mean.jl:19,27)
      double mm2 = 0.0;
      for (int64_t j = 0; j < d; j++) {
        double m = W.mom[j * Cp + c] + (0.5 * fin_grad(F, M, q, part, ns, Cp, c, j)) * eps;
        mm2 += m * m;
      }
      const double wl = exp(W.H0[c] - (-lt_q + 0.5 * mm2));
      for (int64_t j = 0; j < d; j++) W.rb_acc[j * Cp + c] += wl * q[j * Cp + c];
    }
    if (leap < nl_cur) {
      if (!interior_done)
#pragma unroll 4
      for (int64_t j = 0; j < d; j++) {
        double gj = fin_grad(F, M, q, part, ns, Cp, c, j);
        double m = W.mom[j * Cp + c];
        m += (0.5 * gj) * eps;          // end of this leapfrog      HMC.jl:98
        m += (0.5 * gj) * eps;          // start of the next one     HMC.jl:95
        double p = q[j * Cp + c];
        p += eps * m;                   //                           HMC.jl:96
        W.mom[j * Cp + c] = m;
        q[j * Cp + c] = p;
      }
      W.leap[c] = leap;
      W.need_ll[c] = (leap + 1 == nl_cur || W.rb) ? 1 : 0;
      return nev;
    }
    double mm = 0.0;
    for (int64_t j = 0; j < d; j++) {
      double gj = fin_grad(F, M, q, part, ns, Cp, c, j);
      double m = W.mom[j * Cp + c];
      m += (0.5 * gj) * eps;            // HMC.jl:98
      mm += m * m;
    }
    const double H = -lt_q + 0.5 * mm;  // update! HMC.jl:91
    const double e = exp(W.H0[c] - H);
    const double u = uniform(i);
    bool acc; double pacc = 0.0;
    if (kind == MCMCGPU_HMCDA) { pacc = isnan(e) ? 0.0 : (e < 1.0 ? e : 1.0); acc = u < pacc; }  // HMCDA.jl:120-121
    else acc = u < e;                                                                             // HMC.jl:154
    if (acc) {
      for (int64_t j = 0; j < d; j++) {
        W.cur_pars[j * Cp + c] = q[j * Cp + c];
        W.cur_grad[j * Cp + c] = fin_grad(F, M, q, part, ns, Cp, c, j);
      }
      W.cur_lt[c] = lt_q;
      if (S.tuner_on) W.tn_acc[c] += 1;
    }
    if (W.rb && in_range(i, R.first, R.step, R.last)) {   // (sample + sum_k w_k pars_k) / (nleaps + 1), mean.jl:24-30
      const int64_t k = W.kept[c];
      for (int64_t j = 0; j < d; j++) W.rb[(k * d + j) * Cp + c] = (W.cur_pars[j * Cp + c] + W.rb_acc[j * Cp + c]) / (double)(nl_cur + 1);
    }
    store(i, true, acc, eps, nl_cur);
    if (kind == MCMCGPU_HMCDA) {
      if (i < burnin) {                                               // HMCDA.jl:133-138
        const DaStep a = da_adapt(S, i, pacc, W.da_dual[c], W.da_dualH[c], 10.0 * 1.0, 0);
        W.da_dual[c] = a.dual; W.da_dualH[c] = a.dualH; W.da_leapstep[c] = a.leapstep;
      } else {
        W.da_leapstep[c] = W.da_dual[c];                              // :140
      }
    } else if (S.tuner_on && i <= burnin && (i % S.adapt_step) == 0) { // HMC.jl:167-169, adapt! :39-43
      double rate = (double)W.tn_acc[c] / (double)W.tn_prop[c];
      double ts = W.tn_step[c] * (1.0 / (1.0 + exp(-11.0 * (rate - S.target_rate))) + 0.5);
      double cl = ceil(S.target_path / ts);
      W.tn_step[c] = ts;
      W.tn_nleaps[c] = (cl < (double)S.max_step) ? (int64_t)cl : (int64_t)S.max_step;
      W.tn_acc[c] = 0; W.tn_prop[c] = 0;
    }
    i++; begin = true;
  }

  if (begin) {
    if (i > R.last) {
      W.phase[c] = PH_DONE;
      W.istep[c] = i;
      if (W.final_eps) {
        double fe = S.scale;
        if (kind == MCMCGPU_HMCDA) fe = W.da_leapstep[c];
        else if (S.tuner_on) fe = W.tn_step[c];
        W.final_eps[c] = fe;
      }
      atomicSub(W.remaining, 1);
      return nev;
    }
    W.istep[c] = i;
    if (i > W.step_limit) {   // pause: mcmcgpu_run_execute_steps continues from here
      W.phase[c] = PH_PAUSE;
      atomicSub(W.remaining, 1);
      return nev;
    }
    if (kind == MCMCGPU_RAM) {   // the proposal needs the updated factor: ram_kernel makes it
      W.phase[c] = PH_RAM_BEGIN;
      return nev;
    }
    // ---- start step i: draw and write the next pending point ----
    double eps = S.scale; int nl = 0;
    if (kind == MCMCGPU_HMCDA) {
      eps = W.da_leapstep[c];
      double r = round(S.len / eps);                                  // HMCDA.jl:104
      if (!(r >= 1.0)) r = 1.0;
      if (r > (double)S.max_leaps) r = (double)S.max_leaps;
      nl = (int)r;
    } else if (kind == MCMCGPU_HMC) {
      if (S.tuner_on) { W.tn_prop[c] += 1; nl = (int)W.tn_nleaps[c]; eps = W.tn_step[c]; } else nl = S.nleaps;
    } else if (kind == MCMCGPU_MALA) {
      if (S.tuner_on) { W.tn_prop[c] += 1; eps = W.tn_step[c]; }
    }
    const double sq = (kind == MCMCGPU_MALA) ? sqrt(eps) : 0.0;
    double mm = 0.0;
    for (int64_t jb = 0; jb < d; jb += 2) {
      double z0, z1 = 0.0;
      if (W.inj_normals) {
        z0 = W.inj_normals[(i * d + jb) * Cp + c];
        if (jb + 1 < d) z1 = W.inj_normals[(i * d + jb + 1) * Cp + c];
      } else {
        philox_normal_pair(R.seed, gchain, (uint32_t)i, (uint32_t)(jb >> 1), z0, z1);
      }
#pragma unroll
      for (int s = 0; s < 2; s++) {
        const int64_t j = jb + s;
        if (j >= d) break;
        const double z = s ? z1 : z0;
        const double pj = W.cur_pars[j * Cp + c];
        if (kind == MCMCGPU_RWM) {
          q[j * Cp + c] = pj + z * (W.scale[j] * S.scale);            // RWM.jl:52,59
        } else if (kind == MCMCGPU_MALA) {
          double mean = pj + (eps / 2.0) * W.cur_grad[j * Cp + c];    // MALA.jl:98
          q[j * Cp + c] = mean + sq * z;                              // :100
        } else {
          double m = z;                                               // HMC.jl:136
          mm += m * m;
          m += (0.5 * W.cur_grad[j * Cp + c]) * eps;                  // HMC.jl:95
          double p = pj;
          p += eps * m;                                               // HMC.jl:96
          W.mom[j * Cp + c] = m;
          q[j * Cp + c] = p;
        }
      }
    }
    if (hmc_like) {
      if (W.rb) for (int64_t j = 0; j < d; j++) W.rb_acc[j * Cp + c] = 0.0;
      W.H0[c] = -W.cur_lt[c] + 0.5 * mm;                              // update! HMC.jl:91
      W.leap[c] = 0; W.nleaps_cur[c] = nl;
      W.need_ll[c] = (nl == 1 || W.rb) ? 1 : 0;
      W.phase[c] = PH_LEAP;
    } else {
      W.need_ll[c] = 1;
      W.phase[c] = (kind == MCMCGPU_RWM) ? PH_RWM : PH_MALA;
    }
    W.eps_cur[c] = eps;
  }
  return nev;
}

// CTA = TR_CHAINS chains x TR_GROUPS parameter groups.
//   stage A (all threads, element-parallel): chains in the middle of a trajectory -- the bulk of every HMC / HMCDA wave --
//     get the end of leapfrog k and the start of leapfrog k+1 (HMC.jl:98,95,96) for their parameters j = group, group +
//     TR_GROUPS, ...: every load and store is a coalesced 512-byte segment and the machine is full, where one thread per
//     chain walking all d parameters left it latency-bound.  Per element the operations and their order are unchanged.
//   stage B (group 0, one thread per chain): the state machine for everything else (transition_chain).
// Evaluation counts are summed per CTA before the one atomic (one atomic per chain per wave serialised on a single address).
constexpr int TR_CHAINS = 64, TR_GROUPS = 4, TR_UNROLL = 5;
__global__ void __launch_bounds__(TR_CHAINS * TR_GROUPS) transition_kernel(const WaveArgs W) {
  const RunnerDev& R = W.R;
  if (!W.resume && *W.remaining == 0) return;
  const int grp = threadIdx.x / TR_CHAINS;
  const int64_t c = (int64_t)blockIdx.x * TR_CHAINS + (threadIdx.x % TR_CHAINS);
  const int64_t d = W.M.d, Cp = R.Cp;
  bool interior = false;
  if (c < R.C && !W.resume && W.rb == nullptr && W.phase[c] == PH_LEAP) interior = (W.leap[c] + 2 <= W.nleaps_cur[c]);
  __syncthreads();     // every group has read the chain's counters before group 0 advances them in stage B
  if (interior) {
    const ModelDev& M = W.M;
    EvalFin F; F.fam = M.family; F.lt = CUDART_NAN; F.oos = false; F.ginv = 0.0;
    if (M.family == MCMCGPU_FAM_LINEAR || M.family == MCMCGPU_FAM_LOGISTIC) F.oos = sum_part(W.part, W.nsplit, d + 1, d, Cp, c) > 0.0;
    else if (M.family == MCMCGPU_FAM_PROBIT) F.ginv = M.hyper[0] * M.hyper[0];
    const double eps = W.eps_cur[c];
    // TR_UNROLL elements per pass: all loads first (the stores to q / mom could alias them as far as the compiler knows)
    for (int64_t j0 = grp; j0 < d; j0 += TR_GROUPS * TR_UNROLL) {
      double gj[TR_UNROLL], m[TR_UNROLL], p[TR_UNROLL];
#pragma unroll
      for (int u = 0; u < TR_UNROLL; u++) {
        const int64_t j = j0 + (int64_t)u * TR_GROUPS;
        if (j < d) { gj[u] = fin_grad(F, M, W.q, W.part, W.nsplit, Cp, c, j); m[u] = W.mom[j * Cp + c]; p[u] = W.q[j * Cp + c]; }
      }
#pragma unroll
      for (int u = 0; u < TR_UNROLL; u++) {
        const int64_t j = j0 + (int64_t)u * TR_GROUPS;
        if (j < d) {
          m[u] += (0.5 * gj[u]) * eps;          // end of this leapfrog      HMC.jl:98
          m[u] += (0.5 * gj[u]) * eps;          // start of the next one     HMC.jl:95
          p[u] += eps * m[u];                   //                           HMC.jl:96
          W.mom[j * Cp + c] = m[u];
          W.q[j * Cp + c] = p[u];
        }
      }
    }
  }
  int nev = 0;
  if (grp == 0 && c < R.C) nev = transition_chain(W, c, interior);
  const int total = __syncthreads_count(nev);
  if (threadIdx.x == 0 && total) atomicAdd(W.n_evals, (unsigned long long)total);
}

// ---- cooperative transition for the regression families ------------------------------------------------------------
// The regression families are compared with the reference arithmetic within a tolerance by nature (K1 sums X beta and X'r in
// DMMA order), so here the O(d) sums of a decision -- kinetic energy, MALA proposal densities, the prior -- may be formed
// as CO_GROUPS partial sums (added in group order: deterministic, independent of the chain's neighbours).  That lets the
// whole state machine run element-parallel: 64 chains x CO_GROUPS parameter groups per CTA, a group owning the Philox
// pairs k = group (mod CO_GROUPS), i.e. parameters 2k and 2k+1.  Per element every operation and its order is the
// serial kernel's; the scalar decisions are taken by group 0 between the element-parallel stages:
//   A  interior leapfrogs (as in transition_kernel)            B1 partial sums of the pending decision
//   B2 decision, adaptation, keep/thin bookkeeping, next step  B3 accept copy, kept-draw stores, next draw and proposal
//   B4 initial Hamiltonian / phase of the step just started
// (one thread per chain walking all d parameters took 1.01 ms per decision wave at 102 400 chains x d = 100: every
// Box-Muller pair, division and store of a chain in sequence.)
constexpr int CO_CHAINS = 64, CO_GROUPS = 8, CO_UNROLL = 3;
enum { CM_NONE = 0, CM_INTERIOR, CM_FINAL, CM_MALA, CM_RWM, CM_INIT, CM_RESUME };

__global__ void __launch_bounds__(CO_CHAINS * CO_GROUPS, 2) transition_coop_kernel(const WaveArgs W) {
  __shared__ double s_sum[CO_GROUPS][3][CO_CHAINS];      // partial sums [group][slot][chain]
  __shared__ double s_eps[CO_CHAINS];                    // step size of the step being started
  __shared__ long long s_k[CO_CHAINS], s_i[CO_CHAINS];   // kept index of the step just decided (-1: not kept); step being started
  __shared__ int s_acc[CO_CHAINS], s_begin[CO_CHAINS], s_nl[CO_CHAINS];
  const RunnerDev& R = W.R;
  const SamplerDev& S = W.S;
  const ModelDev& M = W.M;
  const int lc = threadIdx.x % CO_CHAINS, grp = threadIdx.x / CO_CHAINS;
  const int64_t c = (int64_t)blockIdx.x * CO_CHAINS + lc;
  const int64_t d = M.d, Cp = R.Cp;
  const int kind = S.kind;
  const bool hmc_like = (kind == MCMCGPU_HMC || kind == MCMCGPU_HMCDA);
  const bool linlog = (M.family == MCMCGPU_FAM_LINEAR || M.family == MCMCGPU_FAM_LOGISTIC);
  const double* part = W.part;
  const int ns = W.nsplit;
  double* q = W.q;
  const int64_t npairs = (d + 1) / 2;

  // ---- stage 0: classify (every group reads the chain's counters; nobody has advanced them yet) ----
  // Every per-chain scalar the kernel will need is loaded HERE, unconditionally and side by side: at small shapes the kernel
  // is a chain of dependent global round trips (remaining -> phase -> leap -> eps -> support flag -> ... : 9 us for an
  // interior wave of 96 chains, 25 us for a decision wave), and the values a later stage needs depend on nothing but c.
  // The arrays are allocated for every run (size Cp), so the speculative reads are in bounds whatever the sampler.
  const bool live = c < R.C;
  const int rem = W.resume ? 1 : *W.remaining;
  int ph = PH_DONE, lp = 0, nlc = 0;
  bool k1d = false;
  double eps_ld = 0.0, oos_sum = 0.0;
  long long istep_ld = 0, kept_ld = 0;              // group 0 only: what stage B2 / B4 consume
  double cur_lt_ld = 0.0, H0_ld = 0.0, ll_ld = 0.0, da_ls_ld = 0.0, da_dual_ld = 0.0, da_dualH_ld = 0.0;
  if (live) {
    ph = W.phase[c]; lp = W.leap[c]; nlc = W.nleaps_cur[c]; eps_ld = W.eps_cur[c];
    if (W.fused_interior) k1d = W.k1_done[c] != 0;
    if (linlog && ns == 1) oos_sum = sum_part(part, ns, d + 1, d, Cp, c);
    if (grp == 0) {
      istep_ld = W.istep[c]; kept_ld = W.kept[c]; cur_lt_ld = W.cur_lt[c]; H0_ld = W.H0[c];
      if (ns == 1) ll_ld = sum_part(part, ns, d, d, Cp, c);
      if (kind == MCMCGPU_HMCDA) { da_ls_ld = W.da_leapstep[c]; da_dual_ld = W.da_dual[c]; da_dualH_ld = W.da_dualH[c]; }
    }
  }
  if (rem == 0) return;                             // uniform over the grid
  int mode = CM_NONE;
  if (live) {
    if (W.resume) mode = (ph == PH_PAUSE) ? CM_RESUME : CM_NONE;
    else if (ph == PH_INIT) mode = CM_INIT;
    else if (ph == PH_RWM) mode = CM_RWM;
    else if (ph == PH_MALA) mode = CM_MALA;
    else if (ph == PH_LEAP) mode = (lp + 2 <= nlc) ? CM_INTERIOR : CM_FINAL;
    // interior leapfrog completed (state and counters) by the likelihood kernel: nothing to do for this chain
    if (W.fused_interior && !W.resume && k1d) mode = CM_NONE;
  }
  const double eps_cur = (mode == CM_INTERIOR || mode == CM_FINAL || mode == CM_MALA) ? eps_ld : 0.0;
  EvalFin F; F.fam = M.family; F.lt = CUDART_NAN; F.oos = false; F.ginv = 0.0;
  if (mode != CM_NONE && mode != CM_RESUME) {
    if (linlog) F.oos = ((ns == 1) ? oos_sum : sum_part(part, ns, d + 1, d, Cp, c)) > 0.0;    // LLAcc: a non-finite likelihood term => zero gradient
    else F.ginv = M.hyper[0] * M.hyper[0];
  }
  __syncthreads();

  // ---- stage A: interior leapfrogs ----
  if (mode == CM_INTERIOR) {
    // CO_UNROLL elements per pass, all loads first (the stores to q / mom could alias them as far as the compiler knows)
    for (int64_t j0 = grp; j0 < d; j0 += CO_GROUPS * CO_UNROLL) {
      double gj[CO_UNROLL], m[CO_UNROLL], p[CO_UNROLL];
#pragma unroll
      for (int u = 0; u < CO_UNROLL; u++) {
        const int64_t j = j0 + (int64_t)u * CO_GROUPS;
        if (j < d) { gj[u] = fin_grad(F, M, q, part, ns, Cp, c, j); m[u] = W.mom[j * Cp + c]; p[u] = q[j * Cp + c]; }
      }
#pragma unroll
      for (int u = 0; u < CO_UNROLL; u++) {
        const int64_t j = j0 + (int64_t)u * CO_GROUPS;
        if (j < d) {
          m[u] += (0.5 * gj[u]) * eps_cur;          // end of this leapfrog      HMC.jl:98
          m[u] += (0.5 * gj[u]) * eps_cur;          // start of the next one     HMC.jl:95
          p[u] += eps_cur * m[u];                   //                           HMC.jl:96
          W.mom[j * Cp + c] = m[u];
          q[j * Cp + c] = p[u];
        }
      }
    }
  }

  // ---- stage B1: partial sums of the pending decision over this group's parameters ----
  const bool decide = (mode == CM_FINAL || mode == CM_MALA || mode == CM_RWM || mode == CM_INIT);
  if (decide) {
    double s0 = 0.0, s1 = 0.0, s2v = 0.0;      // slot 0: kinetic energy / q(new|old); slot 1: prior; slot 2: q(old|new)
    const double psd = M.hyper[0];
    const double lsd = linlog ? log(psd) : 0.0;
    const double h = eps_cur;
    const double lc2 = (mode == CM_MALA) ? log(MG_TWO_PI * h) / 2.0 : 0.0;
    for (int64_t k = grp; k < npairs; k += CO_GROUPS) {
#pragma unroll
      for (int t2 = 0; t2 < 2; t2++) {
        const int64_t j = 2 * k + t2;
        if (j >= d) break;
        const double qj = q[j * Cp + c];
        if (linlog) { const double z = div_by_var(qj - 0.0, psd); s1 += -(MG_LN_SQRT_2PI + 0.5 * z * z + lsd); }   // vars ~ Normal(0, prior_sd)
        else s1 += qj * qj;                                                                               // probit_regression.jl:19-22
        if (mode == CM_FINAL) {
          const double gj = fin_grad(F, M, q, part, ns, Cp, c, j);
          double m = W.mom[j * Cp + c];
          m += (0.5 * gj) * eps_cur;        // HMC.jl:98
          s0 += m * m;
        } else if (mode == CM_MALA) {       // MALA.jl:98,103-105
          const double pj = W.cur_pars[j * Cp + c], gcur = W.cur_grad[j * Cp + c];
          const double mean = pj + (h / 2.0) * gcur;
          const double t1 = mean - qj;   s0 += -(t1 * t1) / (2.0 * h) - lc2;
          const double mean2 = qj + (h / 2.0) * fin_grad(F, M, q, part, ns, Cp, c, j);
          const double t3 = mean2 - pj;  s2v += -(t3 * t3) / (2.0 * h) - lc2;
        }
      }
    }
    s_sum[grp][0][lc] = s0; s_sum[grp][1][lc] = s1; s_sum[grp][2][lc] = s2v;
  }
  __syncthreads();

  // ---- stage B2: the decision (group 0, one thread per chain) ----
  int nev = 0;
  double cur_lt_now = cur_lt_ld;            // the chain's log-target after this wave's decision (group 0; stage B4 reads it)
  if (grp == 0) {
    s_acc[lc] = 0; s_begin[lc] = 0; s_k[lc] = -1; s_nl[lc] = 0; s_eps[lc] = 0.0; s_i[lc] = 0;
    if (mode != CM_NONE) {
      const uint64_t gchain = W.chain_ids ? (uint64_t)W.chain_ids[c] : (uint64_t)(R.chain_offset + c);
      const int64_t burnin = R.first - 1;
      auto uniform = [&](int64_t step) -> double {
        return W.inj_uniforms ? W.inj_uniforms[step * Cp + c] : philox_uniform(R.seed, gchain, (uint32_t)step);
      };
      nev = (mode == CM_RESUME) ? 0 : 1;
      int64_t i = istep_ld;
      bool begin = false, acc = false;
      cur_lt_now = cur_lt_ld;
      double lt_q = CUDART_NAN;
      if (decide) {            // the model-side finish of the evaluation (finalize_eval), from the partial sums
        double pr = 0.0;
        for (int g = 0; g < CO_GROUPS; g++) pr += s_sum[g][1][lc];
        const double ll = (ns == 1) ? ll_ld : sum_part(part, ns, d, d, Cp, c);
        if (linlog) {
          bool oos = F.oos;
          const double a1 = 0.0 + pr;
          if (!isfinite(a1)) oos = true;
          const double a2 = a1 + ll;
          if (!isfinite(a2)) oos = true;
          lt_q = oos ? -CUDART_INF : a2;
        } else {
          const double pvar = F.ginv;
          lt_q = (-0.5 * ((double)d * MG_LOG2PI + (double)d * log(pvar)) - 0.5 * (pr / pvar)) + ll;
        }
      }
      double st_eps = CUDART_NAN; int st_nl = 0; bool stored = false;
      if (mode == CM_RESUME) {
        atomicAdd(W.remaining, 1);
        begin = true;
      } else if (mode == CM_INTERIOR) {
        const int leap = lp + 1;
        W.leap[c] = leap;
        W.need_ll[c] = (leap + 1 == nlc) ? 1 : 0;
      } else if (mode == CM_INIT) {
        if (!isfinite(lt_q)) {     // "Initial values out of model support" RWM.jl:55 MALA.jl:85 HMC.jl:121 HMCDA.jl:88
          W.status[c] = 1; W.phase[c] = PH_DONE; atomicSub(W.remaining, 1);
        } else {
          W.status[c] = 0;
          W.cur_lt[c] = lt_q; cur_lt_now = lt_q;
          if (W.init_lt) W.init_lt[c] = lt_q;
          acc = true;              // "accept" the initial point: stage B3 copies q (and its gradient) into the state
          if (kind == MCMCGPU_HMCDA && !W.restore_da) {                      // HMCDA.jl:90-94
            W.da_leapstep[c] = 1.0; W.da_dual[c] = 1.0; W.da_dualH[c] = 0.0;
            da_ls_ld = 1.0; da_dual_ld = 1.0; da_dualH_ld = 0.0;
          }
          if (S.tuner_on) { W.tn_step[c] = S.scale; W.tn_nleaps[c] = S.nleaps; W.tn_acc[c] = 0; W.tn_prop[c] = 0; }
          i = W.step0 + 1;
          begin = true;
        }
      } else if (mode == CM_RWM) {                                       // RWM.jl:62-70
        const double ratio = lt_q - cur_lt_ld;
        acc = ratio > 0 || ratio > log_lean_normal(uniform(i));
        if (acc) { W.cur_lt[c] = lt_q; cur_lt_now = lt_q; }
        stored = true; st_eps = CUDART_NAN; st_nl = 0;
      } else if (mode == CM_MALA) {                                      // MALA.jl:103-118
        double qno = 0.0, qon = 0.0;
        for (int g = 0; g < CO_GROUPS; g++) { qno += s_sum[g][0][lc]; qon += s_sum[g][2][lc]; }
        const double ratio = lt_q + qon - cur_lt_ld - qno;               // :107
        acc = ratio > 0 || ratio > log_lean_normal(uniform(i));          // :108
        if (acc) { W.cur_lt[c] = lt_q; cur_lt_now = lt_q; if (S.tuner_on) W.tn_acc[c] += 1; }
        stored = true; st_eps = eps_cur; st_nl = 0;
      } else if (mode == CM_FINAL) {                                     // HMC.jl:154 / HMCDA.jl:120-121
        double mm = 0.0;
        for (int g = 0; g < CO_GROUPS; g++) mm += s_sum[g][0][lc];
        const double H = -lt_q + 0.5 * mm;                               // update! HMC.jl:91
        const double e = exp(H0_ld - H);
        const double u = uniform(i);
        double pacc = 0.0;
        if (kind == MCMCGPU_HMCDA) { pacc = isnan(e) ? 0.0 : (e < 1.0 ? e : 1.0); acc = u < pacc; }
        else acc = u < e;
        if (acc) { W.cur_lt[c] = lt_q; cur_lt_now = lt_q; if (S.tuner_on) W.tn_acc[c] += 1; }
        stored = true; st_eps = eps_cur; st_nl = nlc;
        if (kind == MCMCGPU_HMCDA) {
          if (i < burnin) {                                               // HMCDA.jl:133-138
            const DaStep a = da_adapt(S, i, pacc, da_dual_ld, da_dualH_ld, 10.0 * 1.0, 0);
            W.da_dual[c] = a.dual; W.da_dualH[c] = a.dualH; W.da_leapstep[c] = a.leapstep; da_ls_ld = a.leapstep;
          } else {
            W.da_leapstep[c] = da_dual_ld; da_ls_ld = da_dual_ld;         // :140
          }
        }
      }
      if (stored) {
        if (in_range(i, R.first, R.step, R.last)) {                       // SerialMC.jl:49-66
          const int64_t k = kept_ld;
          s_k[lc] = k;
          W.accept[k * Cp + c] = acc ? 1 : 0;
          if (W.logtarget) W.logtarget[k * Cp + c] = cur_lt_now;
          if (W.eps) W.eps[k * Cp + c] = st_eps;
          if (W.nleaps) W.nleaps[k * Cp + c] = st_nl;
          W.kept[c] = k + 1;
        }
        if (S.tuner_on && i <= burnin && (i % S.adapt_step) == 0) {       // MALA.jl:116-118 / HMC.jl:167-169
          const double rate = (double)W.tn_acc[c] / (double)W.tn_prop[c];
          const double ts = W.tn_step[c] * (1.0 / (1.0 + exp(-11.0 * (rate - S.target_rate))) + 0.5);
          W.tn_step[c] = ts;
          if (kind == MCMCGPU_HMC) {
            const double cl = ceil(S.target_path / ts);
            W.tn_nleaps[c] = (cl < (double)S.max_step) ? (int64_t)cl : (int64_t)S.max_step;
          }
          W.tn_acc[c] = 0; W.tn_prop[c] = 0;
        }
        i++; begin = true;
      }
      s_acc[lc] = acc ? 1 : 0;
      if (begin) {
        W.istep[c] = i;
        if (i > R.last) {
          W.phase[c] = PH_DONE;
          if (W.final_eps) W.final_eps[c] = (kind == MCMCGPU_HMCDA) ? da_ls_ld : (S.tuner_on ? W.tn_step[c] : S.scale);
          atomicSub(W.remaining, 1);
        } else if (i > W.step_limit) {
          W.phase[c] = PH_PAUSE;
          atomicSub(W.remaining, 1);
        } else {
          double eps = S.scale; int nl = 0;
          if (kind == MCMCGPU_HMCDA) {
            eps = da_ls_ld;
            double r = round(S.len / eps);                                // HMCDA.jl:104
            if (!(r >= 1.0)) r = 1.0;
            if (r > (double)S.max_leaps) r = (double)S.max_leaps;
            nl = (int)r;
          } else if (kind == MCMCGPU_HMC) {
            if (S.tuner_on) { W.tn_prop[c] += 1; nl = (int)W.tn_nleaps[c]; eps = W.tn_step[c]; } else nl = S.nleaps;
          } else if (kind == MCMCGPU_MALA) {
            if (S.tuner_on) { W.tn_prop[c] += 1; eps = W.tn_step[c]; }
          }
          s_begin[lc] = 1; s_eps[lc] = eps; s_nl[lc] = nl; s_i[lc] = i;
        }
      }
    }
  }
  __syncthreads();

  // ---- stage B3: accept copy, kept-draw stores, next draw and proposal (element-parallel) ----
  const bool acc = s_acc[lc] != 0, begin = s_begin[lc] != 0;
  const long long kk = s_k[lc];
  double mm_part = 0.0;
  if (acc || kk >= 0 || begin) {
    const bool need_grad_state = (kind != MCMCGPU_RWM);
    const double eps = s_eps[lc];
    const int64_t inext = s_i[lc];
    const double sq = (kind == MCMCGPU_MALA) ? sqrt(eps) : 0.0;
    const uint64_t gchain = (W.chain_ids && c < R.C) ? (uint64_t)W.chain_ids[c] : (uint64_t)(R.chain_offset + c);
    for (int64_t k = grp; k < npairs; k += CO_GROUPS) {
      double z0 = 0.0, z1 = 0.0;
      if (begin) {
        if (W.inj_normals) {
          z0 = W.inj_normals[(inext * d + 2 * k) * Cp + c];
          if (2 * k + 1 < d) z1 = W.inj_normals[(inext * d + 2 * k + 1) * Cp + c];
        } else {
          philox_normal_pair(R.seed, gchain, (uint32_t)inext, (uint32_t)k, z0, z1);
        }
      }
      // both elements of the pair: every load first, then every store (the stores go to arrays the loads read from as far
      // as the compiler knows: interleaved, each load is issued only after the preceding store, four round trips per pair)
      double pjv[2] = {0.0, 0.0}, gjv[2] = {0.0, 0.0};
#pragma unroll
      for (int t2 = 0; t2 < 2; t2++) {
        const int64_t j = 2 * k + t2;
        if (j >= d) break;
        if (acc) {
          pjv[t2] = q[j * Cp + c];
          if (need_grad_state) gjv[t2] = fin_grad(F, M, q, part, ns, Cp, c, j);
        } else {
          pjv[t2] = W.cur_pars[j * Cp + c];
          if (need_grad_state) gjv[t2] = W.cur_grad[j * Cp + c];
        }
      }
#pragma unroll
      for (int t2 = 0; t2 < 2; t2++) {
        const int64_t j = 2 * k + t2;
        if (j >= d) break;
        const double pj = pjv[t2], gj = gjv[t2];
        if (acc) {
          W.cur_pars[j * Cp + c] = pj;
          if (need_grad_state) W.cur_grad[j * Cp + c] = gj;
        }
        if (kk >= 0) {                    // the post-decision state is what is kept (SerialMC.jl:49-53)
          W.samples[(kk * d + j) * Cp + c] = pj;
          if (W.grads) W.grads[(kk * d + j) * Cp + c] = need_grad_state ? gj : CUDART_NAN;
        }
        if (begin) {
          const double z = t2 ? z1 : z0;
          if (kind == MCMCGPU_RWM) {
            q[j * Cp + c] = pj + z * (W.scale[j] * S.scale);            // RWM.jl:52,59
          } else if (kind == MCMCGPU_MALA) {
            const double mean = pj + (eps / 2.0) * gj;                   // MALA.jl:98
            q[j * Cp + c] = mean + sq * z;                               // :100
          } else {
            double m = z;                                                // HMC.jl:136
            mm_part += m * m;
            m += (0.5 * gj) * eps;                                       // HMC.jl:95
            double p = pj;
            p += eps * m;                                                // HMC.jl:96
            W.mom[j * Cp + c] = m;
            q[j * Cp + c] = p;
          }
        }
      }
    }
  }
  if (begin && hmc_like) s_sum[grp][0][lc] = mm_part;
  __syncthreads();

  // ---- stage B4: the step just started ----
  if (grp == 0 && begin) {
    if (hmc_like) {
      double mm = 0.0;
      for (int g = 0; g < CO_GROUPS; g++) mm += s_sum[g][0][lc];
      W.H0[c] = -cur_lt_now + 0.5 * mm;                                  // update! HMC.jl:91 (cur_lt_now: this thread's stage B2)
      W.leap[c] = 0; W.nleaps_cur[c] = s_nl[lc];
      W.need_ll[c] = (s_nl[lc] == 1) ? 1 : 0;
      W.phase[c] = PH_LEAP;
    } else {
      W.need_ll[c] = 1;
      W.phase[c] = (kind == MCMCGPU_RWM) ? PH_RWM : PH_MALA;
    }
    W.eps_cur[c] = s_eps[lc];
  }
  const int total = __syncthreads_count(nev);
  if (threadIdx.x == 0 && total) atomicAdd(W.n_evals, (unsigned long long)total);
}

// ---- NUTS: slice NUTS with dual averaging (Hoffman & Gelman 2014, Algorithms 3 and 6), one tree leaf per wave ----------
// The recursion of BuildTree is unrolled into a per-chain state machine: doubling j builds a subtree of 2^j leaves from the
// tree end on side v, one leapfrog (one evaluation) per leaf.  Leaf m of the subtree (1-based) leaves its (theta, p) in
// checkpoint r for every r with (m - 1) mod 2^r == 0 -- the first leaf of every aligned 2^r-leaf block it opens -- and on
// completion runs the U-turn check of every block it closes (m mod 2^r == 0), which is exactly the set of checks the
// recursion makes.  Draws of step i: momentum from the normal blocks, slice uniform u0 from block 0xFFFFFFFF, direction
// of doubling j from NUTS_TREE_BLOCK + 2j, its merge from NUTS_TREE_BLOCK + 2j + 1, candidate choice of the step's leaf
// k (0-based) from NUTS_LEAF_BLOCK + k.  One thread per chain; every array is chain-minor, so a warp's accesses coalesce.
//
// MET: the kind of inverse metric M^-1.  NUTS_DIAG: a diagonal minv (NutsState::minv).  It enters as p = z / sqrt(minv),
// K = 0.5 sum (minv p) p, theta += e (minv m) and the U-turn dots delta . (minv p); with NUTS_UNIT every one of these is
// the identity's operation and minv is never loaded.  (z / 1, 1 * p and 1 * m are exact, so an all-ones metric gives the
// identity's bits.)  NUTS_DENSE: a full matrix A and its lower Cholesky factor L (NutsState::A, L): p = L^-T z by back
// substitution, v = A m (k ascending from 0.0), K = 0.5 sum_j v_j m_j, theta += e v with v = A m taken after the momentum
// half-step, and the U-turn dots delta . v with v stored for both tree ends (NutsState::v) and every checkpoint (ck_p).
// A diagonal A then computes exactly the diagonal metric's products (the zeros add nothing), so it gives their bits.
constexpr int NUTS_UNIT = 0, NUTS_DIAG = 1, NUTS_DENSE = 2;

// minv_j * x, or x itself for the identity metric
template <bool MET>
__device__ __forceinline__ double nuts_mv(const double* minv, int64_t jc, double x) {
  if constexpr (MET) return minv[jc] * x;
  else return x;
}

// continue (true) unless a U-turn: delta = v (theta_m - theta_s), delta . (minv p_s) >= 0 and delta . (minv p_m) >= 0,
// summed in j order
template <bool MET>
__device__ __forceinline__ bool nuts_no_uturn(const double* th_m, const double* p_m, const double* th_s, const double* p_s, double v,
                                              const double* minv, int64_t d, int64_t Cp, int64_t c) {
  double ds = 0.0, dm = 0.0;
  for (int64_t j = 0; j < d; j++) {
    const double delta = v * (th_m[j * Cp + c] - th_s[j * Cp + c]);
    ds += delta * nuts_mv<MET>(minv, j * Cp + c, p_s[j * Cp + c]);
    dm += delta * nuts_mv<MET>(minv, j * Cp + c, p_m[j * Cp + c]);
  }
  return ds >= 0.0 && dm >= 0.0;
}

// Metric adaptation after the dual-averaging update of warm-up step i (Stan's var_adaptation::learn_variance and the
// step-size restart of adapt_diag_e_nuts::transition): the step's final sample joins the window's Welford sums; at a
// window end the variance estimate, regularised towards 1e-3, becomes the metric, the sums restart and the dual averaging
// restarts at mu = log(10 eps) from step i (eps: the step size the update just made, which the next step uses).
__device__ void nuts_adapt_metric(const WaveArgs& W, const int64_t c, int64_t i, double eps) {
  const NutsState& T = W.nuts;
  const int64_t d = W.M.d, Cp = W.R.Cp;
  if (i >= T.win_lo && i <= T.win_hi) {
    const double n = (double)(T.wf_n[c] + 1);
    T.wf_n[c] += 1;
    for (int64_t j = 0; j < d; j++) {
      const double x = W.cur_pars[j * Cp + c];
      double mean = T.wf_mean[j * Cp + c];
      const double delta = x - mean;
      mean += delta / n;
      T.wf_mean[j * Cp + c] = mean;
      T.wf_m2[j * Cp + c] += delta * (x - mean);
    }
  }
  bool end = false;
  for (int k = 0; k < T.n_win; k++) end |= T.win_end[k] == i;
  if (!end) return;
  const double n = (double)T.wf_n[c];
  for (int64_t j = 0; j < d; j++) {
    const double var = n > 1.0 ? T.wf_m2[j * Cp + c] / (n - 1.0) : T.minv[j * Cp + c];   // one draw: the metric stays
    T.minv[j * Cp + c] = (n / (n + 5.0)) * var + 1e-3 * (5.0 / (n + 5.0));
    T.wf_mean[j * Cp + c] = 0.0; T.wf_m2[j * Cp + c] = 0.0;
  }
  T.wf_n[c] = 0;
  T.da_eps0[c] = eps; T.da_i0[c] = i;
  W.da_dual[c] = 1.0; W.da_dualH[c] = 0.0;
}

// v_j = sum_k A[j][k] x_k from 0.0, k ascending; Ac = chain c's A (element (j, k) at (j d + k) ld), x chain-minor
__device__ __forceinline__ double dense_row(const double* Ac, int64_t ld, int64_t j, const double* x, int64_t d, int64_t Cp,
                                           int64_t c) {
  double s = 0.0;
  for (int64_t k = 0; k < d; k++) s += Ac[(j * d + k) * ld] * x[k * Cp + c];
  return s;
}

// the position half of a leapfrog with a dense metric: q_j = th_j + e (A m)_j
__device__ __forceinline__ void dense_position(const double* Ac, int64_t ld, const double* th, const double* m, double* q, double e,
                                               int64_t d, int64_t Cp, int64_t c) {
  for (int64_t j = 0; j < d; j++) {
    double p = th[j * Cp + c];
    p += e * dense_row(Ac, ld, j, m, d, Cp, c);
    q[j * Cp + c] = p;
  }
}

// Lower Cholesky factor l of the matrix whose lower triangle a holds (element (i, j) at (i d + j) ld), in the pinned order:
// for j = 0 .. d-1, s = a_jj, s -= l_jk l_jk for k < j ascending, l_jj = sqrt(s); for i > j, t = a_ij, t -= l_ik l_jk for
// k < j ascending, l_ij = t / l_jj.  False (l partly written) when a pivot s is not finite and > 0.
__device__ bool dense_cholesky(const double* a, double* l, int64_t d, int64_t ld) {
  for (int64_t j = 0; j < d; j++) {
    double s = a[(j * d + j) * ld];
    for (int64_t k = 0; k < j; k++) s -= l[(j * d + k) * ld] * l[(j * d + k) * ld];
    if (!(s > 0.0 && isfinite(s))) return false;
    const double ljj = sqrt(s);
    l[(j * d + j) * ld] = ljj;
    for (int64_t i = j + 1; i < d; i++) {
      double t = a[(i * d + j) * ld];
      for (int64_t k = 0; k < j; k++) t -= l[(i * d + k) * ld] * l[(j * d + k) * ld];
      l[(i * d + j) * ld] = t / ljj;
    }
  }
  return true;
}

// Dense metric adaptation (Stan's covar_adaptation::learn_covariance with welford_covar_estimator), in nuts_adapt_metric's
// order: the step's final sample x joins the window's sums (n += 1, delta = x - mean, mean += delta / n, then
// m2[a][b] += (x_a - mean_a) delta_b with the new mean: full, not symmetrised, as Stan's estimator).  At a window end
// A = (n / (n + 5)) cov + 1e-3 (5 / (n + 5)) I with cov = m2 / (n - 1) (n <= 1: the current A), built in place of m2, and
// L = chol(A); if that Cholesky fails the chain keeps its A, whose factor is recomputed bit for bit.  Then the sums reset
// and the dual averaging restarts as for the diagonal metric.  A, L and m2 are per chain here (ld = Cp).
__device__ void nuts_adapt_dense(const WaveArgs& W, const int64_t c, int64_t i, double eps) {
  const NutsState& T = W.nuts;
  const int64_t d = W.M.d, Cp = W.R.Cp;
  const double* x = W.cur_pars;
  if (i >= T.win_lo && i <= T.win_hi) {
    const double n = (double)(T.wf_n[c] + 1);
    T.wf_n[c] += 1;
    for (int64_t a = 0; a < d; a++) {
      const double xa = x[a * Cp + c], ma = T.wf_mean[a * Cp + c];
      const double ra = xa - (ma + (xa - ma) / n);                      // x_a minus its updated mean
      for (int64_t b = 0; b < d; b++) T.wf_m2[(a * d + b) * Cp + c] += ra * (x[b * Cp + c] - T.wf_mean[b * Cp + c]);
    }
    for (int64_t j = 0; j < d; j++) {
      const double xj = x[j * Cp + c];
      double mean = T.wf_mean[j * Cp + c];
      mean += (xj - mean) / n;
      T.wf_mean[j * Cp + c] = mean;
    }
  }
  bool end = false;
  for (int k = 0; k < T.n_win; k++) end |= T.win_end[k] == i;
  if (!end) return;
  const double n = (double)T.wf_n[c];
  for (int64_t a = 0; a < d; a++)
    for (int64_t b = 0; b < d; b++) {
      const int64_t at = (a * d + b) * Cp + c;
      const double cov = n > 1.0 ? T.wf_m2[at] / (n - 1.0) : T.A[at];
      double an = (n / (n + 5.0)) * cov;
      if (a == b) an = an + 1e-3 * (5.0 / (n + 5.0));
      T.wf_m2[at] = an;
    }
  if (dense_cholesky(T.wf_m2 + c, T.L + c, d, Cp)) {
    for (int64_t k = 0; k < d * d; k++) T.A[k * Cp + c] = T.wf_m2[k * Cp + c];
  } else {
    dense_cholesky(T.A + c, T.L + c, d, Cp);
  }
  for (int64_t k = 0; k < d * d; k++) T.wf_m2[k * Cp + c] = 0.0;
  for (int64_t j = 0; j < d; j++) T.wf_mean[j * Cp + c] = 0.0;
  T.wf_n[c] = 0;
  T.da_eps0[c] = eps; T.da_i0[c] = i;
  W.da_dual[c] = 1.0; W.da_dualH[c] = 0.0;
}

// ---- Stan's multinomial transition (base_nuts::transition / build_tree, pinned in DESIGN.md) ---------------------------
// TR: the transition.  NUTS_TR_SLICE is the slice NUTS above; NUTS_TR_MULTI weights every leaf by exp(H0 - H), samples
// progressively (biased at the tree level) and checks p# . rho > 0 across every pair of neighbouring blocks.  Leaf m
// (1-based) of a subtree is written as a one-leaf block into record rf = ctz(m) -- the level at which it comes to rest, free
// at that moment -- and merged there with the open left halves of records 0 .. rf-1 (the recursion's internal nodes it
// closes, bottom up).  Record rf is then the left half of level rf, or for m = 2^j the finished subtree.
constexpr int NUTS_TR_SLICE = 0, NUTS_TR_MULTI = 1;

__device__ __forceinline__ double nuts_log1p_exp(double x) { return x > 0.0 ? x + log1p(exp(-x)) : log1p(exp(x)); }
// Stan Math's log_sum_exp(a, b)
__device__ __forceinline__ double nuts_log_sum_exp(double a, double b) {
  if (a == -CUDART_INF) return b;
  if (a == CUDART_INF && b == CUDART_INF) return CUDART_INF;
  return a > b ? a + nuts_log1p_exp(b - a) : b + nuts_log1p_exp(a - b);
}

// Leaf leaf of the subtree of doubling jd (its step's 0-based leaf k) has become the tree's end on side `side` with log-weight
// lw = H0 - h: build its block and make the merges it closes.  False when a merge finds a U-turn.
template <int MET>
__device__ bool nuts_mn_leaf(const WaveArgs& W, const int64_t c, const int64_t i, const uint64_t gchain, const int k, const int leaf,
                             const int jd, const int side, double lw, double lt, double h) {
  const NutsState& T = W.nuts;
  const int64_t d = W.M.d, Cp = W.R.Cp, slot = d * Cp;
  const int rf = __ffs(leaf) - 1;
  const double* p_e = T.p[side];                                        // the leaf: p, p# (A p stored, or minv p)
  const double* v_e = MET == NUTS_DENSE ? T.v[side] : nullptr;
  double *rho = T.mn_rho + rf * slot, *pb = T.mn_pb + rf * slot, *th = T.mn_th + rf * slot, *g = T.mn_g + rf * slot;
  double* vb = MET == NUTS_DENSE ? T.mn_vb + rf * slot : nullptr;
  for (int64_t j = 0; j < d; j++) {
    const int64_t jc = j * Cp + c;
    const double pj = p_e[jc];
    rho[jc] = pj; pb[jc] = pj; th[jc] = T.th[side][jc]; g[jc] = T.g[side][jc];
    if constexpr (MET == NUTS_DENSE) vb[jc] = v_e[jc];
  }
  for (int r = 0; r < rf; r++) {                                        // L = record r (built first), R = record rf
    const int64_t lo = r * slot;
    const double lsw = nuts_log_sum_exp(T.mn_lsw[r * Cp + c], lw);
    const bool take_r = lw > lsw ||
        philox_slot_uniform(W.R.seed, gchain, (uint32_t)i, NUTS_LEAF_BLOCK + (uint32_t)(k - (1 << r))) < exp(lw - lsw);
    double a1 = 0.0, b1 = 0.0, a2 = 0.0, b2 = 0.0, a3 = 0.0, b3 = 0.0;
    for (int64_t j = 0; j < d; j++) {
      const int64_t jc = j * Cp + c;
      const double rl = T.mn_rho[lo + jc], rr = rho[jc], pbl = T.mn_pb[lo + jc], pel = T.mn_pe[lo + jc], pbr = pb[jc];
      double sbl, sel, sbr, se;
      if constexpr (MET == NUTS_DENSE) {
        sbl = T.mn_vb[lo + jc]; sel = T.mn_ve[lo + jc]; sbr = vb[jc]; se = v_e[jc];
      } else {
        sbl = nuts_mv<MET == NUTS_DIAG>(T.minv, jc, pbl); sel = nuts_mv<MET == NUTS_DIAG>(T.minv, jc, pel);
        sbr = nuts_mv<MET == NUTS_DIAG>(T.minv, jc, pbr); se = nuts_mv<MET == NUTS_DIAG>(T.minv, jc, p_e[jc]);
      }
      const double rs = rl + rr, x = rl + pbr, y = rr + pel;
      a1 += sbl * rs; b1 += se * rs;                                    // crit(p#[beg L], p#[end R], rho)
      a2 += sbl * x; b2 += sbr * x;                                     // crit(p#[beg L], p#[beg R], rho_L + p[beg R])
      a3 += sel * y; b3 += se * y;                                      // crit(p#[end L], p#[end R], rho_R + p[end L])
      rho[jc] = rs; pb[jc] = pbl;
      if constexpr (MET == NUTS_DENSE) vb[jc] = sbl;
      if (!take_r) { th[jc] = T.mn_th[lo + jc]; g[jc] = T.mn_g[lo + jc]; }
    }
    if (!take_r) { lt = T.mn_lt[r * Cp + c]; h = T.mn_h[r * Cp + c]; }
    lw = lsw;
    if (!(a1 > 0.0 && b1 > 0.0 && a2 > 0.0 && b2 > 0.0 && a3 > 0.0 && b3 > 0.0)) return false;
  }
  T.mn_lsw[rf * Cp + c] = lw; T.mn_lt[rf * Cp + c] = lt; T.mn_h[rf * Cp + c] = h;
  if (rf < jd)                                                          // a left half: keep its last-built leaf
    for (int64_t j = 0; j < d; j++) {
      const int64_t jc = j * Cp + c;
      T.mn_pe[rf * slot + jc] = p_e[jc];
      if constexpr (MET == NUTS_DENSE) T.mn_ve[rf * slot + jc] = v_e[jc];
    }
  return true;
}

// The subtree of doubling jd (record jd) is complete and valid: biased progressive sampling of the step's sample, the tree's
// log-sum-weight, and (when another doubling is allowed) the U-turn checks of the merged tree, which is B (backward) + F
// (forward): the old tree and the subtree by side.  Returns whether the tree goes on.
template <int MET>
__device__ bool nuts_mn_tree(const WaveArgs& W, const int64_t c, const int64_t i, const uint64_t gchain, const int jd, const int side) {
  const NutsState& T = W.nuts;
  const int64_t d = W.M.d, Cp = W.R.Cp, so = jd * W.M.d * W.R.Cp;
  const double lsw_s = T.mn_lsw[jd * Cp + c], lsw_t = T.mn_tlsw[c];
  if (lsw_s > lsw_t ||
      philox_slot_uniform(W.R.seed, gchain, (uint32_t)i, NUTS_TREE_BLOCK + 2u * (uint32_t)jd + 1u) < exp(lsw_s - lsw_t)) {
    for (int64_t j = 0; j < d; j++) { W.cur_pars[j * Cp + c] = T.mn_th[so + j * Cp + c]; W.cur_grad[j * Cp + c] = T.mn_g[so + j * Cp + c]; }
    W.cur_lt[c] = T.mn_lt[jd * Cp + c]; T.mn_sh[c] = T.mn_h[jd * Cp + c];
    T.moved[c] = 1;
  }
  T.mn_tlsw[c] = nuts_log_sum_exp(lsw_t, lsw_s);
  if (jd + 1 >= W.S.nleaps) return false;
  // B- and F+ are the tree's ends; B+ / F- are the old tree's inner end and the subtree's first leaf, by side
  const double* pbp = side ? T.mn_pin : T.mn_pb + so;
  const double* pfm = side ? T.mn_pb + so : T.mn_pin;
  const double* vbp = MET == NUTS_DENSE ? (side ? T.mn_vin : T.mn_vb + so) : nullptr;
  const double* vfm = MET == NUTS_DENSE ? (side ? T.mn_vb + so : T.mn_vin) : nullptr;
  const double* rho_b = side ? T.mn_trho : T.mn_rho + so;
  const double* rho_f = side ? T.mn_rho + so : T.mn_trho;
  double a1 = 0.0, b1 = 0.0, a2 = 0.0, b2 = 0.0, a3 = 0.0, b3 = 0.0;
  for (int64_t j = 0; j < d; j++) {
    const int64_t jc = j * Cp + c;
    const double rb = rho_b[jc], rf = rho_f[jc], pb_p = pbp[jc], pf_m = pfm[jc];
    double sbm, sfp, sbp, sfm;
    if constexpr (MET == NUTS_DENSE) {
      sbm = T.v[0][jc]; sfp = T.v[1][jc]; sbp = vbp[jc]; sfm = vfm[jc];
    } else {
      sbm = nuts_mv<MET == NUTS_DIAG>(T.minv, jc, T.p[0][jc]); sfp = nuts_mv<MET == NUTS_DIAG>(T.minv, jc, T.p[1][jc]);
      sbp = nuts_mv<MET == NUTS_DIAG>(T.minv, jc, pb_p); sfm = nuts_mv<MET == NUTS_DIAG>(T.minv, jc, pf_m);
    }
    const double rs = rb + rf, x = rb + pf_m, y = rf + pb_p;
    a1 += sbm * rs; b1 += sfp * rs;                                     // crit(p#[B-], p#[F+], rho)
    a2 += sbm * x; b2 += sfm * x;                                       // crit(p#[B-], p#[F-], rho_B + p[F-])
    a3 += sbp * y; b3 += sfp * y;                                       // crit(p#[B+], p#[F+], rho_F + p[B+])
    T.mn_trho[jc] = rs;
  }
  return a1 > 0.0 && b1 > 0.0 && a2 > 0.0 && b2 > 0.0 && a3 > 0.0 && b3 > 0.0;
}

template <int MET, int TR>
__device__ int nuts_chain(const WaveArgs& W, const int64_t c) {
  const RunnerDev& R = W.R;
  const SamplerDev& S = W.S;
  const ModelDev& M = W.M;
  const NutsState& T = W.nuts;
  const int ph = W.phase[c];
  if (ph == PH_DONE) return 0;
  if (W.resume) {
    if (ph != PH_PAUSE) return 0;
    atomicAdd(W.remaining, 1);
  } else if (ph == PH_PAUSE) return 0;
  const int64_t d = M.d, Cp = R.Cp;
  const uint64_t gchain = W.chain_ids ? (uint64_t)W.chain_ids[c] : (uint64_t)(R.chain_offset + c);
  const int64_t burnin = R.first - 1;
  double* q = W.q;
  const double* part = W.part;
  const int ns = W.nsplit;
  int64_t i = W.istep[c];
  int nev = 0;
  EvalFin F; F.lt = CUDART_NAN; F.oos = false; F.ginv = 0.0; F.fam = M.family;
  if (ph != PH_PAUSE) { F = finalize_eval(M, q, part, ns, Cp, c, true); nev = 1; }
  bool begin = false, doubling = false;
  int jnext = 0;

  if (ph == PH_PAUSE) {
    begin = true;
  } else if (ph == PH_INIT) {
    if (!isfinite(F.lt)) {   // "Initial values out of model support"
      W.status[c] = 1; W.phase[c] = PH_DONE; atomicSub(W.remaining, 1);
      return nev;
    }
    W.status[c] = 0;
    W.cur_lt[c] = F.lt;
    if (W.init_lt) W.init_lt[c] = F.lt;
    for (int64_t j = 0; j < d; j++) {
      W.cur_pars[j * Cp + c] = q[j * Cp + c];
      W.cur_grad[j * Cp + c] = fin_grad(F, M, q, part, ns, Cp, c, j);
    }
    if (!W.restore_da) { W.da_leapstep[c] = 1.0; W.da_dual[c] = 1.0; W.da_dualH[c] = 0.0; }   // eps0 = 1, as HMCDA
    if constexpr (MET != NUTS_UNIT) if (T.win_end) { T.da_eps0[c] = 1.0; T.da_i0[c] = 0; }
    i = W.step0 + 1;
    begin = true;
  } else {   // PH_NUTS: leaf `leaf` of the subtree of doubling jd has been evaluated at q
    const int jd = T.j[c], side = T.dir[c], leaf = T.leaf[c];
    const double v = side ? 1.0 : -1.0;
    const double e = v * W.eps_cur[c];
    double* th_v = T.th[side];
    double* p_v = T.p[side];
    double* g_v = T.g[side];
    // end of the leapfrog (HMC.jl:98); the leaf becomes the tree's end on side v
    double mm = 0.0;
    for (int64_t j = 0; j < d; j++) {
      const double gj = fin_grad(F, M, q, part, ns, Cp, c, j);
      double m = W.mom[j * Cp + c];
      m += (0.5 * gj) * e;
      if constexpr (MET != NUTS_DENSE) mm += nuts_mv<MET == NUTS_DIAG>(T.minv, j * Cp + c, m) * m;
      th_v[j * Cp + c] = q[j * Cp + c]; p_v[j * Cp + c] = m; g_v[j * Cp + c] = gj;
    }
    if constexpr (MET == NUTS_DENSE)                                    // v = A p of the new end, K = 0.5 v . p
      for (int64_t j = 0; j < d; j++) {
        const double vj = dense_row(T.A + (T.a_ld == 1 ? 0 : c), T.a_ld, j, p_v, d, Cp, c);
        T.v[side][j * Cp + c] = vj;
        mm += vj * p_v[j * Cp + c];
      }
    const double* w_v = MET == NUTS_DENSE ? T.v[side] : p_v;            // what the U-turn dots take: A p, or p
    const double H = -F.lt + 0.5 * mm;                                  // update! HMC.jl:91
    const double H0 = W.H0[c], lu0 = TR == NUTS_TR_SLICE ? T.log_u0[c] : 0.0;
    const int k = T.leaps[c];
    T.leaps[c] = k + 1;
    double alpha;
    bool s, divergent = false;
    if constexpr (TR == NUTS_TR_SLICE) {
      const double ea = exp(H0 - H);
      alpha = T.alpha[c] + (isnan(ea) ? 0.0 : (ea < 1.0 ? ea : 1.0));
      T.alpha[c] = alpha;
      s = H - H0 < 1000.0 - lu0;                                        // false for NaN
      if (lu0 <= H0 - H) {                                              // a valid leaf: candidate with probability 1 / n_sub
        const int nsub = T.n_sub[c] + 1;
        T.n_sub[c] = nsub;
        if (nsub == 1 || philox_slot_uniform(R.seed, gchain, (uint32_t)i, NUTS_LEAF_BLOCK + (uint32_t)k) * (double)nsub < 1.0) {
          for (int64_t j = 0; j < d; j++) { T.sub_pars[j * Cp + c] = th_v[j * Cp + c]; T.sub_grad[j * Cp + c] = g_v[j * Cp + c]; }
          T.sub_lt[c] = F.lt;
        }
      }
      const int64_t slot = d * Cp;
      for (int r = 1; s && r <= jd && (leaf & ((1 << r) - 1)) == 0; r++)      // U-turn checks of the blocks this leaf closes
        s = nuts_no_uturn<MET == NUTS_DIAG>(th_v, w_v, T.ck_th + (r - 1) * slot, T.ck_p + (r - 1) * slot, v, T.minv, d, Cp, c);
    } else {                                                            // Stan's leaf: h, divergence, sum_metro, its block
      const double h = isnan(H) ? CUDART_INF : H;
      divergent = h - H0 > 1000.0;
      alpha = T.alpha[c] + (H0 - h > 0.0 ? 1.0 : exp(H0 - h));
      T.alpha[c] = alpha;
      s = !divergent && nuts_mn_leaf<MET>(W, c, i, gchain, k, leaf, jd, side, H0 - h, F.lt, h);
    }
    bool open = false;
    if (s && leaf < (1 << jd)) {                                        // next leaf of this subtree
      if constexpr (TR == NUTS_TR_SLICE)
        for (int r = 1; r <= jd && ((leaf - 1) & ((1 << r) - 1)) == 0; r++)   // checkpoints of the blocks this leaf opens
          for (int64_t j = 0, slot = d * Cp; j < d; j++) {
            T.ck_th[(r - 1) * slot + j * Cp + c] = th_v[j * Cp + c];
            T.ck_p[(r - 1) * slot + j * Cp + c] = w_v[j * Cp + c];
          }
      for (int64_t j = 0; j < d; j++) {                                 // HMC.jl:95-96 from the end just reached
        double m = p_v[j * Cp + c];
        m += (0.5 * g_v[j * Cp + c]) * e;
        if constexpr (MET == NUTS_DENSE) {
          W.mom[j * Cp + c] = m;
        } else {
          double p = th_v[j * Cp + c];
          p += e * nuts_mv<MET == NUTS_DIAG>(T.minv, j * Cp + c, m);
          W.mom[j * Cp + c] = m; q[j * Cp + c] = p;
        }
      }
      if constexpr (MET == NUTS_DENSE) dense_position(T.A + (T.a_ld == 1 ? 0 : c), T.a_ld, th_v, W.mom, q, e, d, Cp, c);
      T.leaf[c] = leaf + 1;
      return nev;
    } else if (s) {                                                     // the subtree is complete: merge it into the tree
      if constexpr (TR == NUTS_TR_SLICE) {
        const int n = T.n[c], nsub = T.n_sub[c];
        if (philox_slot_uniform(R.seed, gchain, (uint32_t)i, NUTS_TREE_BLOCK + 2u * (uint32_t)jd + 1u) * (double)n < (double)nsub) {
          for (int64_t j = 0; j < d; j++) { W.cur_pars[j * Cp + c] = T.sub_pars[j * Cp + c]; W.cur_grad[j * Cp + c] = T.sub_grad[j * Cp + c]; }
          W.cur_lt[c] = T.sub_lt[c];
          T.moved[c] = 1;
        }
        T.n[c] = n + nsub;
        open = jd + 1 < S.nleaps && nuts_no_uturn<MET == NUTS_DIAG>(T.th[1], MET == NUTS_DENSE ? T.v[1] : T.p[1], T.th[0],
                                                                     MET == NUTS_DENSE ? T.v[0] : T.p[0], 1.0, T.minv, d, Cp, c);
      } else {
        open = nuts_mn_tree<MET>(W, c, i, gchain, jd, side);
      }
    }
    if (open) {
      doubling = true; jnext = jd + 1;
    } else {                                                            // the tree is closed: the step's sample is final
      // slice: alpha / n_alpha of the last doubling; multinomial: sum_metro / n_leapfrog of the step
      const double pacc = alpha / (double)(TR == NUTS_TR_SLICE ? leaf : k + 1);
      if constexpr (TR == NUTS_TR_MULTI)
        if (in_range(i, R.first, R.step, R.last)) {
          const int64_t kk = W.kept[c];
          T.st_accept_stat[kk * Cp + c] = pacc; T.st_energy[kk * Cp + c] = T.mn_sh[c]; T.st_divergent[kk * Cp + c] = divergent ? 1 : 0;
        }
      store_kept(W, c, i, true, T.moved[c] != 0, W.eps_cur[c], k + 1);
      if (i < burnin) {
        double eps0 = 1.0;
        int64_t i0 = 0;
        if constexpr (MET != NUTS_UNIT) if (T.win_end) { eps0 = T.da_eps0[c]; i0 = T.da_i0[c]; }
        const DaStep a = da_adapt(S, i, pacc, W.da_dual[c], W.da_dualH[c], 10.0 * eps0, i0);
        W.da_dual[c] = a.dual; W.da_dualH[c] = a.dualH; W.da_leapstep[c] = a.leapstep;
        if constexpr (MET == NUTS_DIAG) if (T.win_end) nuts_adapt_metric(W, c, i, a.leapstep);
        if constexpr (MET == NUTS_DENSE) if (T.win_end) nuts_adapt_dense(W, c, i, a.leapstep);
      } else {
        W.da_leapstep[c] = W.da_dual[c];
      }
      i++; begin = true;
    }
  }

  if (begin) {
    W.istep[c] = i;
    if (i > R.last) {
      W.phase[c] = PH_DONE;
      if (W.final_eps) W.final_eps[c] = W.da_leapstep[c];
      atomicSub(W.remaining, 1);
      return nev;
    }
    if (i > W.step_limit) {   // pause: mcmcgpu_run_execute_steps continues from here
      W.phase[c] = PH_PAUSE;
      atomicSub(W.remaining, 1);
      return nev;
    }
    // ---- start step i: momentum, H0, slice, a one-point tree at the current state ----
    double mm = 0.0;
    for (int64_t jb = 0; jb < d; jb += 2) {
      double z0, z1;
      philox_normal_pair(R.seed, gchain, (uint32_t)i, (uint32_t)(jb >> 1), z0, z1);
#pragma unroll
      for (int t = 0; t < 2; t++) {
        const int64_t j = jb + t;
        if (j >= d) break;
        double z = t ? z1 : z0;
        if constexpr (MET == NUTS_DIAG) z = z / sqrt(T.minv[j * Cp + c]);     // p = z / sqrt(minv)
        if constexpr (MET != NUTS_DENSE) mm += nuts_mv<MET == NUTS_DIAG>(T.minv, j * Cp + c, z) * z;
        const double pj = W.cur_pars[j * Cp + c], gj = W.cur_grad[j * Cp + c];
        T.th[0][j * Cp + c] = pj; T.th[1][j * Cp + c] = pj;
        T.p[0][j * Cp + c] = z; T.p[1][j * Cp + c] = z;
        T.g[0][j * Cp + c] = gj; T.g[1][j * Cp + c] = gj;
        if constexpr (TR == NUTS_TR_MULTI && MET != NUTS_DENSE) T.mn_trho[j * Cp + c] = z;
      }
    }
    if constexpr (MET == NUTS_DENSE) {   // p = L^-T z by back substitution (Stan's llt().matrixU().solve), v = A p, K = 0.5 v . p
      const double* Lc = T.L + (T.a_ld == 1 ? 0 : c);
      double* p0 = T.p[0];
      for (int64_t j = d - 1; j >= 0; j--) {
        double s = p0[j * Cp + c];
        for (int64_t k = j + 1; k < d; k++) s -= Lc[(k * d + j) * T.a_ld] * p0[k * Cp + c];
        p0[j * Cp + c] = s / Lc[(j * d + j) * T.a_ld];
      }
      for (int64_t j = 0; j < d; j++) {
        const double pj = p0[j * Cp + c];
        const double vj = dense_row(T.A + (T.a_ld == 1 ? 0 : c), T.a_ld, j, p0, d, Cp, c);
        mm += vj * pj;
        T.p[1][j * Cp + c] = pj; T.v[0][j * Cp + c] = vj; T.v[1][j * Cp + c] = vj;
        if constexpr (TR == NUTS_TR_MULTI) T.mn_trho[j * Cp + c] = pj;
      }
    }
    W.H0[c] = -W.cur_lt[c] + 0.5 * mm;                                  // update! HMC.jl:91
    if constexpr (TR == NUTS_TR_SLICE) {
      T.log_u0[c] = log(philox_uniform(R.seed, gchain, (uint32_t)i));
      T.n[c] = 1;
    } else {                                                            // the one-point tree: log-weight 0, sample H = H0
      T.mn_tlsw[c] = 0.0; T.mn_sh[c] = W.H0[c]; T.alpha[c] = 0.0;
    }
    T.leaps[c] = 0; T.moved[c] = 0;
    W.eps_cur[c] = W.da_leapstep[c];
    doubling = true; jnext = 0;
  }
  if (doubling) {   // doubling jnext: direction, then the first leaf of its subtree from the end on that side
    const int side = philox_slot_uniform(R.seed, gchain, (uint32_t)i, NUTS_TREE_BLOCK + 2u * (uint32_t)jnext) >= 0.5 ? 1 : 0;
    T.j[c] = jnext; T.dir[c] = side; T.leaf[c] = 1;
    if constexpr (TR == NUTS_TR_SLICE) { T.n_sub[c] = 0; T.alpha[c] = 0.0; }
    else                                                                // the old tree's end on this side becomes its inner end
      for (int64_t j = 0; j < d; j++) {
        T.mn_pin[j * Cp + c] = T.p[side][j * Cp + c];
        if constexpr (MET == NUTS_DENSE) T.mn_vin[j * Cp + c] = T.v[side][j * Cp + c];
      }
    const double e = (side ? 1.0 : -1.0) * W.eps_cur[c];
    const double* th_v = T.th[side];
    const double* p_v = T.p[side];
    const double* g_v = T.g[side];
    for (int64_t j = 0; j < d; j++) {
      double m = p_v[j * Cp + c];
      m += (0.5 * g_v[j * Cp + c]) * e;                                 // HMC.jl:95
      if constexpr (MET == NUTS_DENSE) {
        W.mom[j * Cp + c] = m;
      } else {
        double p = th_v[j * Cp + c];
        p += e * nuts_mv<MET == NUTS_DIAG>(T.minv, j * Cp + c, m);      // HMC.jl:96
        W.mom[j * Cp + c] = m; q[j * Cp + c] = p;
      }
    }
    if constexpr (MET == NUTS_DENSE) dense_position(T.A + (T.a_ld == 1 ? 0 : c), T.a_ld, th_v, W.mom, q, e, d, Cp, c);   // HMC.jl:96
    W.need_ll[c] = 1;
    W.phase[c] = PH_NUTS;
  }
  return nev;
}

constexpr int NUTS_THREADS = 128;
template <int MET, int TR>
__global__ void __launch_bounds__(NUTS_THREADS) nuts_kernel(const WaveArgs W) {
  if (!W.resume && *W.remaining == 0) return;
  const int64_t c = (int64_t)blockIdx.x * NUTS_THREADS + threadIdx.x;
  const int nev = (c < W.R.C) ? nuts_chain<MET, TR>(W, c) : 0;
  const int total = __syncthreads_count(nev);
  if (threadIdx.x == 0 && total) atomicAdd(W.n_evals, (unsigned long long)total);
}

cudaError_t launch_transition(const WaveArgs& W, cudaStream_t st) {
  if (W.S.kind == MCMCGPU_NUTS) {
    const unsigned blocks = (unsigned)((W.R.C + NUTS_THREADS - 1) / NUTS_THREADS);
    if (W.nuts.mn_rho) {
      if (W.nuts.A) nuts_kernel<NUTS_DENSE, NUTS_TR_MULTI><<<blocks, NUTS_THREADS, 0, st>>>(W);
      else if (W.nuts.minv) nuts_kernel<NUTS_DIAG, NUTS_TR_MULTI><<<blocks, NUTS_THREADS, 0, st>>>(W);
      else nuts_kernel<NUTS_UNIT, NUTS_TR_MULTI><<<blocks, NUTS_THREADS, 0, st>>>(W);
    } else if (W.nuts.A) nuts_kernel<NUTS_DENSE, NUTS_TR_SLICE><<<blocks, NUTS_THREADS, 0, st>>>(W);
    else if (W.nuts.minv) nuts_kernel<NUTS_DIAG, NUTS_TR_SLICE><<<blocks, NUTS_THREADS, 0, st>>>(W);
    else nuts_kernel<NUTS_UNIT, NUTS_TR_SLICE><<<blocks, NUTS_THREADS, 0, st>>>(W);
    return cudaGetLastError();
  }
  const bool regression = (W.M.family == MCMCGPU_FAM_LINEAR || W.M.family == MCMCGPU_FAM_LOGISTIC || W.M.family == MCMCGPU_FAM_PROBIT);
  if (regression && W.S.kind != MCMCGPU_RAM && W.rb == nullptr) {
    int blocks = (int)((W.R.C + CO_CHAINS - 1) / CO_CHAINS);
    transition_coop_kernel<<<blocks, CO_CHAINS * CO_GROUPS, 0, st>>>(W);
    return cudaGetLastError();
  }
  int blocks = (int)((W.R.C + TR_CHAINS - 1) / TR_CHAINS);
  transition_kernel<<<blocks, TR_CHAINS * TR_GROUPS, 0, st>>>(W);
  return cudaGetLastError();
}


// L = chol(A) for n dense metrics at pitch ld (mcmcgpu_run_set_dense_metric); bad[c] = 1 where a pivot fails
__global__ void __launch_bounds__(128) dense_factor_kernel(const double* A, double* L, int64_t d, int64_t n, int64_t ld, int32_t* bad) {
  const int64_t c = (int64_t)blockIdx.x * 128 + threadIdx.x;
  if (c < n) bad[c] = dense_cholesky(A + c, L + c, d, ld) ? 0 : 1;
}
cudaError_t launch_dense_factor(const double* A, double* L, int64_t d, int64_t n, int64_t ld, int32_t* bad, cudaStream_t st) {
  dense_factor_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(A, L, d, n, ld, bad);
  return cudaGetLastError();
}

// ---- RAM (robust adaptive Metropolis) for the wave engine ----------------------------------------------
__global__ void __launch_bounds__(128) ram_kernel(const WaveArgs W, int init) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const RunnerDev& R = W.R;
  if (c >= R.C) return;
  const int d = (int)W.M.d;
  const int64_t Cp = R.Cp;
  constexpr int MD = RAM_WAVE_MAX_D;
  if (init) {                                                   // RAM.jl:50,55: S = diag(model.scale * sampler.scale)
    for (int a = 0; a < d; a++)
      for (int b = 0; b < d; b++) W.ram_S[((int64_t)a * d + b) * Cp + c] = (a == b) ? W.scale[a] * W.S.scale : 0.0;
    W.ram_pending[c] = 0;
    return;
  }
  const int ph = W.phase[c];
  if (!W.ram_pending[c] && ph != PH_RAM_BEGIN) return;
  double Sm[MD * MD], Am[MD * MD], Bm[MD * MD], z[MD];
  for (int a = 0; a < d; a++)
    for (int b = 0; b < d; b++) Sm[a * d + b] = W.ram_S[((int64_t)a * d + b) * Cp + c];
  if (W.ram_pending[c]) {                                       // RAM.jl:73-78 for the step just decided
    const int64_t i = W.istep[c] - 1;
    for (int a = 0; a < d; a++) z[a] = W.mom[(int64_t)a * Cp + c];
    double eta = (double)d * pow((double)i, -2.0 / 3.0);
    if (!(eta < 1.0)) eta = 1.0;
    const double al = W.ram_al[c];
    double zz = 0.0;
    for (int a = 0; a < d; a++) zz += z[a] * z[a];
    for (int a = 0; a < d; a++)
      for (int b = 0; b < d; b++) Am[a * d + b] = ((a == b) ? 1.0 : 0.0) + (z[a] * z[b]) / zz * eta * (al - W.S.rate);
    for (int a = 0; a < d; a++)
      for (int b = 0; b < d; b++) {
        double s2 = 0.0;
        for (int k = 0; k < d; k++) s2 += Sm[a * d + k] * Am[k * d + b];
        Bm[a * d + b] = s2;
      }
    for (int a = 0; a < d; a++)
      for (int b = 0; b < d; b++) {
        double s2 = 0.0;
        for (int k = 0; k < d; k++) s2 += Bm[a * d + k] * Sm[b * d + k];
        Am[a * d + b] = s2;
      }
    for (int a = 0; a < d; a++)
      for (int b = 0; b < d; b++) {
        if (b > a) { Sm[a * d + b] = 0.0; continue; }
        double s2 = Am[a * d + b];
        for (int k = 0; k < b; k++) s2 -= Sm[a * d + k] * Sm[b * d + k];
        Sm[a * d + b] = (a == b) ? sqrt(s2) : s2 / Sm[b * d + b];
      }
    for (int a = 0; a < d; a++)
      for (int b = 0; b < d; b++) W.ram_S[((int64_t)a * d + b) * Cp + c] = Sm[a * d + b];
    W.ram_pending[c] = 0;
  }
  if (ph != PH_RAM_BEGIN) return;
  // RAM.jl:59-60: rvec = randn(d); proposedPars = pars + S * rvec
  const int64_t i = W.istep[c];
  const uint64_t gchain = (uint64_t)(R.chain_offset + c);
  for (int jb = 0; jb < d; jb += 2) {
    double z0, z1 = 0.0;
    if (W.inj_normals) {
      z0 = W.inj_normals[(i * d + jb) * Cp + c];
      if (jb + 1 < d) z1 = W.inj_normals[(i * d + jb + 1) * Cp + c];
    } else {
      philox_normal_pair(R.seed, gchain, (uint32_t)i, (uint32_t)(jb >> 1), z0, z1);
    }
    z[jb] = z0;
    if (jb + 1 < d) z[jb + 1] = z1;
  }
  for (int a = 0; a < d; a++) {
    double acc = 0.0;
    for (int b = 0; b < d; b++) acc += Sm[a * d + b] * z[b];
    W.q[(int64_t)a * Cp + c] = W.cur_pars[(int64_t)a * Cp + c] + acc;
    W.mom[(int64_t)a * Cp + c] = z[a];
  }
  W.need_ll[c] = 1;
  W.eps_cur[c] = W.S.scale;
  W.phase[c] = PH_RWM;
}

// RAM for d > RAM_WAVE_MAX_D: one CTA per chain; the factor and three d x d work matrices live in global memory (L2).
// Every matrix element is formed by ONE thread with the reference's serial sum over k (RAM.jl:76-78 restated literally:
// A = I + eta (alpha - rate) z z'/|z|^2, B = S A, M = B S', S = chol(M)' column by column), so the result does not depend
// on the thread count and equals the one-thread kernel's -- and the oracle's -- operation for operation.
constexpr int RAMB_THREADS = 256;
__global__ void __launch_bounds__(RAMB_THREADS) ram_big_kernel(const WaveArgs W, int init) {
  const int64_t c = blockIdx.x;
  const RunnerDev& R = W.R;
  const int d = (int)W.M.d, tid = threadIdx.x;
  const int64_t Cp = R.Cp, dd = (int64_t)d * d;
  double* S = W.ram_Sb + c * dd;
  double* A = W.ram_scratch + c * 3 * dd;
  double* B = A + dd;
  double* Mx = B + dd;
  __shared__ double z[RAM_BIG_MAX_D];
  __shared__ double s_scal[2];
  if (init) {                                                   // RAM.jl:50,55: S = diag(model.scale * sampler.scale)
    for (int64_t e = tid; e < dd; e += RAMB_THREADS) { const int a = (int)(e / d), b = (int)(e % d); S[e] = (a == b) ? W.scale[a] * W.S.scale : 0.0; }
    if (tid == 0) W.ram_pending[c] = 0;
    return;
  }
  const int ph = W.phase[c];
  const bool pending = W.ram_pending[c] != 0;
  if (!pending && ph != PH_RAM_BEGIN) return;
  if (pending) {                                                // RAM.jl:73-78 for the step just decided
    for (int a = tid; a < d; a += RAMB_THREADS) z[a] = W.mom[(int64_t)a * Cp + c];
    __syncthreads();
    if (tid == 0) {
      const int64_t i = W.istep[c] - 1;
      double eta = (double)d * pow((double)i, -2.0 / 3.0);
      if (!(eta < 1.0)) eta = 1.0;
      double zz = 0.0;
      for (int a = 0; a < d; a++) zz += z[a] * z[a];
      s_scal[0] = zz; s_scal[1] = eta * (W.ram_al[c] - W.S.rate);
    }
    __syncthreads();
    const double zz = s_scal[0];
    const int64_t ii = W.istep[c] - 1;
    double eta = (double)d * pow((double)ii, -2.0 / 3.0);
    if (!(eta < 1.0)) eta = 1.0;
    const double dal = W.ram_al[c] - W.S.rate;
    for (int64_t e = tid; e < dd; e += RAMB_THREADS) {
      const int a = (int)(e / d), b = (int)(e % d);
      A[e] = ((a == b) ? 1.0 : 0.0) + (z[a] * z[b]) / zz * eta * dal;
    }
    __syncthreads();
    for (int64_t e = tid; e < dd; e += RAMB_THREADS) {          // B = S * A
      const int a = (int)(e / d), b = (int)(e % d);
      double s2 = 0.0;
      for (int k = 0; k < d; k++) s2 += S[a * d + k] * A[k * d + b];
      B[e] = s2;
    }
    __syncthreads();
    for (int64_t e = tid; e < dd; e += RAMB_THREADS) {          // M = B * S'
      const int a = (int)(e / d), b = (int)(e % d);
      double s2 = 0.0;
      for (int k = 0; k < d; k++) s2 += B[a * d + k] * S[b * d + k];
      Mx[e] = s2;
    }
    __syncthreads();
    // S = chol(M)' (lower factor), column by column: the diagonal first, then the rows below it in parallel; each element is
    // M[a][b] - sum_{k<b} S[a][k] S[b][k] in the reference's order
    for (int b = 0; b < d; b++) {
      if (tid == 0) {
        double s2 = Mx[b * d + b];
        for (int k = 0; k < b; k++) s2 -= S[b * d + k] * S[b * d + k];
        S[b * d + b] = sqrt(s2);
      }
      __syncthreads();
      const double dg = S[b * d + b];
      for (int a = b + 1 + tid; a < d; a += RAMB_THREADS) {
        double s2 = Mx[a * d + b];
        for (int k = 0; k < b; k++) s2 -= S[a * d + k] * S[b * d + k];
        S[a * d + b] = s2 / dg;
      }
      for (int a = tid; a < b; a += RAMB_THREADS) S[a * d + b] = 0.0;     // upper part (b > a)
      __syncthreads();
    }
    if (tid == 0) W.ram_pending[c] = 0;
  }
  if (ph != PH_RAM_BEGIN) return;
  // RAM.jl:59-60: rvec = randn(d); proposedPars = pars + S * rvec
  const int64_t i = W.istep[c];
  const uint64_t gchain = W.chain_ids ? (uint64_t)W.chain_ids[c] : (uint64_t)(R.chain_offset + c);
  __syncthreads();
  for (int k = tid; 2 * k < d; k += RAMB_THREADS) {
    double z0, z1 = 0.0;
    if (W.inj_normals) {
      z0 = W.inj_normals[(i * d + 2 * k) * Cp + c];
      if (2 * k + 1 < d) z1 = W.inj_normals[(i * d + 2 * k + 1) * Cp + c];
    } else {
      philox_normal_pair(R.seed, gchain, (uint32_t)i, (uint32_t)k, z0, z1);
    }
    z[2 * k] = z0;
    if (2 * k + 1 < d) z[2 * k + 1] = z1;
  }
  __syncthreads();
  for (int a = tid; a < d; a += RAMB_THREADS) {
    double acc = 0.0;
    for (int b = 0; b < d; b++) acc += S[a * d + b] * z[b];
    W.q[(int64_t)a * Cp + c] = W.cur_pars[(int64_t)a * Cp + c] + acc;
    W.mom[(int64_t)a * Cp + c] = z[a];
  }
  if (tid == 0) { W.need_ll[c] = 1; W.eps_cur[c] = W.S.scale; W.phase[c] = PH_RWM; }
}

cudaError_t launch_ram(const WaveArgs& W, bool init, cudaStream_t st) {
  if (W.ram_Sb) ram_big_kernel<<<(unsigned)W.R.C, RAMB_THREADS, 0, st>>>(W, init ? 1 : 0);
  else ram_kernel<<<(unsigned)((W.R.C + 127) / 128), 128, 0, st>>>(W, init ? 1 : 0);
  return cudaGetLastError();
}

// ---- closed-form families through the wave engine ---------------------------------------------
__global__ void eval_closed_kernel(const ModelDev M, const double* q, double* part, int64_t C, int64_t Cp,
                                   const int32_t* phase, const int32_t* remaining) {
  extern __shared__ double sh_series[];
  if (remaining && *remaining == 0) return;
  if (M.family == MCMCGPU_FAM_OU) {
    for (int64_t t = threadIdx.x; t < M.N; t += blockDim.x) sh_series[t] = M.series[t];
    __syncthreads();
  }
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  if (phase && phase[c] >= PH_PAUSE) return;
  const int64_t d = M.d;
  if (M.family == MCMCGPU_FAM_NORMAL_FN) {
    double s = 0.0;
    for (int64_t j = 0; j < d; j++) { double v = q[j * Cp + c]; s += v * v; part[j * Cp + c] = -2.0 * v; }
    part[d * Cp + c] = -s;
  } else if (M.family == MCMCGPU_FAM_NORMAL_DSL) {
    const double mu = M.hyper[0], sigma = M.hyper[1];
    double s = 0.0;
    for (int64_t j = 0; j < d; j++) s += logpdf_normal(q[j * Cp + c], mu, sigma);
    double acc = 0.0 + s;
    bool oos = !isfinite(acc);
    for (int64_t j = 0; j < d; j++) part[j * Cp + c] = oos ? 0.0 : (mu - q[j * Cp + c]) / (sigma * sigma);
    part[d * Cp + c] = oos ? -CUDART_INF : acc;
  } else if (M.family == MCMCGPU_FAM_ABS_NORMAL) {
    const double mu = M.hyper[0], sigma = M.hyper[1];
    double s = 0.0;
    for (int64_t j = 0; j < d; j++) s += logpdf_normal(fabs(q[j * Cp + c]), mu, sigma);
    double acc = 0.0 + s;
    bool oos = !isfinite(acc);
    for (int64_t j = 0; j < d; j++) {
      double v = q[j * Cp + c];
      double sg = (v > 0.0) ? 1.0 : ((v < 0.0) ? -1.0 : 0.0);
      part[j * Cp + c] = oos ? 0.0 : sg * ((mu - fabs(v)) / (sigma * sigma));
    }
    part[d * Cp + c] = oos ? -CUDART_INF : acc;
  } else {  // OU
    double v[3] = {q[c], q[Cp + c], q[2 * Cp + c]}, g[3];
    double lt = Family<MCMCGPU_FAM_OU, 3>::evalallg(M, sh_series, 3, v, g);
    part[c] = g[0]; part[Cp + c] = g[1]; part[2 * Cp + c] = g[2];
    part[3 * Cp + c] = lt;
  }
  part[(d + 1) * Cp + c] = 0.0;
}

cudaError_t launch_eval_closed(const ModelDev& M, const double* q, double* part, int64_t C, int64_t Cp,
                               const int32_t* phase, const int32_t* remaining, cudaStream_t st) {
  size_t smem = (M.family == MCMCGPU_FAM_OU) ? sizeof(double) * (size_t)M.N : 0;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(eval_closed_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  eval_closed_kernel<<<(unsigned)((C + 127) / 128), 128, smem, st>>>(M, q, part, C, Cp, phase, remaining);
  return cudaGetLastError();
}

__global__ void finalize_kernel(const ModelDev M, const double* q, const double* part, int nsplit, int64_t C, int64_t Cp,
                                double* lt, double* grad) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  EvalFin F = finalize_eval(M, q, part, nsplit, Cp, c, true);
  lt[c] = F.lt;
  if (grad) for (int64_t j = 0; j < M.d; j++) grad[j * Cp + c] = fin_grad(F, M, q, part, nsplit, Cp, c, j);
}
cudaError_t launch_finalize(const ModelDev& M, const double* q, const double* part, int nsplit, int64_t C, int64_t Cp,
                            double* lt, double* grad, cudaStream_t st) {
  finalize_kernel<<<(unsigned)((C + 127) / 128), 128, 0, st>>>(M, q, part, nsplit, C, Cp, lt, grad);
  return cudaGetLastError();
}

// Fold of the row-split partials: red[i] = sum over splits of part[sp][i].  RS_GROUPS threads share one element, each
// summing every RS_GROUPS-th split in order, and their partial sums are added in group order: a fixed association for a
// given split count (the split count itself already fixes K1's own summation order), 8 dependent loads instead of 63
// for a small problem spread over 63 splits.
constexpr int RS_GROUPS = 8, RS_ELEMS = 32;
__global__ void __launch_bounds__(RS_GROUPS * RS_ELEMS) reduce_splits_kernel(const double* __restrict__ part, int nsplit, int64_t n,
                                                                              double* __restrict__ red) {
  __shared__ double sh[RS_GROUPS][RS_ELEMS];
  const int e = threadIdx.x % RS_ELEMS, g = threadIdx.x / RS_ELEMS;
  const int64_t i = (int64_t)blockIdx.x * RS_ELEMS + e;
  double s = 0.0;
  if (i < n) for (int sp = g; sp < nsplit; sp += RS_GROUPS) s += part[(int64_t)sp * n + i];
  sh[g][e] = s;
  __syncthreads();
  if (g == 0 && i < n) {
    double t = sh[0][e];
#pragma unroll
    for (int k = 1; k < RS_GROUPS; k++) t += sh[k][e];
    red[i] = t;
  }
}
cudaError_t launch_reduce_splits(const double* part, int nsplit, int64_t rows, int64_t Cp, double* red, cudaStream_t st) {
  int64_t n = rows * Cp;
  reduce_splits_kernel<<<(unsigned)((n + RS_ELEMS - 1) / RS_ELEMS), RS_GROUPS * RS_ELEMS, 0, st>>>(part, nsplit, n, red);
  return cudaGetLastError();
}

// ---- layout kernels ---------------------------------------------------------------------------
template <typename T>
__global__ void transpose_kernel(const T* in, T* out, int64_t rows_in, int64_t cols_in, int64_t in_pitch, int64_t out_pitch,
                                 int64_t in_col0) {
  // out[cidx][r] = in[r][in_col0 + cidx] for r < rows_in, cidx < cols_in  (generic tiled transpose)
  __shared__ T tile[32][33];
  int64_t bx = (int64_t)blockIdx.x * 32, by = (int64_t)blockIdx.y * 32;
  for (int k = threadIdx.y; k < 32; k += blockDim.y) {
    int64_t r = by + k, cc = bx + threadIdx.x;
    if (r < rows_in && cc < cols_in) tile[k][threadIdx.x] = in[r * in_pitch + in_col0 + cc];
  }
  __syncthreads();
  for (int k = threadIdx.y; k < 32; k += blockDim.y) {
    int64_t cc = bx + k, r = by + threadIdx.x;
    if (r < rows_in && cc < cols_in) out[cc * out_pitch + r] = tile[threadIdx.x][k];
  }
}
static dim3 tgrid(int64_t rows, int64_t cols) { return dim3((unsigned)((cols + 31) / 32), (unsigned)((rows + 31) / 32)); }

cudaError_t transpose_to_chain_minor(const double* in, double* out, int64_t C, int64_t K, int64_t Cp, cudaStream_t st) {
  // in [C][K] -> out [K][Cp]
  dim3 g = tgrid(C, K);
  if (g.y > 65535) return cudaErrorInvalidValue;
  transpose_kernel<double><<<g, dim3(32, 8), 0, st>>>(in, out, C, K, K, Cp, 0);
  return cudaGetLastError();
}
cudaError_t transpose_to_chain_major(const double* in, double* out, int64_t c0, int64_t nc, int64_t K, int64_t Cp, cudaStream_t st) {
  // in [K][Cp] (columns c0..c0+nc) -> out [nc][K]
  for (int64_t k0 = 0; k0 < K; k0 += 65535LL * 32) {
    int64_t kk = K - k0 < 65535LL * 32 ? K - k0 : 65535LL * 32;
    transpose_kernel<double><<<tgrid(kk, nc), dim3(32, 8), 0, st>>>(in + k0 * Cp, out + k0, kk, nc, Cp, K, c0);
  }
  return cudaGetLastError();
}
cudaError_t transpose_to_chain_major_u8(const uint8_t* in, uint8_t* out, int64_t c0, int64_t nc, int64_t K, int64_t Cp, cudaStream_t st) {
  for (int64_t k0 = 0; k0 < K; k0 += 65535LL * 32) {
    int64_t kk = K - k0 < 65535LL * 32 ? K - k0 : 65535LL * 32;
    transpose_kernel<uint8_t><<<tgrid(kk, nc), dim3(32, 8), 0, st>>>(in + k0 * Cp, out + k0, kk, nc, Cp, K, c0);
  }
  return cudaGetLastError();
}

__global__ void philox_dump_kernel(uint64_t seed, int64_t chain_offset, int64_t C, int64_t d, int64_t last,
                                   double* normals, double* uniforms) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= C * (last + 1)) return;
  const int64_t c = idx / (last + 1), i = idx % (last + 1);
  const uint64_t gchain = (uint64_t)(chain_offset + c);
  for (int64_t jb = 0; jb < d; jb += 2) {
    double z0, z1;
    philox_normal_pair(seed, gchain, (uint32_t)i, (uint32_t)(jb >> 1), z0, z1);
    normals[(c * (last + 1) + i) * d + jb] = z0;
    if (jb + 1 < d) normals[(c * (last + 1) + i) * d + jb + 1] = z1;
  }
  uniforms[c * (last + 1) + i] = philox_uniform(seed, gchain, (uint32_t)i);
}
cudaError_t launch_philox_dump(uint64_t seed, int64_t chain_offset, int64_t C, int64_t d, int64_t last,
                               double* normals, double* uniforms, cudaStream_t st) {
  int64_t n = C * (last + 1);
  philox_dump_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(seed, chain_offset, C, d, last, normals, uniforms);
  return cudaGetLastError();
}

__global__ void fill_kernel(double* p, double v, int64_t n) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}
__global__ void broadcast_kernel(const double* src, double* dst, int64_t K, int64_t C, int64_t Cp) {
  const int64_t n = K * C;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x)
    dst[(t / C) * Cp + t % C] = src[t / C];
}
cudaError_t broadcast_to_chain_minor(const double* src, double* dst, int64_t K, int64_t C, int64_t Cp, cudaStream_t st) {
  const int64_t n = K * C;
  const int64_t blocks = (n + 255) / 256;
  broadcast_kernel<<<(unsigned)(blocks < 8192 ? blocks : 8192), 256, 0, st>>>(src, dst, K, C, Cp);
  return cudaGetLastError();
}
cudaError_t launch_fill(double* p, double v, int64_t n, cudaStream_t st) {
  fill_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(p, v, n);
  return cudaGetLastError();
}

}  // namespace mg
