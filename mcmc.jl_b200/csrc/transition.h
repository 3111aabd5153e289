#pragma once
#include "common.cuh"
namespace mg {

// per-chain phases of the wave engine
constexpr int PH_INIT = 0;   // q = init has been evaluated
constexpr int PH_RWM = 1;    // q = RWM proposal has been evaluated
constexpr int PH_MALA = 2;   // q = MALA proposal has been evaluated
constexpr int PH_LEAP = 3;   // q = position after a leapfrog position update has been evaluated
constexpr int PH_RAM_BEGIN = 4;  // RAM: the next proposal is made by ram_kernel (after the factor update)
constexpr int PH_NUTS = 5;   // q = NUTS tree leaf (position after a leapfrog position update) has been evaluated
constexpr int PH_PAUSE = 98;  // reached the step limit of this execute call; resumes at the next one
constexpr int PH_DONE = 99;

// NUTS per-chain state, chain-minor at pitch Cp (sides: 0 = backward end of the tree, 1 = forward end)
constexpr int NUTS_MAX_DOUBLINGS = 10;
struct NutsState {
  double* th[2];               // [d][Cp] position of each tree end
  double* p[2];                // [d][Cp] momentum of each tree end
  double* g[2];                // [d][Cp] gradient of each tree end
  double *sub_pars, *sub_grad; // [d][Cp] candidate of the subtree being built
  double* sub_lt;              // [Cp]
  double *ck_th, *ck_p;        // [maxdoublings][d][Cp] U-turn checkpoints: the first leaf of the open 2^r-leaf block, r = 1..j
  double *log_u0, *alpha;      // [Cp] log slice uniform of the step; sum of min(1, exp(H0 - H)) over the current doubling
  int32_t *j, *leaf, *leaps;   // [Cp] doubling, leaf in the subtree (1-based), leapfrogs made in the step
  int32_t *n, *n_sub;          // [Cp] valid leaves of the tree / of the subtree
  int32_t *dir;                // [Cp] 1: the current subtree grows forward, 0: backward
  uint8_t* moved;              // [Cp] the step's sample is no longer the starting point
  // diagonal inverse metric M^-1 (mcmcgpu_run_set_metric / _set_metric_adaptation).  Null: the identity, and nuts_kernel's
  // identity instantiation, which loads nothing
  double* minv;                // [d][Cp]
  // metric adaptation in Stan's windows (null win_end: off).  Steps win_lo..win_hi add their final sample to the Welford
  // sums; at each of the n_win window-end steps the metric is re-estimated and the dual averaging restarts
  double *wf_mean, *wf_m2;     // [d][Cp] Welford mean and sum of squared deviations of the current window
  int64_t* wf_n;               // [Cp] samples in the current window
  double* da_eps0;             // [Cp] step size of the last restart: the dual averaging's mu = log(10 da_eps0)
  int64_t* da_i0;              // [Cp] step of the last restart (the dual averaging counts steps from it)
  const int64_t* win_end;      // [n_win] ascending
  int64_t win_lo, win_hi;
  int32_t n_win;  // dense inverse metric (mcmcgpu_run_set_dense_metric; null A: none).  Element (j, k) of chain c's matrix at
  // (j*d + k)*a_ld + c with a_ld = Cp, or at (j*d + k) for one matrix every chain reads (a_ld = 1: a fixed shared metric).
  // With adaptation A and L are per chain and wf_m2 is [d*d][Cp] (the full Welford sum of cross products).
  double* A;                   // M^-1
  double* L;                   // lower Cholesky factor of A (the upper triangle is not used)
  double* v[2];                // [d][Cp] A p of each tree end; with a dense metric ck_p holds A p instead of p
  int64_t a_ld;
  // Stan's multinomial transition (mcmcgpu_run_set_nuts_transition; null mn_rho: slice NUTS).  Block records, one per level
  // r = 0 .. maxdoublings-1, each [maxdoublings][d][Cp]: record r holds the open left half of 2^r leaves of the subtree being
  // built, and record j the finished subtree of doubling j.  A block keeps the sum of its momenta, the momentum p of its
  // first- and last-built leaves (pb, pe), its proposal (theta, grad) and, with a dense metric, A p of both end leaves (vb,
  // ve); p# = minv p is recomputed for the identity and diagonal metrics.  alpha sums the Metropolis statistic over the step.
  double *mn_rho, *mn_pb, *mn_pe, *mn_th, *mn_g, *mn_vb, *mn_ve;
  double *mn_lsw, *mn_lt, *mn_h;        // [maxdoublings][Cp] log-sum-weight, proposal's log-target and H
  double *mn_trho, *mn_pin, *mn_vin;    // [d][Cp] the tree's momentum sum; p (A p) of the old tree's end on the growing side
  double *mn_tlsw, *mn_sh;              // [Cp] the tree's log-sum-weight; H of the step's sample
  double *st_accept_stat, *st_energy;   // [S][Cp] per kept step: sum_metro / n_leapfrog, H of the sample
  uint8_t* st_divergent;                // [S][Cp] the step's last subtree stopped at a divergent leaf
};

struct WaveArgs {
  ModelDev M;
  SamplerDev S;
  RunnerDev R;
  int32_t nsplit;              // partial buffers to sum (1 after an all-reduce)
  int32_t resume;              // 1: this launch only restarts paused chains (no evaluation is consumed)
  int32_t restore_da;          // 1: HMCDA adaptation state was set by the host (mcmcgpu_run_set_state)
  int64_t step0;               // chains start at step step0 + 1
  int64_t step_limit;          // chains pause before starting a step > step_limit
  int32_t fused_interior;      // 1: the likelihood kernel has already made the interior leapfrog updates (K1Args::fuse_leap)
  uint8_t* k1_done;            // [Cp] with fused_interior: 1 for the chains the likelihood kernel has fully advanced this wave
                               // (it writes the flag of every chain it evaluates, every wave)
  // evaluation in/out
  double* q;                   // [d][Cp]
  const double* part;          // [nsplit][d+2][Cp]
  // chain state
  double *cur_pars, *cur_grad, *cur_lt, *mom, *H0;
  int32_t *phase, *leap, *nleaps_cur;
  int64_t *istep, *kept;
  double *eps_cur;
  double *da_leapstep, *da_dual, *da_dualH;
  double *tn_step; int64_t *tn_nleaps, *tn_acc, *tn_prop;
  double* ram_S;               // RAM: [d*d][Cp] lower-triangular proposal factor (row-major index a*d+b), d <= RAM_WAVE_MAX_D
  double* ram_Sb;              // RAM, d > RAM_WAVE_MAX_D: [C][d*d] chain-major factor (one CTA per chain), else null
  double* ram_scratch;         // RAM, d > RAM_WAVE_MAX_D: [C][3][d*d] work matrices
  double* ram_al;              // RAM: min(1, exp(ratio)) of the step just decided
  uint8_t* ram_pending;        // RAM: factor update pending for that step
  uint8_t* need_ll;
  int32_t* status;
  int32_t* remaining;
  unsigned long long* n_evals;
  // inputs
  const double* init; const double* scale; const double* inj_normals; const double* inj_uniforms;
  // outputs
  double* samples; double* grads; uint8_t* accept; double* logtarget; double* eps; int32_t* nleaps;
  double* final_eps;
  double* rb;                  // [S][d][Cp] Rao-Blackwell sums (store_rb) or null
  double* rb_acc;              // [d][Cp] running sum_k w_k pars_k of the current trajectory
  double* init_lt;             // [Cp] log-target at the initial point, or null
  const int64_t* chain_ids;    // [Cp] global chain id of every chain (Philox key), or null = chain_offset + position
  NutsState nuts;              // NUTS runs only
};

cudaError_t launch_transition(const WaveArgs& W, cudaStream_t st);   // NUTS runs: nuts_kernel
constexpr int RAM_WAVE_MAX_D = 16;    // one thread per chain, factor in local memory; larger d: one CTA per chain (ram_big_kernel)
constexpr int RAM_BIG_MAX_D = 128;
cudaError_t launch_ram(const WaveArgs& W, bool init, cudaStream_t st);   // RAM.jl:50-60,73-78 for the wave engine
// closed-form families through the wave engine: writes part[0][(d+2)][Cp] directly (final lt / grad)
cudaError_t launch_eval_closed(const ModelDev& M, const double* q, double* part, int64_t C, int64_t Cp,
                               const int32_t* phase, const int32_t* remaining, cudaStream_t st);
// finalize an evaluation outside a run (mcmcgpu_logtarget_grad): part -> lt[Cp], grad[d][Cp]
cudaError_t launch_finalize(const ModelDev& M, const double* q, const double* part, int nsplit, int64_t C, int64_t Cp,
                            double* lt, double* grad, cudaStream_t st);
cudaError_t launch_reduce_splits(const double* part, int nsplit, int64_t rows, int64_t Cp, double* red, cudaStream_t st);
// layout changes between the host's chain-major arrays and the device's chain-minor arrays
cudaError_t transpose_to_chain_minor(const double* in /*[C][K]*/, double* out /*[K][Cp]*/, int64_t C, int64_t K, int64_t Cp, cudaStream_t st);
cudaError_t transpose_to_chain_major(const double* in /*[K][Cp]*/, double* out /*[nc][K]*/, int64_t c0, int64_t nc, int64_t K, int64_t Cp, cudaStream_t st);
cudaError_t transpose_to_chain_major_u8(const uint8_t* in, uint8_t* out, int64_t c0, int64_t nc, int64_t K, int64_t Cp, cudaStream_t st);
cudaError_t launch_philox_dump(uint64_t seed, int64_t chain_offset, int64_t C, int64_t d, int64_t last,
                               double* normals /*[C][last+1][d]*/, double* uniforms /*[C][last+1]*/, cudaStream_t st);
cudaError_t launch_fill(double* p, double v, int64_t n, cudaStream_t st);
// dense metric: L = chol(A) of n matrices at pitch ld, bad[c] = 1 where that fails; src [K] copied to every chain of dst [K][Cp]
cudaError_t launch_dense_factor(const double* A, double* L, int64_t d, int64_t n, int64_t ld, int32_t* bad, cudaStream_t st);
cudaError_t broadcast_to_chain_minor(const double* src, double* dst, int64_t K, int64_t C, int64_t Cp, cudaStream_t st);

}  // namespace mg
