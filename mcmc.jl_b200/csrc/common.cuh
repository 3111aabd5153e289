// common.cuh -- shared device helpers of libmcmcgpu: Philox4x32-10 draws, family formulas, layouts.
// All sampler arithmetic is FP64 and written in the reference's operation order (SURVEY.md 8a); the
// translation units that include the sampler code are compiled with -fmad=false so that no
// multiply-add is contracted (bit-level agreement with the CPU restatement on closed-form targets).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include <math_constants.h>
#include "../../include/mcmcgpu.h"
#include "log_table.h"

#define MG_LOG2PI 1.8378770664093453
#define MG_LN_SQRT_2PI 0.91893853320467274178
#define MG_TWO_PI 6.283185307179586
#define MG_SQRT1_2 0.70710678118654752440

namespace mg {

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11).  Engine convention: key = (seed lo, seed hi);
// counter = (chain lo, chain hi, step, block).  Normal block b gives normals 2b and 2b+1
// (Box-Muller); block 0xFFFFFFFF gives the uniform of the Metropolis test.  Step 0 is the
// pre-loop draw of HMCDA (HMCDA.jl:90).
// ---------------------------------------------------------------------------------------------
struct u4 { uint32_t x, y, z, w; };

__host__ __device__ __forceinline__ u4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                     uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; r++) {
#ifdef __CUDA_ARCH__
    uint32_t hi0 = __umulhi(M0, c0), lo0 = M0 * c0, hi1 = __umulhi(M1, c2), lo1 = M1 * c2;
#else
    uint64_t p0 = (uint64_t)M0 * c0, p1 = (uint64_t)M1 * c2;
    uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0, hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
#endif
    uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += W0; k1 += W1;
  }
  u4 o; o.x = c0; o.y = c1; o.z = c2; o.w = c3;
  return o;
}

// uniform from 53 random bits: (b + 0.5) / 2^53 in (0, 1]; exact for b < 2^52, while for b >= 2^52 the sum b + 0.5 is
// rounded to even (so 1.0 itself occurs with probability 2^-54; harmless: log(1) = 0, and `u < p` then rejects)
__host__ __device__ __forceinline__ double u01(uint32_t hi, uint32_t lo) {
  uint64_t b = (((uint64_t)hi << 21) ^ ((uint64_t)lo >> 11)) & ((1ull << 53) - 1);
  return ((double)b + 0.5) * (1.0 / 9007199254740992.0);
}

// ---- lean, branch-free exp / reciprocal / log (|x| < 700 for exp) ---------------------------------------------------
// The link epilogue shares the FP64 pipe with DMMA, so every FP64 instruction counts; libm's exp and the IEEE division
// also carry slow-path branches that keep the compiler from interleaving the independent elements of a thread.
//   exp(x) = 2^k * (e^(r/2))^2,  k = rint(x*log2 e) (magic-number add), r = x - k*ln2 (hi/lo), degree-11 Taylor in r/2
//   (truncation 2e-18; measured against mpmath: 3.3e-16 relative);  1/d by rcp.approx + two Newton steps (<= 2e-16).
__device__ __forceinline__ double exp_lean(double x) {
  const double t = fma(x, 1.4426950408889634, 6755399441055744.0);
  const int k = __double2loint(t);
  const double kf = t - 6755399441055744.0;
  double r = fma(kf, -6.93147180369123816490e-01, x);
  r = fma(kf, -1.90821492927058770002e-10, r);
  const double h = 0.5 * r;
  double p = 2.50521083854417187751e-08;            // 1/11!
  p = fma(p, h, 2.75573192239858906526e-07);        // 1/10!
  p = fma(p, h, 2.75573192239858906526e-06);        // 1/9!
  p = fma(p, h, 2.48015873015873015873e-05);        // 1/8!
  p = fma(p, h, 1.98412698412698412698e-04);        // 1/7!
  p = fma(p, h, 1.38888888888888888889e-03);        // 1/6!
  p = fma(p, h, 8.33333333333333333333e-03);        // 1/5!
  p = fma(p, h, 4.16666666666666666667e-02);        // 1/4!
  p = fma(p, h, 1.66666666666666666667e-01);        // 1/3!
  p = fma(p, h, 0.5);
  p = fma(p, h, 1.0);
  p = fma(p, h, 1.0);
  const double e = p * p;
  return __hiloint2double(__double2hiint(e) + (k << 20), __double2loint(e));   // * 2^k, |k| <= 1010: stays normal
}
__device__ __forceinline__ double rcp_lean(double d) {     // d in [1, 1e305]
  double y;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(d));
  double e = fma(-d, y, 1.0);
  y = fma(y, e, y);
  e = fma(-d, y, 1.0);
  return fma(y, e, y);
}

// log(x) for x in the normal positive range, after fdlibm's e_log.c (argument reduction to sqrt(2)/2 < m < sqrt(2),
// s = f/(2+f), degree-7 even/odd polynomial in s^2; 1.4e-16 relative against mpmath), the division replaced by
// rcp_lean; zero, denormal, negative, infinite and NaN arguments go to libm's log (they decide the support test).
template <bool CHECKED>
__device__ __forceinline__ double log_lean_t(double x) {
  int hx = __double2hiint(x);
  if (CHECKED && (unsigned)(hx - 0x00100000) >= (unsigned)(0x7ff00000 - 0x00100000)) return log(x);
  int k = (hx >> 20) - 1023;
  hx &= 0x000fffff;
  const int i = (hx + 0x95f64) & 0x100000;
  k += i >> 20;
  const double m = __hiloint2double(hx | (i ^ 0x3ff00000), __double2loint(x));
  const double f = m - 1.0;
  const double sq = f * rcp_lean(2.0 + f);
  const double dk = (double)k;
  const double z = sq * sq, w = z * z;
  const double t1 = w * fma(w, fma(w, 1.531383769920937332e-01, 2.222219843214978396e-01), 3.999999999940941908e-01);
  const double t2 = z * fma(w, fma(w, fma(w, 1.479819860511658591e-01, 1.818357216161805012e-01), 2.857142874366239149e-01), 6.666666666666735130e-01);
  const double R = t2 + t1;
  const double hfsq = 0.5 * f * f;
  return dk * 6.93147180369123816490e-01 - ((hfsq - fma(sq, hfsq + R, dk * 1.90821492927058770002e-10)) - f);
}


// log(x) for normal positive x from the 129-interval table of (1/c_j, log c_j) (tools/gen_log_table.py; the table K1's
// logistic link keeps in shared memory, read here through the read-only cache: the load/store unit is idle in the sampler
// kernels): fdlibm's reduction to sqrt(2)/2 <= m < sqrt(2), u = m/c_j - 1 by one fused multiply-add, log1p(u) of degree 6:
// 11 FP64 instructions instead of log_lean's 28; 2.3e-16 relative, 2e-18 absolute where the logarithm vanishes (x -> 1).
static __device__ const double mg_log_tab[2 * LOG_NINT] = {LOG_TABLE_VALUES};
__device__ __forceinline__ double log_tab_normal(double x) {
  int hx = __double2hiint(x);
  int k = (hx >> 20) - 1023;
  hx &= 0x000fffff;
  const int i = (hx + 0x95f64) & 0x100000;
  k += i >> 20;
  const int hm = hx | (i ^ 0x3ff00000);
  const double m = __hiloint2double(hm, __double2loint(x));
  const int t = (hm - LOG_BASE_HI) >> LOG_SHIFT;
  const double rinv = __ldg(mg_log_tab + 2 * t), lc = __ldg(mg_log_tab + 2 * t + 1);
  const double u = fma(m, rinv, -1.0);
  double p = fma(-1.0 / 6.0, u, 0.2);
  p = fma(p, u, -0.25);
  p = fma(p, u, 1.0 / 3.0);
  p = fma(p, u, -0.5);
  const double l1 = fma(p, u * u, u);
  const double dk = __hiloint2double(0x43300000, k ^ 0x80000000) - 4503601774854144.0;   // (double)k without a conversion
  return fma(dk, 6.93147180369123816490e-01, lc) + fma(dk, 1.90821492927058770002e-10, l1);
}

__device__ __forceinline__ double log_lean(double x) { return log_lean_t<true>(x); }
// for arguments known to be normal positive numbers (e.g. the 53-bit uniforms in (0, 1)): no fallback branch at all
__device__ __forceinline__ double log_lean_normal(double x) { return log_tab_normal(x); }

// exp for any argument: the lean path inside (-700, 700), libm outside (overflow, underflow, NaN)
__device__ __forceinline__ double exp_any(double x) {
  return ((__double2hiint(x) & 0x7fffffff) < 0x4085E000) ? exp_lean(x) : exp(x);
}

__device__ __forceinline__ void philox_normal_pair(uint64_t seed, uint64_t chain, uint32_t step, uint32_t block,
                                                   double& z0, double& z1) {
  u4 o = philox4x32_10((uint32_t)chain, (uint32_t)(chain >> 32), step, block, (uint32_t)seed, (uint32_t)(seed >> 32));
  double u1 = u01(o.x, o.y), u2 = u01(o.z, o.w);
  // u1 in [2^-54, 1]: always a normal number; at u1 = 1 (probability 2^-54) the table log is +-1e-18, hence the clamp
  double r = sqrt(fmax(-2.0 * log_lean_normal(u1), 0.0));
  double s, c;
  sincospi(2.0 * u2, &s, &c);
  z0 = r * c; z1 = r * s;
}
__device__ __forceinline__ double philox_uniform(uint64_t seed, uint64_t chain, uint32_t step) {
  u4 o = philox4x32_10((uint32_t)chain, (uint32_t)(chain >> 32), step, 0xFFFFFFFFu, (uint32_t)seed, (uint32_t)(seed >> 32));
  return u01(o.x, o.y);
}
// uniform of an arbitrary block of step `step`: NUTS draws its tree directions (blocks 0x80000000 + 2j), subtree merges
// (0x80000000 + 2j + 1) and leaf candidates (0x40000000 + k) here; the normal blocks 0 .. (d-1)/2 and the Metropolis
// block 0xFFFFFFFF stay apart from them
__device__ __forceinline__ double philox_slot_uniform(uint64_t seed, uint64_t chain, uint32_t step, uint32_t block) {
  u4 o = philox4x32_10((uint32_t)chain, (uint32_t)(chain >> 32), step, block, (uint32_t)seed, (uint32_t)(seed >> 32));
  return u01(o.x, o.y);
}
constexpr uint32_t NUTS_LEAF_BLOCK = 0x40000000u, NUTS_TREE_BLOCK = 0x80000000u;

// ---------------------------------------------------------------------------------------------
// scalar log-densities (Distributions.jl 2013 == Rmath dnorm4 / dunif / pnorm log scale)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double logpdf_normal(double x, double mu, double sigma) {
  double z = (x - mu) / sigma;
  return -(MG_LN_SQRT_2PI + 0.5 * z * z + log(sigma));
}
__device__ __forceinline__ double logpdf_uniform(double x, double a, double b) {
  return (a <= x && x <= b) ? -log(b - a) : -CUDART_INF;
}
// log Phi(x): logcdf(Normal(), x) of examples/probit_regression.jl:29
__device__ __forceinline__ double log_ndtr(double x) {
  if (x > 0.0) return log1p(-0.5 * erfc(x * MG_SQRT1_2));
  if (x > -37.0) return log(0.5 * erfc(-x * MG_SQRT1_2));
  double x2 = x * x, r = 1.0 / x2;
  double s = 1.0 - r * (1.0 - 3.0 * r * (1.0 - 5.0 * r * (1.0 - 7.0 * r * (1.0 - 9.0 * r))));
  return -0.5 * x2 - MG_LN_SQRT_2PI - log(-x) + log(s);
}

// in(i, first:step:last)  (SerialMC.jl:49) and the kept index
__host__ __device__ __forceinline__ bool in_range(int64_t i, int64_t first, int64_t step, int64_t last) {
  return i >= first && i <= last && ((i - first) % step) == 0;
}

// model description as the kernels see it
struct ModelDev {
  int32_t family;
  int64_t N, d;
  double hyper[4];
  const double* series;  // OU: x[0..N-1] on the device
};

// sampler + runner description as the kernels see it
struct SamplerDev {
  int32_t kind, nleaps;
  double scale, rate, len, shrinkage, t0, step;
  int64_t max_leaps;
  int32_t tuner_on, adapt_step, max_step;
  double target_path, target_rate;
};
struct RunnerDev {
  int64_t first, step, last, S;
  int64_t C, Cp;          // chains, padded chain count (array pitch)
  int64_t chain_offset;
  uint64_t seed;
  int32_t init_per_chain, store_grad, store_lt, store_rb;
};

}  // namespace mg
