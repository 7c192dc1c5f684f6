// bayes.cuh — the terms of Bayesian problems, shared by Sampler/TMCMC (tmcmc.cu) and Optimizer/CMAES (objective.cu): the per-variable
// log-prior and the per-point log-likelihood terms of Bayesian/Reference (definitions in include/ktmcmc.h). Both files are compiled with
// --fmad=false, so every caller rounds each term the same way.
#pragma once
#include <math.h>

#include "../../include/kcma.h"
#include "common.cuh"

namespace kc {

constexpr double kHalfLog2Pi = 0.91893853320467274178;
constexpr double kInvSqrt2 = 0.70710678118654752440;
constexpr double kPi = 3.14159265358979323846;

// Per-variable constant of the prior: -log(b - a) (Uniform) or log(b) (Normal).
__device__ __forceinline__ double prior_const(int type, double a, double b) { return type == KCMA_PRIOR_UNIFORM ? -log(b - a) : log(b); }
// log-prior term of x given the constant c = prior_const(type, a, b); callers that evaluate many rows compute c once per variable
__device__ __forceinline__ double prior_term_c(int type, double a, double b, double c, double x) {
  if (type == KCMA_PRIOR_UNIFORM) return (x >= a && x <= b) ? c : -INFINITY;
  const double z = (x - a) / b;
  return -0.5 * (z * z) - c - kHalfLog2Pi;
}
__device__ __forceinline__ double prior_term(int type, double a, double b, double x) { return prior_term_c(type, a, b, prior_const(type, a, b), x); }
// log-prior of one row: lane-strided partials, xor butterfly (all lanes return the same bits)
__device__ __forceinline__ double log_prior_row(const double* __restrict__ x, int n, const int* __restrict__ type,
                                                const double* __restrict__ pa, const double* __restrict__ pb, int lane) {
  double p = 0.0;
  for (int d = lane; d < n; d += 32) p = p + prior_term(type[d], pa[d], pb[d], x[d]);
  return warp_sum_butterfly(p);
}

// Bayesian/Reference terms (tests/helpers/otmcmc_reference.c restates them in the same operation order)
__device__ __forceinline__ double log_ndtr(double u) {
  if (u >= -1.0) return log(0.5 * erfc(-u * kInvSqrt2));
  return log(0.5 * erfcx(-u * kInvSqrt2)) - 0.5 * (u * u);
}
__device__ __forceinline__ double student_t_const(double nu) {   // lgamma((nu + 1) / 2) - lgamma(nu / 2) - log(nu pi) / 2
  if (nu < 50.0) return lgamma(0.5 * (nu + 1.0)) - lgamma(0.5 * nu) - 0.5 * log(nu * kPi);
  const double ix = 1.0 / (0.5 * nu), y = ix * ix;
  return ix * (-0.125 + y * (1.0 / 192.0 + y * (-1.0 / 640.0 + y * (17.0 / 14336.0)))) - kHalfLog2Pi;
}
// Codes of a bad model output, smallest first when one row has several
enum { kRefNonFinite = 0, kRefParameter = 1, kRefPoissonMean = 2 };
// Term j of a row: prediction gj, per-point parameters p (read only for a likelihood that has one), datum dj, lgamma(dj + 1) in DC[j]
// (Poisson). A bad output lowers `bad` to its code and gives NaN.
template <int LIK>
__device__ __forceinline__ double reference_term(double gj, const double* __restrict__ p, int j, double dj, const double* __restrict__ DC, int& bad) {
  double t;
  if (!isfinite(gj)) { bad = min(bad, (int)kRefNonFinite); t = NAN; }
  else if (LIK == KCMA_LIK_POISSON) {
    if (gj < 0.0) { bad = min(bad, (int)kRefPoissonMean); t = NAN; }
    else t = dj == 0.0 ? -gj : (gj == 0.0 ? -INFINITY : dj * log(gj) - gj - __ldg(DC + j));
  } else {
    const double pj = p[j], r = dj - gj;
    if (!(pj > 0.0) || !isfinite(pj)) { bad = min(bad, (int)kRefParameter); t = NAN; }
    else if (LIK == KCMA_LIK_STUDENT_T) t = student_t_const(pj) - 0.5 * (pj + 1.0) * log1p(r * r / pj);
    else {
      const double z = r / pj;
      t = -kHalfLog2Pi - log(pj) - 0.5 * (z * z);
      if (LIK == KCMA_LIK_POSITIVE_NORMAL) { t = t - log_ndtr(gj / pj); if (t != t) t = -INFINITY; }
    }
  }
  return t;
}

}  // namespace kc
