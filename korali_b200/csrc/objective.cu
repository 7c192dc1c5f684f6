// objective.cu — K3: the batched device-objective conduit. One launch evaluates F(x_i) for every sample of the
// local population shard; it replaces the per-sample Conduit dispatch of runGeneration (CMAES.cpp.base:205-224:
// build Sample JSON, KORALI_START, KORALI_WAITALL, read "F(x)") and Optimization::evaluate
// (optimization.cpp.base:26-34, non-finite F(x) is an error).
//
// x_i = m + sigma*y_i is recomputed from the stored y ("BDZ Matrix") with the reference's rounding
// (round(sigma*y) then round(m + .), CMAES.cpp.base:512), so X need not be materialised.
// One warp per sample; summation order = 32 lane-strided partials + xor butterfly, identical to the CPU oracle
// (oracle/okcma.c objective_one) => polynomial objectives are bit-identical to the oracle's.
// This file is compiled with --fmad=false.
#include "bayes.cuh"
#include "common.cuh"
#include "kernels.h"
#include "../../include/kcma.h"

namespace kc {

struct XRow {
  const double* y;     // row of Y (or of X when from_x)
  const double* mean;
  double ssigma;       // +-sigma
  bool from_x;
  __device__ __forceinline__ double operator()(int d) const {
    return from_x ? y[d] : __dadd_rn(mean[d], __dmul_rn(ssigma, y[d]));
  }
};

// PRIOR (Bayesian problems): the log-prior of the same row is summed from the values the objective loads, in the order of
// log_prior_row (lane d % 32 sums its variables ascending, then the butterfly), into *lp.
template <int OBJ, bool PRIOR = false>
__device__ __forceinline__ double eval_row(const XRow& x, int n, const double* __restrict__ coef, int lane, const PriorCols* pr = nullptr,
                                           double* lp = nullptr) {
  double p = 0.0, p2 = 0.0, q = 0.0;
  auto tap = [&](int d, double v) {
    if constexpr (PRIOR) q = q + prior_term_c(pr->type[d], pr->a[d], pr->b[d], pr->c[d], v);
  };
  // The lane-strided partial sums are accumulated in index order (the canonical order shared with the oracle); the loads of
  // 8 consecutive terms are issued together so that every warp keeps 2 KB in flight (HBM latency x bandwidth).
  if (OBJ == KCMA_OBJ_NEG_SPHERE || OBJ == KCMA_OBJ_NEG_SUMSQ) {
    int i = lane;
    for (; i + 32 * 7 < n; i += 32 * 8) {
      double v[8];
#pragma unroll
      for (int k = 0; k < 8; k++) v[k] = x(i + 32 * k);
#pragma unroll
      for (int k = 0; k < 8; k++) { p = __dadd_rn(p, __dmul_rn(v[k], v[k])); tap(i + 32 * k, v[k]); }
    }
    for (; i < n; i += 32) { const double v = x(i); p = __dadd_rn(p, __dmul_rn(v, v)); tap(i, v); }
    const double s = warp_sum_butterfly(p);
    if constexpr (PRIOR) *lp = warp_sum_butterfly(q);
    return OBJ == KCMA_OBJ_NEG_SPHERE ? __dmul_rn(-0.5, s) : -s;
  } else if (OBJ == KCMA_OBJ_NEG_ELLIPSOID) {
    int i = lane;
    for (; i + 32 * 7 < n; i += 32 * 8) {
      double v[8], c[8];
#pragma unroll
      for (int k = 0; k < 8; k++) { v[k] = x(i + 32 * k); c[k] = coef[i + 32 * k]; }
#pragma unroll
      for (int k = 0; k < 8; k++) { p = __dadd_rn(p, __dmul_rn(c[k], __dmul_rn(v[k], v[k]))); tap(i + 32 * k, v[k]); }
    }
    for (; i < n; i += 32) { const double v = x(i); p = __dadd_rn(p, __dmul_rn(coef[i], __dmul_rn(v, v))); tap(i, v); }
    if constexpr (PRIOR) *lp = warp_sum_butterfly(q);
    return -warp_sum_butterfly(p);
  } else if (OBJ == KCMA_OBJ_NEG_ROSENBROCK) {
    int i = lane;
    for (; i + 1 < n; i += 32) {
      const double xi = x(i), xn = x(i + 1);
      tap(i, xi);
      const double a = __dmul_rn(xi, xi);
      const double b = __dsub_rn(xn, a);
      const double c = __dmul_rn(b, b);
      const double d = __dmul_rn(100.0, c);
      const double e = __dsub_rn(1.0, xi);
      const double f = __dmul_rn(e, e);
      p = __dadd_rn(p, __dadd_rn(d, f));
    }
    if constexpr (PRIOR) {
      if (i < n) tap(i, x(i));   // the last variable, which only enters as x_{i+1}
      *lp = warp_sum_butterfly(q);
    }
    return -warp_sum_butterfly(p);
  } else if (OBJ == KCMA_OBJ_NEG_ACKLEY) {
    const double c = 2.0 * 3.14159265358979323846;
    for (int i = lane; i < n; i += 32) {
      const double v = x(i);
      p = __dadd_rn(p, __dmul_rn(v, v));
      p2 = __dadd_rn(p2, cos(__dmul_rn(c, v)));
      tap(i, v);
    }
    if constexpr (PRIOR) *lp = warp_sum_butterfly(q);
    const double sum1 = warp_sum_butterfly(p) / (double)n;
    const double sum2 = warp_sum_butterfly(p2) / (double)n;
    const double r1 = __dmul_rn(20.0, exp(__dmul_rn(-0.2, sqrt(sum1))));
    const double r2 = exp(sum2);
    return __dsub_rn(__dsub_rn(__dadd_rn(r1, r2), 20.0), exp(1.0));
  } else {  // KCMA_OBJ_NEG_SPHERE_SIN2
    for (int i = lane; i < n; i += 32) {
      const double v = x(i);
      const double s = sin(v);
      p = __dadd_rn(p, __dadd_rn(__dmul_rn(v, v), __dmul_rn(s, s)));
      tap(i, v);
    }
    if constexpr (PRIOR) *lp = warp_sum_butterfly(q);
    return -warp_sum_butterfly(p);
  }
}

// Samples are in LOCAL order: sample s uses z-row s (or s/2 when mirrored, odd s with -sigma).
template <int OBJ>
__global__ void __launch_bounds__(256)
objective_kernel(const double* __restrict__ Y, int ldy, long long samples, int n, int mirrored, int from_x,
                 const double* __restrict__ mean, DevScalars* __restrict__ sc, const double* __restrict__ coef,
                 double* __restrict__ f, int evaluate) {
  const int lane = threadIdx.x & 31;
  const long long warp = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  const double sigma = sc->sigma;
  for (long long s = warp; s < samples; s += nwarps) {
    XRow x;
    x.from_x = from_x != 0;
    x.mean = mean;
    if (from_x) { x.y = Y + (size_t)s * ldy; x.ssigma = sigma; }
    else if (mirrored) { x.y = Y + (size_t)(s >> 1) * ldy; x.ssigma = (s & 1) ? -sigma : sigma; }
    else { x.y = Y + (size_t)s * ldy; x.ssigma = sigma; }
    if (evaluate) {
      const double v = eval_row<OBJ>(x, n, coef, lane);
      if (lane == 0) {
        f[s] = v;
        if (!isfinite(v)) atomicExch(&sc->nonfinite, 1);
      }
    }
  }
}

// ---- Bayesian problems (include/kcma.h) ----------------------------------------------------------------------------------------
// F from the log-prior p and the log-likelihood l of global sample `sample`: -inf outside the prior's support whatever l is; else
// p + l, where a NaN or +inf sets the error flag and names the sample.
__device__ __forceinline__ double log_posterior(double p, double l, unsigned long long sample, DevScalars* sc) {
  if (p == -INFINITY) return -INFINITY;
  const double f = p + l;
  if (f != f || f == INFINITY) {
    atomicExch(&sc->nonfinite, 1);
    atomicMax(&sc->post_err, ~((sample << 3) | (unsigned long long)(f == INFINITY ? kPostPosInf : kPostNaN)));
  }
  return f;
}

__global__ void prior_constants_kernel(int n, const int* __restrict__ type, const double* __restrict__ a, const double* __restrict__ b,
                                       double* __restrict__ c) {
  const int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d < n) c[d] = prior_const(type[d], a[d], b[d]);
}

// objective_kernel for a built-in log-likelihood: the log-prior of the same reconstructed x = m +- sigma y is reduced in the one pass
// over Y, then F = log_posterior (X is never materialised for it). Without a bound the prior's loads and terms take 78 registers
// (3 CTAs per SM, against 6 for objective_kernel); 4 CTAs per SM cost 56 bytes of stack and measured 0.250 instead of 0.281 ms at
// N = 1000, lambda = 65536 (profiles/r05_bench_cmaes_bayesian_launch_bounds.log); 5 or 6 spill more.
template <int OBJ>
__global__ void __launch_bounds__(256, 4)
posterior_objective_kernel(const double* __restrict__ Y, int ldy, long long samples, int n, int mirrored, int from_x,
                           const double* __restrict__ mean, DevScalars* __restrict__ sc, const double* __restrict__ coef, PriorCols pr,
                           double* __restrict__ f, unsigned long long row0) {
  const int lane = threadIdx.x & 31;
  const long long warp = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  const double sigma = sc->sigma;
  for (long long s = warp; s < samples; s += nwarps) {
    XRow x;
    x.from_x = from_x != 0;
    x.mean = mean;
    if (from_x) { x.y = Y + (size_t)s * ldy; x.ssigma = sigma; }
    else if (mirrored) { x.y = Y + (size_t)(s >> 1) * ldy; x.ssigma = (s & 1) ? -sigma : sigma; }
    else { x.y = Y + (size_t)s * ldy; x.ssigma = sigma; }
    double lp;
    const double l = eval_row<OBJ, true>(x, n, coef, lane, &pr, &lp);
    if (lane == 0) f[s] = log_posterior(lp, l, row0 + (unsigned long long)s, sc);
  }
}

// The log-posterior of materialised rows (a host / device model or a computational model wrote its outputs): one warp per row. The
// log-prior first; outside the support F = -inf and the model's outputs for the row are not read. Otherwise l is F[i] as the model
// wrote it (LIK = 0) or the sum of the M Bayesian/Reference terms (lane k sums j = k, k + 32, ... ascending, then the butterfly, as
// tm_reference_loglik_kernel); a bad model output is recorded like TMCMC's ref_err.
template <int LIK>
__global__ void __launch_bounds__(256)
posterior_rows_kernel(long long rows, int n, const double* __restrict__ X, int ldx, PriorCols pr, int m, long long ldm,
                      const double* __restrict__ G, const double* __restrict__ P, const double* __restrict__ D,
                      const double* __restrict__ DC, double* __restrict__ f, unsigned long long row0, DevScalars* __restrict__ sc) {
  const int lane = threadIdx.x & 31;
  const long long warp = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long i = warp; i < rows; i += nwarps) {
    const double* x = X + (size_t)i * ldx;
    double q = 0.0;
    for (int d = lane; d < n; d += 32) q = q + prior_term_c(pr.type[d], pr.a[d], pr.b[d], pr.c[d], x[d]);
    const double lp = warp_sum_butterfly(q);
    if (lp == -INFINITY) {
      if (lane == 0) f[i] = -INFINITY;
      continue;
    }
    double l;
    if (LIK == 0) {
      l = f[i];
    } else {
      const double* g = G + i * ldm;
      const double* p = LIK == KCMA_LIK_POISSON ? nullptr : P + i * ldm;
      double s = 0.0;
      int bad = 4;
      for (int j = lane; j < m; j += 32) s = s + reference_term<LIK>(g[j], p, j, __ldg(D + j), DC, bad);
      if (bad < 4) {
        atomicExch(&sc->nonfinite, 1);
        atomicMax(&sc->post_err, ~(((row0 + (unsigned long long)i) << 3) | (unsigned)bad));
      }
      l = warp_sum_butterfly(s);
    }
    if (lane == 0) f[i] = log_posterior(lp, l, row0 + (unsigned long long)i, sc);
  }
}

// dF/dx of the built-in objectives for every sample ("Evaluate With Gradients", CMAES.cpp.base:199-200,226-228: the
// reference reads sample["Gradient"] from the user model, examples/optimization/stochastic/_model/model.py:10-63).
// One warp per sample; same formulas as oracle/okcma.c objective_gradient_one.
__global__ void __launch_bounds__(256)
objective_gradient_kernel(int objective, const double* __restrict__ Y, int ldy, long long samples, int n, int mirrored, int from_x,
                          const double* __restrict__ mean, const DevScalars* __restrict__ sc, const double* __restrict__ coef,
                          double* __restrict__ G, int ldg) {
  const int lane = threadIdx.x & 31;
  const long long warp = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  const double sigma = sc->sigma;
  for (long long s = warp; s < samples; s += nwarps) {
    XRow x;
    x.from_x = from_x != 0;
    x.mean = mean;
    if (from_x) { x.y = Y + (size_t)s * ldy; x.ssigma = sigma; }
    else if (mirrored) { x.y = Y + (size_t)(s >> 1) * ldy; x.ssigma = (s & 1) ? -sigma : sigma; }
    else { x.y = Y + (size_t)s * ldy; x.ssigma = sigma; }
    double* g = G + (size_t)s * ldg;
    double e1 = 0.0, e2 = 0.0, r = 0.0;
    const double c = 2.0 * 3.14159265358979323846;
    if (objective == KCMA_OBJ_NEG_ACKLEY) {
      double s1 = 0.0, s2 = 0.0;
      for (int i = lane; i < n; i += 32) { const double v = x(i); s1 += v * v; s2 += cos(c * v); }
      s1 = warp_sum_butterfly(s1); s2 = warp_sum_butterfly(s2);
      r = sqrt(s1 / (double)n);
      e1 = 20.0 * exp(-0.2 * r); e2 = exp(s2 / (double)n);
    }
    for (int i = lane; i < n; i += 32) {
      const double v = x(i);
      double d;
      switch (objective) {
        case KCMA_OBJ_NEG_SPHERE: d = -v; break;
        case KCMA_OBJ_NEG_SUMSQ: d = -2.0 * v; break;
        case KCMA_OBJ_NEG_ELLIPSOID: d = -2.0 * coef[i] * v; break;
        case KCMA_OBJ_NEG_ROSENBROCK: {
          double a = 0.0;
          if (i + 1 < n) a += -400.0 * v * (x(i + 1) - v * v) - 2.0 * (1.0 - v);
          if (i > 0) { const double w = x(i - 1); a += 200.0 * (v - w * w); }
          d = -a;
          break;
        }
        case KCMA_OBJ_NEG_ACKLEY: d = (r > 0.0 ? e1 * (-0.2) * v / ((double)n * r) : 0.0) + e2 * (-c * sin(c * v)) / (double)n; break;
        default: d = -(2.0 * v + 2.0 * sin(v) * cos(v)); break;   // KCMA_OBJ_NEG_SPHERE_SIN2
      }
      g[i] = d;
    }
  }
}

// isSampleFeasible (optimizer.cpp.base:5-14) for every sample + optional materialisation of X ("Sample Population").
__global__ void __launch_bounds__(256)
feasibility_kernel(const double* __restrict__ Y, int ldy, long long samples, int n, int mirrored,
                   const double* __restrict__ mean, const DevScalars* __restrict__ sc, const double* __restrict__ lower,
                   const double* __restrict__ upper, unsigned char* __restrict__ infeasible, double* __restrict__ X, int ldx,
                   const int* __restrict__ row_list) {
  const int lane = threadIdx.x & 31;
  const long long warp = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  const double sigma = sc->sigma;
  for (long long li = warp; li < samples; li += nwarps) {
    const long long s = row_list ? row_list[li] : li;
    const double* y = Y + (size_t)(mirrored ? (s >> 1) : s) * ldy;
    const double ss = (mirrored && (s & 1)) ? -sigma : sigma;
    bool bad = false;
    for (int d = lane; d < n; d += 32) {
      const double v = __dadd_rn(mean[d], __dmul_rn(ss, y[d]));
      if (X) X[(size_t)s * ldx + d] = v;
      if (lower) bad |= !isfinite(v) || v < lower[d] || v > upper[d];
    }
    if (infeasible) {
      const unsigned m = __ballot_sync(0xffffffffu, bad);
      if (lane == 0) infeasible[s] = m ? 1 : 0;
    }
  }
}

// Built-in constraint family KCMA_CON_HALFSPACE: g_c(x) = -(x_c - shift_c); G is [n_con][ldg].
__global__ void __launch_bounds__(256)
constraints_halfspace_kernel(const double* __restrict__ Y, int ldy, long long samples, int n, const double* __restrict__ mean,
                             DevScalars* __restrict__ sc, const double* __restrict__ shift, int n_con,
                             double* __restrict__ G, long long ldg, const int* __restrict__ row_list) {
  const double sigma = sc->sigma;
  const long long total = samples * n_con;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const long long li = idx / n_con;
    const int c = (int)(idx - li * n_con);
    const long long s = row_list ? row_list[li] : li;
    const int d = c % n;
    const double x = __dadd_rn(mean[d], __dmul_rn(sigma, Y[(size_t)s * ldy + d]));
    const double g = -__dsub_rn(x, shift[c]);
    if (!isfinite(g)) atomicExch(&sc->nonfinite, 1);
    G[(size_t)c * ldg + s] = g;
  }
}

static int grid_for_warps(long long warps, int num_sms) {
  long long blocks = (warps + 7) / 8;
  const long long cap = (long long)num_sms * 8;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

int launch_objective(cudaStream_t st, int objective, const double* Y, int ldy, long long samples, int n, int mirrored,
                     int from_x, const double* mean, DevScalars* sc, const double* coef, double* f, int num_sms) {
  if (samples <= 0) return 0;
  const int grid = grid_for_warps(samples, num_sms);
#define LAUNCH(ID) objective_kernel<ID><<<grid, 256, 0, st>>>(Y, ldy, samples, n, mirrored, from_x, mean, sc, coef, f, 1)
  switch (objective) {
    case KCMA_OBJ_NEG_SPHERE: LAUNCH(KCMA_OBJ_NEG_SPHERE); break;
    case KCMA_OBJ_NEG_ROSENBROCK: LAUNCH(KCMA_OBJ_NEG_ROSENBROCK); break;
    case KCMA_OBJ_NEG_ACKLEY: LAUNCH(KCMA_OBJ_NEG_ACKLEY); break;
    case KCMA_OBJ_NEG_ELLIPSOID: LAUNCH(KCMA_OBJ_NEG_ELLIPSOID); break;
    case KCMA_OBJ_NEG_SUMSQ: LAUNCH(KCMA_OBJ_NEG_SUMSQ); break;
    case KCMA_OBJ_NEG_SPHERE_SIN2: LAUNCH(KCMA_OBJ_NEG_SPHERE_SIN2); break;
    default: return 1;
  }
#undef LAUNCH
  return 0;
}

void launch_prior_constants(cudaStream_t st, int n, const int* type, const double* a, const double* b, double* c) {
  prior_constants_kernel<<<(n + 127) / 128, 128, 0, st>>>(n, type, a, b, c);
}

int launch_posterior_objective(cudaStream_t st, int objective, const double* Y, int ldy, long long samples, int n, int mirrored, int from_x,
                               const double* mean, DevScalars* sc, const double* coef, const PriorCols& pr, double* f,
                               unsigned long long row0, int num_sms) {
  if (samples <= 0) return 0;
  const int grid = grid_for_warps(samples, num_sms);
#define LAUNCH(ID) posterior_objective_kernel<ID><<<grid, 256, 0, st>>>(Y, ldy, samples, n, mirrored, from_x, mean, sc, coef, pr, f, row0)
  switch (objective) {
    case KCMA_OBJ_NEG_SPHERE: LAUNCH(KCMA_OBJ_NEG_SPHERE); break;
    case KCMA_OBJ_NEG_ROSENBROCK: LAUNCH(KCMA_OBJ_NEG_ROSENBROCK); break;
    case KCMA_OBJ_NEG_ACKLEY: LAUNCH(KCMA_OBJ_NEG_ACKLEY); break;
    case KCMA_OBJ_NEG_ELLIPSOID: LAUNCH(KCMA_OBJ_NEG_ELLIPSOID); break;
    case KCMA_OBJ_NEG_SUMSQ: LAUNCH(KCMA_OBJ_NEG_SUMSQ); break;
    case KCMA_OBJ_NEG_SPHERE_SIN2: LAUNCH(KCMA_OBJ_NEG_SPHERE_SIN2); break;
    default: return 1;
  }
#undef LAUNCH
  return 0;
}

void launch_posterior_rows(cudaStream_t st, int lik, long long rows, int n, const double* X, int ldx, const PriorCols& pr, int m,
                           long long ldm, const double* G, const double* P, const double* D, const double* DC, double* f,
                           unsigned long long row0, DevScalars* sc, int num_sms) {
  if (rows <= 0) return;
  const int grid = grid_for_warps(rows, num_sms);
#define LAUNCH(LIK) posterior_rows_kernel<LIK><<<grid, 256, 0, st>>>(rows, n, X, ldx, pr, m, ldm, G, P, D, DC, f, row0, sc)
  switch (lik) {
    case KCMA_LIK_NORMAL: LAUNCH(KCMA_LIK_NORMAL); break;
    case KCMA_LIK_POSITIVE_NORMAL: LAUNCH(KCMA_LIK_POSITIVE_NORMAL); break;
    case KCMA_LIK_STUDENT_T: LAUNCH(KCMA_LIK_STUDENT_T); break;
    case KCMA_LIK_POISSON: LAUNCH(KCMA_LIK_POISSON); break;
    default: LAUNCH(0); break;
  }
#undef LAUNCH
}

void launch_objective_gradient(cudaStream_t st, int objective, const double* Y, int ldy, long long samples, int n, int mirrored, int from_x,
                               const double* mean, const DevScalars* sc, const double* coef, double* G, int ldg, int num_sms) {
  if (samples <= 0) return;
  objective_gradient_kernel<<<grid_for_warps(samples, num_sms), 256, 0, st>>>(objective, Y, ldy, samples, n, mirrored, from_x, mean, sc, coef, G, ldg);
}

void launch_feasibility(cudaStream_t st, const double* Y, int ldy, long long samples, int n, int mirrored, const double* mean,
                        const DevScalars* sc, const double* lower, const double* upper, unsigned char* infeasible,
                        double* X, int ldx, const int* row_list, int num_sms) {
  if (samples <= 0) return;
  feasibility_kernel<<<grid_for_warps(samples, num_sms), 256, 0, st>>>(Y, ldy, samples, n, mirrored, mean, sc, lower, upper,
                                                                       infeasible, X, ldx, row_list);
}

void launch_constraints_halfspace(cudaStream_t st, const double* Y, int ldy, long long samples, int n, const double* mean,
                                  DevScalars* sc, const double* shift, int n_con, double* G, long long ldg,
                                  const int* row_list, int num_sms) {
  if (samples <= 0 || n_con <= 0) return;
  long long blocks = (samples * n_con + 255) / 256;
  if (blocks > (long long)num_sms * 8) blocks = (long long)num_sms * 8;
  constraints_halfspace_kernel<<<(int)blocks, 256, 0, st>>>(Y, ldy, samples, n, mean, sc, shift, n_con, G, ldg, row_list);
}

}  // namespace kc
