// mocma.cu — multi-objective CMA-ES generation loop on the device (include/kmocma.h): the sibling solver "Optimizer/MOCMAES"
// (MOCMAES.cpp.base) on the conventions of the CMA-ES path. One CTA per individual: every individual carries its own covariance
// matrix, evolution path, step size and success probability, so the natural unit of parallelism is (individual, matrix entry).
//
//   kmocma_ask    mo_sample_kernel     parent index (Philox), Cholesky factor of the parent's covariance in shared memory (column by
//                                      column, every entry's sum in ascending index like the oracle), z (Philox + Box-Muller),
//                                      x = parent + sigma L z, redraw until inside the bounds, inherit C / sigma / path / p_succ
//   kmocma_eval   mo_objective_kernel  built-in models (one thread per sample, the reference's summation order) or the host conduit
//   kmocma_tell   mo_sort_kernel       sortSampleIndices :232-342 on the 2 lambda merged values: non-dominance levels, then
//                                      contributing hypervolume inside a level (one CTA; the inner maxima in parallel)
//                 mo_update_kernel     success probability, evolution path, rank-1 covariance update, step size :356-391
//                 mo_parents_kernel    the mu best of (offspring + previous offspring) become the parents :393-417
//                 mo_stats_kernel      per-objective bests, standard deviations, non-dominated flags :420-481
//                 (host)               archive of non-dominated samples ("Sample Collection", :483-519): grows without bound, result
//                                      bookkeeping — kept on the host from the lambda x (n + K) values copied back per generation
// Compiled with --fmad=false: the arithmetic rounds like the reference's scalar code and like oracle/omocma.c (bit-identical given
// the same z; the device's log / sincospi / exp may differ from libm in the last bit, so device vs oracle is compared to 1e-9 over a free run).
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/kmocma.h"
#include "common.cuh"
#include "handle.cuh"

namespace {

using namespace kc;

__device__ __forceinline__ void mo_philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t out[4]) {
#pragma unroll
  for (int r = 0; r < 10; r++) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
__device__ __forceinline__ double mo_unit(uint32_t lo, uint32_t hi) {
  const unsigned long long v = ((unsigned long long)hi << 32) | lo;
  return (double)(v >> 12) * 0x1.0p-52 + 0x1.0p-53;
}
__device__ __forceinline__ void mo_block(unsigned long long seed, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t r[4]) {
  mo_philox(c0, c1, c2, c3, (uint32_t)seed, (uint32_t)(seed >> 32) ^ 0x4d4f434du, r);
}

struct MoScalars {
  unsigned long long nondom;
  int chol_failed, no_feasible, nonfinite, pad;
};

// sampleSingle :191-230. One CTA per offspring; dynamic shared memory: L (n x n) | z (n + 1) | x (n).
__global__ void __launch_bounds__(128)
mo_sample_kernel(int n, int lambda, int mu, unsigned long long seed, unsigned generation, const double* __restrict__ lower,
                 const double* __restrict__ upper, const double* __restrict__ pX, const double* __restrict__ pS, const double* __restrict__ pC,
                 const double* __restrict__ pP, const double* __restrict__ pPS, double* __restrict__ cX, double* __restrict__ cS,
                 double* __restrict__ cC, double* __restrict__ cP, double* __restrict__ cPS, double* __restrict__ parent_index,
                 MoScalars* __restrict__ sc) {
  extern __shared__ double sm[];
  double* L = sm;
  double* z = sm + (size_t)n * n;
  double* x = z + n + 1;
  __shared__ int s_parent;
  const int i = blockIdx.x, tid = threadIdx.x;
  if (tid == 0) {
    int p = i;
    if (mu != lambda) {
      uint32_t r[4];
      mo_block(seed, 0u, (uint32_t)i, 0u, generation, r);
      const double u = mo_unit(r[0], r[1]);
      const unsigned long long nd = sc->nondom;
      p = (int)floor((double)((unsigned long long)mu < nd ? (unsigned long long)mu : nd) * u);
    }
    s_parent = p;
    parent_index[i] = (double)p;
  }
  __syncthreads();
  const int p = s_parent;
  const double* A = pC + (size_t)p * n * n;
  for (int e = tid; e < n * n; e += blockDim.x) L[e] = 0.0;
  __syncthreads();
  // Cholesky, column by column; entry (r, j): A[r][j] - sum_{k < j} L[r][k] L[j][k] in ascending k (the oracle's order)
  for (int j = 0; j < n; j++) {
    if (tid == 0) {
      double s = A[(size_t)j * n + j];
      for (int k = 0; k < j; k++) s -= L[j * n + k] * L[j * n + k];
      if (!(s > 0.0)) { sc->chol_failed = 1; s = 1.0; }
      L[j * n + j] = sqrt(s);
    }
    __syncthreads();
    const double ljj = L[j * n + j];
    for (int r = j + 1 + tid; r < n; r += blockDim.x) {
      double s = A[(size_t)r * n + j];
      for (int k = 0; k < j; k++) s -= L[r * n + k] * L[j * n + k];
      L[r * n + j] = s / ljj;
    }
    __syncthreads();
  }
  const double sig = pS[p];
  for (unsigned attempt = 0;; attempt++) {
    for (int pr = tid; 2 * pr < n; pr += blockDim.x) {
      uint32_t r[4];
      mo_block(seed, (1u << 20) + (uint32_t)pr, (uint32_t)i, attempt, generation, r);
      const double u1 = mo_unit(r[0], r[1]), u2 = mo_unit(r[2], r[3]);
      const double rad = sqrt(-2.0 * log(u1));
      double s, c;
      sincospi(2.0 * u2, &s, &c);
      z[2 * pr] = rad * c; z[2 * pr + 1] = rad * s;
    }
    __syncthreads();
    int ok = 1;
    for (int d = tid; d < n; d += blockDim.x) {
      double y = 0.0;
      for (int e = 0; e < d; e++) y += (L[d * n + e] * sig) * z[e];
      y += z[d] * (L[d * n + d] * sig);
      const double xd = y + pX[(size_t)p * n + d];
      x[d] = xd;
      if (xd < lower[d] || xd > upper[d]) ok = 0;
    }
    if (__syncthreads_and(ok)) break;
    if (attempt > 1000000u) { if (tid == 0) sc->no_feasible = 1; break; }
  }
  for (int d = tid; d < n; d += blockDim.x) { cX[(size_t)i * n + d] = x[d]; cP[(size_t)i * n + d] = pP[(size_t)p * n + d]; }
  for (int e = tid; e < n * n; e += blockDim.x) cC[(size_t)i * n * n + e] = A[e];
  if (tid == 0) { cS[i] = sig; cPS[i] = pPS[p]; }
}

// examples/optimization/multiobjective/_model/model.py:5-38, one thread per sample (the reference's loops)
__global__ void mo_objective_kernel(int id, int n, int lambda, int K, const double* __restrict__ X, double* __restrict__ F, MoScalars* __restrict__ sc) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= lambda) return;
  const double* x = X + (size_t)i * n;
  double r1 = 0., r2 = 0., r3 = 0.;
  for (int d = 0; d + 1 < n; d++) r1 += 100 * ((x[d + 1] - x[d] * x[d]) * (x[d + 1] - x[d] * x[d])) + (1 - x[d]) * (1 - x[d]);
  for (int d = 0; d < n; d++) r2 += x[d] * x[d];
  F[(size_t)i * K] = -r1; F[(size_t)i * K + 1] = -r2;
  if (id == KMOCMA_OBJ_NEG_ROSENBROCK_AND_TWO_SPHERES) {
    for (int d = 0; d < n; d++) r3 += (x[d] - 2) * (x[d] - 2);
    F[(size_t)i * K + 2] = -r3;
  }
  for (int k = 0; k < K; k++) if (!isfinite(F[(size_t)i * K + k])) sc->nonfinite = 1;
}
__global__ void mo_check_finite_kernel(const double* __restrict__ F, int count, MoScalars* __restrict__ sc) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count && !isfinite(F[i])) sc->nonfinite = 1;
}

// sortSampleIndices :232-342. values = [current | previous] (n2 x K, larger is better). One CTA; shared: rank, max_nb, list (int, n2 each),
// hv (double, n2). sorted[i] = position of sample i in the order (worst first).
__global__ void __launch_bounds__(1024)
mo_sort_kernel(const double* __restrict__ Fcur, const double* __restrict__ Fprev, int lambda, int K, int* __restrict__ sorted) {
  extern __shared__ double smd[];
  const int n2 = 2 * lambda, tid = threadIdx.x;
  double* hv = smd;
  int* rank = (int*)(smd + n2);
  int* max_nb = rank + n2;
  int* list = max_nb + n2;
  __shared__ int s_min_max, s_min_rank, s_left, s_m;
  __shared__ double s_ref[KMOCMA_MAX_OBJECTIVES];
  auto val = [&](int i, int k) { return i < lambda ? Fcur[(size_t)i * K + k] : Fprev[(size_t)(i - lambda) * K + k]; };
  for (int i = tid; i < n2; i += blockDim.x) { rank[i] = 0; sorted[i] = -1; }
  if (tid == 0) { s_min_rank = n2; s_left = n2; }
  __syncthreads();
  for (int r = n2; r >= 1 && s_left > 0; --r) {
    if (tid == 0) s_min_max = K;
    __syncthreads();
    for (int i = tid; i < n2; i += blockDim.x) {
      int mnb = 0;
      if (rank[i] == 0) {
        for (int j = 0; j < n2; ++j)
          if (i != j && rank[j] == 0) {
            int nb = 0;
            for (int k = 0; k < K; ++k)
              if (val(i, k) < val(j, k)) nb++;
            if (nb > mnb) mnb = nb;
          }
        atomicMin(&s_min_max, mnb);
      }
      max_nb[i] = mnb;
    }
    __syncthreads();
    int assigned = 0;
    for (int i = tid; i < n2; i += blockDim.x)
      if (rank[i] == 0 && max_nb[i] == s_min_max) { rank[i] = r; assigned++; }
    if (assigned) { atomicMin(&s_min_rank, r); atomicSub(&s_left, assigned); }
    __syncthreads();
  }
  const int min_rank = s_min_rank, max_rank = n2 - min_rank;
  for (int i = tid; i < n2; i += blockDim.x) rank[i] -= min_rank;
  if (tid < K) {
    double ref = INFINITY;
    for (int i = 0; i < n2; ++i) { const double v = val(i, tid); if (v < ref) ref = v; }
    s_ref[tid] = ref;
  }
  __syncthreads();
  int order = 0;
  for (int r = 0; r <= max_rank; ++r) {
    for (;;) {
      if (tid == 0) {
        int m = 0;
        for (int i = 0; i < n2; ++i)
          if (rank[i] == r && sorted[i] == -1) list[m++] = i;
        s_m = m;
      }
      __syncthreads();
      const int m = s_m;
      if (m == 0) break;
      for (int a = tid; a < m; a += blockDim.x) {
        double h = 0.0;
        for (int k = 0; k < K; ++k) {
          double ub = -INFINITY;
          for (int b = 0; b < m; ++b)
            if (a != b) { const double v = val(list[b], k); if (v > ub) ub = v; }
          h += (ub - s_ref[k]);
        }
        hv[a] = h;
      }
      __syncthreads();
      if (tid == 0) {
        int next = list[0];
        double best = hv[0];
        for (int a = 1; a < m; ++a)
          if (hv[a] > best) { best = hv[a]; next = list[a]; }
        sorted[next] = order;
      }
      order++;
      __syncthreads();
    }
    __syncthreads();
  }
}

// updateDistribution :356-391, one CTA per offspring
__global__ void __launch_bounds__(128)
mo_update_kernel(int n, int lambda, int mu, double cc, double ccov, double cp, double target, const int* __restrict__ sorted,
                 const double* __restrict__ parent_index, const double* __restrict__ pX, const double* __restrict__ cX, double* __restrict__ cS,
                 double* __restrict__ cC, double* __restrict__ cP, double* __restrict__ cPS) {
  __shared__ double s_len, s_ps;
  extern __shared__ double pcs[];
  const int i = blockIdx.x, tid = threadIdx.x, n2 = 2 * lambda;
  double* C = cC + (size_t)i * n * n;
  double* pc = cP + (size_t)i * n;
  const double path_factor = sqrt(cc * (2. - cc));
  const double dd = 1.0 + 2.0 * fmax(0.0, sqrt(((double)mu - 1.) / ((double)n + 1.)) - 1.0) + cc;
  const double chi_n = sqrt((double)n) * (1. - 1. / (4. * (double)n) + 1. / (21. * (double)n * (double)n));
  if (tid == 0) {
    double ps = cPS[i] * (1. - cp);
    if (sorted[i] >= n2 - mu) ps += cp;
    ps = fmin(ps, 1.0);
    cPS[i] = ps; s_ps = ps;
  }
  const double* parent = pX + (size_t)((int)parent_index[i]) * n;
  const double sig = cS[i];
  for (int d = tid; d < n; d += blockDim.x) {
    double v = (1. - cc) * pc[d];
    v += path_factor / sqrt(C[(size_t)d * n + d]) * (cX[(size_t)i * n + d] - parent[d]) / sig;
    pc[d] = v; pcs[d] = v;
  }
  __syncthreads();
  if (tid == 0) {
    double len = 0.;
    for (int d = 0; d < n; ++d) len += pcs[d] * pcs[d];
    s_len = sqrt(len);
  }
  __syncthreads();
  const bool extra = s_ps >= target;
  for (int e = tid; e < n * n; e += blockDim.x) {
    const int d = e / n, f = e - d * n;
    double c = (1. - ccov) * C[e] + ccov * pcs[d] * pcs[f];
    if (extra) c += ccov * path_factor * path_factor * c;
    C[e] = c;
  }
  if (tid == 0) cS[i] = sig * exp(cc / dd * (s_len / chi_n - 1.0));
}

// parents update :393-417, one CTA per merged sample
__global__ void __launch_bounds__(128)
mo_parents_kernel(int n, int lambda, int mu, const int* __restrict__ sorted, const double* __restrict__ cX, const double* __restrict__ cS,
                  const double* __restrict__ cC, const double* __restrict__ cP, const double* __restrict__ cPS, const double* __restrict__ vX,
                  const double* __restrict__ vS, const double* __restrict__ vC, const double* __restrict__ vP, const double* __restrict__ vPS,
                  double* __restrict__ pX, double* __restrict__ pS, double* __restrict__ pC, double* __restrict__ pP, double* __restrict__ pPS) {
  const int i = blockIdx.x, tid = threadIdx.x, n2 = 2 * lambda;
  if (sorted[i] < n2 - mu) return;
  const int pidx = n2 - sorted[i] - 1;
  const bool cur = i < lambda;
  const int s = cur ? i : i - lambda;
  const double *X = cur ? cX : vX, *S = cur ? cS : vS, *C = cur ? cC : vC, *P = cur ? cP : vP, *PS = cur ? cPS : vPS;
  for (int d = tid; d < n; d += blockDim.x) { pX[(size_t)pidx * n + d] = X[(size_t)s * n + d]; pP[(size_t)pidx * n + d] = P[(size_t)s * n + d]; }
  for (int e = tid; e < n * n; e += blockDim.x) pC[(size_t)pidx * n * n + e] = C[(size_t)s * n * n + e];
  if (tid == 0) { pS[pidx] = S[s]; pPS[pidx] = PS[s]; }
}

// updateStatistics :420-481 (the archive merge :483-519 runs on the host). One CTA.
__global__ void __launch_bounds__(256)
mo_stats_kernel(int n, int lambda, int K, const double* __restrict__ F, const double* __restrict__ cX, const double* __restrict__ cS,
                const double* __restrict__ cC, double* __restrict__ best_ever, double* __restrict__ best_ever_x, double* __restrict__ prev_best,
                double* __restrict__ prev_best_x, double* __restrict__ cur_best, double* __restrict__ cur_best_x, double* __restrict__ val_diff,
                double* __restrict__ var_diff, double* __restrict__ min_sd, double* __restrict__ max_sd, unsigned char* __restrict__ nondom_flag,
                MoScalars* __restrict__ sc) {
  const int tid = threadIdx.x;
  __shared__ int s_count;
  if (tid == 0) s_count = 0;
  if (tid < K) {
    const int k = tid;
    prev_best[k] = cur_best[k];
    for (int d = 0; d < n; d++) prev_best_x[(size_t)k * n + d] = cur_best_x[(size_t)k * n + d];
    double cb = -INFINITY;
    for (int i = 0; i < lambda; ++i)
      if (F[(size_t)i * K + k] > cb) {
        cb = F[(size_t)i * K + k];
        double l2 = 0.;
        for (int d = 0; d < n; ++d) {
          const double xv = cX[(size_t)i * n + d];
          cur_best_x[(size_t)k * n + d] = xv;
          const double df = prev_best_x[(size_t)k * n + d] - xv;
          l2 += df * df;     // std::pow(x, 2.) is x * x
        }
        val_diff[k] = cb - prev_best[k];
        var_diff[k] = sqrt(l2);
      }
    cur_best[k] = cb;
    if (cb > best_ever[k]) {
      best_ever[k] = cb;
      for (int d = 0; d < n; d++) best_ever_x[(size_t)k * n + d] = cur_best_x[(size_t)k * n + d];
    }
  }
  __syncthreads();
  for (int i = tid; i < lambda; i += blockDim.x) {
    double mn = INFINITY, mx = -INFINITY;
    for (int d = 0; d < n; ++d) {   // :452-461 indexes _currentSigma by the dimension; restated as written, clamped to the array
      const double sdev = cS[d < lambda ? d : lambda - 1] * sqrt(cC[(size_t)i * n * n + (size_t)d * n + d]);
      if (sdev > mx) mx = sdev;
      if (sdev < mn) mn = sdev;
    }
    min_sd[i] = mn; max_sd[i] = mx;
    bool dominated = false;
    for (int j = 0; j < lambda && !dominated; ++j)
      if (j != i) {
        int nd = 0;
        for (int k = 0; k < K; ++k)
          if (F[(size_t)j * K + k] > F[(size_t)i * K + k]) nd++;
        if (nd == K) dominated = true;
      }
    nondom_flag[i] = dominated ? 0 : 1;
    if (!dominated) atomicAdd(&s_count, 1);
  }
  __syncthreads();
  if (tid == 0) sc->nondom = (unsigned long long)s_count;
}

}  // namespace

struct kmocma : Handle<kmocma, MoScalars> {
  kmocma_cfg cfg;
  int N = 0, lambda = 0, mu = 0, K = 0;
  uint64_t model_evals = 0;
  double cc = 0, ccov = 0, cp = 0, target = 0;
  double *dLower = nullptr, *dUpper = nullptr;
  double *dX[3] = {}, *dS[3] = {}, *dC[3] = {}, *dP[3] = {}, *dPS[3] = {};
  double *dF = nullptr, *dFprev = nullptr, *dParentIndex = nullptr;
  int* dSorted = nullptr;
  double *dBestEver = nullptr, *dBestEverX = nullptr, *dPrevBest = nullptr, *dPrevBestX = nullptr, *dCurBest = nullptr, *dCurBestX = nullptr,
         *dValDiff = nullptr, *dVarDiff = nullptr, *dMinSd = nullptr, *dMaxSd = nullptr;
  unsigned char* dFlag = nullptr;
  std::vector<double> coll_x, coll_f;   // archive of non-dominated samples (host)
  std::vector<double> hX, hF;
  double tc_min_value_diff = -INFINITY, tc_min_var_diff = -INFINITY, tc_min_sd = -INFINITY, tc_max_sd = INFINITY, tc_max_generations = 1e10,
         tc_max_model_evaluations = 1e9;
  kmocma_host_objective_fn host_obj = nullptr; void* host_obj_user = nullptr;
  bool have_inj_f = false;
};
enum { CUR = 0, PREV = 1, PAR = 2 };

namespace {
size_t sample_smem(int n) { return sizeof(double) * ((size_t)n * n + 2 * (size_t)n + 2); }
const HostScalar<kmocma> kHostScalars[] = {
    {"Evolution Path Adaption Strength", &kmocma::cc, false},
    {"Covariance Learning Rate", &kmocma::ccov, false},
    {"Termination Criteria/Min Value Difference Threshold", &kmocma::tc_min_value_diff, true},
    {"Termination Criteria/Min Variable Difference Threshold", &kmocma::tc_min_var_diff, true},
    {"Termination Criteria/Min Standard Deviation", &kmocma::tc_min_sd, true},
    {"Termination Criteria/Max Standard Deviation", &kmocma::tc_max_sd, true},
    {"Termination Criteria/Max Generations", &kmocma::tc_max_generations, true},
    {"Termination Criteria/Max Model Evaluations", &kmocma::tc_max_model_evaluations, true},
};
bool find_array(kmocma* h, const char* key, Array* r) {
  const size_t N = h->N, L = h->lambda, mu = h->mu, K = h->K;
  static const char* pop[3] = {"Current", "Previous", "Parent"};
  for (int s = 0; s < 3; s++) {
    const size_t rows = s == PAR ? mu : L;
    const std::string p = pop[s];
    if (p + " Sample Population" == key) { *r = dense(h->dX[s], rows * N); return true; }
    if (p + " Sigma" == key) { *r = dense(h->dS[s], rows); return true; }
    if (p + " Covariance Matrix" == key) { *r = dense(h->dC[s], rows * N * N); return true; }
    if (p + " Evolution Paths" == key) { *r = dense(h->dP[s], rows * N); return true; }
    if (p + " Success Probabilities" == key) { *r = dense(h->dPS[s], rows); return true; }
  }
#define A(KEY, ARR) if (!strcmp(key, KEY)) { *r = ARR; return true; }
  A("Current Values", dense(h->dF, L * K)) A("Previous Values", dense(h->dFprev, L * K)) A("Parent Index", dense(h->dParentIndex, L))
  A("Best Ever Values", dense(h->dBestEver, K)) A("Current Best Values", dense(h->dCurBest, K)) A("Previous Best Values", dense(h->dPrevBest, K))
  A("Best Ever Variables Vector", dense(h->dBestEverX, K * N)) A("Current Best Variables Vector", dense(h->dCurBestX, K * N))
  A("Current Best Value Differences", dense(h->dValDiff, K)) A("Current Best Variable Differences", dense(h->dVarDiff, K))
  A("Current Min Standard Deviations", dense(h->dMinSd, L)) A("Current Max Standard Deviations", dense(h->dMaxSd, L))
  A("Sorted Indices", dense(h->dSorted, 2 * L, Elem::i32))
#undef A
  if (!strcmp(key, "Sample Collection")) { *r = dense(h->coll_x.data(), h->coll_x.size()); r->host = true; return true; }
  if (!strcmp(key, "Sample Value Collection")) { *r = dense(h->coll_f.data(), h->coll_f.size()); r->host = true; return true; }
  return false;
}
}  // namespace

extern "C" {

void kmocma_cfg_defaults(kmocma_cfg* c) {
  memset(c, 0, sizeof(*c));
  c->abi_version = KMOCMA_ABI_VERSION;
  c->num_objectives = 2;
  c->evolution_path_adaption_strength = -1.0; c->covariance_learning_rate = -1.0;
  c->target_success_rate = 0.175; c->threshold_probability = 0.44; c->success_learning_rate = 0.08;
}

const char* kmocma_last_error(const kmocma_t* h) { return h ? h->err.c_str() : kmocma::create_err; }

void kmocma_destroy(kmocma_t* h) { delete h; }

// setInitialConfiguration :10-144
int kmocma_create(const kmocma_cfg* cfg, kmocma_t** out) {
  if (!cfg || !out) return fail<kmocma>(nullptr, "null argument");
  if (cfg->abi_version != KMOCMA_ABI_VERSION) return fail<kmocma>(nullptr, "kmocma_cfg ABI version mismatch");
  if (cfg->n < 1) return fail<kmocma>(nullptr, "no variables");
  if (cfg->num_objectives < 2 || cfg->num_objectives > KMOCMA_MAX_OBJECTIVES)
    return fail<kmocma>(nullptr, "Problem requires multiple objectives, 'Num Objectives' is set to %zu\n.", (size_t)cfg->num_objectives);
  const uint64_t N = cfg->n, K = cfg->num_objectives;
  uint64_t lambda = cfg->population_size, mu = cfg->mu_value;
  if (lambda == 0) lambda = (uint64_t)ceil(4. + floor(3. * log((double)N)));
  if (mu == 0) mu = (uint64_t)(lambda / 2.);
  if (mu > lambda) return fail<kmocma>(nullptr, "Number of parents ('Mu Value' %zu) must be smaller or equal with population size (%zu).\n", (size_t)mu, (size_t)lambda);
  if (cfg->success_learning_rate <= 0. || cfg->success_learning_rate > 1.)
    return fail<kmocma>(nullptr, "Invalid Global Success Learning Rate (%f), must be greater than 0.0 and less or equal to 1.0\n", cfg->success_learning_rate);
  if (cfg->target_success_rate <= 0. || cfg->target_success_rate > 1.)
    return fail<kmocma>(nullptr, "Invalid Target Success Rate (%f), must be greater than 0.0 and less or equal to 1.0\n", cfg->target_success_rate);
  if (sample_smem((int)N) > 200 * 1024) return fail<kmocma>(nullptr, "Optimizer/MOCMAES on the device holds one covariance factor per CTA in shared memory: n <= 158");
  if (2 * lambda * (sizeof(double) + 3 * sizeof(int)) > 200 * 1024) return fail<kmocma>(nullptr, "Optimizer/MOCMAES: the ranking of the 2 lambda merged samples runs in one CTA's shared memory: population size <= 5120");
  if (cfg->objective != KMOCMA_OBJ_EXTERNAL) {
    const uint64_t want = cfg->objective == KMOCMA_OBJ_NEG_ROSENBROCK_AND_TWO_SPHERES ? 3 : 2;
    if (cfg->objective != KMOCMA_OBJ_NEG_ROSENBROCK_AND_SPHERE && cfg->objective != KMOCMA_OBJ_NEG_ROSENBROCK_AND_TWO_SPHERES)
      return fail<kmocma>(nullptr, "unknown objective id %d", cfg->objective);
    if (K != want) return fail<kmocma>(nullptr, "the built-in objective has %zu objectives, 'Num Objectives' is %zu", (size_t)want, (size_t)K);
  }
  std::vector<double> lower(N), upper(N), sd(N);
  double trace = 0., min_sdev = INFINITY, max_sdev = -INFINITY;
  for (uint64_t i = 0; i < N; i++) {
    lower[i] = cfg->lower_bound ? cfg->lower_bound[i] : -INFINITY;
    upper[i] = cfg->upper_bound ? cfg->upper_bound[i] : INFINITY;
    const double iv = cfg->initial_value ? cfg->initial_value[i] : NAN;
    double s = cfg->initial_stddev ? cfg->initial_stddev[i] : NAN;
    if (!std::isfinite(iv) && (!std::isfinite(lower[i]) || !std::isfinite(upper[i])))
      return fail<kmocma>(nullptr, "Initial (Mean) Value of variable %zu not defined, and cannot be inferred because a variable bound is not finite.\n", (size_t)i);
    if (!std::isfinite(s)) {
      if (!std::isfinite(lower[i]) || !std::isfinite(upper[i]))
        return fail<kmocma>(nullptr, "Initial Standard Deviation of variable %zu not defined, and cannot be inferred because a variable bound is not finite.\n", (size_t)i);
      s = (upper[i] - lower[i]) * 0.3;
    }
    sd[i] = s;
    trace += s * s;
    if (s < min_sdev) min_sdev = s;
    if (s > max_sdev) max_sdev = s;
  }
  // (the configuration checks above come first, like the reference's; the device is needed from here on)
  if (open_device<kmocma>(cfg->device)) return 1;
  kmocma* h = new kmocma();
  h->cfg = *cfg;
  h->cfg.lower_bound = h->cfg.upper_bound = h->cfg.initial_value = h->cfg.initial_stddev = nullptr;
  h->N = (int)N; h->lambda = (int)lambda; h->mu = (int)mu; h->K = (int)K; h->device = cfg->device;
  h->cp = cfg->success_learning_rate; h->target = cfg->target_success_rate;
  h->cc = cfg->evolution_path_adaption_strength < 0. ? 2. / ((double)N + 2.) : cfg->evolution_path_adaption_strength;
  h->ccov = cfg->covariance_learning_rate < 0. ? 2. / ((double)N * (double)N + 6.) : cfg->covariance_learning_rate;
  CREATE_OK(h, cudaFuncSetAttribute(mo_sample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sample_smem((int)N)));
  CREATE_OK(h, cudaFuncSetAttribute(mo_sort_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(2 * lambda * (sizeof(double) + 3 * sizeof(int)))));
  const uint64_t rows[3] = {lambda, lambda, mu};
  for (int s = 0; s < 3; s++) {
    CREATE_OK(h, alloc(h->mem, &h->dX[s], rows[s] * N)); CREATE_OK(h, alloc(h->mem, &h->dS[s], rows[s])); CREATE_OK(h, alloc(h->mem, &h->dC[s], rows[s] * N * N));
    CREATE_OK(h, alloc(h->mem, &h->dP[s], rows[s] * N)); CREATE_OK(h, alloc(h->mem, &h->dPS[s], rows[s]));
  }
  CREATE_OK(h, alloc(h->mem, &h->dLower, N)); CREATE_OK(h, alloc(h->mem, &h->dUpper, N));
  CREATE_OK(h, alloc(h->mem, &h->dF, lambda * K)); CREATE_OK(h, alloc(h->mem, &h->dFprev, lambda * K)); CREATE_OK(h, alloc(h->mem, &h->dParentIndex, lambda));
  CREATE_OK(h, alloc(h->mem, &h->dSorted, 2 * lambda));
  CREATE_OK(h, alloc(h->mem, &h->dBestEver, K)); CREATE_OK(h, alloc(h->mem, &h->dPrevBest, K)); CREATE_OK(h, alloc(h->mem, &h->dCurBest, K));
  CREATE_OK(h, alloc(h->mem, &h->dBestEverX, K * N)); CREATE_OK(h, alloc(h->mem, &h->dPrevBestX, K * N)); CREATE_OK(h, alloc(h->mem, &h->dCurBestX, K * N));
  CREATE_OK(h, alloc(h->mem, &h->dValDiff, K)); CREATE_OK(h, alloc(h->mem, &h->dVarDiff, K)); CREATE_OK(h, alloc(h->mem, &h->dMinSd, lambda)); CREATE_OK(h, alloc(h->mem, &h->dMaxSd, lambda));
  CREATE_OK(h, alloc(h->mem, &h->dFlag, lambda)); CREATE_OK(h, alloc(h->mem, &h->dSc, 1)); CREATE_OK(h, alloc_host(h->mem, &h->hSc, 1));
  auto up = [&](double* d, const std::vector<double>& v) { return cudaMemcpy(d, v.data(), sizeof(double) * v.size(), cudaMemcpyHostToDevice); };
  CREATE_OK(h, up(h->dLower, lower)); CREATE_OK(h, up(h->dUpper, upper));
  std::vector<double> ninf(lambda * K, -INFINITY), kinf(K, INFINITY), kninf(K, -INFINITY);
  CREATE_OK(h, up(h->dF, ninf)); CREATE_OK(h, up(h->dFprev, ninf));
  CREATE_OK(h, up(h->dBestEver, kninf)); CREATE_OK(h, up(h->dPrevBest, kninf)); CREATE_OK(h, up(h->dCurBest, kninf));
  CREATE_OK(h, up(h->dValDiff, kinf)); CREATE_OK(h, up(h->dVarDiff, kinf));
  CREATE_OK(h, up(h->dMinSd, std::vector<double>(lambda, min_sdev))); CREATE_OK(h, up(h->dMaxSd, std::vector<double>(lambda, max_sdev)));
  const double sigma0 = sqrt(trace / (double)N);
  std::vector<double> pc((size_t)mu * N * N, 0.0);
  for (uint64_t i = 0; i < mu; i++)
    for (uint64_t d = 0; d < N; d++) pc[i * N * N + d * N + d] = sd[d] * sd[d] / (sigma0 * sigma0);
  CREATE_OK(h, up(h->dC[PAR], pc));
  CREATE_OK(h, up(h->dS[PAR], std::vector<double>(mu, sigma0))); CREATE_OK(h, up(h->dPS[PAR], std::vector<double>(mu, h->target)));
  h->hSc->nondom = 1;
  CREATE_OK(h, cudaMemcpy(h->dSc, h->hSc, sizeof(MoScalars), cudaMemcpyHostToDevice));
  *out = h;
  return 0;
}

// prepareGeneration :177-189 + sampleSingle :191-230
int kmocma_ask(kmocma_t* h) {
  if (!h) return fail(h, "null solver handle");
  CUDA_OK(h, cudaSetDevice(h->device));
  const size_t N = h->N, L = h->lambda;
  CUDA_OK(h, cudaMemcpyAsync(h->dFprev, h->dF, sizeof(double) * L * h->K, cudaMemcpyDeviceToDevice, h->stream));
  CUDA_OK(h, cudaMemcpyAsync(h->dX[PREV], h->dX[CUR], sizeof(double) * L * N, cudaMemcpyDeviceToDevice, h->stream));
  CUDA_OK(h, cudaMemcpyAsync(h->dS[PREV], h->dS[CUR], sizeof(double) * L, cudaMemcpyDeviceToDevice, h->stream));
  CUDA_OK(h, cudaMemcpyAsync(h->dC[PREV], h->dC[CUR], sizeof(double) * L * N * N, cudaMemcpyDeviceToDevice, h->stream));
  CUDA_OK(h, cudaMemcpyAsync(h->dP[PREV], h->dP[CUR], sizeof(double) * L * N, cudaMemcpyDeviceToDevice, h->stream));
  CUDA_OK(h, cudaMemcpyAsync(h->dPS[PREV], h->dPS[CUR], sizeof(double) * L, cudaMemcpyDeviceToDevice, h->stream));
  mo_sample_kernel<<<h->lambda, 128, sample_smem(h->N), h->stream>>>(h->N, h->lambda, h->mu, h->cfg.seed, (unsigned)h->gen, h->dLower, h->dUpper,
                                                                    h->dX[PAR], h->dS[PAR], h->dC[PAR], h->dP[PAR], h->dPS[PAR], h->dX[CUR], h->dS[CUR],
                                                                    h->dC[CUR], h->dP[CUR], h->dPS[CUR], h->dParentIndex, h->dSc);
  h->launches++;
  if (pull(h)) return 1;
  if (h->hSc->chol_failed) return fail(h, "Error during Cholesky decomposition of covariance matrix.\n");
  if (h->hSc->no_feasible) return fail(h, "no feasible sample after 10^6 draws");
  return 0;
}

int kmocma_set_host_objective(kmocma_t* h, kmocma_host_objective_fn fn, void* user) {
  if (!h) return fail(h, "null solver handle");
  h->host_obj = fn; h->host_obj_user = user;
  return 0;
}

int kmocma_inject_f(kmocma_t* h, const double* f, size_t count) {
  if (!h) return fail(h, "null solver handle");
  if (count != (size_t)h->lambda * h->K) return fail(h, "inject_f: %zu values for %d x %d", count, h->lambda, h->K);
  CUDA_OK(h, cudaSetDevice(h->device));
  CUDA_OK(h, cudaMemcpyAsync(h->dF, f, sizeof(double) * count, cudaMemcpyHostToDevice, h->stream));
  CUDA_OK(h, cudaStreamSynchronize(h->stream));
  h->have_inj_f = true;
  return 0;
}

// runGeneration :152-170
int kmocma_eval(kmocma_t* h) {
  if (!h) return fail(h, "null solver handle");
  CUDA_OK(h, cudaSetDevice(h->device));
  h->model_evals += h->lambda;
  const int L = h->lambda, K = h->K, N = h->N;
  if (h->have_inj_f) {
    h->have_inj_f = false;
  } else if (h->host_obj) {
    h->hX.resize((size_t)L * N); h->hF.resize((size_t)L * K);
    CUDA_OK(h, cudaMemcpyAsync(h->hX.data(), h->dX[CUR], sizeof(double) * L * N, cudaMemcpyDeviceToHost, h->stream));
    CUDA_OK(h, cudaStreamSynchronize(h->stream));
    h->host_obj(h->host_obj_user, h->hX.data(), (uint64_t)L, (uint64_t)N, h->hF.data(), (uint64_t)K);
    CUDA_OK(h, cudaMemcpyAsync(h->dF, h->hF.data(), sizeof(double) * L * K, cudaMemcpyHostToDevice, h->stream));
  } else if (h->cfg.objective == KMOCMA_OBJ_EXTERNAL) {
    return fail(h, "objective is External: inject the values or set a host objective before eval");
  } else {
    mo_objective_kernel<<<(L + 127) / 128, 128, 0, h->stream>>>(h->cfg.objective, N, L, K, h->dX[CUR], h->dF, h->dSc);
    h->launches++;
  }
  mo_check_finite_kernel<<<(L * K + 255) / 256, 256, 0, h->stream>>>(h->dF, L * K, h->dSc);
  h->launches++;
  if (pull(h)) return 1;
  if (h->hSc->nonfinite) return fail(h, "Non finite value of function evaluation detected\n");
  return 0;
}

// updateDistribution :344-418 + updateStatistics :420-520
int kmocma_tell(kmocma_t* h) {
  if (!h) return fail(h, "null solver handle");
  CUDA_OK(h, cudaSetDevice(h->device));
  const int L = h->lambda, K = h->K, N = h->N, mu = h->mu;
  mo_sort_kernel<<<1, 1024, (size_t)2 * L * (sizeof(double) + 3 * sizeof(int)), h->stream>>>(h->dF, h->dFprev, L, K, h->dSorted);
  mo_update_kernel<<<L, 128, sizeof(double) * N, h->stream>>>(N, L, mu, h->cc, h->ccov, h->cp, h->target, h->dSorted, h->dParentIndex, h->dX[PAR],
                                                               h->dX[CUR], h->dS[CUR], h->dC[CUR], h->dP[CUR], h->dPS[CUR]);
  mo_parents_kernel<<<2 * L, 128, 0, h->stream>>>(N, L, mu, h->dSorted, h->dX[CUR], h->dS[CUR], h->dC[CUR], h->dP[CUR], h->dPS[CUR], h->dX[PREV],
                                                  h->dS[PREV], h->dC[PREV], h->dP[PREV], h->dPS[PREV], h->dX[PAR], h->dS[PAR], h->dC[PAR], h->dP[PAR],
                                                  h->dPS[PAR]);
  mo_stats_kernel<<<1, 256, 0, h->stream>>>(N, L, K, h->dF, h->dX[CUR], h->dS[CUR], h->dC[CUR], h->dBestEver, h->dBestEverX, h->dPrevBest,
                                            h->dPrevBestX, h->dCurBest, h->dCurBestX, h->dValDiff, h->dVarDiff, h->dMinSd, h->dMaxSd, h->dFlag, h->dSc);
  h->launches += 4;
  // archive of non-dominated samples (:483-519) on the host
  std::vector<unsigned char> flag(L);
  h->hX.resize((size_t)L * N); h->hF.resize((size_t)L * K);
  CUDA_OK(h, cudaMemcpyAsync(flag.data(), h->dFlag, L, cudaMemcpyDeviceToHost, h->stream));
  CUDA_OK(h, cudaMemcpyAsync(h->hX.data(), h->dX[CUR], sizeof(double) * L * N, cudaMemcpyDeviceToHost, h->stream));
  CUDA_OK(h, cudaMemcpyAsync(h->hF.data(), h->dF, sizeof(double) * L * K, cudaMemcpyDeviceToHost, h->stream));
  CUDA_OK(h, cudaStreamSynchronize(h->stream));
  CUDA_OK(h, cudaGetLastError());
  std::vector<int> cand;
  for (int i = 0; i < L; i++) if (flag[i]) cand.push_back(i);
  const size_t ncoll = h->coll_f.size() / K;
  std::vector<char> keep_c(cand.size(), 1), keep_s(ncoll, 1);
  for (size_t a = 0; a < cand.size(); ++a)
    for (size_t j = 0; j < ncoll; ++j) {
      int cdom = 0, sdom = 0;
      for (int k = 0; k < K; ++k) {
        if (h->hF[(size_t)cand[a] * K + k] > h->coll_f[j * K + k]) cdom++;
        if (h->hF[(size_t)cand[a] * K + k] < h->coll_f[j * K + k]) sdom++;
      }
      if (cdom == K) keep_s[j] = 0;
      if (sdom == K) keep_c[a] = 0;
    }
  std::vector<double> nx, nf;
  for (size_t j = 0; j < ncoll; ++j)
    if (keep_s[j]) { nx.insert(nx.end(), h->coll_x.begin() + j * N, h->coll_x.begin() + (j + 1) * N); nf.insert(nf.end(), h->coll_f.begin() + j * K, h->coll_f.begin() + (j + 1) * K); }
  for (size_t a = 0; a < cand.size(); ++a)
    if (keep_c[a]) {
      nx.insert(nx.end(), h->hX.begin() + (size_t)cand[a] * N, h->hX.begin() + (size_t)(cand[a] + 1) * N);
      nf.insert(nf.end(), h->hF.begin() + (size_t)cand[a] * K, h->hF.begin() + (size_t)(cand[a] + 1) * K);
    }
  h->coll_x.swap(nx); h->coll_f.swap(nf);
  h->gen++;
  return 0;
}

int kmocma_run_generation(kmocma_t* h) { return kmocma_ask(h) || kmocma_eval(h) || kmocma_tell(h); }

int kmocma_check_termination(kmocma_t* h, int* finished, const char** reason) {
  if (!h) return fail(h, "null solver handle");
  if (!finished) return fail(h, "null argument");
  CUDA_OK(h, cudaSetDevice(h->device));
  h->reason.clear();
  int fin = 0;
  const int K = h->K, L = h->lambda;
  if (h->gen > 1) {
    std::vector<double> vd(K), xd(K), mn(L), mx(L);
    CUDA_OK(h, cudaMemcpy(vd.data(), h->dValDiff, sizeof(double) * K, cudaMemcpyDeviceToHost));
    CUDA_OK(h, cudaMemcpy(xd.data(), h->dVarDiff, sizeof(double) * K, cudaMemcpyDeviceToHost));
    CUDA_OK(h, cudaMemcpy(mn.data(), h->dMinSd, sizeof(double) * L, cudaMemcpyDeviceToHost));
    CUDA_OK(h, cudaMemcpy(mx.data(), h->dMaxSd, sizeof(double) * L, cudaMemcpyDeviceToHost));
    // (the first criterion reads the BASE class threshold _minValueDifferenceThreshold, MOCMAES.config "Termination Criteria")
    if (fabs(*std::max_element(vd.begin(), vd.end())) < h->tc_min_value_diff) { h->reason += "Min Max Value Difference Threshold;"; fin = 1; }
    if (*std::max_element(xd.begin(), xd.end()) < h->tc_min_var_diff) { h->reason += "Min Variable Difference Threshold;"; fin = 1; }
    if (*std::max_element(mn.begin(), mn.end()) <= h->tc_min_sd) { h->reason += "Min Standard Deviation;"; fin = 1; }
    if (*std::min_element(mx.begin(), mx.end()) >= h->tc_max_sd) { h->reason += "Max Standard Deviation;"; fin = 1; }
  }
  if (h->tc_max_model_evaluations <= (double)h->model_evals) { h->reason += "solver['Max Model Evaluations'];"; fin = 1; }
  if ((double)h->gen > h->tc_max_generations) { h->reason += "solver['Max Generations'];"; fin = 1; }
  *finished = fin;
  if (reason) *reason = h->reason.c_str();
  return 0;
}

int kmocma_run(kmocma_t* h, uint64_t max_generations, uint64_t* done) {
  return run(h, max_generations, done, kmocma_check_termination, kmocma_run_generation);
}

int kmocma_get_array(kmocma_t* h, const char* key, double* out, size_t cap, size_t* count) {
  if (!h) return fail(h, "null solver handle");
  if (!key) return fail(h, "null argument");
  CUDA_OK(h, cudaSetDevice(h->device));
  Array r;
  if (!find_array(h, key, &r)) return fail(h, "unknown array key '%s'", key);
  return copy_out(h, key, r, out, cap, count, "get_array(%s): capacity %zu < %zu");
}

int kmocma_get_scalar(kmocma_t* h, const char* key, double* out) {
  if (!h) return fail(h, "null solver handle");
  if (!key || !out) return fail(h, "null argument");
  if (double* p = host_scalar(h, kHostScalars, key, false)) *out = *p;
  else if (!strcmp(key, "Current Non Dominated Sample Count")) {
    CUDA_OK(h, cudaSetDevice(h->device));
    if (pull(h)) return 1;
    *out = (double)h->hSc->nondom;
  } else if (!strcmp(key, "Infeasible Sample Count")) *out = 0.0;   // :216 counts nothing (the increment is commented out in the reference)
  else if (!strcmp(key, "Model Evaluation Count")) *out = (double)h->model_evals;
  else if (!strcmp(key, "Current Generation")) *out = (double)h->gen;
  else if (!strcmp(key, "Sample Collection Size")) *out = (double)(h->coll_f.size() / h->K);
  else if (!strcmp(key, "Population Size")) *out = (double)h->lambda;
  else if (!strcmp(key, "Mu Value")) *out = (double)h->mu;
  else return fail(h, "unknown scalar key '%s'", key);
  return 0;
}

int kmocma_set_scalar(kmocma_t* h, const char* key, double v) {
  if (!h) return fail(h, "null solver handle");
  if (!key) return fail(h, "null argument");
  double* p = host_scalar(h, kHostScalars, key, true);
  if (!p) return fail(h, "unknown scalar key '%s'", key);
  *p = v;
  return 0;
}

uint64_t kmocma_launch_count(const kmocma_t* h) { return h ? h->launches : 0; }

}  // extern "C"
