// tmcmc.cu — transitional MCMC on the device (include/ktmcmc.h): "Sampler/TMCMC" for "Bayesian/Custom" problems on the kernels and
// conventions of the CMA-ES path. Everything outside the likelihood model stays in HBM; inside a generation the host reads one
// thing, the chain count and the longest chain after the resampling, which fixes the number of MCMC steps.
//
//   ktmcmc_anneal    tm_anneal_kernel        l_max, bisection of CoV(D) = target (one CTA, fixed-order sums, no host sync per
//                                            iteration), weights w~, cumsum(w~), LogEvidence
//                    tm_mean_partial_kernel  weighted mean over 64 row chunks, tm_mean_final_kernel: the chunk sums in order
//   (+ kernels.h)    tm_rows_kernel          rows sqrt(w~_i)(x_i - mean) for launch_syrk; launch_reduce_splits; tm_cov_kernel: s * P
//                    eigensolver             launch_eigen_small (N <= 24) or launch_eigen_tridiag + launch_eig_sign / launch_eig_order
//                                            + tm_commit_kernel (eigenvalues below 0 clamped to 0): the proposal factor A = B D
//   ktmcmc_resample  tm_draw_kernel          inverse-CDF search of Philox uniforms, integer histogram (deterministic)
//                    tm_chains_kernel        integer scans into chain and database offsets (one CTA)
//                    tm_chain_init_kernel    chains start at their leader's (x, l, p)
//   ktmcmc_propose   tm_z_kernel + launch_gemm_tn (x' = x + A z for every chain) + tm_epilogue_kernel (log-prior, support flag)
//                    + tm_compact_kernel / tm_gather_kernel (the in-support proposals of active chains, packed in chain order)
//   ktmcmc_eval      launch_objective (built-in models) or the host / device conduit on the packed rows; Bayesian/Reference: the
//                    host / device computational model writes G (and P), then tm_reference_loglik_kernel<LIK> reduces them to l
//   ktmcmc_accept    tm_accept_kernel        Metropolis test, database append, acceptance statistics
// Compiled with --fmad=false: the arithmetic rounds like oracle/otmcmc.c (the device's exp / log / sincospi may differ from libm in
// the last bit; the GEMM and the SYRK sum in their own order).
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/ktmcmc.h"
#include "bayes.cuh"
#include "common.cuh"
#include "handle.cuh"
#include "kernels.h"

namespace {

using namespace kc;

constexpr int kThreads = 1024;        // one-CTA reductions and scans: thread t owns a fixed slice (restated by the oracle)
constexpr int kMeanChunks = 64;       // row chunks of the weighted mean
constexpr uint32_t kKeyTag = 0x544d434du;   // "TMCM"

__device__ __forceinline__ void tm_philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, unsigned long long seed, uint32_t out[4]) {
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32) ^ kKeyTag;
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
__device__ __forceinline__ double tm_unit(uint32_t lo, uint32_t hi) {
  const unsigned long long v = ((unsigned long long)hi << 32) | lo;
  return (double)(v >> 12) * 0x1.0p-52 + 0x1.0p-53;
}
__device__ __forceinline__ void tm_box_muller(const uint32_t r[4], double& z0, double& z1) {
  const double u1 = tm_unit(r[0], r[1]), u2 = tm_unit(r[2], r[3]);
  const double rad = sqrt(-2.0 * log(u1));
  double s, c;
  sincospi(2.0 * u2, &s, &c);
  z0 = rad * c; z1 = rad * s;
}

struct TmScalars {
  double rho, rho_prev, delta, cov, logev, llmax;
  unsigned long long evals;          // in-support proposals evaluated (all generations)
  unsigned long long step_evals;     // rows of the current evaluation
  unsigned long long accepted, proposals;   // this generation
  int chain_count, max_len, leaders, last_pos;
  int nan_flag, allinf_flag;
  unsigned long long ref_err;        // Bayesian/Reference: ~(row << 2 | code) of the first bad model output (atomicMax), 0 = none
};

// Generation 1: one warp per sample; lanes over the Box-Muller pairs, then the log-prior of the row.
__global__ void __launch_bounds__(256)
tm_prior_kernel(int n, int lambda, unsigned long long seed, const int* __restrict__ type, const double* __restrict__ pa,
                const double* __restrict__ pb, double* __restrict__ X, int ld, double* __restrict__ LP) {
  const int lane = threadIdx.x & 31;
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (i >= lambda) return;
  double* x = X + (size_t)i * ld;
  for (int p = lane; 2 * p < n; p += 32) {
    uint32_t r[4];
    tm_philox((1u << 20) + (uint32_t)p, (uint32_t)i, 0u, 0u, seed, r);
    double z0, z1;
    tm_box_muller(r, z0, z1);
    const double u[2] = {tm_unit(r[0], r[1]), tm_unit(r[2], r[3])};
    const double z[2] = {z0, z1};
    for (int h = 0; h < 2 && 2 * p + h < n; h++) {
      const int d = 2 * p + h;
      x[d] = type[d] == KTMCMC_PRIOR_UNIFORM ? pa[d] + (pb[d] - pa[d]) * u[h] : pa[d] + pb[d] * z[h];
    }
  }
  __syncwarp();
  const double lp = log_prior_row(x, n, type, pa, pb, lane);
  if (lane == 0) LP[i] = lp;
}

// fixed-order block sum of kThreads per-thread partials: xor butterfly inside each warp, then over the 32 warp sums
__device__ __forceinline__ double block_sum(double v, double* red) {
  const int tid = threadIdx.x;
  v = warp_sum_butterfly(v);
  __syncthreads();
  if ((tid & 31) == 0) red[tid >> 5] = v;
  __syncthreads();
  if (tid < 32) {
    double s = warp_sum_butterfly(red[tid]);
    if (tid == 0) red[32] = s;
  }
  __syncthreads();
  return red[32];
}

__device__ __forceinline__ double weight(double l, double D, double llmax) { return l == -INFINITY ? 0.0 : exp(D * (l - llmax)); }

// Steps 1-2 and the cumulative weights of step 4, one CTA of kThreads threads.
__global__ void __launch_bounds__(kThreads, 1)
tm_anneal_kernel(const double* __restrict__ LL, int lambda, double target, double dmin, double dmax, double* __restrict__ W,
                 double* __restrict__ Cum, TmScalars* __restrict__ sc) {
  __shared__ double red[80];
  __shared__ double smax[32];
  __shared__ int snan, sfin, slast;
  __shared__ double sprefix[kThreads + 1];
  const int tid = threadIdx.x;
  if (tid == 0) { snan = 0; sfin = 0; slast = -1; }
  __syncthreads();
  double mx = -INFINITY;
  int nan = 0, fin = 0;
  for (int i = tid; i < lambda; i += kThreads) {
    const double l = LL[i];
    if (l != l) nan = 1;
    else if (l != -INFINITY) { fin = 1; mx = fmax(mx, l); }
  }
  if (nan) atomicOr(&snan, 1);
  if (fin) atomicOr(&sfin, 1);
  mx = warp_max(mx);
  if ((tid & 31) == 0) smax[tid >> 5] = mx;
  __syncthreads();
  if (snan || !sfin) {
    if (tid == 0) { sc->nan_flag |= snan; sc->allinf_flag |= !sfin; sc->delta = 0.0; sc->rho_prev = sc->rho; }
    return;
  }
  double llmax = -INFINITY;
  for (int w = 0; w < 32; w++) llmax = fmax(llmax, smax[w]);
  const double rho = sc->rho, rem = 1.0 - rho;
  const double fl = (double)lambda;
  auto cov_of = [&](double D, double& s1) {
    double p1 = 0.0, p2 = 0.0;
#pragma unroll 1
    for (int i = tid; i < lambda; i += kThreads) { const double w = weight(LL[i], D, llmax); p1 = p1 + w; p2 = p2 + w * w; }
    s1 = block_sum(p1, red);
    const double s2 = block_sum(p2, red + 40);
    return sqrt(fmax(0.0, fl * s2 / (s1 * s1) - 1.0));
  };
  double s1;
  double D = rem;
  if (cov_of(rem, s1) > target) {
    double lo = 0.0, hi = rem;
#pragma unroll 1
    for (int it = 0; it < 64; it++) {
      const double mid = 0.5 * (lo + hi);
      if (cov_of(mid, s1) > target) hi = mid; else lo = mid;
    }
    D = lo;
  }
  D = fmin(fmax(D, dmin), dmax);
  double rho_new;
  if (D >= rem) { D = rem; rho_new = 1.0; } else rho_new = rho + D;
  const double cov = cov_of(D, s1);
  for (int i = tid; i < lambda; i += kThreads) W[i] = weight(LL[i], D, llmax) / s1;
  __syncthreads();
  // cumsum(w~): contiguous chunks, sequential inside, chunk totals prefix-summed in order
  const int chunk = (lambda + kThreads - 1) / kThreads;
  const int b0 = min(lambda, tid * chunk), b1 = min(lambda, b0 + chunk);
  double tot = 0.0;
  int last = -1;
  for (int i = b0; i < b1; i++) { tot = tot + W[i]; if (W[i] > 0.0) last = i; }
  sprefix[tid] = tot;
  if (last >= 0) atomicMax(&slast, last);
  __syncthreads();
  if (tid == 0) {
    double run = 0.0;
    for (int t = 0; t < kThreads; t++) { const double v = sprefix[t]; sprefix[t] = run; run = run + v; }
  }
  __syncthreads();
  const double pre = sprefix[tid];
  double loc = 0.0;
  for (int i = b0; i < b1; i++) { loc = loc + W[i]; Cum[i] = pre + loc; }
  if (tid == 0) {
    sc->rho_prev = rho; sc->rho = rho_new; sc->delta = D; sc->cov = cov; sc->llmax = llmax;
    sc->logev = sc->logev + (log(s1 / fl) + D * llmax);
    sc->last_pos = slast;
  }
}

// weighted mean, pass 1: partial[c][d] = sum over the rows of chunk c (ascending) of w~_i x_id
__global__ void __launch_bounds__(128)
tm_mean_partial_kernel(const double* __restrict__ X, int ld, int n, int lambda, const double* __restrict__ W, double* __restrict__ part) {
  const int d = blockIdx.x * blockDim.x + threadIdx.x, c = blockIdx.y;
  if (d >= n) return;
  const int rows = (lambda + kMeanChunks - 1) / kMeanChunks;
  const int r0 = min(lambda, c * rows), r1 = min(lambda, r0 + rows);
  double p = 0.0;
  for (int i = r0; i < r1; i++) p = p + W[i] * X[(size_t)i * ld + d];
  part[(size_t)c * ld + d] = p;
}
__global__ void tm_mean_final_kernel(const double* __restrict__ part, int ld, int n, double* __restrict__ mean) {
  const int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= n) return;
  double m = 0.0;
  for (int c = 0; c < kMeanChunks; c++) m = m + part[(size_t)c * ld + d];
  mean[d] = m;
}
// rows of the SYRK: S_i = sqrt(w~_i) (x_i - mean)
__global__ void __launch_bounds__(256)
tm_rows_kernel(const double* __restrict__ X, int ld, int n, int lambda, const double* __restrict__ W, const double* __restrict__ mean,
               double* __restrict__ S) {
  const long long total = (long long)lambda * n;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const long long i = idx / n;
    const int d = (int)(idx - i * n);
    S[(size_t)i * ld + d] = sqrt(W[i]) * (X[(size_t)i * ld + d] - mean[d]);
  }
}
// Sigma = s P from the lower triangle of P
__global__ void tm_cov_kernel(const double* __restrict__ P, int ld, int n, double s, double* __restrict__ Cv) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x, d = blockIdx.y;
  if (e >= n) return;
  Cv[(size_t)d * ld + e] = s * (e <= d ? P[(size_t)d * ld + e] : P[(size_t)e * ld + d]);
}
// A[d][e] = B[d][e] sqrt(max(ev, 0)) with B[d][e] = sign * VT[perm[e]][d] (ascending |eigenvalue|, as eig_commit_kernel)
__global__ void tm_commit_kernel(const double* __restrict__ VT, int ld, int n, const int* __restrict__ perm, const double* __restrict__ ev,
                                 const double* __restrict__ sign, double* __restrict__ A) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x, d = blockIdx.y;
  if (e >= n) return;
  const int p = perm[e];
  A[(size_t)d * ld + e] = sign[p] * VT[(size_t)p * ld + d] * sqrt(fmax(ev[p], 0.0));
}

// step 4: leader of draw k = first index with cumsum >= u_k
__global__ void tm_draw_kernel(const double* __restrict__ Cum, int lambda, unsigned long long seed, unsigned generation,
                               const TmScalars* __restrict__ sc, int* __restrict__ counts) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= lambda) return;
  uint32_t r[4];
  tm_philox(0u, (uint32_t)k, 0u, generation, seed, r);
  const double u = tm_unit(r[0], r[1]);
  int lo = 0, hi = lambda;   // first i in [lo, hi) with Cum[i] >= u
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (Cum[mid] >= u) hi = mid; else lo = mid + 1;
  }
  if (lo >= lambda) lo = sc->last_pos;
  atomicAdd(&counts[lo], 1);
}
// integer scans of counts into chains (ascending leader) and database offsets; one CTA
__global__ void __launch_bounds__(kThreads)
tm_chains_kernel(const int* __restrict__ counts, int lambda, int L, int* __restrict__ leader, int* __restrict__ len, int* __restrict__ dbstart,
                 TmScalars* __restrict__ sc) {
  __shared__ int sch[kThreads], sdb[kThreads];
  __shared__ int smaxc, sleaders;
  const int tid = threadIdx.x;
  if (tid == 0) { smaxc = 0; sleaders = 0; }
  const int chunk = (lambda + kThreads - 1) / kThreads;
  const int b0 = min(lambda, tid * chunk), b1 = min(lambda, b0 + chunk);
  int nch = 0, ndb = 0, mc = 0, nl = 0;
  for (int i = b0; i < b1; i++) {
    const int c = counts[i];
    nch += (c + L - 1) / L; ndb += c; mc = max(mc, c); nl += c > 0;
  }
  sch[tid] = nch; sdb[tid] = ndb;
  __syncthreads();
  atomicMax(&smaxc, mc); atomicAdd(&sleaders, nl);
  if (tid == 0) {
    int a = 0, b = 0;
    for (int t = 0; t < kThreads; t++) { const int x = sch[t], y = sdb[t]; sch[t] = a; sdb[t] = b; a += x; b += y; }
    sc->chain_count = a;
  }
  __syncthreads();
  int k = sch[tid], db = sdb[tid];
  for (int i = b0; i < b1; i++) {
    const int c = counts[i];
    for (int j = 0; j * L < c; j++) { leader[k] = i; len[k] = min(L, c - j * L); dbstart[k] = db + j * L; k++; }
    db += c;
  }
  if (tid == 0) { sc->max_len = min(L, smaxc); sc->leaders = sleaders; sc->accepted = 0; sc->proposals = 0; }
}
__global__ void __launch_bounds__(256)
tm_chain_init_kernel(const TmScalars* __restrict__ sc, const int* __restrict__ leader, const double* __restrict__ X, const double* __restrict__ LL,
                     const double* __restrict__ LP, int ld, int n, double* __restrict__ CX, double* __restrict__ CLL, double* __restrict__ CLP) {
  const int lane = threadIdx.x & 31;
  const int k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (k >= sc->chain_count) return;
  const int i = leader[k];
  for (int d = lane; d < n; d += 32) CX[(size_t)k * ld + d] = X[(size_t)i * ld + d];
  if (lane == 0) { CLL[k] = LL[i]; CLP[k] = LP[i]; }
}

// z of chain k at step t: one thread per (chain, pair)
__global__ void __launch_bounds__(256)
tm_z_kernel(double* __restrict__ Z, int ld, int chains, int n, unsigned long long seed, unsigned step, unsigned generation) {
  const int npairs = (n + 1) >> 1;
  const long long total = (long long)chains * npairs;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(idx / npairs), p = (int)(idx - (long long)k * npairs);
    uint32_t r[4];
    tm_philox((1u << 20) + (uint32_t)p, (uint32_t)k, step, generation, seed, r);
    double z0, z1;
    tm_box_muller(r, z0, z1);
    double* dst = Z + (size_t)k * ld + 2 * p;
    dst[0] = z0;
    if (2 * p + 1 < n) dst[1] = z1;
  }
}
// x' = x + y, log-prior, support flag of the active chains (one warp per chain)
__global__ void __launch_bounds__(256)
tm_epilogue_kernel(int chains, int n, int ld, int step, int burn, const int* __restrict__ len, const double* __restrict__ CX,
                   const double* __restrict__ Y, const int* __restrict__ type, const double* __restrict__ pa, const double* __restrict__ pb,
                   double* __restrict__ XP, double* __restrict__ LPP, int* __restrict__ flag) {
  const int lane = threadIdx.x & 31;
  const int k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (k >= chains) return;
  const bool active = step < burn + len[k];
  double* xp = XP + (size_t)k * ld;
  if (active)
    for (int d = lane; d < n; d += 32) xp[d] = CX[(size_t)k * ld + d] + Y[(size_t)k * ld + d];
  __syncwarp();
  const double lp = active ? log_prior_row(xp, n, type, pa, pb, lane) : -INFINITY;
  if (lane == 0) { LPP[k] = lp; flag[k] = !active ? -1 : (lp != -INFINITY ? 1 : 0); }
}
// evaluation slots of the in-support proposals in chain order; one CTA
__global__ void __launch_bounds__(kThreads)
tm_compact_kernel(const int* __restrict__ flag, int chains, int* __restrict__ slot, TmScalars* __restrict__ sc) {
  __shared__ int spre[kThreads];
  __shared__ int sact;
  const int tid = threadIdx.x;
  if (tid == 0) sact = 0;
  const int chunk = (chains + kThreads - 1) / kThreads;
  const int b0 = min(chains, tid * chunk), b1 = min(chains, b0 + chunk);
  int c = 0, a = 0;
  for (int k = b0; k < b1; k++) { c += flag[k] == 1; a += flag[k] >= 0; }
  spre[tid] = c;
  __syncthreads();
  atomicAdd(&sact, a);
  if (tid == 0) {
    int run = 0;
    for (int t = 0; t < kThreads; t++) { const int v = spre[t]; spre[t] = run; run += v; }
    sc->step_evals = (unsigned long long)run;
    sc->evals += (unsigned long long)run;
  }
  __syncthreads();
  int s = spre[tid];
  for (int k = b0; k < b1; k++) slot[k] = flag[k] == 1 ? s++ : -1;
  if (tid == 0) sc->proposals += (unsigned long long)sact;
}
__global__ void __launch_bounds__(256)
tm_gather_kernel(int chains, int n, int ld, const int* __restrict__ slot, const double* __restrict__ XP, double* __restrict__ EX) {
  const int lane = threadIdx.x & 31;
  const int k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (k >= chains) return;
  const int s = slot[k];
  if (s < 0) return;
  for (int d = lane; d < n; d += 32) EX[(size_t)s * ld + d] = XP[(size_t)k * ld + d];
}
// Metropolis test and database append (one warp per chain)
__global__ void __launch_bounds__(256)
tm_accept_kernel(int chains, int n, int ld, int step, int burn, unsigned long long seed, unsigned generation, const int* __restrict__ len,
                 const int* __restrict__ dbstart, const int* __restrict__ slot, const double* __restrict__ XP, const double* __restrict__ LPP,
                 const double* __restrict__ EF, double* __restrict__ CX, double* __restrict__ CLL, double* __restrict__ CLP,
                 double* __restrict__ DX, double* __restrict__ DLL, double* __restrict__ DLP, int* __restrict__ acc_flag,
                 TmScalars* __restrict__ sc) {
  const int lane = threadIdx.x & 31;
  const int k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (k >= chains) return;
  if (step >= burn + len[k]) return;
  int acc = 0;
  if (lane == 0) {
    const int s = slot[k];
    if (s >= 0) {
      const double l = EF[s];
      if (l != l) atomicExch(&sc->nan_flag, 1);
      uint32_t r[4];
      tm_philox(1u, (uint32_t)k, (uint32_t)step, generation, seed, r);
      const double u = tm_unit(r[0], r[1]);
      acc = log(u) < sc->rho * (l - CLL[k]) + (LPP[k] - CLP[k]);
      if (acc) { CLL[k] = l; CLP[k] = LPP[k]; atomicAdd(&sc->accepted, 1ull); }
    }
    acc_flag[k] = acc;
  }
  acc = __shfl_sync(0xffffffffu, acc, 0);
  if (acc)
    for (int d = lane; d < n; d += 32) CX[(size_t)k * ld + d] = XP[(size_t)k * ld + d];
  __syncwarp();
  if (step >= burn) {
    const int row = dbstart[k] + step - burn;
    for (int d = lane; d < n; d += 32) DX[(size_t)row * ld + d] = CX[(size_t)k * ld + d];
    if (lane == 0) { DLL[row] = CLL[k]; DLP[row] = CLP[k]; }
  }
}
__global__ void tm_check_nan_kernel(const double* __restrict__ F, int count, TmScalars* __restrict__ sc) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count && F[i] != F[i]) sc->nan_flag = 1;
}

// l of each evaluated row from its M predictions G (and parameters P): one warp per row, lane k sums j = k, k + 32, ... ascending,
// then the xor butterfly. Reads rows * M * 8 bytes of G (and of P) once, coalesced; the data (and, for Poisson, lgamma(d + 1) in
// DC) through the read-only path. A bad output is recorded in sc->ref_err and leaves its term NaN.
template <int LIK>
__global__ void __launch_bounds__(256)
tm_reference_loglik_kernel(int rows, int m, long long ldm, const double* __restrict__ G, const double* __restrict__ P,
                           const double* __restrict__ D, const double* __restrict__ DC, double* __restrict__ EF, TmScalars* __restrict__ sc) {
  const int lane = threadIdx.x & 31;
  const long long i = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  if (i >= rows) return;
  const double* g = G + i * ldm;
  const double* p = LIK == KTMCMC_LIK_POISSON ? nullptr : P + i * ldm;
  double s = 0.0;
  int bad = 4;
  for (int j = lane; j < m; j += 32) s = s + reference_term<LIK>(g[j], p, j, __ldg(D + j), DC, bad);
  if (bad < 4) atomicMax(&sc->ref_err, ~(((unsigned long long)i << 2) | (unsigned)bad));
  s = warp_sum_butterfly(s);
  if (lane == 0) EF[i] = s;
}
template <int LIK>
void launch_reference(cudaStream_t st, int rows, int m, long long ldm, const double* G, const double* P, const double* D, const double* DC,
                      double* EF, TmScalars* sc) {
  tm_reference_loglik_kernel<LIK><<<(unsigned)(((long long)rows * 32 + 255) / 256), 256, 0, st>>>(rows, m, ldm, G, P, D, DC, EF, sc);
}

unsigned grid_for(long long threads, int per) { return (unsigned)std::max<long long>(1, (threads + per - 1) / per); }

}  // namespace

struct ktmcmc : Handle<ktmcmc, TmScalars> {
  ktmcmc_cfg cfg;
  int N = 0, ld = 0, lambda = 0, num_sms = 148, L = 1;
  std::vector<uint64_t> burn_in;
  int *dType = nullptr, *dCounts = nullptr, *dLeader = nullptr, *dLen = nullptr, *dDbStart = nullptr, *dFlag = nullptr, *dSlot = nullptr,
      *dAcc = nullptr, *dPerm = nullptr;
  double *dPa = nullptr, *dPb = nullptr, *dCoef = nullptr;
  double *dX = nullptr, *dLL = nullptr, *dLP = nullptr;            // population
  double *dDX = nullptr, *dDLL = nullptr, *dDLP = nullptr;         // database (next population)
  double *dCX = nullptr, *dCLL = nullptr, *dCLP = nullptr;         // chain states
  double *dZ = nullptr, *dY = nullptr, *dXP = nullptr, *dLPP = nullptr, *dEX = nullptr, *dEF = nullptr;
  double *dW = nullptr, *dCum = nullptr, *dPart = nullptr, *dMean = nullptr, *dS = nullptr, *dWs = nullptr, *dP = nullptr, *dCov = nullptr;
  double *dVT = nullptr, *dGT = nullptr, *dB = nullptr, *dA = nullptr, *dD = nullptr, *dSign = nullptr;
  long long s_rows = 0;
  DevScalars* dDsc = nullptr;
  TridiagWs* tri = nullptr;
  // generation state on the host
  int chains = 0, steps = 0, step = 0, burn = 0, eval_rows = 0;
  bool in_generation = false, proposed = false, evaluated = false, have_inj = false;
  uint64_t init_evals = 0;
  double tc_target = 1.0, tc_max_generations = 1e10, tc_max_model_evaluations = 1e9;
  ktmcmc_host_loglik_fn host_fn = nullptr; void* host_user = nullptr;
  kcma_device_objective_fn dev_fn = nullptr; void* dev_user = nullptr;
  // Bayesian/Reference (lik = 0: Bayesian/Custom): data, lgamma(data + 1) for Poisson, model outputs G and parameters Pr (s_rows x ldm)
  int lik = 0, ef_rows = 0;
  long long m = 0, ldm = 0;
  double *dData = nullptr, *dDataC = nullptr, *dG = nullptr, *dPr = nullptr;
  bool have_ref_inj = false;
  ktmcmc_host_reference_fn host_ref_fn = nullptr; void* host_ref_user = nullptr;
  ktmcmc_device_reference_fn dev_ref_fn = nullptr; void* dev_ref_user = nullptr;
  std::vector<double> hX, hF, hG, hP;
  ~ktmcmc() {
    cudaSetDevice(device);
    cudaStreamSynchronize(stream);
    if (tri) tridiag_ws_destroy(tri);
  }
};

namespace {
const HostScalar<ktmcmc> kHostScalars[] = {
    {"Termination Criteria/Target Annealing Exponent", &ktmcmc::tc_target, true},
    {"Termination Criteria/Max Generations", &ktmcmc::tc_max_generations, true},
    {"Termination Criteria/Max Model Evaluations", &ktmcmc::tc_max_model_evaluations, true},
};
// every pull also reports a failed launch since the last one
int tm_pull(ktmcmc* h) {
  if (pull(h)) return 1;
  CUDA_OK(h, cudaGetLastError());
  return 0;
}
const char* tm_param_key(int lik) { return lik == KTMCMC_LIK_STUDENT_T ? "Degrees Of Freedom" : "Standard Deviation"; }
int tm_check_flags(ktmcmc* h) {
  if (h->hSc->ref_err) {
    const unsigned long long e = ~h->hSc->ref_err;
    const long long row = (long long)(e >> 2);
    const int code = (int)(e & 3);
    if (code == kRefNonFinite)
      return fail(h, "Bayesian/Reference: 'Reference Evaluations' of sample %lld contains a non-finite value\n", row);
    if (code == kRefParameter)
      return fail(h, "Bayesian/Reference: '%s' of sample %lld contains a value that is not positive and finite\n", tm_param_key(h->lik), row);
    return fail(h, "Bayesian/Reference: 'Reference Evaluations' of sample %lld contains a negative Poisson mean\n", row);
  }
  if (h->hSc->nan_flag) return fail(h, "A NaN log-likelihood was produced by the likelihood model\n");
  if (h->hSc->allinf_flag) return fail(h, "Every sample of the population has a log-likelihood of -inf: the annealing step is undefined\n");
  return 0;
}
}  // namespace

extern "C" {

void ktmcmc_cfg_defaults(ktmcmc_cfg* c) {
  memset(c, 0, sizeof(*c));
  c->abi_version = KTMCMC_ABI_VERSION;
  c->population_size = 0;
  c->max_chain_length = 1;
  c->target_cov = 1.0;
  c->covariance_scaling = 0.04;
  c->min_annealing_update = 1e-5;
  c->max_annealing_update = 1.0;
  c->loglik = KCMA_OBJ_EXTERNAL;
}

const char* ktmcmc_last_error(const ktmcmc_t* h) { return h ? h->err.c_str() : ktmcmc::create_err; }

void ktmcmc_destroy(ktmcmc_t* h) { delete h; }

int ktmcmc_create(const ktmcmc_cfg* cfg, ktmcmc_t** out) {
  if (!cfg || !out) return fail<ktmcmc>(nullptr, "null argument");
  if (cfg->abi_version != KTMCMC_ABI_VERSION) return fail<ktmcmc>(nullptr, "ktmcmc_cfg ABI version mismatch");
  if (cfg->n < 1) return fail<ktmcmc>(nullptr, "Bayesian problems require at least one variable.\n");
  if (cfg->population_size < 2) return fail<ktmcmc>(nullptr, "Sampler/TMCMC: 'Population Size' must be at least 2 (got %zu)\n", (size_t)cfg->population_size);
  if (cfg->population_size > (1u << 30)) return fail<ktmcmc>(nullptr, "Sampler/TMCMC: 'Population Size' above 2^30 is not supported\n");
  if (cfg->max_chain_length < 1) return fail<ktmcmc>(nullptr, "Sampler/TMCMC: 'Max Chain Length' must be at least 1\n");
  if (!(cfg->target_cov > 0.0)) return fail<ktmcmc>(nullptr, "Sampler/TMCMC: 'Target Coefficient Of Variation' must be positive\n");
  if (!(cfg->covariance_scaling > 0.0)) return fail<ktmcmc>(nullptr, "Sampler/TMCMC: 'Covariance Scaling' must be positive\n");
  if (!(cfg->min_annealing_update > 0.0) || !(cfg->max_annealing_update >= cfg->min_annealing_update))
    return fail<ktmcmc>(nullptr, "Sampler/TMCMC: need 0 < 'Min Annealing Exponent Update' <= 'Max Annealing Exponent Update'\n");
  if (!cfg->prior_type || !cfg->prior_a || !cfg->prior_b) return fail<ktmcmc>(nullptr, "Sampler/TMCMC: every variable needs a prior distribution\n");
  const int N = (int)cfg->n;
  for (int d = 0; d < N; d++) {
    const int t = cfg->prior_type[d];
    const double a = cfg->prior_a[d], b = cfg->prior_b[d];
    if (t == KTMCMC_PRIOR_UNIFORM) {
      if (!std::isfinite(a) || !std::isfinite(b) || !(b > a)) return fail<ktmcmc>(nullptr, "Univariate/Uniform prior of variable %d: need finite Minimum < Maximum\n", d);
    } else if (t == KTMCMC_PRIOR_NORMAL) {
      if (!std::isfinite(a) || !std::isfinite(b) || !(b > 0.0)) return fail<ktmcmc>(nullptr, "Univariate/Normal prior of variable %d: need a finite Mean and a positive Standard Deviation\n", d);
    } else return fail<ktmcmc>(nullptr, "unknown prior type %d of variable %d", t, d);
  }
  if (cfg->loglik != KCMA_OBJ_EXTERNAL && (cfg->loglik < KCMA_OBJ_NEG_SPHERE || cfg->loglik > KCMA_OBJ_NEG_SPHERE_SIN2))
    return fail<ktmcmc>(nullptr, "unknown log-likelihood model id %d", cfg->loglik);
  if (!eigen_use_small(N) && !eigen_tridiag_fits(N)) return fail<ktmcmc>(nullptr, "Sampler/TMCMC: n = %d is above the tridiagonal eigensolver's size\n", N);
  if (open_device<ktmcmc>(cfg->device)) return 1;
  ktmcmc* h = new ktmcmc();
  h->cfg = *cfg;
  h->burn_in.assign(cfg->per_generation_burn_in, cfg->per_generation_burn_in + (cfg->per_generation_burn_in ? cfg->burn_in_count : 0));
  h->cfg.per_generation_burn_in = nullptr; h->cfg.prior_type = nullptr; h->cfg.prior_a = h->cfg.prior_b = h->cfg.loglik_coef = nullptr;
  h->N = N; h->ld = (N + 15) / 16 * 16; h->lambda = (int)cfg->population_size; h->device = cfg->device;
  h->L = (int)std::min<uint64_t>(cfg->max_chain_length, cfg->population_size);
  cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, h->device);
  const size_t ld = h->ld, lam = h->lambda, rows = (lam + 15) / 16 * 16 + 16;
  h->s_rows = (long long)rows;
  CREATE_OK(h, alloc(h->mem, &h->dType, N)); CREATE_OK(h, alloc(h->mem, &h->dPa, N)); CREATE_OK(h, alloc(h->mem, &h->dPb, N)); CREATE_OK(h, alloc(h->mem, &h->dCoef, N));
  for (double** p : {&h->dX, &h->dDX, &h->dCX, &h->dZ, &h->dY, &h->dXP, &h->dEX, &h->dS}) CREATE_OK(h, alloc(h->mem, p, rows * ld));
  for (double** p : {&h->dLL, &h->dLP, &h->dDLL, &h->dDLP, &h->dCLL, &h->dCLP, &h->dLPP, &h->dEF, &h->dW, &h->dCum}) CREATE_OK(h, alloc(h->mem, p, lam));
  for (int** p : {&h->dCounts, &h->dLeader, &h->dLen, &h->dDbStart, &h->dFlag, &h->dSlot, &h->dAcc}) CREATE_OK(h, alloc(h->mem, p, lam));
  CREATE_OK(h, alloc(h->mem, &h->dPerm, 2 * (size_t)N + 64));
  CREATE_OK(h, alloc(h->mem, &h->dPart, (size_t)kMeanChunks * ld)); CREATE_OK(h, alloc(h->mem, &h->dMean, ld));
  CREATE_OK(h, alloc(h->mem, &h->dWs, (size_t)16 * N * ld));
  for (double** p : {&h->dP, &h->dCov, &h->dVT, &h->dGT, &h->dB, &h->dA}) CREATE_OK(h, alloc(h->mem, p, (size_t)N * ld));
  CREATE_OK(h, alloc(h->mem, &h->dD, ld)); CREATE_OK(h, alloc(h->mem, &h->dSign, ld));
  CREATE_OK(h, alloc(h->mem, &h->dDsc, 1)); CREATE_OK(h, alloc(h->mem, &h->dSc, 1));
  CREATE_OK(h, alloc_host(h->mem, &h->hSc, 1));
  std::vector<int> type(cfg->prior_type, cfg->prior_type + N);
  std::vector<double> coef(N);
  for (int d = 0; d < N; d++) coef[d] = cfg->loglik_coef ? cfg->loglik_coef[d] : pow(10.0, 6.0 * d / (double)std::max(N - 1, 1));
  CREATE_OK(h, cudaMemcpy(h->dType, type.data(), sizeof(int) * N, cudaMemcpyHostToDevice));
  CREATE_OK(h, cudaMemcpy(h->dPa, cfg->prior_a, sizeof(double) * N, cudaMemcpyHostToDevice));
  CREATE_OK(h, cudaMemcpy(h->dPb, cfg->prior_b, sizeof(double) * N, cudaMemcpyHostToDevice));
  CREATE_OK(h, cudaMemcpy(h->dCoef, coef.data(), sizeof(double) * N, cudaMemcpyHostToDevice));
  DevScalars ds; memset(&ds, 0, sizeof(ds)); ds.sigma = 1.0;
  CREATE_OK(h, cudaMemcpy(h->dDsc, &ds, sizeof(ds), cudaMemcpyHostToDevice));
  launch_set_identity(h->stream, h->dVT, (int)ld, N);
  launch_set_identity(h->stream, h->dB, (int)ld, N);
  if (!eigen_use_small(N)) {
    char msg[512] = "";
    h->tri = tridiag_ws_create(N, (int)ld, h->num_sms, msg, sizeof(msg));
    if (!h->tri) return create_fail(h, "%s", msg);
  }
  CREATE_OK(h, cudaStreamSynchronize(h->stream));
  CREATE_OK(h, cudaGetLastError());
  *out = h;
  return 0;
}

int ktmcmc_set_host_loglik(ktmcmc_t* h, ktmcmc_host_loglik_fn fn, void* user) {
  if (!h) return fail(h, "null solver handle");
  h->host_fn = fn; h->host_user = user;
  return 0;
}
int ktmcmc_set_device_loglik(ktmcmc_t* h, kcma_device_objective_fn fn, void* user) {
  if (!h) return fail(h, "null solver handle");
  h->dev_fn = fn; h->dev_user = user;
  return 0;
}

int ktmcmc_set_reference(ktmcmc_t* h, int32_t likelihood, const double* data, uint64_t m) {
  if (!h) return fail(h, "null solver handle");
  if (h->lik) return fail(h, "set_reference: the reference data are already set");
  if (h->gen != 1 || h->proposed) return fail(h, "set_reference: call it before generation 1");
  if (h->cfg.loglik != KCMA_OBJ_EXTERNAL) return fail(h, "set_reference: the log-likelihood must be External (KCMA_OBJ_EXTERNAL)");
  if (likelihood < KTMCMC_LIK_NORMAL || likelihood > KTMCMC_LIK_POISSON) return fail(h, "set_reference: unknown likelihood %d", likelihood);
  if (!data || m < 1 || m > (uint64_t)INT32_MAX) return fail(h, "set_reference: need 1 <= m < 2^31 reference data (got %zu)", (size_t)m);
  std::vector<double> dc(m, 0.0);
  for (uint64_t j = 0; j < m; j++) {
    const double d = data[j];
    if (!std::isfinite(d)) return fail(h, "Bayesian/Reference: 'Reference Data' %zu is not finite\n", (size_t)j);
    if (likelihood == KTMCMC_LIK_POISSON && (d < 0.0 || d != floor(d)))
      return fail(h, "Bayesian/Reference: 'Reference Data' %zu (%g) must be a non-negative integer for the Poisson likelihood\n", (size_t)j, d);
    if (likelihood == KTMCMC_LIK_POSITIVE_NORMAL && d < 0.0)
      return fail(h, "Bayesian/Reference: 'Reference Data' %zu (%g) must be >= 0 for the Positive Normal likelihood\n", (size_t)j, d);
    if (likelihood == KTMCMC_LIK_POISSON) dc[j] = lgamma(d + 1.0);
  }
  CUDA_OK(h, cudaSetDevice(h->device));
  const long long ldm = ((long long)m + 3) / 4 * 4;   // 32-byte aligned rows
  const bool param = likelihood != KTMCMC_LIK_POISSON;
  const size_t each = (size_t)h->s_rows * ldm;
  const double gib = (double)each * sizeof(double) * (param ? 2 : 1) / (double)(1ull << 30);
  if (alloc(h->mem, &h->dG, each) != cudaSuccess || (param && alloc(h->mem, &h->dPr, each) != cudaSuccess)) {
    cudaGetLastError();
    return fail(h, "Bayesian/Reference: cannot allocate the model outputs of %d samples x %zu reference points (%.2f GiB)\n", h->lambda,
                   (size_t)m, gib);
  }
  CUDA_OK(h, alloc(h->mem, &h->dData, m));
  CUDA_OK(h, alloc(h->mem, &h->dDataC, m));
  CUDA_OK(h, cudaMemcpy(h->dData, data, sizeof(double) * m, cudaMemcpyHostToDevice));
  CUDA_OK(h, cudaMemcpy(h->dDataC, dc.data(), sizeof(double) * m, cudaMemcpyHostToDevice));
  h->lik = likelihood; h->m = (long long)m; h->ldm = ldm;
  return 0;
}
int ktmcmc_set_host_reference_model(ktmcmc_t* h, ktmcmc_host_reference_fn fn, void* user) {
  if (!h) return fail(h, "null solver handle");
  h->host_ref_fn = fn; h->host_ref_user = user;
  return 0;
}
int ktmcmc_set_device_reference_model(ktmcmc_t* h, ktmcmc_device_reference_fn fn, void* user) {
  if (!h) return fail(h, "null solver handle");
  h->dev_ref_fn = fn; h->dev_ref_user = user;
  return 0;
}

// steps 1-3
int ktmcmc_anneal(ktmcmc_t* h) {
  if (!h) return fail(h, "null solver handle");
  if (h->gen < 2 || h->in_generation) return fail(h, "anneal: expected the start of a generation after the first");
  CUDA_OK(h, cudaSetDevice(h->device));
  const int N = h->N, ld = h->ld, lam = h->lambda;
  cudaStream_t st = h->stream;
  tm_anneal_kernel<<<1, kThreads, 0, st>>>(h->dLL, lam, h->cfg.target_cov, h->cfg.min_annealing_update, h->cfg.max_annealing_update, h->dW, h->dCum, h->dSc);
  tm_mean_partial_kernel<<<dim3((N + 127) / 128, kMeanChunks), 128, 0, st>>>(h->dX, ld, N, lam, h->dW, h->dPart);
  tm_mean_final_kernel<<<(N + 127) / 128, 128, 0, st>>>(h->dPart, ld, N, h->dMean);
  tm_rows_kernel<<<std::min(grid_for((long long)lam * N, 256), (unsigned)h->num_sms * 16), 256, 0, st>>>(h->dX, ld, N, lam, h->dW, h->dMean, h->dS);
  const int splits = launch_syrk(st, N, lam, nullptr, h->dS, ld, h->s_rows, h->dWs, ld, lam, h->num_sms, 16);
  launch_reduce_splits(st, h->dWs, ld, splits, N, h->dP);
  tm_cov_kernel<<<dim3((N + 127) / 128, N), 128, 0, st>>>(h->dP, ld, N, h->cfg.covariance_scaling, h->dCov);
  h->launches += 8;
  if (!h->tri) {
    const double tol = 4.0 * 2.220446049250313e-16 * sqrt((double)N);
    launch_eigen_small(st, h->dCov, ld, N, h->dVT, h->dGT, h->dB, h->dA, h->dD, tol, 40, h->dDsc);
    h->launches += 2;
  } else {
    double *vt = nullptr, *ev = nullptr;
    int l = 0;
    if (!launch_eigen_tridiag(st, h->tri, h->dCov, &vt, &ev, &l))
      return fail(h, "the tridiagonal eigensolver could not be launched: %s", cudaGetErrorString(cudaGetLastError()));
    launch_eig_sign(st, vt, ld, N, h->dSign);
    launch_eig_order(st, ev, N, h->dPerm, h->dDsc);
    tm_commit_kernel<<<dim3((N + 127) / 128, N), 128, 0, st>>>(vt, ld, N, h->dPerm, ev, h->dSign, h->dA);
    h->launches += l + 4;
  }
  CUDA_OK(h, cudaGetLastError());
  h->in_generation = true;
  h->chains = 0;
  return 0;
}

// step 4; reads the chain count and the longest chain (the number of MCMC steps)
int ktmcmc_resample(ktmcmc_t* h) {
  if (!h) return fail(h, "null solver handle");
  if (!h->in_generation || h->chains) return fail(h, "resample: call ktmcmc_anneal first");
  CUDA_OK(h, cudaSetDevice(h->device));
  const int lam = h->lambda;
  cudaStream_t st = h->stream;
  CUDA_OK(h, cudaMemsetAsync(h->dCounts, 0, sizeof(int) * lam, st));
  tm_draw_kernel<<<grid_for(lam, 256), 256, 0, st>>>(h->dCum, lam, h->cfg.seed, (unsigned)h->gen, h->dSc, h->dCounts);
  tm_chains_kernel<<<1, kThreads, 0, st>>>(h->dCounts, lam, h->L, h->dLeader, h->dLen, h->dDbStart, h->dSc);
  tm_chain_init_kernel<<<grid_for((long long)lam * 32, 256), 256, 0, st>>>(h->dSc, h->dLeader, h->dX, h->dLL, h->dLP, h->ld, h->N, h->dCX, h->dCLL, h->dCLP);
  h->launches += 3;
  if (tm_pull(h)) return 1;
  if (tm_check_flags(h)) return 1;
  h->chains = h->hSc->chain_count;
  h->burn = (int)(h->gen < h->burn_in.size() ? h->burn_in[h->gen] : h->cfg.default_burn_in);
  h->steps = h->burn + h->hSc->max_len;
  h->step = 0;
  h->proposed = h->evaluated = false;
  return 0;
}

int ktmcmc_propose(ktmcmc_t* h) {
  if (!h) return fail(h, "null solver handle");
  CUDA_OK(h, cudaSetDevice(h->device));
  const int N = h->N, ld = h->ld;
  cudaStream_t st = h->stream;
  if (h->gen == 1) {
    if (h->proposed) return fail(h, "propose: the prior draws of generation 1 are waiting for eval / accept");
    tm_prior_kernel<<<grid_for((long long)h->lambda * 32, 256), 256, 0, st>>>(N, h->lambda, h->cfg.seed, h->dType, h->dPa, h->dPb, h->dEX, ld, h->dLP);
    h->launches++;
    h->eval_rows = h->lambda;
  } else {
    if (!h->in_generation || !h->chains || h->step >= h->steps || h->proposed) return fail(h, "propose: no MCMC step pending (anneal and resample first)");
    const int K = h->chains;
    const long long pairs = (long long)K * ((N + 1) / 2);
    tm_z_kernel<<<std::min(grid_for(pairs, 256), (unsigned)h->num_sms * 16), 256, 0, st>>>(h->dZ, ld, K, N, h->cfg.seed, (unsigned)h->step, (unsigned)h->gen);
    launch_gemm_tn(st, K, N, N, h->dZ, ld, h->dA, ld, h->dY, ld);
    tm_epilogue_kernel<<<grid_for((long long)K * 32, 256), 256, 0, st>>>(K, N, ld, h->step, h->burn, h->dLen, h->dCX, h->dY, h->dType, h->dPa, h->dPb,
                                                                        h->dXP, h->dLPP, h->dFlag);
    tm_compact_kernel<<<1, kThreads, 0, st>>>(h->dFlag, K, h->dSlot, h->dSc);
    tm_gather_kernel<<<grid_for((long long)K * 32, 256), 256, 0, st>>>(K, N, ld, h->dSlot, h->dXP, h->dEX);
    h->launches += 5;
    h->eval_rows = -1;   // known on the device; read only when a host or device conduit needs it
  }
  CUDA_OK(h, cudaGetLastError());
  h->proposed = true;
  h->evaluated = false;
  return 0;
}

int ktmcmc_inject_loglik(ktmcmc_t* h, const double* l, size_t count) {
  if (!h) return fail(h, "null solver handle");
  if (!h->proposed || h->evaluated) return fail(h, "inject_loglik: no proposals waiting for an evaluation");
  CUDA_OK(h, cudaSetDevice(h->device));
  if (h->eval_rows < 0) { if (tm_pull(h)) return 1; h->eval_rows = (int)h->hSc->step_evals; }
  if (count != (size_t)h->eval_rows) return fail(h, "inject_loglik: %zu values for %d evaluation rows", count, h->eval_rows);
  if (count) CUDA_OK(h, cudaMemcpyAsync(h->dEF, l, sizeof(double) * count, cudaMemcpyHostToDevice, h->stream));
  CUDA_OK(h, cudaStreamSynchronize(h->stream));
  h->have_inj = true;
  return 0;
}

int ktmcmc_inject_reference(ktmcmc_t* h, const double* g, const double* p, size_t count) {
  if (!h) return fail(h, "null solver handle");
  if (!h->lik) return fail(h, "inject_reference: no reference data (ktmcmc_set_reference)");
  if (!h->proposed || h->evaluated) return fail(h, "inject_reference: no proposals waiting for an evaluation");
  if (!g || (h->lik != KTMCMC_LIK_POISSON) != (p != nullptr)) return fail(h, "inject_reference: need g, and p exactly when the likelihood has a parameter");
  CUDA_OK(h, cudaSetDevice(h->device));
  if (h->eval_rows < 0) { if (tm_pull(h)) return 1; h->eval_rows = (int)h->hSc->step_evals; }
  if (count != (size_t)h->eval_rows * h->m) return fail(h, "inject_reference: %zu values for %d evaluation rows x %lld", count, h->eval_rows, h->m);
  const size_t row = sizeof(double) * h->m, pitch = sizeof(double) * h->ldm;
  if (count) {
    CUDA_OK(h, cudaMemcpy2DAsync(h->dG, pitch, g, row, row, h->eval_rows, cudaMemcpyHostToDevice, h->stream));
    if (p) CUDA_OK(h, cudaMemcpy2DAsync(h->dPr, pitch, p, row, row, h->eval_rows, cudaMemcpyHostToDevice, h->stream));
  }
  CUDA_OK(h, cudaStreamSynchronize(h->stream));
  h->have_ref_inj = true;
  return 0;
}

int ktmcmc_inject_factor(ktmcmc_t* h, const double* a, size_t count) {
  if (!h) return fail(h, "null solver handle");
  if (count != (size_t)h->N * h->N) return fail(h, "inject_factor: %zu values for %d x %d", count, h->N, h->N);
  CUDA_OK(h, cudaSetDevice(h->device));
  CUDA_OK(h, cudaMemcpy2DAsync(h->dA, sizeof(double) * h->ld, a, sizeof(double) * h->N, sizeof(double) * h->N, h->N, cudaMemcpyHostToDevice, h->stream));
  CUDA_OK(h, cudaStreamSynchronize(h->stream));
  return 0;
}

int ktmcmc_eval(ktmcmc_t* h) {
  if (!h) return fail(h, "null solver handle");
  if (!h->proposed || h->evaluated) return fail(h, "eval: call ktmcmc_propose first");
  CUDA_OK(h, cudaSetDevice(h->device));
  const int N = h->N, ld = h->ld;
  cudaStream_t st = h->stream;
  h->ef_rows = h->eval_rows;
  if (h->have_inj) {
    h->have_inj = false;
  } else if (h->lik) {
    // Bayesian/Reference: injected outputs, or the device / host computational model, then the likelihood kernel
    if (h->eval_rows < 0) { if (tm_pull(h)) return 1; h->eval_rows = (int)h->hSc->step_evals; }
    const int rows = h->ef_rows = h->eval_rows;
    const long long m = h->m, ldm = h->ldm;
    double* dp = h->lik == KTMCMC_LIK_POISSON ? nullptr : h->dPr;
    if (h->have_ref_inj) {
      h->have_ref_inj = false;
    } else if (rows > 0 && h->dev_ref_fn) {
      h->dev_ref_fn(h->dev_ref_user, h->dEX, (uint64_t)rows, (uint64_t)N, (uint64_t)ld, h->dG, dp, (uint64_t)m, (uint64_t)ldm, (void*)st);
    } else if (rows > 0 && h->host_ref_fn) {
      const size_t row = sizeof(double) * m, pitch = sizeof(double) * ldm;
      h->hX.resize((size_t)rows * N); h->hG.resize((size_t)rows * m); h->hP.resize(dp ? (size_t)rows * m : 0);
      CUDA_OK(h, cudaMemcpy2DAsync(h->hX.data(), sizeof(double) * N, h->dEX, sizeof(double) * ld, sizeof(double) * N, rows, cudaMemcpyDeviceToHost, st));
      CUDA_OK(h, cudaStreamSynchronize(st));
      h->host_ref_fn(h->host_ref_user, h->hX.data(), (uint64_t)rows, (uint64_t)N, h->hG.data(), dp ? h->hP.data() : nullptr, (uint64_t)m);
      CUDA_OK(h, cudaMemcpy2DAsync(h->dG, pitch, h->hG.data(), row, row, rows, cudaMemcpyHostToDevice, st));
      if (dp) CUDA_OK(h, cudaMemcpy2DAsync(dp, pitch, h->hP.data(), row, row, rows, cudaMemcpyHostToDevice, st));
    } else if (rows > 0) {
      return fail(h, "Bayesian/Reference: inject the model outputs or set a host / device computational model before eval");
    }
    if (rows > 0) {
      switch (h->lik) {
        case KTMCMC_LIK_NORMAL: launch_reference<KTMCMC_LIK_NORMAL>(st, rows, (int)m, ldm, h->dG, dp, h->dData, h->dDataC, h->dEF, h->dSc); break;
        case KTMCMC_LIK_POSITIVE_NORMAL: launch_reference<KTMCMC_LIK_POSITIVE_NORMAL>(st, rows, (int)m, ldm, h->dG, dp, h->dData, h->dDataC, h->dEF, h->dSc); break;
        case KTMCMC_LIK_STUDENT_T: launch_reference<KTMCMC_LIK_STUDENT_T>(st, rows, (int)m, ldm, h->dG, dp, h->dData, h->dDataC, h->dEF, h->dSc); break;
        default: launch_reference<KTMCMC_LIK_POISSON>(st, rows, (int)m, ldm, h->dG, dp, h->dData, h->dDataC, h->dEF, h->dSc); break;
      }
      h->launches++;
    }
  } else if (h->cfg.loglik != KCMA_OBJ_EXTERNAL) {
    const long long rows = h->gen == 1 ? h->lambda : h->chains;   // rows past the packed ones are evaluated and never read
    launch_objective(st, h->cfg.loglik, h->dEX, ld, rows, N, 0, 1, nullptr, h->dDsc, h->dCoef, h->dEF, h->num_sms);
    h->launches++;
  } else if (h->host_fn || h->dev_fn) {
    if (h->eval_rows < 0) { if (tm_pull(h)) return 1; h->eval_rows = (int)h->hSc->step_evals; }
    const int rows = h->eval_rows;
    if (rows > 0) {
      if (h->dev_fn) {
        h->dev_fn(h->dev_user, h->dEX, (uint64_t)rows, (uint64_t)N, (uint64_t)ld, h->dEF, (void*)st);
      } else {
        h->hX.resize((size_t)rows * N); h->hF.resize(rows);
        CUDA_OK(h, cudaMemcpy2DAsync(h->hX.data(), sizeof(double) * N, h->dEX, sizeof(double) * ld, sizeof(double) * N, rows, cudaMemcpyDeviceToHost, st));
        CUDA_OK(h, cudaStreamSynchronize(st));
        h->host_fn(h->host_user, h->hX.data(), (uint64_t)rows, (uint64_t)N, h->hF.data());
        CUDA_OK(h, cudaMemcpyAsync(h->dEF, h->hF.data(), sizeof(double) * rows, cudaMemcpyHostToDevice, st));
      }
    }
  } else {
    return fail(h, "the log-likelihood is External: inject the values or set a host / device model before eval");
  }
  CUDA_OK(h, cudaGetLastError());
  h->evaluated = true;
  return 0;
}

int ktmcmc_accept(ktmcmc_t* h) {
  if (!h) return fail(h, "null solver handle");
  if (!h->evaluated) return fail(h, "accept: call ktmcmc_eval first");
  CUDA_OK(h, cudaSetDevice(h->device));
  const int N = h->N, ld = h->ld, lam = h->lambda;
  cudaStream_t st = h->stream;
  h->proposed = h->evaluated = false;
  if (h->gen == 1) {
    CUDA_OK(h, cudaMemcpyAsync(h->dX, h->dEX, sizeof(double) * lam * ld, cudaMemcpyDeviceToDevice, st));
    CUDA_OK(h, cudaMemcpyAsync(h->dLL, h->dEF, sizeof(double) * lam, cudaMemcpyDeviceToDevice, st));
    tm_check_nan_kernel<<<grid_for(lam, 256), 256, 0, st>>>(h->dLL, lam, h->dSc);
    h->launches++;
    h->init_evals = lam;
    if (tm_pull(h) || tm_check_flags(h)) return 1;
    h->gen = 2;
    return 0;
  }
  const int K = h->chains;
  tm_accept_kernel<<<grid_for((long long)K * 32, 256), 256, 0, st>>>(K, N, ld, h->step, h->burn, h->cfg.seed, (unsigned)h->gen, h->dLen, h->dDbStart,
                                                                    h->dSlot, h->dXP, h->dLPP, h->dEF, h->dCX, h->dCLL, h->dCLP, h->dDX, h->dDLL,
                                                                    h->dDLP, h->dAcc, h->dSc);
  h->launches++;
  CUDA_OK(h, cudaGetLastError());
  if (++h->step < h->steps) return 0;
  std::swap(h->dX, h->dDX); std::swap(h->dLL, h->dDLL); std::swap(h->dLP, h->dDLP);
  h->in_generation = false;
  if (tm_pull(h) || tm_check_flags(h)) return 1;
  h->gen++;
  return 0;
}

int ktmcmc_run_generation(ktmcmc_t* h) {
  if (!h) return fail(h, "null solver handle");
  if (h->gen == 1) return ktmcmc_propose(h) || ktmcmc_eval(h) || ktmcmc_accept(h);
  if (ktmcmc_anneal(h) || ktmcmc_resample(h)) return 1;
  while (h->in_generation)
    if (ktmcmc_propose(h) || ktmcmc_eval(h) || ktmcmc_accept(h)) return 1;
  return 0;
}

int ktmcmc_check_termination(ktmcmc_t* h, int* finished, const char** reason) {
  if (!h) return fail(h, "null solver handle");
  if (!finished) return fail(h, "null argument");
  CUDA_OK(h, cudaSetDevice(h->device));
  if (tm_pull(h)) return 1;
  h->reason.clear();
  int fin = 0;
  if (h->gen > 1 && h->hSc->rho >= h->tc_target) { h->reason += "Target Annealing Exponent;"; fin = 1; }
  if (h->tc_max_model_evaluations <= (double)(h->init_evals + h->hSc->evals)) { h->reason += "solver['Max Model Evaluations'];"; fin = 1; }
  if ((double)h->gen > h->tc_max_generations) { h->reason += "solver['Max Generations'];"; fin = 1; }
  *finished = fin;
  if (reason) *reason = h->reason.c_str();
  return 0;
}

int ktmcmc_run(ktmcmc_t* h, uint64_t max_generations, uint64_t* done) {
  return run(h, max_generations, done, ktmcmc_check_termination, ktmcmc_run_generation);
}

int ktmcmc_get_array(ktmcmc_t* h, const char* key, double* out, size_t cap, size_t* count) {
  if (!h) return fail(h, "null solver handle");
  if (!key) return fail(h, "null argument");
  CUDA_OK(h, cudaSetDevice(h->device));
  CUDA_OK(h, cudaStreamSynchronize(h->stream));
  const size_t N = h->N, ld = h->ld, lam = h->lambda, chains = h->chains;
  Array r;
  if (!strcmp(key, "Sample Database")) r = pitched(h->dX, lam, N, ld);
  else if (!strcmp(key, "Sample LogLikelihood Database")) r = dense(h->dLL, lam);
  else if (!strcmp(key, "Sample LogPrior Database")) r = dense(h->dLP, lam);
  else if (!strcmp(key, "Covariance Matrix")) r = pitched(h->dCov, N, N, ld);
  else if (!strcmp(key, "Proposal Factor")) r = pitched(h->dA, N, N, ld);
  else if (!strcmp(key, "Mean Theta")) r = dense(h->dMean, N);
  else if (!strcmp(key, "Weights")) r = dense(h->dW, lam);
  else if (!strcmp(key, "Selection Counts")) r = dense(h->dCounts, lam, Elem::i32);
  else if (!strcmp(key, "Chain Leaders")) r = dense(h->dLeader, chains, Elem::i32);
  else if (!strcmp(key, "Chain Lengths")) r = dense(h->dLen, chains, Elem::i32);
  else if (!strcmp(key, "Proposal Support")) r = dense(h->dFlag, chains, Elem::i32);
  else if (!strcmp(key, "Accept Flags")) r = dense(h->dAcc, chains, Elem::i32);
  else if (!strcmp(key, "Evaluation Rows")) {
    if (h->proposed && h->eval_rows < 0) { if (tm_pull(h)) return 1; h->eval_rows = (int)h->hSc->step_evals; }
    r = pitched(h->dEX, h->proposed ? (size_t)h->eval_rows : 0, N, ld);
  } else if (!strcmp(key, "Evaluation LogLikelihoods")) {
    if (h->ef_rows < 0) { if (tm_pull(h)) return 1; h->ef_rows = (int)h->hSc->step_evals; }
    r = dense(h->dEF, (size_t)h->ef_rows);
  } else return fail(h, "unknown array key '%s'", key);
  return copy_out(h, key, r, out, cap, count, "get_array(%s): capacity %zu < %zu");
}

int ktmcmc_get_scalar(ktmcmc_t* h, const char* key, double* out) {
  if (!h) return fail(h, "null solver handle");
  if (!key || !out) return fail(h, "null argument");
  CUDA_OK(h, cudaSetDevice(h->device));
  if (tm_pull(h)) return 1;
  const TmScalars& s = *h->hSc;
  if (double* p = host_scalar(h, kHostScalars, key, false)) *out = *p;
  else if (!strcmp(key, "Annealing Exponent")) *out = s.rho;
  else if (!strcmp(key, "Previous Annealing Exponent")) *out = s.rho_prev;
  else if (!strcmp(key, "Annealing Exponent Update")) *out = s.delta;
  else if (!strcmp(key, "Coefficient Of Variation")) *out = s.cov;
  else if (!strcmp(key, "LogEvidence")) *out = s.logev;
  else if (!strcmp(key, "Max Loglikelihood")) *out = s.llmax;
  else if (!strcmp(key, "Chain Count")) *out = (double)s.chain_count;
  else if (!strcmp(key, "Max Chain Steps")) *out = (double)h->steps;
  else if (!strcmp(key, "Current Step")) *out = (double)h->step;
  else if (!strcmp(key, "Proposals Acceptance Rate")) *out = s.proposals ? (double)s.accepted / (double)s.proposals : 0.0;
  else if (!strcmp(key, "Selection Acceptance Rate")) *out = (double)s.leaders / (double)h->lambda;
  else if (!strcmp(key, "Model Evaluation Count")) *out = (double)(h->init_evals + s.evals);
  else if (!strcmp(key, "Current Generation")) *out = (double)h->gen;
  else if (!strcmp(key, "Population Size")) *out = (double)h->lambda;
  else if (!strcmp(key, "Burn In")) *out = (double)h->burn;
  else return fail(h, "unknown scalar key '%s'", key);
  return 0;
}

int ktmcmc_set_scalar(ktmcmc_t* h, const char* key, double v) {
  if (!h) return fail(h, "null solver handle");
  if (!key) return fail(h, "null argument");
  double* p = host_scalar(h, kHostScalars, key, true);
  if (!p) return fail(h, "unknown scalar key '%s'", key);
  *p = v;
  return 0;
}

uint64_t ktmcmc_launch_count(const ktmcmc_t* h) { return h ? h->launches : 0; }

}  // extern "C"
