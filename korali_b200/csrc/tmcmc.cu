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
//   ktmcmc_eval      launch_objective (built-in models) or the host / device conduit on the packed rows
//   ktmcmc_accept    tm_accept_kernel        Metropolis test, database append, acceptance statistics
// Compiled with --fmad=false: the arithmetic rounds like oracle/otmcmc.c (the device's exp / log / sincospi may differ from libm in
// the last bit; the GEMM and the SYRK sum in their own order).
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/ktmcmc.h"
#include "common.cuh"
#include "kernels.h"

namespace {

using namespace kc;

constexpr int kThreads = 1024;        // one-CTA reductions and scans: thread t owns a fixed slice (restated by the oracle)
constexpr int kMeanChunks = 64;       // row chunks of the weighted mean
constexpr uint32_t kKeyTag = 0x544d434du;   // "TMCM"
constexpr double kHalfLog2Pi = 0.91893853320467274178;

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
  int nan_flag, allinf_flag, pad0, pad1;
};

__device__ __forceinline__ double prior_term(int type, double a, double b, double x) {
  if (type == KTMCMC_PRIOR_UNIFORM) return (x >= a && x <= b) ? -log(b - a) : -INFINITY;
  const double z = (x - a) / b;
  return -0.5 * (z * z) - log(b) - kHalfLog2Pi;
}
// log-prior of one row: lane-strided partials, xor butterfly (all lanes return the same bits)
__device__ __forceinline__ double log_prior_row(const double* __restrict__ x, int n, const int* __restrict__ type,
                                                const double* __restrict__ pa, const double* __restrict__ pb, int lane) {
  double p = 0.0;
  for (int d = lane; d < n; d += 32) p = p + prior_term(type[d], pa[d], pb[d], x[d]);
  return warp_sum_butterfly(p);
}

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

unsigned grid_for(long long threads, int per) { return (unsigned)std::max<long long>(1, (threads + per - 1) / per); }

}  // namespace

struct ktmcmc {
  ktmcmc_cfg cfg;
  int N = 0, ld = 0, lambda = 0, device = 0, num_sms = 148, L = 1;
  uint64_t gen = 1, launches = 0;
  std::vector<uint64_t> burn_in;
  cudaStream_t stream = 0;
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
  TmScalars* dSc = nullptr;
  TmScalars* hSc = nullptr;          // pinned
  TridiagWs* tri = nullptr;
  // generation state on the host
  int chains = 0, steps = 0, step = 0, burn = 0, eval_rows = 0;
  bool in_generation = false, proposed = false, evaluated = false, have_inj = false;
  uint64_t init_evals = 0;
  double tc_target = 1.0, tc_max_generations = 1e10, tc_max_model_evaluations = 1e9;
  ktmcmc_host_loglik_fn host_fn = nullptr; void* host_user = nullptr;
  kcma_device_objective_fn dev_fn = nullptr; void* dev_user = nullptr;
  std::vector<double> hX, hF;
  std::string err, reason;
  std::vector<void*> allocs;
};

namespace {
char g_tm_err[512] = "";
int tm_fail(ktmcmc* h, const char* fmt, ...) {
  char buf[512];
  va_list ap; va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (h) h->err = buf; else snprintf(g_tm_err, sizeof(g_tm_err), "%s", buf);
  return 1;
}
#define TM_CUDA(h, call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return tm_fail(h, "CUDA error %s at %s:%d", cudaGetErrorString(e_), __FILE__, __LINE__); } while (0)
template <typename T>
cudaError_t tm_alloc(ktmcmc* h, T** p, size_t count) {
  cudaError_t e = cudaMalloc((void**)p, sizeof(T) * (count ? count : 1));
  if (e == cudaSuccess) { h->allocs.push_back(*p); e = cudaMemset(*p, 0, sizeof(T) * (count ? count : 1)); }
  return e;
}
int tm_pull(ktmcmc* h) {
  TM_CUDA(h, cudaMemcpyAsync(h->hSc, h->dSc, sizeof(TmScalars), cudaMemcpyDeviceToHost, h->stream));
  TM_CUDA(h, cudaStreamSynchronize(h->stream));
  TM_CUDA(h, cudaGetLastError());
  return 0;
}
int tm_check_flags(ktmcmc* h) {
  if (h->hSc->nan_flag) return tm_fail(h, "A NaN log-likelihood was produced by the likelihood model\n");
  if (h->hSc->allinf_flag) return tm_fail(h, "Every sample of the population has a log-likelihood of -inf: the annealing step is undefined\n");
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

const char* ktmcmc_last_error(const ktmcmc_t* h) { return h ? h->err.c_str() : g_tm_err; }

void ktmcmc_destroy(ktmcmc_t* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);
  if (h->tri) tridiag_ws_destroy(h->tri);
  for (void* p : h->allocs) cudaFree(p);
  if (h->hSc) cudaFreeHost(h->hSc);
  delete h;
}

int ktmcmc_create(const ktmcmc_cfg* cfg, ktmcmc_t** out) {
  if (!cfg || !out) return tm_fail(nullptr, "null argument");
  if (cfg->abi_version != KTMCMC_ABI_VERSION) return tm_fail(nullptr, "ktmcmc_cfg ABI version mismatch");
  if (cfg->n < 1) return tm_fail(nullptr, "Bayesian problems require at least one variable.\n");
  if (cfg->population_size < 2) return tm_fail(nullptr, "Sampler/TMCMC: 'Population Size' must be at least 2 (got %zu)\n", (size_t)cfg->population_size);
  if (cfg->population_size > (1u << 30)) return tm_fail(nullptr, "Sampler/TMCMC: 'Population Size' above 2^30 is not supported\n");
  if (cfg->max_chain_length < 1) return tm_fail(nullptr, "Sampler/TMCMC: 'Max Chain Length' must be at least 1\n");
  if (!(cfg->target_cov > 0.0)) return tm_fail(nullptr, "Sampler/TMCMC: 'Target Coefficient Of Variation' must be positive\n");
  if (!(cfg->covariance_scaling > 0.0)) return tm_fail(nullptr, "Sampler/TMCMC: 'Covariance Scaling' must be positive\n");
  if (!(cfg->min_annealing_update > 0.0) || !(cfg->max_annealing_update >= cfg->min_annealing_update))
    return tm_fail(nullptr, "Sampler/TMCMC: need 0 < 'Min Annealing Exponent Update' <= 'Max Annealing Exponent Update'\n");
  if (!cfg->prior_type || !cfg->prior_a || !cfg->prior_b) return tm_fail(nullptr, "Sampler/TMCMC: every variable needs a prior distribution\n");
  const int N = (int)cfg->n;
  for (int d = 0; d < N; d++) {
    const int t = cfg->prior_type[d];
    const double a = cfg->prior_a[d], b = cfg->prior_b[d];
    if (t == KTMCMC_PRIOR_UNIFORM) {
      if (!std::isfinite(a) || !std::isfinite(b) || !(b > a)) return tm_fail(nullptr, "Univariate/Uniform prior of variable %d: need finite Minimum < Maximum\n", d);
    } else if (t == KTMCMC_PRIOR_NORMAL) {
      if (!std::isfinite(a) || !std::isfinite(b) || !(b > 0.0)) return tm_fail(nullptr, "Univariate/Normal prior of variable %d: need a finite Mean and a positive Standard Deviation\n", d);
    } else return tm_fail(nullptr, "unknown prior type %d of variable %d", t, d);
  }
  if (cfg->loglik != KCMA_OBJ_EXTERNAL && (cfg->loglik < KCMA_OBJ_NEG_SPHERE || cfg->loglik > KCMA_OBJ_NEG_SPHERE_SIN2))
    return tm_fail(nullptr, "unknown log-likelihood model id %d", cfg->loglik);
  if (!eigen_use_small(N) && !eigen_tridiag_fits(N)) return tm_fail(nullptr, "Sampler/TMCMC: n = %d is above the tridiagonal eigensolver's size\n", N);
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) return tm_fail(nullptr, "no CUDA device: korali_b200 has no CPU fallback");
  if (cfg->device < 0 || cfg->device >= ndev) return tm_fail(nullptr, "invalid device %d", cfg->device);
  ktmcmc* h = new ktmcmc();
  h->cfg = *cfg;
  h->burn_in.assign(cfg->per_generation_burn_in, cfg->per_generation_burn_in + (cfg->per_generation_burn_in ? cfg->burn_in_count : 0));
  h->cfg.per_generation_burn_in = nullptr; h->cfg.prior_type = nullptr; h->cfg.prior_a = h->cfg.prior_b = h->cfg.loglik_coef = nullptr;
  h->N = N; h->ld = (N + 15) / 16 * 16; h->lambda = (int)cfg->population_size; h->device = cfg->device;
  h->L = (int)std::min<uint64_t>(cfg->max_chain_length, cfg->population_size);
#define CREATE_CUDA(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { tm_fail(nullptr, "CUDA error %s at %s:%d", cudaGetErrorString(e_), __FILE__, __LINE__); ktmcmc_destroy(h); return 1; } } while (0)
  CREATE_CUDA(cudaSetDevice(h->device));
  cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, h->device);
  const size_t ld = h->ld, lam = h->lambda, rows = (lam + 15) / 16 * 16 + 16;
  h->s_rows = (long long)rows;
  CREATE_CUDA(tm_alloc(h, &h->dType, N)); CREATE_CUDA(tm_alloc(h, &h->dPa, N)); CREATE_CUDA(tm_alloc(h, &h->dPb, N)); CREATE_CUDA(tm_alloc(h, &h->dCoef, N));
  for (double** p : {&h->dX, &h->dDX, &h->dCX, &h->dZ, &h->dY, &h->dXP, &h->dEX, &h->dS}) CREATE_CUDA(tm_alloc(h, p, rows * ld));
  for (double** p : {&h->dLL, &h->dLP, &h->dDLL, &h->dDLP, &h->dCLL, &h->dCLP, &h->dLPP, &h->dEF, &h->dW, &h->dCum}) CREATE_CUDA(tm_alloc(h, p, lam));
  for (int** p : {&h->dCounts, &h->dLeader, &h->dLen, &h->dDbStart, &h->dFlag, &h->dSlot, &h->dAcc}) CREATE_CUDA(tm_alloc(h, p, lam));
  CREATE_CUDA(tm_alloc(h, &h->dPerm, 2 * (size_t)N + 64));
  CREATE_CUDA(tm_alloc(h, &h->dPart, (size_t)kMeanChunks * ld)); CREATE_CUDA(tm_alloc(h, &h->dMean, ld));
  CREATE_CUDA(tm_alloc(h, &h->dWs, (size_t)16 * N * ld));
  for (double** p : {&h->dP, &h->dCov, &h->dVT, &h->dGT, &h->dB, &h->dA}) CREATE_CUDA(tm_alloc(h, p, (size_t)N * ld));
  CREATE_CUDA(tm_alloc(h, &h->dD, ld)); CREATE_CUDA(tm_alloc(h, &h->dSign, ld));
  CREATE_CUDA(tm_alloc(h, &h->dDsc, 1)); CREATE_CUDA(tm_alloc(h, &h->dSc, 1));
  CREATE_CUDA(cudaMallocHost((void**)&h->hSc, sizeof(TmScalars)));
  memset(h->hSc, 0, sizeof(TmScalars));
  std::vector<int> type(cfg->prior_type, cfg->prior_type + N);
  std::vector<double> coef(N);
  for (int d = 0; d < N; d++) coef[d] = cfg->loglik_coef ? cfg->loglik_coef[d] : pow(10.0, 6.0 * d / (double)std::max(N - 1, 1));
  CREATE_CUDA(cudaMemcpy(h->dType, type.data(), sizeof(int) * N, cudaMemcpyHostToDevice));
  CREATE_CUDA(cudaMemcpy(h->dPa, cfg->prior_a, sizeof(double) * N, cudaMemcpyHostToDevice));
  CREATE_CUDA(cudaMemcpy(h->dPb, cfg->prior_b, sizeof(double) * N, cudaMemcpyHostToDevice));
  CREATE_CUDA(cudaMemcpy(h->dCoef, coef.data(), sizeof(double) * N, cudaMemcpyHostToDevice));
  DevScalars ds; memset(&ds, 0, sizeof(ds)); ds.sigma = 1.0;
  CREATE_CUDA(cudaMemcpy(h->dDsc, &ds, sizeof(ds), cudaMemcpyHostToDevice));
  launch_set_identity(h->stream, h->dVT, (int)ld, N);
  launch_set_identity(h->stream, h->dB, (int)ld, N);
  if (!eigen_use_small(N)) {
    char msg[512] = "";
    h->tri = tridiag_ws_create(N, (int)ld, h->num_sms, msg, sizeof(msg));
    if (!h->tri) { tm_fail(nullptr, "%s", msg); ktmcmc_destroy(h); return 1; }
  }
  CREATE_CUDA(cudaStreamSynchronize(h->stream));
  CREATE_CUDA(cudaGetLastError());
#undef CREATE_CUDA
  *out = h;
  return 0;
}

int ktmcmc_set_host_loglik(ktmcmc_t* h, ktmcmc_host_loglik_fn fn, void* user) {
  if (!h) return tm_fail(nullptr, "null solver handle");
  h->host_fn = fn; h->host_user = user;
  return 0;
}
int ktmcmc_set_device_loglik(ktmcmc_t* h, kcma_device_objective_fn fn, void* user) {
  if (!h) return tm_fail(nullptr, "null solver handle");
  h->dev_fn = fn; h->dev_user = user;
  return 0;
}

// steps 1-3
int ktmcmc_anneal(ktmcmc_t* h) {
  if (!h) return tm_fail(nullptr, "null solver handle");
  if (h->gen < 2 || h->in_generation) return tm_fail(h, "anneal: expected the start of a generation after the first");
  TM_CUDA(h, cudaSetDevice(h->device));
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
      return tm_fail(h, "the tridiagonal eigensolver could not be launched: %s", cudaGetErrorString(cudaGetLastError()));
    launch_eig_sign(st, vt, ld, N, h->dSign);
    launch_eig_order(st, ev, N, h->dPerm, h->dDsc);
    tm_commit_kernel<<<dim3((N + 127) / 128, N), 128, 0, st>>>(vt, ld, N, h->dPerm, ev, h->dSign, h->dA);
    h->launches += l + 4;
  }
  TM_CUDA(h, cudaGetLastError());
  h->in_generation = true;
  h->chains = 0;
  return 0;
}

// step 4; reads the chain count and the longest chain (the number of MCMC steps)
int ktmcmc_resample(ktmcmc_t* h) {
  if (!h) return tm_fail(nullptr, "null solver handle");
  if (!h->in_generation || h->chains) return tm_fail(h, "resample: call ktmcmc_anneal first");
  TM_CUDA(h, cudaSetDevice(h->device));
  const int lam = h->lambda;
  cudaStream_t st = h->stream;
  TM_CUDA(h, cudaMemsetAsync(h->dCounts, 0, sizeof(int) * lam, st));
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
  if (!h) return tm_fail(nullptr, "null solver handle");
  TM_CUDA(h, cudaSetDevice(h->device));
  const int N = h->N, ld = h->ld;
  cudaStream_t st = h->stream;
  if (h->gen == 1) {
    if (h->proposed) return tm_fail(h, "propose: the prior draws of generation 1 are waiting for eval / accept");
    tm_prior_kernel<<<grid_for((long long)h->lambda * 32, 256), 256, 0, st>>>(N, h->lambda, h->cfg.seed, h->dType, h->dPa, h->dPb, h->dEX, ld, h->dLP);
    h->launches++;
    h->eval_rows = h->lambda;
  } else {
    if (!h->in_generation || !h->chains || h->step >= h->steps || h->proposed) return tm_fail(h, "propose: no MCMC step pending (anneal and resample first)");
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
  TM_CUDA(h, cudaGetLastError());
  h->proposed = true;
  h->evaluated = false;
  return 0;
}

int ktmcmc_inject_loglik(ktmcmc_t* h, const double* l, size_t count) {
  if (!h) return tm_fail(nullptr, "null solver handle");
  if (!h->proposed || h->evaluated) return tm_fail(h, "inject_loglik: no proposals waiting for an evaluation");
  TM_CUDA(h, cudaSetDevice(h->device));
  if (h->eval_rows < 0) { if (tm_pull(h)) return 1; h->eval_rows = (int)h->hSc->step_evals; }
  if (count != (size_t)h->eval_rows) return tm_fail(h, "inject_loglik: %zu values for %d evaluation rows", count, h->eval_rows);
  if (count) TM_CUDA(h, cudaMemcpyAsync(h->dEF, l, sizeof(double) * count, cudaMemcpyHostToDevice, h->stream));
  TM_CUDA(h, cudaStreamSynchronize(h->stream));
  h->have_inj = true;
  return 0;
}

int ktmcmc_inject_factor(ktmcmc_t* h, const double* a, size_t count) {
  if (!h) return tm_fail(nullptr, "null solver handle");
  if (count != (size_t)h->N * h->N) return tm_fail(h, "inject_factor: %zu values for %d x %d", count, h->N, h->N);
  TM_CUDA(h, cudaSetDevice(h->device));
  TM_CUDA(h, cudaMemcpy2DAsync(h->dA, sizeof(double) * h->ld, a, sizeof(double) * h->N, sizeof(double) * h->N, h->N, cudaMemcpyHostToDevice, h->stream));
  TM_CUDA(h, cudaStreamSynchronize(h->stream));
  return 0;
}

int ktmcmc_eval(ktmcmc_t* h) {
  if (!h) return tm_fail(nullptr, "null solver handle");
  if (!h->proposed || h->evaluated) return tm_fail(h, "eval: call ktmcmc_propose first");
  TM_CUDA(h, cudaSetDevice(h->device));
  const int N = h->N, ld = h->ld;
  cudaStream_t st = h->stream;
  if (h->have_inj) {
    h->have_inj = false;
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
        TM_CUDA(h, cudaMemcpy2DAsync(h->hX.data(), sizeof(double) * N, h->dEX, sizeof(double) * ld, sizeof(double) * N, rows, cudaMemcpyDeviceToHost, st));
        TM_CUDA(h, cudaStreamSynchronize(st));
        h->host_fn(h->host_user, h->hX.data(), (uint64_t)rows, (uint64_t)N, h->hF.data());
        TM_CUDA(h, cudaMemcpyAsync(h->dEF, h->hF.data(), sizeof(double) * rows, cudaMemcpyHostToDevice, st));
      }
    }
  } else {
    return tm_fail(h, "the log-likelihood is External: inject the values or set a host / device model before eval");
  }
  TM_CUDA(h, cudaGetLastError());
  h->evaluated = true;
  return 0;
}

int ktmcmc_accept(ktmcmc_t* h) {
  if (!h) return tm_fail(nullptr, "null solver handle");
  if (!h->evaluated) return tm_fail(h, "accept: call ktmcmc_eval first");
  TM_CUDA(h, cudaSetDevice(h->device));
  const int N = h->N, ld = h->ld, lam = h->lambda;
  cudaStream_t st = h->stream;
  h->proposed = h->evaluated = false;
  if (h->gen == 1) {
    TM_CUDA(h, cudaMemcpyAsync(h->dX, h->dEX, sizeof(double) * lam * ld, cudaMemcpyDeviceToDevice, st));
    TM_CUDA(h, cudaMemcpyAsync(h->dLL, h->dEF, sizeof(double) * lam, cudaMemcpyDeviceToDevice, st));
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
  TM_CUDA(h, cudaGetLastError());
  if (++h->step < h->steps) return 0;
  std::swap(h->dX, h->dDX); std::swap(h->dLL, h->dDLL); std::swap(h->dLP, h->dDLP);
  h->in_generation = false;
  if (tm_pull(h) || tm_check_flags(h)) return 1;
  h->gen++;
  return 0;
}

int ktmcmc_run_generation(ktmcmc_t* h) {
  if (!h) return tm_fail(nullptr, "null solver handle");
  if (h->gen == 1) return ktmcmc_propose(h) || ktmcmc_eval(h) || ktmcmc_accept(h);
  if (ktmcmc_anneal(h) || ktmcmc_resample(h)) return 1;
  while (h->in_generation)
    if (ktmcmc_propose(h) || ktmcmc_eval(h) || ktmcmc_accept(h)) return 1;
  return 0;
}

int ktmcmc_check_termination(ktmcmc_t* h, int* finished, const char** reason) {
  if (!h || !finished) return tm_fail(h, "null argument");
  TM_CUDA(h, cudaSetDevice(h->device));
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
  if (!h) return tm_fail(nullptr, "null solver handle");
  uint64_t g = 0;
  for (; g < max_generations; g++) {
    int fin; const char* why;
    if (ktmcmc_check_termination(h, &fin, &why)) return 1;
    if (fin) break;
    if (ktmcmc_run_generation(h)) return 1;
  }
  if (done) *done = g;
  return 0;
}

int ktmcmc_get_array(ktmcmc_t* h, const char* key, double* out, size_t cap, size_t* count) {
  if (!h || !key) return tm_fail(h, "null argument");
  TM_CUDA(h, cudaSetDevice(h->device));
  TM_CUDA(h, cudaStreamSynchronize(h->stream));
  const size_t N = h->N, ld = h->ld, lam = h->lambda;
  const double* src = nullptr;
  const int* isrc = nullptr;
  size_t rows = 0, width = 1, pitch = 1;
  if (!strcmp(key, "Sample Database")) { src = h->dX; rows = lam; width = N; pitch = ld; }
  else if (!strcmp(key, "Sample LogLikelihood Database")) { src = h->dLL; rows = lam; }
  else if (!strcmp(key, "Sample LogPrior Database")) { src = h->dLP; rows = lam; }
  else if (!strcmp(key, "Covariance Matrix")) { src = h->dCov; rows = N; width = N; pitch = ld; }
  else if (!strcmp(key, "Proposal Factor")) { src = h->dA; rows = N; width = N; pitch = ld; }
  else if (!strcmp(key, "Mean Theta")) { src = h->dMean; rows = 1; width = N; pitch = ld; }
  else if (!strcmp(key, "Weights")) { src = h->dW; rows = lam; }
  else if (!strcmp(key, "Selection Counts")) { isrc = h->dCounts; rows = lam; }
  else if (!strcmp(key, "Chain Leaders")) { isrc = h->dLeader; rows = h->chains; }
  else if (!strcmp(key, "Chain Lengths")) { isrc = h->dLen; rows = h->chains; }
  else if (!strcmp(key, "Proposal Support")) { isrc = h->dFlag; rows = h->chains; }
  else if (!strcmp(key, "Accept Flags")) { isrc = h->dAcc; rows = h->chains; }
  else if (!strcmp(key, "Evaluation Rows")) {
    if (h->proposed && h->eval_rows < 0) { if (tm_pull(h)) return 1; h->eval_rows = (int)h->hSc->step_evals; }
    src = h->dEX; rows = h->proposed ? (size_t)h->eval_rows : 0; width = N; pitch = ld;
  } else return tm_fail(h, "unknown array key '%s'", key);
  const size_t n = rows * width;
  if (count) *count = n;
  if (!out) return 0;
  if (cap < n) return tm_fail(h, "get_array(%s): capacity %zu < %zu", key, cap, n);
  if (n == 0) return 0;
  if (isrc) {
    std::vector<int> tmp(n);
    TM_CUDA(h, cudaMemcpy(tmp.data(), isrc, sizeof(int) * n, cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < n; i++) out[i] = (double)tmp[i];
  } else {
    TM_CUDA(h, cudaMemcpy2D(out, sizeof(double) * width, src, sizeof(double) * pitch, sizeof(double) * width, rows, cudaMemcpyDeviceToHost));
  }
  return 0;
}

int ktmcmc_get_scalar(ktmcmc_t* h, const char* key, double* out) {
  if (!h || !key || !out) return tm_fail(h, "null argument");
  TM_CUDA(h, cudaSetDevice(h->device));
  if (tm_pull(h)) return 1;
  const TmScalars& s = *h->hSc;
  if (!strcmp(key, "Annealing Exponent")) *out = s.rho;
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
  else if (!strcmp(key, "Termination Criteria/Target Annealing Exponent")) *out = h->tc_target;
  else if (!strcmp(key, "Termination Criteria/Max Generations")) *out = h->tc_max_generations;
  else if (!strcmp(key, "Termination Criteria/Max Model Evaluations")) *out = h->tc_max_model_evaluations;
  else return tm_fail(h, "unknown scalar key '%s'", key);
  return 0;
}

int ktmcmc_set_scalar(ktmcmc_t* h, const char* key, double v) {
  if (!h || !key) return tm_fail(h, "null argument");
  if (!strcmp(key, "Termination Criteria/Target Annealing Exponent")) h->tc_target = v;
  else if (!strcmp(key, "Termination Criteria/Max Generations")) h->tc_max_generations = v;
  else if (!strcmp(key, "Termination Criteria/Max Model Evaluations")) h->tc_max_model_evaluations = v;
  else return tm_fail(h, "unknown scalar key '%s'", key);
  return 0;
}

uint64_t ktmcmc_launch_count(const ktmcmc_t* h) { return h ? h->launches : 0; }

}  // extern "C"
