// dea.cu — Differential Evolution generation loop on the B200 behind include/kdea.h: the sibling population solver of SURVEY 8f-4 on
// the kernels of the CMA-ES path (Philox streams, batched device objectives, batched host conduit). Replaces DEA.cpp.base:
//   initSamples :91-101          dea_init_kernel        one thread per (sample, dimension)
//   mutateSingle :123-186        dea_mutate_kernel      one warp per sample: lane 0 draws the parent indices (rejection loops of
//   fixInfeasible :188-201                              :125-133, :161-166), the lanes walk the dimensions (crossover draw per dimension,
//   isSampleFeasible                                    fix of the out-of-bounds part on redraws), warp vote = feasibility flag
//   prepareGeneration :103-121   rounds: every infeasible candidate is mutated again (attempt r of sample i = Philox(i, r): the same
//                                draws as the reference's per-sample do-while, whose iterations do not depend on other samples)
//   runGeneration :72-85         objective_kernel (X read directly) or the batched host conduit
//   updateSolver :203-282        dea_best_kernel (first maximum), dea_accept_kernel (the four accept rules; "Iterative" through a
//                                running maximum), dea_mean_kernel (mean in sample order, max - min per dimension)
// All arithmetic with explicit roundings (no FMA contraction): populations are bit-identical to oracle/odea.c.
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/kdea.h"
#include "common.cuh"
#include "handle.cuh"
#include "kernels.h"

namespace kc {
namespace {

__device__ __forceinline__ void dea_philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t out[4]) {
#pragma unroll
  for (int r = 0; r < 10; r++) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
__device__ __forceinline__ double dea_unit(uint32_t lo, uint32_t hi) {
  const unsigned long long v = ((unsigned long long)hi << 32) | lo;
  return (double)(v >> 12) * 0x1.0p-52 + 0x1.0p-53;
}
constexpr uint32_t DEA_IDX = 0u, DEA_CROSS = 1u << 20, DEA_FIX = 1u << 21;
// include/kdea.h: key = { seed_lo, seed_hi ^ "DEA!" }, ctr = { base + (k >> 1), sample, attempt, generation }, half (k & 1)
__device__ __forceinline__ double dea_uniform(unsigned long long seed, unsigned generation, unsigned attempt, unsigned long long sample, uint32_t base,
                                              uint32_t k) {
  uint32_t r[4];
  dea_philox(base + (k >> 1), (uint32_t)sample, attempt, generation, (uint32_t)seed, (uint32_t)(seed >> 32) ^ 0x44454121u, r);
  return (k & 1u) ? dea_unit(r[2], r[3]) : dea_unit(r[0], r[1]);
}

struct DeaScalars {
  double best_ever_value, prev_best_ever_value, cur_best_value, prev_best_value, min_step;
  unsigned long long infeasible, best_idx;
  int redo_count, pad;
};

// initSamples (:91-101): candidate = lower + width * u, sample = candidate
__global__ void __launch_bounds__(256)
dea_init_kernel(double* __restrict__ X, double* __restrict__ Xc, int ld, long long lambda, int n, const double* __restrict__ lower,
                const double* __restrict__ upper, unsigned long long seed) {
  const long long total = lambda * n;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const long long i = idx / n;
    const int d = (int)(idx - i * n);
    const double width = __dsub_rn(upper[d], lower[d]);
    const double v = __dadd_rn(lower[d], __dmul_rn(width, dea_uniform(seed, 0u, 0u, (unsigned long long)i, DEA_CROSS, (uint32_t)d)));
    Xc[(size_t)i * ld + d] = v;
    X[(size_t)i * ld + d] = v;
  }
}

// mutateSingle (:123-186) + fixInfeasible (:188-201, on redraws: the flag of the PREVIOUS attempt decides, :113) + isSampleFeasible.
// One warp per listed sample (rows == nullptr: all samples, attempt 0).
__global__ void __launch_bounds__(256)
dea_mutate_kernel(const double* __restrict__ X, double* __restrict__ Xc, int ld, long long lambda, int n, const int* __restrict__ rows, int count,
                  const unsigned* __restrict__ attempt, const double* __restrict__ lower, const double* __restrict__ upper, double crossover_rate,
                  double mutation_rate, int parent_rule, int fix_infeasible, unsigned long long seed, unsigned generation,
                  const DeaScalars* __restrict__ sc, unsigned char* __restrict__ infeasible) {
  const int lane = threadIdx.x & 31;
  const long long w = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  if (w >= count) return;
  const long long i = rows ? rows[w] : w;
  const unsigned att = attempt ? attempt[i] : 0u;
  unsigned long long a = 0, b = 0, c = 0, rn = 0;
  if (lane == 0) {
    uint32_t k = 0;
    do { a = (unsigned long long)(dea_uniform(seed, generation, att, i, DEA_IDX, k++) * (double)lambda); } while (a == (unsigned long long)i);
    do { b = (unsigned long long)(dea_uniform(seed, generation, att, i, DEA_IDX, k++) * (double)lambda); } while (b == (unsigned long long)i || b == a);
    if (parent_rule == KDEA_PARENT_RANDOM) {
      do { c = (unsigned long long)(dea_uniform(seed, generation, att, i, DEA_IDX, k++) * (double)lambda); } while (c == (unsigned long long)i || c == a || c == b);
    } else {
      c = sc->best_idx;
    }
    rn = (unsigned long long)(dea_uniform(seed, generation, att, i, DEA_IDX, k++) * (double)n);
  }
  a = __shfl_sync(0xffffffffu, a, 0); b = __shfl_sync(0xffffffffu, b, 0); c = __shfl_sync(0xffffffffu, c, 0); rn = __shfl_sync(0xffffffffu, rn, 0);
  const double* xa = X + (size_t)a * ld;
  const double* xb = X + (size_t)b * ld;
  const double* xp = X + (size_t)c * ld;
  const double* xi = X + (size_t)i * ld;
  double* out = Xc + (size_t)i * ld;
  const bool fix = fix_infeasible && att > 0;
  bool ok = true;
  for (int d = lane; d < n; d += 32) {
    double v;
    if ((dea_uniform(seed, generation, att, i, DEA_CROSS, (uint32_t)d) < crossover_rate) || ((unsigned long long)d == rn))
      v = __dadd_rn(xp[d], __dmul_rn(mutation_rate, __dsub_rn(xa[d], xb[d])));
    else
      v = xi[d];
    if (fix) {
      double len = 0.0;
      if (v < lower[d]) len = __dsub_rn(v, lower[d]);
      if (v > upper[d]) len = __dsub_rn(v, upper[d]);
      v = __dsub_rn(xi[d], __dmul_rn(len, dea_uniform(seed, generation, att, i, DEA_FIX, (uint32_t)d)));
    }
    out[d] = v;
    ok = ok && isfinite(v) && !(v < lower[d]) && !(v > upper[d]);
  }
  ok = __all_sync(0xffffffffu, ok);
  if (lane == 0) infeasible[i] = ok ? 0 : 1;
}

// infeasible flags -> list of samples to mutate again (any order: the mutation of a sample depends on no other candidate), their
// attempt counters, the infeasible counter (:116). Warp-aggregated atomics on the counter in DeaScalars (zeroed by the caller).
__global__ void __launch_bounds__(256)
dea_compact_kernel(const unsigned char* __restrict__ flags, long long lambda, int* __restrict__ rows, unsigned* __restrict__ attempt, DeaScalars* __restrict__ sc) {
  const int lane = threadIdx.x & 31;
  for (long long base = (long long)blockIdx.x * blockDim.x; base < lambda; base += (long long)gridDim.x * blockDim.x) {
    const long long j = base + threadIdx.x;
    const bool take = j < lambda && flags[j] != 0;
    const unsigned m = __ballot_sync(0xffffffffu, take);
    if (m == 0) continue;
    int pos = 0;
    if (lane == 0) {
      pos = atomicAdd(&sc->redo_count, __popc(m));
      atomicAdd(&sc->infeasible, (unsigned long long)__popc(m));
    }
    pos = __shfl_sync(0xffffffffu, pos, 0);
    if (take) { rows[pos + __popc(m & ((1u << lane) - 1u))] = (int)j; attempt[j]++; }
  }
}
__global__ void dea_zero_redo_kernel(DeaScalars* sc) { sc->redo_count = 0; }

// _bestSampleIndex = first maximum of F (std::max_element, :209), previous / current best values (:210-212). Single block.
__global__ void __launch_bounds__(1024)
dea_best_kernel(const double* __restrict__ F, long long lambda, DeaScalars* __restrict__ sc) {
  __shared__ double sv[32];
  __shared__ long long si[32];
  double bv = -INFINITY;
  long long bi = 0x7fffffffffffffffll;
  for (long long j = threadIdx.x; j < lambda; j += blockDim.x) {
    const double v = F[j];
    if (bi == 0x7fffffffffffffffll || v > bv) { bv = v; bi = j; }   // per thread: ascending j, strict > keeps the first maximum
  }
  for (int off = 16; off >= 1; off >>= 1) {
    const double ov = __shfl_xor_sync(0xffffffffu, bv, off);
    const long long oi = __shfl_xor_sync(0xffffffffu, bi, off);
    if (oi != 0x7fffffffffffffffll && (bi == 0x7fffffffffffffffll || ov > bv || (ov == bv && oi < bi))) { bv = ov; bi = oi; }
  }
  if ((threadIdx.x & 31) == 0) { sv[threadIdx.x >> 5] = bv; si[threadIdx.x >> 5] = bi; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 0; w < (int)(blockDim.x >> 5); w++)
      if (si[w] != 0x7fffffffffffffffll && (bi == 0x7fffffffffffffffll || sv[w] > bv || (sv[w] == bv && si[w] < bi))) { bv = sv[w]; bi = si[w]; }
    sc->best_idx = (unsigned long long)bi;
    sc->prev_best_ever_value = sc->best_ever_value;
    sc->prev_best_value = sc->cur_best_value;
    sc->cur_best_value = bv;
  }
}

// "Iterative" (:258-267): sample i is accepted iff F[i] > the running best-ever value, which then becomes F[i]:
// accept_i = F[i] > max(best_ever_0, max_{j<i} F[j]). Exclusive running maximum by one block (chunked scan).
__global__ void __launch_bounds__(1024)
dea_running_max_kernel(const double* __restrict__ F, long long lambda, const DeaScalars* __restrict__ sc, unsigned char* __restrict__ accept) {
  __shared__ double wmax[32];
  __shared__ double carry;
  if (threadIdx.x == 0) carry = sc->best_ever_value;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (long long base = 0; base < lambda; base += 1024) {
    const long long j = base + threadIdx.x;
    const double v = j < lambda ? F[j] : -INFINITY;
    double incl = v;   // inclusive max scan inside the warp
    for (int off = 1; off < 32; off <<= 1) { const double y = __shfl_up_sync(0xffffffffu, incl, off); if (lane >= off) incl = fmax(incl, y); }
    if (lane == 31) wmax[warp] = incl;
    __syncthreads();
    if (warp == 0) {
      double x = wmax[lane];
      for (int off = 1; off < 32; off <<= 1) { const double y = __shfl_up_sync(0xffffffffu, x, off); if (lane >= off) x = fmax(x, y); }
      wmax[lane] = x;
    }
    __syncthreads();
    double excl = __shfl_up_sync(0xffffffffu, incl, 1);
    if (lane == 0) excl = -INFINITY;
    excl = fmax(excl, carry);
    if (warp > 0) excl = fmax(excl, wmax[warp - 1]);
    if (j < lambda) accept[j] = v > excl ? 1 : 0;
    __syncthreads();
    if (threadIdx.x == 0) carry = fmax(carry, wmax[31]);
    __syncthreads();
  }
}

// current best / best ever variables (:214, :219) and the accept rules (:222-267); one thread per (sample, dimension) element.
__global__ void __launch_bounds__(256)
dea_accept_kernel(double* __restrict__ X, const double* __restrict__ Xc, int ld, long long lambda, int n, const double* __restrict__ F,
                  const double* __restrict__ Fprev, int rule, const unsigned char* __restrict__ iter_accept, const DeaScalars* __restrict__ sc,
                  double* __restrict__ cur_best, double* __restrict__ best_ever) {
  const double best_ever_value = sc->best_ever_value, cur_best_value = sc->cur_best_value;
  const long long best = (long long)sc->best_idx;
  const long long total = lambda * n;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const long long i = idx / n;
    const int d = (int)(idx - i * n);
    const double cand = Xc[(size_t)i * ld + d];
    if (i == best) {
      cur_best[d] = cand;
      if (cur_best_value > best_ever_value) best_ever[d] = cand;
    }
    bool acc;
    if (rule == KDEA_ACCEPT_BEST) acc = (i == best) && (cur_best_value > best_ever_value);
    else if (rule == KDEA_ACCEPT_GREEDY) acc = F[i] > Fprev[i];
    else if (rule == KDEA_ACCEPT_IMPROVED) acc = F[i] > best_ever_value;
    else acc = iter_accept[i] != 0;
    if (acc) X[(size_t)i * ld + d] = cand;
  }
}

// best-ever value after the accept rules (:227, :238, :250, :264): the maximum seen so far in every rule that fired
__global__ void dea_best_ever_kernel(DeaScalars* sc) {
  if (sc->cur_best_value > sc->best_ever_value) sc->best_ever_value = sc->cur_best_value;
  sc->min_step = INFINITY;   // :280-281: the result of std::min is discarded in the reference — the value stays +Inf
}

// mean in sample order (:271-273: every term divided by lambda, added for i = 0, 1, ...), max - min per dimension (:275-285).
// The additions of a dimension are one dependent chain (the reference's rounding), lambda x 8 cycles long; everything else is taken
// off that chain: a block owns 32 dimensions, all 256 threads fetch the next tile of 256 samples x 32 dimensions (32 loads in flight
// per thread, coalesced) and divide, while warp 0 adds the current tile from shared memory, one lane per dimension.
constexpr int DM_TS = 256, DM_NT = 256, DM_LD = 33;
__global__ void __launch_bounds__(DM_NT)
dea_mean_kernel(const double* __restrict__ X, int ld, long long lambda, int n, double* __restrict__ mean, double* __restrict__ prev_mean,
                double* __restrict__ maxdist) {
  extern __shared__ double tile[];                 // DM_TS x DM_LD quotients
  __shared__ double smx[DM_NT], smn[DM_NT];
  const int tid = threadIdx.x, dd = tid & 31, srow = tid >> 5, d0 = blockIdx.x * 32, d = d0 + dd;
  const double inv = (double)lambda;
  constexpr int PER = DM_TS * 32 / DM_NT;          // 32 elements per thread and tile: samples srow, srow + 8, ...
  double m = 0.0, mx = -INFINITY, mn = INFINITY;
  double reg[PER];
  auto fetch = [&](long long t0) {
#pragma unroll
    for (int k = 0; k < PER; k++) {
      const long long i = t0 + srow + 8 * k;
      reg[k] = (i < lambda && d < n) ? X[(size_t)i * ld + d] : 0.0;
    }
  };
  fetch(0);
  for (long long t0 = 0; t0 < lambda; t0 += DM_TS) {
#pragma unroll
    for (int k = 0; k < PER; k++) {
      const long long i = t0 + srow + 8 * k;
      if (i < lambda && d < n) { if (reg[k] > mx) mx = reg[k]; if (reg[k] < mn) mn = reg[k]; }
      tile[(srow + 8 * k) * DM_LD + dd] = __ddiv_rn(reg[k], inv);
    }
    __syncthreads();
    if (t0 + DM_TS < lambda) fetch(t0 + DM_TS);    // in flight while warp 0 walks the chain
    if (tid < 32) {
      const int cnt = (int)min((long long)DM_TS, lambda - t0);
      int sidx = 0;
      for (; sidx + 16 <= cnt; sidx += 16) {   // 16 quotients loaded together, added in order: the chain runs at the DADD latency
        double q[16];
#pragma unroll
        for (int k = 0; k < 16; k++) q[k] = tile[(sidx + k) * DM_LD + dd];
#pragma unroll
        for (int k = 0; k < 16; k++) m = __dadd_rn(m, q[k]);
      }
      for (; sidx < cnt; sidx++) m = __dadd_rn(m, tile[sidx * DM_LD + dd]);
    }
    __syncthreads();
  }
  smx[tid] = mx; smn[tid] = mn;
  __syncthreads();
  if (tid < 32 && d < n) {
    for (int k = 1; k < 8; k++) { mx = fmax(mx, smx[tid + 32 * k]); mn = fmin(mn, smn[tid + 32 * k]); }
    prev_mean[d] = mean[d];
    mean[d] = m;
    maxdist[d] = __dsub_rn(mx, mn);
  }
}
void launch_dea_mean(cudaStream_t st, const double* X, int ld, long long lambda, int n, double* mean, double* prev_mean, double* maxdist) {
  static std::atomic<unsigned long long> attr{0};
  const size_t smem = sizeof(double) * DM_TS * DM_LD;
  if (first_call_on_device(attr)) cudaFuncSetAttribute(dea_mean_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  dea_mean_kernel<<<(n + 31) / 32, DM_NT, smem, st>>>(X, ld, lambda, n, mean, prev_mean, maxdist);
}

}  // namespace
}  // namespace kc

using namespace kc;

struct kdea : Handle<kdea, DeaScalars> {
  kdea_cfg cfg;
  int N = 0, ld = 0, num_sms = 148;
  long long lambda = 0;
  std::vector<double> lower, upper, coef;
  double *dX = nullptr, *dXc = nullptr, *dF = nullptr, *dFprev = nullptr, *dMean = nullptr, *dPrevMean = nullptr, *dBestEver = nullptr,
         *dCurBest = nullptr, *dMaxDist = nullptr, *dLower = nullptr, *dUpper = nullptr, *dCoef = nullptr;
  int* dRows = nullptr;
  unsigned* dAttempt = nullptr;
  unsigned char *dInfeasible = nullptr, *dIterAccept = nullptr;
  DevScalars* dObjSc = nullptr;   // sigma / nonfinite block the objective kernels expect
  uint64_t model_evals = 0;
  bool have_inj_f = false;
  kcma_host_objective_fn host_obj = nullptr; void* host_obj_user = nullptr;
  std::vector<double> hX, hF;
  double tc_max_infeasible = 1e7, tc_min_value = -INFINITY, tc_min_step = -INFINITY, tc_max_value = INFINITY, tc_min_value_diff = -INFINITY,
         tc_max_generations = 1e10, tc_max_model_evaluations = 1e9;
};

namespace {
const HostScalar<kdea> kHostScalars[] = {
    {"Termination Criteria/Max Infeasible Resamplings", &kdea::tc_max_infeasible, true},
    {"Termination Criteria/Min Value", &kdea::tc_min_value, true},
    {"Termination Criteria/Min Step Size", &kdea::tc_min_step, true},
    {"Termination Criteria/Max Value", &kdea::tc_max_value, true},
    {"Termination Criteria/Min Value Difference Threshold", &kdea::tc_min_value_diff, true},
    {"Termination Criteria/Max Generations", &kdea::tc_max_generations, true},
    {"Termination Criteria/Max Model Evaluations", &kdea::tc_max_model_evaluations, true},
};
bool find_array(kdea* h, const char* key, Array* r) {
  const size_t N = h->N, L = (size_t)h->lambda, ld = h->ld;
#define A(K, ARR) if (!strcmp(key, K)) { *r = ARR; return true; }
  A("Sample Population", pitched(h->dX, L, N, ld)) A("Candidate Population", pitched(h->dXc, L, N, ld))
  A("Value Vector", dense(h->dF, L)) A("Previous Value Vector", dense(h->dFprev, L))
  A("Current Mean", dense(h->dMean, N)) A("Previous Mean", dense(h->dPrevMean, N)) A("Best Ever Variables", dense(h->dBestEver, N))
  A("Current Best Variables", dense(h->dCurBest, N)) A("Max Distances", dense(h->dMaxDist, N))
#undef A
  return false;
}
double* find_dev_scalar(kdea* h, const char* key) {
  DeaScalars* s = h->hSc;
#define S(K, F) if (!strcmp(key, K)) return &s->F;
  S("Best Ever Value", best_ever_value) S("Current Best Value", cur_best_value) S("Previous Best Value", prev_best_value)
  S("Previous Best Ever Value", prev_best_ever_value) S("Current Minimum Step Size", min_step)
#undef S
  return nullptr;
}
}  // namespace

extern "C" {

void kdea_cfg_defaults(kdea_cfg* c) {
  memset(c, 0, sizeof(*c));
  c->abi_version = KDEA_ABI_VERSION;
  c->population_size = 200; c->crossover_rate = 0.9; c->mutation_rate = 0.5;
  c->mutation_rule = KDEA_MUTATION_FIXED; c->parent_selection_rule = KDEA_PARENT_RANDOM; c->accept_rule = KDEA_ACCEPT_GREEDY;
  c->fix_infeasible = 1;
}

const char* kdea_last_error(const kdea_t* h) { return h ? h->err.c_str() : kdea::create_err; }

void kdea_destroy(kdea_t* h) { delete h; }

// setInitialConfiguration (:15-64)
int kdea_create(const kdea_cfg* cfg, kdea_t** out) {
  if (!cfg || !out) return fail<kdea>(nullptr, "kdea_create: null argument");
  if (cfg->abi_version != KDEA_ABI_VERSION) return fail<kdea>(nullptr, "kdea_cfg ABI version %u, library %u", cfg->abi_version, KDEA_ABI_VERSION);
  if (open_device<kdea>(cfg->device)) return 1;
  if (cfg->n == 0) return fail<kdea>(nullptr, "Optimization Evaluation problems require at least one variable.\n");
  if (cfg->n > (1u << 20)) return fail<kdea>(nullptr, "too many variables for the Philox sub-streams of DEA (%lu > 2^20)", (unsigned long)cfg->n);
  if (cfg->population_size < 4) return fail<kdea>(nullptr, "DEA needs a Population Size of at least 4 (three distinct partners per sample, DEA.cpp.base:125-166)");
  if (cfg->population_size > 0x7fffffffull) return fail<kdea>(nullptr, "Population Size too large");
  if (cfg->mutation_rule != KDEA_MUTATION_FIXED) return fail<kdea>(nullptr, "Mutation Rule 'Self Adaptive' is not built (its rates are global state updated sample by sample, DEA.cpp.base:136-156)");
  if (cfg->parent_selection_rule != KDEA_PARENT_RANDOM && cfg->parent_selection_rule != KDEA_PARENT_BEST) return fail<kdea>(nullptr, "Parent Selection Rule not recognized");
  if (cfg->accept_rule < KDEA_ACCEPT_BEST || cfg->accept_rule > KDEA_ACCEPT_ITERATIVE) return fail<kdea>(nullptr, "Accept Rule (%d) not recognized.\n", cfg->accept_rule);
  if (!cfg->lower_bound || !cfg->upper_bound) return fail<kdea>(nullptr, "DEA needs Lower Bound and Upper Bound for every variable (the initial population is uniform in the box)");
  kdea* h = new kdea();
  h->cfg = *cfg;
  h->N = (int)cfg->n; h->ld = (h->N + 15) / 16 * 16; h->lambda = (long long)cfg->population_size; h->device = cfg->device;
  const int N = h->N, ld = h->ld;
  h->lower.assign(cfg->lower_bound, cfg->lower_bound + N);
  h->upper.assign(cfg->upper_bound, cfg->upper_bound + N);
  for (int d = 0; d < N; d++) {
    if (!std::isfinite(h->lower[d]) || !std::isfinite(h->upper[d])) return create_fail(h, "DEA: variable %d needs finite bounds", d);
    if (h->upper[d] < h->lower[d]) return create_fail(h, "Lower Bound (%.4f) of variable %d exceeds Upper Bound (%.4f).\n", h->lower[d], d, h->upper[d]);
  }
  h->coef.resize(N);
  for (int d = 0; d < N; d++) h->coef[d] = cfg->objective_coef ? cfg->objective_coef[d] : pow(10.0, 6.0 * (double)d / (double)(N > 1 ? N - 1 : 1));
  h->cfg.lower_bound = h->cfg.upper_bound = h->cfg.objective_coef = nullptr;
  cudaDeviceProp prop;
  CREATE_OK(h, cudaGetDeviceProperties(&prop, h->device));
  h->num_sms = prop.multiProcessorCount;
  const size_t L = (size_t)h->lambda, mat = L * ld;
  Allocations& m = h->mem;
  CREATE_OK(h, alloc(m, &h->dX, mat)); CREATE_OK(h, alloc(m, &h->dXc, mat));
  CREATE_OK(h, alloc(m, &h->dF, L)); CREATE_OK(h, alloc(m, &h->dFprev, L));
  CREATE_OK(h, alloc(m, &h->dMean, ld)); CREATE_OK(h, alloc(m, &h->dPrevMean, ld));
  CREATE_OK(h, alloc(m, &h->dBestEver, ld)); CREATE_OK(h, alloc(m, &h->dCurBest, ld));
  CREATE_OK(h, alloc(m, &h->dMaxDist, ld)); CREATE_OK(h, alloc(m, &h->dLower, ld));
  CREATE_OK(h, alloc(m, &h->dUpper, ld)); CREATE_OK(h, alloc(m, &h->dCoef, ld));
  CREATE_OK(h, alloc(m, &h->dRows, L)); CREATE_OK(h, alloc(m, &h->dAttempt, L));
  CREATE_OK(h, alloc(m, &h->dInfeasible, L)); CREATE_OK(h, alloc(m, &h->dIterAccept, L));
  CREATE_OK(h, alloc(m, &h->dSc, 1)); CREATE_OK(h, alloc(m, &h->dObjSc, 1));
  CREATE_OK(h, alloc_host(m, &h->hSc, 1));
  CREATE_OK(h, cudaMemcpy(h->dLower, h->lower.data(), sizeof(double) * N, cudaMemcpyHostToDevice));
  CREATE_OK(h, cudaMemcpy(h->dUpper, h->upper.data(), sizeof(double) * N, cudaMemcpyHostToDevice));
  CREATE_OK(h, cudaMemcpy(h->dCoef, h->coef.data(), sizeof(double) * N, cudaMemcpyHostToDevice));
  h->hSc->best_ever_value = h->hSc->prev_best_ever_value = h->hSc->cur_best_value = h->hSc->prev_best_value = -INFINITY;
  h->hSc->min_step = INFINITY;
  CREATE_OK(h, cudaMemcpy(h->dSc, h->hSc, sizeof(DeaScalars), cudaMemcpyHostToDevice));
  std::vector<double> ninf(L, -INFINITY);   // _valueVector = -Inf (:37)
  CREATE_OK(h, cudaMemcpy(h->dF, ninf.data(), sizeof(double) * L, cudaMemcpyHostToDevice));
  CREATE_OK(h, cudaMemcpy(h->dFprev, ninf.data(), sizeof(double) * L, cudaMemcpyHostToDevice));
  dea_init_kernel<<<h->num_sms * 4, 256, 0, h->stream>>>(h->dX, h->dXc, ld, h->lambda, N, h->dLower, h->dUpper, cfg->seed);
  launch_dea_mean(h->stream, h->dX, ld, h->lambda, N, h->dMean, h->dPrevMean, h->dMaxDist);   // :60-63
  CREATE_OK(h, cudaMemset(h->dPrevMean, 0, sizeof(double) * ld));
  CREATE_OK(h, cudaMemset(h->dMaxDist, 0, sizeof(double) * ld));
  h->launches += 2;
  CREATE_OK(h, cudaDeviceSynchronize());
  *out = h;
  return 0;
}

int kdea_set_host_objective(kdea_t* h, kcma_host_objective_fn fn, void* user) {
  if (!h) return fail(h, "null solver handle");
  h->host_obj = fn; h->host_obj_user = user;
  return 0;
}

int kdea_inject_f(kdea_t* h, const double* f, size_t count) {
  if (!h) return fail(h, "null solver handle");
  if (count != (size_t)h->lambda) return fail(h, "inject F: expected %zu values", (size_t)h->lambda);
  for (size_t i = 0; i < count; i++) if (!std::isfinite(f[i])) return fail(h, "Non finite value of function evaluation detected: %f\n", f[i]);
  CUDA_OK(h, cudaSetDevice(h->device));
  h->hF.assign(f, f + count);
  h->have_inj_f = true;
  return 0;
}

// prepareGeneration (:103-121)
int kdea_ask(kdea_t* h) {
  if (!h) return fail(h, "null solver handle");
  CUDA_OK(h, cudaSetDevice(h->device));
  const int N = h->N, ld = h->ld;
  const long long L = h->lambda;
  if (h->gen > 1) {
    CUDA_OK(h, cudaMemsetAsync(h->dAttempt, 0, sizeof(unsigned) * (size_t)L, h->stream));
    const int wpb = 8;
    dea_mutate_kernel<<<(unsigned)((L + wpb - 1) / wpb), 256, 0, h->stream>>>(h->dX, h->dXc, ld, L, N, nullptr, (int)L, nullptr, h->dLower, h->dUpper,
                                                                            h->cfg.crossover_rate, h->cfg.mutation_rate, h->cfg.parent_selection_rule,
                                                                            h->cfg.fix_infeasible, h->cfg.seed, (unsigned)h->gen, h->dSc, h->dInfeasible);
    h->launches++;
    for (int round = 0;; round++) {
      dea_zero_redo_kernel<<<1, 1, 0, h->stream>>>(h->dSc);
      dea_compact_kernel<<<(unsigned)std::min<long long>((L + 255) / 256, (long long)h->num_sms * 4), 256, 0, h->stream>>>(h->dInfeasible, L, h->dRows, h->dAttempt, h->dSc);
      h->launches += 2;
      h->scalars_fresh = false;
      if (pull_cached(h)) return 1;
      const int cnt = h->hSc->redo_count;
      if (cnt == 0) break;
      if (round >= 100000) return fail(h, "a sample never becomes feasible (100000 mutations)");
      dea_mutate_kernel<<<(unsigned)((cnt + wpb - 1) / wpb), 256, 0, h->stream>>>(h->dX, h->dXc, ld, L, N, h->dRows, cnt, h->dAttempt, h->dLower, h->dUpper,
                                                                                h->cfg.crossover_rate, h->cfg.mutation_rate, h->cfg.parent_selection_rule,
                                                                                h->cfg.fix_infeasible, h->cfg.seed, (unsigned)h->gen, h->dSc, h->dInfeasible);
      h->launches++;
    }
  }
  CUDA_OK(h, cudaMemcpyAsync(h->dFprev, h->dF, sizeof(double) * (size_t)L, cudaMemcpyDeviceToDevice, h->stream));   // :120
  return 0;
}

// runGeneration :72-85 as one batched evaluation
int kdea_eval(kdea_t* h) {
  if (!h) return fail(h, "null solver handle");
  CUDA_OK(h, cudaSetDevice(h->device));
  const int N = h->N, ld = h->ld;
  const size_t L = (size_t)h->lambda;
  h->model_evals += L;
  if (h->have_inj_f) {
    h->have_inj_f = false;
    CUDA_OK(h, cudaMemcpyAsync(h->dF, h->hF.data(), sizeof(double) * L, cudaMemcpyHostToDevice, h->stream));
    CUDA_OK(h, cudaStreamSynchronize(h->stream));
    return 0;
  }
  if (h->host_obj) {
    h->hX.resize(L * N); h->hF.resize(L);
    CUDA_OK(h, cudaMemcpy2DAsync(h->hX.data(), sizeof(double) * N, h->dXc, sizeof(double) * ld, sizeof(double) * N, L, cudaMemcpyDeviceToHost, h->stream));
    CUDA_OK(h, cudaStreamSynchronize(h->stream));
    h->host_obj(h->host_obj_user, h->hX.data(), (uint64_t)L, (uint64_t)N, h->hF.data());
    for (size_t i = 0; i < L; i++)
      if (!std::isfinite(h->hF[i])) return fail(h, "Non finite value of function evaluation detected: %f\n", h->hF[i]);
    CUDA_OK(h, cudaMemcpyAsync(h->dF, h->hF.data(), sizeof(double) * L, cudaMemcpyHostToDevice, h->stream));
    CUDA_OK(h, cudaStreamSynchronize(h->stream));
    return 0;
  }
  if (h->cfg.objective == KCMA_OBJ_EXTERNAL) return fail(h, "objective is External: set a host objective or inject the Value Vector before eval");
  if (launch_objective(h->stream, h->cfg.objective, h->dXc, ld, (long long)L, N, 0, 1, h->dMean, h->dObjSc, h->dCoef, h->dF, h->num_sms))
    return fail(h, "unknown objective id %d", h->cfg.objective);
  h->launches++;
  int bad = 0;
  CUDA_OK(h, cudaMemcpyAsync(&bad, &h->dObjSc->nonfinite, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  CUDA_OK(h, cudaStreamSynchronize(h->stream));
  if (bad) {
    cudaMemsetAsync(&h->dObjSc->nonfinite, 0, sizeof(int), h->stream);
    return fail(h, "Non finite value of function evaluation detected: nan\n");
  }
  return 0;
}

// updateSolver (:203-282)
int kdea_tell(kdea_t* h) {
  if (!h) return fail(h, "null solver handle");
  CUDA_OK(h, cudaSetDevice(h->device));
  const int N = h->N, ld = h->ld;
  const long long L = h->lambda;
  dea_best_kernel<<<1, 1024, 0, h->stream>>>(h->dF, L, h->dSc);
  if (h->cfg.accept_rule == KDEA_ACCEPT_ITERATIVE) { dea_running_max_kernel<<<1, 1024, 0, h->stream>>>(h->dF, L, h->dSc, h->dIterAccept); h->launches++; }
  dea_accept_kernel<<<h->num_sms * 4, 256, 0, h->stream>>>(h->dX, h->dXc, ld, L, N, h->dF, h->dFprev, h->cfg.accept_rule, h->dIterAccept, h->dSc,
                                                         h->dCurBest, h->dBestEver);
  dea_best_ever_kernel<<<1, 1, 0, h->stream>>>(h->dSc);
  launch_dea_mean(h->stream, h->dX, ld, L, N, h->dMean, h->dPrevMean, h->dMaxDist);
  h->launches += 4;
  h->scalars_fresh = false;
  h->gen++;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(h, "CUDA error after generation: %s", cudaGetErrorString(e));
  return 0;
}

int kdea_run_generation(kdea_t* h) { return kdea_ask(h) || kdea_eval(h) || kdea_tell(h); }

// generated checkTermination: DEA.config:62-83, optimizer.config, solver.config
int kdea_check_termination(kdea_t* h, int* finished, const char** reason) {
  if (!h) return fail(h, "null solver handle");
  CUDA_OK(h, cudaSetDevice(h->device));
  if (pull_cached(h)) return 1;
  const DeaScalars& s = *h->hSc;
  int fin = 0;
  h->reason.clear();
  const uint64_t gen = h->gen;
  if ((double)s.infeasible > h->tc_max_infeasible) { h->reason += "DEA['Max Infeasible Resamplings'];"; fin = 1; }
  if (gen > 1 && (-s.best_ever_value < h->tc_min_value)) { h->reason += "DEA['Min Value'];"; fin = 1; }
  if (s.min_step < h->tc_min_step) { h->reason += "DEA['Min Step Size'];"; fin = 1; }
  if (gen > 1 && (+s.best_ever_value > h->tc_max_value)) { h->reason += "optimizer['Max Value'];"; fin = 1; }
  if (gen > 1 && (fabs(s.cur_best_value - s.prev_best_value) < h->tc_min_value_diff)) { h->reason += "optimizer['Min Value Difference Threshold'];"; fin = 1; }
  if (h->tc_max_model_evaluations <= (double)h->model_evals) { h->reason += "solver['Max Model Evaluations'];"; fin = 1; }
  if ((double)gen > h->tc_max_generations) { h->reason += "solver['Max Generations'];"; fin = 1; }
  *finished = fin;
  if (reason) *reason = h->reason.c_str();
  return 0;
}

int kdea_run(kdea_t* h, uint64_t max_generations, uint64_t* done) {
  return run(h, max_generations, done, kdea_check_termination, kdea_run_generation);
}

int kdea_get_array(kdea_t* h, const char* key, double* out, size_t cap, size_t* count) {
  if (!h) return fail(h, "null solver handle");
  CUDA_OK(h, cudaSetDevice(h->device));
  Array r;
  if (!find_array(h, key, &r)) return fail(h, "unknown array key '%s'", key);
  return copy_out(h, key, r, out, cap, count, "buffer too small for '%s' (%zu < %zu)");
}

int kdea_set_array(kdea_t* h, const char* key, const double* in, size_t count) {
  if (!h) return fail(h, "null solver handle");
  CUDA_OK(h, cudaSetDevice(h->device));
  Array r;
  if (!find_array(h, key, &r)) return fail(h, "unknown array key '%s'", key);
  return copy_in(h, key, r, in, count);
}

int kdea_get_scalar(kdea_t* h, const char* key, double* out) {
  if (!h) return fail(h, "null solver handle");
  CUDA_OK(h, cudaSetDevice(h->device));
  if (double* p = host_scalar(h, kHostScalars, key, false)) { *out = *p; return 0; }
  if (pull_cached(h)) return 1;
  if (double* p = find_dev_scalar(h, key)) { *out = *p; return 0; }
  if (!strcmp(key, "Best Sample Index")) { *out = (double)h->hSc->best_idx; return 0; }
  if (!strcmp(key, "Infeasible Sample Count")) { *out = (double)h->hSc->infeasible; return 0; }
  if (!strcmp(key, "Current Generation")) { *out = (double)(h->gen - 1); return 0; }
  if (!strcmp(key, "Model Evaluation Count")) { *out = (double)h->model_evals; return 0; }
  if (!strcmp(key, "Variable Count")) { *out = (double)h->N; return 0; }
  return fail(h, "unknown scalar key '%s'", key);
}

int kdea_set_scalar(kdea_t* h, const char* key, double v) {
  if (!h) return fail(h, "null solver handle");
  CUDA_OK(h, cudaSetDevice(h->device));
  if (double* p = host_scalar(h, kHostScalars, key, true)) { *p = v; return 0; }
  if (pull_cached(h)) return 1;
  if (double* p = find_dev_scalar(h, key)) { *p = v; return push(h); }
  if (!strcmp(key, "Best Sample Index")) { h->hSc->best_idx = (unsigned long long)v; return push(h); }
  if (!strcmp(key, "Infeasible Sample Count")) { h->hSc->infeasible = (unsigned long long)v; return push(h); }
  if (!strcmp(key, "Current Generation")) { h->gen = (uint64_t)v + 1; return 0; }
  if (!strcmp(key, "Model Evaluation Count")) { h->model_evals = (uint64_t)v; return 0; }
  return fail(h, "unknown scalar key '%s'", key);
}

uint64_t kdea_launch_count(const kdea_t* h) { return h ? h->launches : 0; }

}  // extern "C"
