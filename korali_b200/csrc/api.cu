// api.cu — the C ABI of libkcma.so (include/kcma.h) and the host-side orchestration of one CMA-ES generation.
// The host code only sequences kernel launches on one stream; all solver state stays in HBM.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <math.h>
#include <nccl.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <string>
#include <vector>

#include "../../include/kcma.h"
#include "common.cuh"
#include "handle.cuh"
#include "kernels.h"

using namespace kc;
namespace kc { extern long long* g_jacobi_dbg; }

namespace {

// ---- NCCL through dlopen: no link-time dependency; prefers the copy torch already loaded ---------------
struct NcclApi {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  bool load(std::string& err) {
    if (lib) return true;
    lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);
    if (!lib) lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) { err = std::string("cannot load libnccl.so.2: ") + dlerror(); return false; }
#define SYM(F) F = (decltype(F))dlsym(lib, "nccl" #F); if (!F) { err = "missing symbol nccl" #F; return false; }
    SYM(GetUniqueId) SYM(CommInitRank) SYM(CommDestroy) SYM(GroupStart) SYM(GroupEnd) SYM(AllGather) SYM(AllReduce) SYM(GetErrorString)
#undef SYM
    return true;
  }
} g_nccl;

inline int round_up(int v, int m) { return (v + m - 1) / m * m; }

struct Phase { double ms = 0; uint64_t calls = 0; };

}  // namespace

struct kcma : Handle<kcma, DevScalars> {
  kcma_cfg cfg;
  int N = 0, ld = 0, num_sms = 148;
  std::vector<double> lower, upper, init_val, init_sd, min_sd, coef, con_shift;
  bool has_bounds = false, any_min_sd = false;
  uint64_t lambda = 0, mu = 0, vlambda = 0, vmu = 0, cur_lambda = 0, cur_mu = 0, s_max = 0, mu_max = 0;
  uint64_t shard_lo = 0, shard_hi = 0;       // this rank's samples of the CURRENT population
  // Constraint path on several ranks: the correction loop of handleConstraints (:774-832) updates the constraint normals sample by
  // sample in population order, so every rank draws and corrects the WHOLE population (same Philox counters, same arithmetic:
  // bitwise the one-GPU run) and only the model evaluations are sharded: rank r evaluates [eval_lo, eval_hi), F is all-gathered.
  bool repl = false;
  uint64_t eval_lo = 0, eval_hi = 0;
  uint64_t max_local = 0, max_zrows = 0;     // allocation bounds
  double mueff = 0, cs = 0, cc = 0, damp = 0, chi_n = 0, trace = 0;
  std::vector<double> h_weights;
  double tc_max_condition = INFINITY, tc_min_sd = -INFINITY, tc_max_sd = INFINITY, tc_max_value = INFINITY,
         tc_min_value_diff = -INFINITY, tc_max_model_evaluations = 1e9, tc_max_generations = 1e10;
  uint64_t model_evals = 0;
  int is_viability = 0, has_constraints = 0;
  uint64_t n_con = 0;
  // device state
  double *dC = nullptr, *dB = nullptr, *dA = nullptr, *dD = nullptr, *dVT = nullptr, *dVTw = nullptr, *dGT = nullptr, *dEv = nullptr;
  int* dPerm = nullptr;
  double *dMean = nullptr, *dMeanOld = nullptr, *dMeanUpd = nullptr, *dT = nullptr, *dPs = nullptr, *dPc = nullptr;
  double *dZ = nullptr, *dY = nullptr, *dX = nullptr, *dF = nullptr;
  double* dGrad = nullptr;   // "Gradients" of the local samples (Use Gradient Information), max_local x ld
  // discrete variables ("Granularity"): per-variable granularity, masking matrices, "Discrete Mutations" (max_local x ld)
  bool has_discrete = false;
  std::vector<double> gran;
  double *dGran = nullptr, *dMask = nullptr, *dMaskSigma = nullptr, *dDiscMut = nullptr;
  unsigned* dIdx = nullptr;
  unsigned char* dSortWs = nullptr;
  double *dW = nullptr, *dSelW = nullptr;
  int *dSelS = nullptr, *dCount = nullptr;
  double *dS = nullptr, *dPartial = nullptr, *dWsplit = nullptr, *dRed = nullptr;
  double *dBestEver = nullptr, *dCurBest = nullptr;
  double *dLower = nullptr, *dUpper = nullptr, *dMinSd = nullptr, *dCoef = nullptr, *dShift = nullptr;
  double* dSigmaSampling = nullptr;
  unsigned char* dInfeasible = nullptr;
  unsigned char* dFresh = nullptr;              // mirrored resampling rounds: pair was drawn in the previous round
  unsigned long long* dRound = nullptr;         // {infeasible members, rows to redraw} of a resampling round (all-reduced over the ranks)
  unsigned long long* hRound = nullptr;         // pinned
  unsigned long long* dRoundV = nullptr;        // one slot per rank (settling the resampling budget)
  // constraint path (K9)
  double *dG = nullptr, *dBounds = nullptr, *dNormal = nullptr, *dCaux = nullptr, *dBestCon = nullptr, *dU = nullptr;
  unsigned long long* dViol = nullptr;
  unsigned char* dIndicator = nullptr;
  int *dEvSample = nullptr, *dEvCon = nullptr, *dVioRows = nullptr;
  unsigned* dAttempt = nullptr;
  long long ldg = 0; int u_rows = 0;
  double normal_lr = -1.0, cov_adaption_factor = -1.0;
  double* dFlush = nullptr; size_t flush_bytes = 0;
  int* hCount = nullptr;      // pinned
  int s_rows_padded = 0, rows_per_cta = 64, max_splits = 16, cur_splits = 1;
  bool sampled_pending = false;  // ask done, tell not yet: X uses (mean, sigma); afterwards (mean_old, sigma_sampling)
  // injections
  bool inj_z = false, inj_bd = false, inj_y = false, inj_x = false, inj_f = false, inj_grad = false;
  bool vt_valid = false;
  // batched host conduit
  kcma_host_objective_fn host_obj = nullptr; void* host_obj_user = nullptr;
  kcma_host_objective_grad_fn host_obj_grad = nullptr;
  std::vector<double> hGrad;
  kcma_host_constraints_fn host_con = nullptr; void* host_con_user = nullptr;
  kcma_device_objective_fn dev_obj = nullptr; void* dev_obj_user = nullptr;   // user objective on the device pointer of X
  std::vector<double> hX, hF, hG;
  // tridiagonalisation-based eigensolver (created on first use)
  kc::TridiagWs* tri = nullptr;
  // nccl
  ncclComm_t comm = nullptr;
  bool comm_in_process = false;   // kcma_comm_init_all: the ranks are threads of one process (no graph replay there, see graph_eligible)
  // timing
  bool timing = false;
  std::map<std::string, Phase> phases;
  struct Pending { std::string name; cudaEvent_t a, b; };
  std::vector<Pending> pending;
  std::vector<cudaEvent_t> event_pool;
  uint64_t sweeps_base = 0;   // DevScalars::jacobi_sweeps_total at the last kcma_timing_reset
  // CUDA graph of one whole generation (ask + eval + tell) for the launch-latency-bound configurations
  cudaStream_t cap_stream = nullptr;
  cudaGraphExec_t gexec = nullptr;
  bool capturing = false, graph_failed = false;
  uint64_t dev_gen = ~0ull;   // value DevScalars::gen is known to hold on the device (~0 = unknown): the graph replay reads it
  uint64_t g_launches = 0, g_evals = 0;   // host-side counters one replay stands for
  std::string warn;
  char warn_out[4096];
  ~kcma();
};

namespace {

struct PhaseTimer {
  kcma* h; const char* name; cudaEvent_t a = nullptr, b = nullptr;
  PhaseTimer(kcma* h_, const char* n) : h(h_), name(n) {
    if (!h->timing) return;
    auto get = [&]() { cudaEvent_t e; if (!h->event_pool.empty()) { e = h->event_pool.back(); h->event_pool.pop_back(); } else cudaEventCreate(&e); return e; };
    a = get(); b = get();
    cudaEventRecord(a, h->stream);
  }
  ~PhaseTimer() {
    if (!h->timing) return;
    cudaEventRecord(b, h->stream);
    h->pending.push_back({name, a, b});
  }
};

void resolve_timers(kcma* h) {
  for (auto& p : h->pending) {
    cudaEventSynchronize(p.b);
    float ms = 0;
    cudaEventElapsedTime(&ms, p.a, p.b);
    auto& ph = h->phases[p.name];
    ph.ms += ms; ph.calls++;
    h->event_pool.push_back(p.a); h->event_pool.push_back(p.b);
  }
  h->pending.clear();
}

// ref: CMAES.cpp.base:233-284 (host arithmetic identical to the oracle's so the constants are bit-equal)
int init_mu_weights(kcma* h, uint64_t numsamplesmu) {
  const uint64_t N = h->N;
  std::vector<double>& w = h->h_weights;
  std::fill(w.begin(), w.end(), 0.0);
  switch (h->cfg.mu_type) {
    case KCMA_MU_LINEAR: for (uint64_t i = 0; i < numsamplesmu; i++) w[i] = (double)(numsamplesmu - i); break;
    case KCMA_MU_EQUAL: for (uint64_t i = 0; i < numsamplesmu; i++) w[i] = 1.; break;
    case KCMA_MU_LOGARITHMIC:
      for (uint64_t i = 0; i < numsamplesmu; i++) w[i] = log(std::max((double)numsamplesmu, 0.5 * h->cur_lambda) + 0.5) - log(i + 1.);
      break;
    case KCMA_MU_PROPORTIONAL: for (uint64_t i = 0; i < numsamplesmu; i++) w[i] = 1.; break;
    default: return fail(h, "Invalid setting of Mu Type (%d) (Linear, Equal, Logarithmic, or Proportional accepted).", h->cfg.mu_type);
  }
  double s1 = 0.0, s2 = 0.0;
  for (uint64_t i = 0; i < numsamplesmu; i++) { s1 += w[i]; s2 += w[i] * w[i]; }
  h->mueff = s1 * s1 / s2;
  for (uint64_t i = 0; i < numsamplesmu; i++) w[i] /= s1;
  if ((h->cfg.initial_cumulative_covariance <= 0) || (h->cfg.initial_cumulative_covariance > 1))
    h->cc = (4.0 + h->mueff / (1.0 * N)) / (N + 4.0 + 2.0 * h->mueff / (1.0 * N));
  else
    h->cc = h->cfg.initial_cumulative_covariance;
  h->cs = h->cfg.initial_sigma_cumulation_factor;
  if (h->cs <= 0 || h->cs >= 1) {
    if (h->has_constraints) h->cs = sqrt(h->mueff) / (sqrt(h->mueff) + sqrt((double)N));
    else h->cs = (h->mueff + 2.0) / (N + h->mueff + 3.0);
  }
  h->damp = h->cfg.initial_damp_factor;
  if (h->damp <= 0.0) h->damp = (1.0 + 2 * std::max(0.0, sqrt((h->mueff - 1.0) / (N + 1.0)) - 1)) + h->cs;
  cudaMemcpyAsync(h->dW, w.data(), sizeof(double) * h->mu_max, cudaMemcpyHostToDevice, h->stream);
  return 0;
}

// ref: CMAES.cpp.base:286-313. Only diagonals of C and B are written (SURVEY Q10).
int init_covariance(kcma* h) {
  const int N = h->N, ld = h->ld;
  h->trace = 0.0;
  for (int i = 0; i < N; ++i) h->trace += h->init_sd[i] * h->init_sd[i];
  const double sigma = sqrt(h->trace / N);
  std::vector<double> D(N), Cd(N), one(N, 1.0);
  for (int i = 0; i < N; ++i) {
    D[i] = h->init_sd[i] * sqrt(N / h->trace);
    Cd[i] = D[i];
    Cd[i] *= Cd[i];
  }
  cudaStreamSynchronize(h->stream);
  // diagonals via strided 2D copies
  cudaMemcpy2D(h->dC, sizeof(double) * (ld + 1), Cd.data(), sizeof(double), sizeof(double), N, cudaMemcpyHostToDevice);
  cudaMemcpy2D(h->dB, sizeof(double) * (ld + 1), one.data(), sizeof(double), sizeof(double), N, cudaMemcpyHostToDevice);
  cudaMemcpy(h->dD, D.data(), sizeof(double) * N, cudaMemcpyHostToDevice);
  // B is only meaningful until the next eigen(); restart the warm-started solver from the identity basis
  launch_set_identity(h->stream, h->dVT, ld, N);
  cudaStreamSynchronize(h->stream);
  h->vt_valid = true;
  double mn = D[0], mx = D[0];
  for (int i = 1; i < N; i++) { mn = std::min(mn, D[i]); mx = std::max(mx, D[i]); }
  double maxd = Cd[0], mind = Cd[0];
  for (int i = 1; i < N; i++) { maxd = std::max(maxd, Cd[i]); mind = std::min(mind, Cd[i]); }
  cudaMemcpy(h->hSc, h->dSc, sizeof(DevScalars), cudaMemcpyDeviceToHost);
  h->hSc->sigma = sigma;
  h->hSc->min_eig = mn * mn; h->hSc->max_eig = mx * mx;
  h->hSc->max_diag_c = maxd; h->hSc->min_diag_c = mind;
  cudaMemcpy(h->dSc, h->hSc, sizeof(DevScalars), cudaMemcpyHostToDevice);
  h->scalars_fresh = true;
  return 0;
}

int nccl_check(kcma* h, ncclResult_t r, const char* what) {
  if (r == ncclSuccess) return 0;
  return fail(h, "NCCL error in %s: %s", what, g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?");
}

int push_scalars(kcma* h) {
  h->hSc->gen = h->gen - 1;   // device copy of the generation counter = last completed generation
  if (push(h)) return 1;
  h->dev_gen = h->gen - 1;
  return 0;
}

void set_population(kcma* h, uint64_t lambda, uint64_t mu) {
  h->cur_lambda = lambda;
  h->cur_mu = mu;
  kcma_shard_range(lambda, h->cfg.mirrored_sampling, h->cfg.rank, h->cfg.nranks, &h->shard_lo, &h->shard_hi);
  h->eval_lo = h->shard_lo; h->eval_hi = h->shard_hi;
  if (h->repl) { h->shard_lo = 0; h->shard_hi = lambda; }
}

uint64_t local_samples(const kcma* h) { return h->shard_hi - h->shard_lo; }
uint64_t eval_samples(const kcma* h) { return h->eval_hi - h->eval_lo; }
uint64_t eval_row0(const kcma* h) { return h->eval_lo - h->shard_lo; }     // first evaluated row of the local X / Y
uint64_t local_zrows(const kcma* h) { return h->cfg.mirrored_sampling ? local_samples(h) / 2 : local_samples(h); }

// VT = B^T (vectors as rows) after B was set from outside the eigensolver.
__global__ void transpose_kernel(const double* __restrict__ in, double* __restrict__ out, int ld, int n) {
  __shared__ double tile[32][33];
  const int x0 = blockIdx.x * 32, y0 = blockIdx.y * 32, tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int r = ty; r < 32; r += 8) tile[r][tx] = (y0 + r < n && x0 + tx < n) ? in[(size_t)(y0 + r) * ld + x0 + tx] : 0.0;
  __syncthreads();
  for (int r = ty; r < 32; r += 8)
    if (x0 + r < n && y0 + tx < n) out[(size_t)(x0 + r) * ld + y0 + tx] = tile[tx][r];
}

__global__ void copy_sigma_kernel(const DevScalars* sc, double* out) { *out = sc->sigma; }
__global__ void fold_error_flag_kernel(double* slot, DevScalars* sc, int unfold) {
  if (!unfold) *slot = sc->nonfinite ? 1.0 : 0.0;
  else if (*slot > 0.0) sc->nonfinite = 1;
}
__global__ void check_finite_kernel(const double* __restrict__ f, long long n, DevScalars* sc) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    if (!isfinite(f[i])) atomicExch(&sc->nonfinite, 1);
}
void launch_check_finite(cudaStream_t st, const double* f, long long n, DevScalars* sc) {
  if (n > 0) check_finite_kernel<<<(int)std::min<long long>((n + 255) / 256, 1024), 256, 0, st>>>(f, n, sc);
}

// infeasible flags -> list of z-rows to resample + counters (prepareGeneration :455-459, :484-490). Single block.
__global__ void __launch_bounds__(1024)
infeasible_compact_kernel(const unsigned char* __restrict__ flags, int samples, int mirrored, int* __restrict__ rows,
                          int* __restrict__ count_out, DevScalars* __restrict__ sc, unsigned char* __restrict__ fresh,
                          unsigned long long* __restrict__ round_out) {
  __shared__ int warp_tot[32];
  __shared__ int carry;
  __shared__ unsigned long long bad_total;
  if (threadIdx.x == 0) { carry = 0; bad_total = 0; }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int items = mirrored ? samples / 2 : samples;
  for (int base = 0; base < items; base += 1024) {
    const int j = base + threadIdx.x;
    int bad = 0; bool take = false;
    if (j < items) {
      if (mirrored) { bad = flags[2 * j] + flags[2 * j + 1]; take = (bad == 2); }
      else { bad = flags[j]; take = bad != 0; }
      // the reference counts an infeasible member once per DRAW (:457, :485-487): a mirrored pair with one feasible member is
      // accepted and not drawn again, so it must not be counted again in the following rounds
      if (fresh) { if (!fresh[j]) bad = 0; fresh[j] = take ? 1 : 0; }
    }
    if (bad) atomicAdd(&bad_total, (unsigned long long)bad);
    const unsigned m = __ballot_sync(0xffffffffu, take);
    if (lane == 0) warp_tot[warp] = __popc(m);
    __syncthreads();
    if (warp == 0) {
      int x = warp_tot[lane];
      for (int off = 1; off < 32; off <<= 1) { const int y = __shfl_up_sync(0xffffffffu, x, off); if (lane >= off) x += y; }
      warp_tot[lane] = x;
    }
    __syncthreads();
    const int c = carry;
    if (take) rows[c + (warp ? warp_tot[warp - 1] : 0) + __popc(m & ((1u << lane) - 1u))] = j;
    __syncthreads();
    if (threadIdx.x == 0) carry = c + warp_tot[31];
    __syncthreads();
  }
  if (threadIdx.x == 0) { *count_out = carry; sc->infeasible_this_round = bad_total; round_out[0] = bad_total; round_out[1] = (unsigned long long)carry; }
}

__global__ void bump_attempts_kernel(unsigned* attempt, const int* rows, int count) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) attempt[rows[i]]++;
}

// y_row = A z_row for listed rows (resampling only; one warp per output element).
__global__ void __launch_bounds__(256)
resample_rows_kernel(const double* __restrict__ Z, double* __restrict__ Y, int ld, const double* __restrict__ A, int n,
                     const int* __restrict__ rows, int diagonal, const double* __restrict__ D) {
  const int lane = threadIdx.x & 31;
  const int d = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (d >= n) return;
  const int row = rows[blockIdx.y];
  const double* z = Z + (size_t)row * ld;
  double a = 0.0;
  if (diagonal) { if (lane == 0) a = D[d] * z[d]; }
  else for (int e = lane; e < n; e += 32) a += A[(size_t)d * ld + e] * z[e];
  a = warp_sum_butterfly(a);
  if (lane == 0) Y[(size_t)row * ld + d] = a;
}

// Diagonal Covariance sampling (:498-502): y = D o z.
__global__ void __launch_bounds__(256)
diag_sample_kernel(const double* __restrict__ Z, double* __restrict__ Y, int ld, long long rows, int n, const double* __restrict__ D) {
  const long long total = rows * ld;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int d = (int)(i % ld);
    Y[i] = d < n ? D[d] * Z[i] : 0.0;
  }
}

__global__ void add_infeasible_from_round_kernel(DevScalars* sc, const unsigned long long* round) { sc->infeasible_sample_count += round[0]; }
__global__ void flush_kernel(double* p, size_t n) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = (double)i;
}
__global__ void expand_mirrored_kernel(const double* Y, double* out, int ld, long long samples, int n) {
  const long long total = samples * n;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long s = i / n; const int d = (int)(i - s * n);
    const double v = Y[(size_t)(s >> 1) * ld + d];
    out[i] = (s & 1) ? -v : v;
  }
}

int ensure_vt(kcma* h) {
  if (h->vt_valid) return 0;
  dim3 grid((h->N + 31) / 32, (h->N + 31) / 32);
  transpose_kernel<<<grid, 256, 0, h->stream>>>(h->dB, h->dVT, h->ld, h->N);
  launch_scale_bd(h->stream, h->dB, h->ld, h->dD, h->dA, h->ld, h->N);
  h->launches += 2;
  h->vt_valid = true;
  return 0;
}

// Which eigensolver runs above the single-CTA size: the tridiagonal one, or the warm-started one-sided Jacobi kernels on the
// constraint path and beyond the tridiagonal solver's size. KCMA_EIGEN=tridiag | jacobi forces one of the two, so that tests can
// compare them on the same input; read per call so that one process can run both.
bool eigen_use_tridiag(const kcma* h) {
  const char* e = getenv("KCMA_EIGEN");
  if (e && !strcmp(e, "jacobi")) return false;
  // The constraint path decomposes C_aux once per correction round (handleConstraints :774-832): nearly the same matrix again and
  // again, which the warm-started one-sided Jacobi finishes in a sweep or two (config 5: 3.9 instead of 6.1 ms per generation)
  if (h->has_constraints && h->N <= 1184 && !(e && !strcmp(e, "tridiag"))) return false;
  return eigen_tridiag_fits(h->N);
}

// updateEigensystem (CMAES.cpp.base:869-890) + eigen (:896-938)
int update_eigensystem(kcma* h, const double* dM) {
  PhaseTimer t(h, "eigen");
  const int N = h->N, ld = h->ld;
  if (h->inj_bd) { h->inj_bd = false; return ensure_vt(h); }
  if (h->cfg.diagonal_covariance) {
    launch_eig_diagonal(h->stream, dM, ld, N, h->dD, h->dSc);
    h->launches += 1;
    h->scalars_fresh = false;
    return 0;
  }
  ensure_vt(h);
  const double tol = 4.0 * 2.220446049250313e-16 * sqrt((double)N);
  const int max_sweeps = 40;
  if (eigen_use_small(N)) {  // the whole solver in one launch, everything in one SM's shared memory
    launch_eigen_small(h->stream, dM, ld, N, h->dVT, h->dGT, h->dB, h->dA, h->dD, tol, max_sweeps, h->dSc);
    h->launches += 2;
    h->scalars_fresh = false;
    return 0;
  }
  if (eigen_use_tridiag(h)) {
    // Householder tridiagonalisation + divide & conquer + WY back-transform (tridiag.cu, dc.cu); no host round trip
    if (!h->tri) {
      char msg[512] = "";
      h->tri = tridiag_ws_create(N, ld, h->num_sms, msg, sizeof(msg));
      if (!h->tri) return fail(h, "%s", msg);
    }
    int l = 4;
    bool ok;
    { PhaseTimer t1(h, "eigen_sytrd"); ok = tridiag_stage_sytrd(h->stream, h->tri, dM); }
    if (ok) ok = tridiag_stage_back_fork(h->stream, h->tri, &l);   // Q accumulation on the side stream, next to stage 2
    if (ok) { PhaseTimer t2(h, "eigen_dc"); ok = tridiag_stage_dc(h->stream, h->tri, &l); }
    if (ok) { PhaseTimer t3(h, "eigen_back"); ok = tridiag_stage_back_join(h->stream, h->tri, &l); }
    if (!ok) return fail(h, "the tridiagonal eigensolver could not be launched: %s", cudaGetErrorString(cudaGetLastError()));
    const double* vt = tridiag_result_vectors(h->tri);
    const double* ev = tridiag_result_values(h->tri);
    launch_eig_sign(h->stream, vt, ld, N, h->dT);   // dT (scratch of tell()) holds the signs here
    launch_eig_order(h->stream, ev, N, h->dPerm, h->dSc);
    launch_eig_commit(h->stream, vt, ld, N, h->dPerm, ev, h->dT, h->dB, h->dA, h->dD, h->dVT, h->dSc);
    h->launches += l + 4;
    h->scalars_fresh = false;
    return 0;
  }
  CUDA_OK(h, cudaMemcpyAsync(h->dVTw, h->dVT, sizeof(double) * (size_t)N * ld, cudaMemcpyDeviceToDevice, h->stream));
  // GT = VT * M  (M symmetric): GT[i][j] = sum_k VT[i][k] M[j][k]
  launch_gemm_tn(h->stream, N, N, N, h->dVTw, ld, dM, ld, h->dGT, ld);
  h->launches += 1;
  const bool persistent = launch_jacobi_persistent(h->stream, h->dGT, h->dVTw, ld, N, tol, max_sweeps, h->dSc, h->num_sms, (unsigned*)h->dPerm);
  if (persistent) {
    h->launches += 1;
    h->scalars_fresh = false;
    // (sweep count: accumulated on the device in DevScalars::jacobi_sweeps_total and read by kcma_timing_get, no sync here)
  } else
  for (int sweep = 0; sweep < max_sweeps; sweep++) {
    int l = 0;
    h->phases["eigen_sweeps"].calls++;
    launch_jacobi_block_sweep(h->stream, h->dGT, h->dVTw, ld, N, tol, h->dSc, &l);
    h->launches += l;
    h->scalars_fresh = false;
    if (pull_cached(h)) return 1;
    if (h->hSc->jacobi_rotations == 0) break;
    // quadratic convergence: once every pair of the sweep was already orthogonal to 1e-8 (KC_QUAD_TAIL), what is left after
    // this sweep is ~1e-16 * lambda / gap and the confirmation sweep (a full pass that rotates nothing) can be skipped
    double max_rel;
    memcpy(&max_rel, &h->hSc->jacobi_max_rel_bits, sizeof(double));
    if (max_rel < 1e-20) break;   // the kernels record the SQUARED cosine
  }
  if (!persistent) { int l = 0; launch_jacobi_block_flush(h->stream, h->dGT, h->dVTw, ld, N, tol, h->dSc, &l); h->launches += l; }
  launch_rayleigh(h->stream, h->dGT, h->dVTw, ld, N, h->dEv, h->dT);   // dT (scratch of tell()) holds the signs here
  launch_eig_order(h->stream, h->dEv, N, h->dPerm, h->dSc);
  launch_eig_commit(h->stream, h->dVTw, ld, N, h->dPerm, h->dEv, h->dT, h->dB, h->dA, h->dD, h->dVT, h->dSc);
  h->launches += 4;
  h->scalars_fresh = false;
  return 0;
}

// by-value generation argument of the kernels; while a graph is being captured the kernels read DevScalars::gen instead
unsigned gen_arg(const kcma* h) { return h->capturing ? kGenFromDevice : (unsigned)h->gen; }

// ---- bounds rejection (prepareGeneration :439-492) ------------------------------------------------------------------------------
// The reference redraws ONE sample at a time until it is feasible or the cumulative 'Infeasible Sample Count' reaches 'Max
// Infeasible Resamplings' (:459, :490). The draws are Philox(sample, attempt), so the attempts of a sample do not depend on the
// order in which samples are visited: the device redraws ALL infeasible samples once per ROUND (attempt r in round r) until every
// sample is feasible, which gives the reference's population and counter whenever the budget is not exhausted. When it is, the
// reference's visiting order matters (samples before the exhaustion point are fully resampled, the one that exhausts the budget
// keeps an infeasible draw, every later sample keeps its FIRST draw): settle_resampling_budget() replays that order on the host
// from the per-sample attempt counts and re-generates the draws the reference would have kept.
int settle_resampling_budget(kcma* h, long long ls, unsigned long long zrow_begin, unsigned long long count_before,
                             unsigned long long local_counted, unsigned long long cap) {
  const int N = h->N, ld = h->ld, mirrored = h->cfg.mirrored_sampling;
  const unsigned long long maxres = h->cfg.max_infeasible_resamplings;
  const long long zrows = mirrored ? ls / 2 : ls;
  const int nr = h->repl ? 1 : h->cfg.nranks, rank = h->repl ? 0 : h->cfg.rank;
  std::vector<unsigned> att((size_t)zrows);
  std::vector<unsigned char> flag((size_t)ls);
  CUDA_OK(h, cudaMemcpyAsync(att.data(), h->dAttempt, sizeof(unsigned) * zrows, cudaMemcpyDeviceToHost, h->stream));
  CUDA_OK(h, cudaMemcpyAsync(flag.data(), h->dInfeasible, (size_t)ls, cudaMemcpyDeviceToHost, h->stream));
  CUDA_OK(h, cudaStreamSynchronize(h->stream));
  // count at the first sample of this rank if every earlier rank resampled to the end (exact as long as no earlier rank exhausts it)
  std::vector<unsigned long long> per_rank((size_t)nr, 0ull);
  per_rank[rank] = local_counted;
  if (nr > 1) {
    CUDA_OK(h, cudaMemcpyAsync(h->dRoundV, per_rank.data(), sizeof(unsigned long long) * nr, cudaMemcpyHostToDevice, h->stream));
    if (nccl_check(h, g_nccl.AllReduce(h->dRoundV, h->dRoundV, nr, ncclUint64, ncclSum, h->comm, h->stream), "all-reduce(resampling per rank)")) return 1;
    CUDA_OK(h, cudaMemcpyAsync(per_rank.data(), h->dRoundV, sizeof(unsigned long long) * nr, cudaMemcpyDeviceToHost, h->stream));
    CUDA_OK(h, cudaStreamSynchronize(h->stream));
  }
  unsigned long long c = count_before;
  for (int q = 0; q < rank; q++) c += per_rank[q];   // >= maxres once an earlier rank exhausted the budget: then only "c >= maxres" matters
  const unsigned long long c_start = c;
  std::vector<int> rows;            // z rows whose kept draw is not the one the rounds ended with
  std::vector<unsigned> keep;       // ... and the attempt the reference keeps
  for (long long j = 0; j < zrows; j++) {
    const unsigned k = att[j];      // failed draws before the current one
    unsigned long long t;
    unsigned final_att;
    if (!mirrored) {
      const bool feasible_now = flag[j] == 0;
      const unsigned long long kk = feasible_now ? k : (unsigned long long)k + 1;   // infeasible draws seen so far (all of them if never feasible)
      const bool endless = !feasible_now;                                            // still infeasible at the cap: treat as "never"
      if (kk == 0) continue;
      const unsigned long long room = c < maxres ? maxres - c : 0ull;
      t = std::max(1ull, room);                                   // infeasible draws the reference makes before it gives up
      if (!endless && kk < t) { c += kk; continue; }              // feasible before the budget runs out: the rounds' draw stands
      if (endless && t > kk) t = kk;                              // (cannot happen with cap >= maxres; keeps the index in range)
      c += t;
      final_att = (unsigned)(t - 1);
    } else {
      const int m = flag[2 * j] + flag[2 * j + 1];                // infeasible members of the current draw
      const bool accepted = m < 2;
      const unsigned long long kf = accepted ? k : (unsigned long long)k + 1;        // draws with BOTH members infeasible
      if (kf == 0) { c += (unsigned long long)m; continue; }
      const unsigned long long room = c < maxres ? maxres - c : 0ull;
      t = std::max(1ull, (room + 1) / 2);                         // smallest t >= 1 with c + 2 t >= maxres
      if (accepted && kf < t) { c += 2 * kf + (unsigned long long)m; continue; }
      if (t > kf) t = kf;
      c += 2 * t;
      final_att = (unsigned)(t - 1);
    }
    if (final_att != k) { rows.push_back((int)j); keep.push_back(final_att); }
  }
  const unsigned long long contributed = c - c_start;
  // exact global counter = before + sum of what every rank contributes under the reference's order
  unsigned long long total = count_before + contributed;
  if (nr > 1) {
    std::fill(per_rank.begin(), per_rank.end(), 0ull);
    per_rank[rank] = contributed;
    CUDA_OK(h, cudaMemcpyAsync(h->dRoundV, per_rank.data(), sizeof(unsigned long long) * nr, cudaMemcpyHostToDevice, h->stream));
    if (nccl_check(h, g_nccl.AllReduce(h->dRoundV, h->dRoundV, nr, ncclUint64, ncclSum, h->comm, h->stream), "all-reduce(resampling settled)")) return 1;
    CUDA_OK(h, cudaMemcpyAsync(per_rank.data(), h->dRoundV, sizeof(unsigned long long) * nr, cudaMemcpyDeviceToHost, h->stream));
    CUDA_OK(h, cudaStreamSynchronize(h->stream));
    total = count_before;
    for (int q = 0; q < nr; q++) total += per_rank[q];
  }
  (void)cap;
  if (!rows.empty()) {   // re-generate the draws the reference keeps: z = Philox(row, attempt), y = B D z, x, feasibility flags
    const int cnt = (int)rows.size();
    for (int i = 0; i < cnt; i++) att[rows[i]] = keep[i];
    int* dRows = (int*)h->dSelS;
    CUDA_OK(h, cudaMemcpyAsync(h->dAttempt, att.data(), sizeof(unsigned) * zrows, cudaMemcpyHostToDevice, h->stream));
    CUDA_OK(h, cudaMemcpyAsync(dRows, rows.data(), sizeof(int) * cnt, cudaMemcpyHostToDevice, h->stream));
    launch_philox_normal(h->stream, h->dZ, ld, cnt, N, h->cfg.seed, (unsigned)h->gen, zrow_begin, h->dAttempt, dRows, h->num_sms);
    dim3 grid((N + 7) / 8, cnt);
    resample_rows_kernel<<<grid, 256, 0, h->stream>>>(h->dZ, h->dY, ld, h->dA, N, dRows, h->cfg.diagonal_covariance, h->dD);
    launch_feasibility(h->stream, h->dY, ld, ls, N, mirrored, h->dMean, h->dSc, h->dLower, h->dUpper, h->dInfeasible,
                       h->cfg.keep_population ? h->dX : nullptr, ld, nullptr, h->num_sms);
    h->launches += 3;
    CUDA_OK(h, cudaStreamSynchronize(h->stream));   // `att` / `rows` are host vectors
  }
  h->scalars_fresh = false;
  if (pull_cached(h)) return 1;
  h->hSc->infeasible_sample_count = total;
  return push_scalars(h);
}

int resample_infeasible(kcma* h, long long ls, unsigned long long zrow_begin) {
  const int N = h->N, ld = h->ld;
  int* dRows = (int*)h->dSelS;                     // reuse: the selection list is rebuilt in tell()
  unsigned* dAttempt = h->dAttempt;                // zeroed per generation
  const unsigned long long maxres = h->cfg.max_infeasible_resamplings;
  const bool multi = h->cfg.nranks > 1 && !h->repl;
  unsigned char* dFresh = (h->cfg.mirrored_sampling && maxres != 0) ? h->dFresh : nullptr;
  if (dFresh) CUDA_OK(h, cudaMemsetAsync(dFresh, 1, local_zrows(h), h->stream));
  unsigned long long count_before = 0, local_counted = 0;
  if (maxres != 0) {
    if (pull_cached(h)) return 1;
    count_before = h->hSc->infeasible_sample_count;
  }
  // no sample needs more redraws than the budget holds; the hard cap keeps a never-feasible sample from spinning forever
  const unsigned long long cap = std::min<unsigned long long>(maxres, 100000ull);
  for (unsigned long long round = 0;; round++) {
    infeasible_compact_kernel<<<1, 1024, 0, h->stream>>>(h->dInfeasible, (int)ls, h->cfg.mirrored_sampling, dRows, h->dCount, h->dSc, dFresh,
                                                         h->dRound);
    // 'Infeasible Sample Count' and the decision to go on resampling are GLOBAL: every rank must leave this loop in the same
    // round (the loop holds a collective) and must see the same counter in the termination chain
    if (multi && nccl_check(h, g_nccl.AllReduce(h->dRound, h->dRound, 2, ncclUint64, ncclSum, h->comm, h->stream), "all-reduce(infeasible)")) return 1;
    add_infeasible_from_round_kernel<<<1, 1, 0, h->stream>>>(h->dSc, h->dRound);
    h->launches += 2;
    h->scalars_fresh = false;
    if (maxres == 0) return 0;  // reference release build: size_t(Infinity) == 0 -> never resamples (SURVEY Q2)
    CUDA_OK(h, cudaMemcpyAsync(h->hCount, h->dCount, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CUDA_OK(h, cudaMemcpyAsync(h->hRound, h->dRound, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
    if (pull_cached(h)) return 1;
    local_counted += h->hSc->infeasible_this_round;
    const int cnt = *h->hCount;
    if (h->hRound[1] == 0 || round >= cap) break;
    if (cnt > 0) {
      bump_attempts_kernel<<<(cnt + 255) / 256, 256, 0, h->stream>>>(dAttempt, dRows, cnt);
      launch_philox_normal(h->stream, h->dZ, ld, cnt, N, h->cfg.seed, (unsigned)h->gen, zrow_begin, dAttempt, dRows, h->num_sms);
      dim3 grid((N + 7) / 8, cnt);
      resample_rows_kernel<<<grid, 256, 0, h->stream>>>(h->dZ, h->dY, ld, h->dA, N, dRows, h->cfg.diagonal_covariance, h->dD);
      // re-check (sample list = z-rows, or both members when mirrored)
      launch_feasibility(h->stream, h->dY, ld, ls, N, h->cfg.mirrored_sampling, h->dMean, h->dSc, h->dLower, h->dUpper,
                         h->dInfeasible, h->cfg.keep_population ? h->dX : nullptr, ld, nullptr, h->num_sms);
      h->launches += 4;
    }
  }
  if (h->hSc->infeasible_sample_count >= maxres) return settle_resampling_budget(h, ls, zrow_begin, count_before, local_counted, cap);
  return 0;
}

int sample_population(kcma* h) {
  const int N = h->N, ld = h->ld;
  const long long zrows = (long long)local_zrows(h);
  const unsigned long long zrow_begin = h->cfg.mirrored_sampling ? h->shard_lo / 2 : h->shard_lo;
  if (!h->inj_y && !h->inj_x) {
    if (!h->inj_z) {
      PhaseTimer t(h, "rng");
      launch_philox_normal(h->stream, h->dZ, ld, zrows, N, h->cfg.seed, gen_arg(h), zrow_begin, nullptr, nullptr, h->num_sms, h->dSc);
      h->launches++;
    }
    h->inj_z = false;
    PhaseTimer t(h, "sample_gemm");
    if (h->cfg.diagonal_covariance) {
      diag_sample_kernel<<<h->num_sms * 8, 256, 0, h->stream>>>(h->dZ, h->dY, ld, zrows, N, h->dD);
    } else {
      launch_gemm_tn(h->stream, (int)zrows, N, N, h->dZ, ld, h->dA, ld, h->dY, ld);
    }
    h->launches++;
  }
  copy_sigma_kernel<<<1, 1, 0, h->stream>>>(h->dSc, h->dSigmaSampling);
  h->launches++;
  CUDA_OK(h, cudaMemsetAsync(h->dAttempt, 0, sizeof(unsigned) * (size_t)(zrows > 0 ? zrows : 1), h->stream));
  // feasibility (isSampleFeasible) and resampling
  const long long ls = (long long)local_samples(h);
  if ((h->has_bounds || h->cfg.keep_population) && !h->inj_x) {
    PhaseTimer t(h, "feasibility");
    launch_feasibility(h->stream, h->dY, ld, ls, N, h->cfg.mirrored_sampling, h->dMean, h->dSc,
                       h->has_bounds ? h->dLower : nullptr, h->dUpper, h->has_bounds ? h->dInfeasible : nullptr,
                       h->cfg.keep_population ? h->dX : nullptr, ld, nullptr, h->num_sms);
    h->launches++;
    if (h->has_discrete) {   // :515-544 + discretize (:453, :478-481); from here on X (not mean + sigma y) is the population
      launch_discrete_mutation(h->stream, h->dX, ld, ls, N, h->shard_lo, h->cfg.mirrored_sampling, h->dSc, h->dMask, h->dGran, h->dBestEver,
                               h->cfg.seed, gen_arg(h), h->dAttempt, h->dDiscMut);
      h->launches++;
      if (h->has_bounds) { launch_feasibility_x(h->stream, h->dX, ld, ls, N, h->dLower, h->dUpper, h->dInfeasible, h->num_sms); h->launches++; }
    }
    if (h->has_bounds && resample_infeasible(h, ls, zrow_begin)) return 1;
  }
  h->inj_y = false;
  if (h->has_discrete) h->inj_x = true;   // eval / tell read the materialised X (same mode as an injected population)
  h->sampled_pending = true;
  return 0;
}

__global__ void gather_rows_kernel(const double* __restrict__ X, int ld, int n, const int* __restrict__ rows, int count, double* __restrict__ out) {
  const long long total = (long long)count * n;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int li = (int)(i / n), d = (int)(i - (long long)li * n);
    out[i] = X[(size_t)rows[li] * ld + d];
  }
}
__global__ void scatter_g_kernel(const double* __restrict__ gin, int count, int n_con, const int* __restrict__ rows, double* __restrict__ G,
                                 long long ldg, DevScalars* sc) {
  const long long total = (long long)count * n_con;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i / count), li = (int)(i - (long long)c * count);
    const double g = gin[i];
    if (!isfinite(g)) atomicExch(&sc->nonfinite, 1);
    G[(size_t)c * ldg + (rows ? rows[li] : li)] = g;
  }
}

// Constraint evaluations of the listed samples (rows == nullptr: all `count` samples) into dG, either with the built-in
// device family or through the batched host conduit (X -> host, user functions, G -> device).
int evaluate_constraints(kcma* h, const int* dRows, int count) {
  const int N = h->N, ld = h->ld, nc = (int)h->n_con;
  if (count <= 0) return 0;
  if (!h->host_con) {
    launch_constraints_halfspace(h->stream, h->dY, ld, count, N, h->dMean, h->dSc, h->dShift, nc, h->dG, h->ldg, dRows, h->num_sms);
    h->launches++;
    return 0;
  }
  // X of these samples is current in dX (keep_population is forced on with a host conduit)
  h->hX.resize((size_t)count * N); h->hG.resize((size_t)count * nc);
  double* dTmp = h->dU;  // scratch: at least n_con*s_max rows x ld
  if (dRows) {
    gather_rows_kernel<<<h->num_sms * 4, 256, 0, h->stream>>>(h->dX, ld, N, dRows, count, dTmp);
    CUDA_OK(h, cudaMemcpyAsync(h->hX.data(), dTmp, sizeof(double) * (size_t)count * N, cudaMemcpyDeviceToHost, h->stream));
  } else {
    CUDA_OK(h, cudaMemcpy2DAsync(h->hX.data(), sizeof(double) * N, h->dX, sizeof(double) * ld, sizeof(double) * N, count, cudaMemcpyDeviceToHost, h->stream));
  }
  CUDA_OK(h, cudaStreamSynchronize(h->stream));
  h->host_con(h->host_con_user, h->hX.data(), (uint64_t)count, (uint64_t)N, h->hG.data(), (uint64_t)nc);
  CUDA_OK(h, cudaMemcpyAsync(dTmp, h->hG.data(), sizeof(double) * (size_t)count * nc, cudaMemcpyHostToDevice, h->stream));
  scatter_g_kernel<<<h->num_sms * 2, 256, 0, h->stream>>>(dTmp, count, nc, dRows, h->dG, h->ldg, h->dSc);
  h->launches += 2;
  return 0;
}

// checkMeanAndSetRegime (CMAES.cpp.base:315-345)
int check_mean_and_set_regime(kcma* h) {
  if (!h->is_viability) return 0;
  if (h->host_con) {
    std::vector<double> m(h->N), g(h->n_con);
    CUDA_OK(h, cudaMemcpyAsync(m.data(), h->dMean, sizeof(double) * h->N, cudaMemcpyDeviceToHost, h->stream));
    CUDA_OK(h, cudaStreamSynchronize(h->stream));
    h->host_con(h->host_con_user, m.data(), 1, (uint64_t)h->N, g.data(), h->n_con);
    if (pull_cached(h)) return 1;
    h->hSc->constraint_evaluation_count += 1;
    int ok = 1;
    for (uint64_t c = 0; c < h->n_con; c++) {
      if (!std::isfinite(g[c])) return fail(h, "Non finite value of constraint evaluation %lu detected: %f\n", (unsigned long)c, g[c]);
      if (g[c] > 0.0) ok = 0;
    }
    h->hSc->mean_feasible = ok;
    if (push_scalars(h)) return 1;
  } else {
    if (h->cfg.constraint_family != KCMA_CON_HALFSPACE) return fail(h, "no constraint functions defined");
    launch_constraints_mean(h->stream, h->dMean, h->dShift, h->N, (int)h->n_con, h->dSc);
    h->launches++;
    h->scalars_fresh = false;
    if (pull_cached(h)) return 1;
  }
  if (h->hSc->nonfinite) return fail(h, "Non finite value of constraint evaluation detected\n");
  if (!h->hSc->mean_feasible) return 0;
  // mean inside the domain: leave the viability regime for good and re-initialise (:336-344)
  h->is_viability = 0;
  CUDA_OK(h, cudaMemsetAsync(h->dBounds, 0, sizeof(double) * h->n_con, h->stream));
  set_population(h, h->lambda, h->mu);
  if (init_mu_weights(h, h->cur_mu)) return 1;
  return init_covariance(h);
}

// re-draw the listed samples: z (next Philox attempt), y = A z, x; bounds-rejection rounds bounded by the cumulative
// _resampledParameterCount (:816-826). nv = number of listed rows (host copy).
int resample_violators(kcma* h, int nv) {
  const int N = h->N, ld = h->ld;
  if (nv <= 0) return 0;
  launch_add_resampled(h->stream, h->dSc, h->dCount);
  bump_attempts_kernel<<<(nv + 255) / 256, 256, 0, h->stream>>>(h->dAttempt, h->dVioRows, nv);
  launch_philox_normal(h->stream, h->dZ, ld, nv, N, h->cfg.seed, (unsigned)h->gen, h->shard_lo, h->dAttempt, h->dVioRows, h->num_sms);
  dim3 grid((N + 7) / 8, nv);
  resample_rows_kernel<<<grid, 256, 0, h->stream>>>(h->dZ, h->dY, ld, h->dA, N, h->dVioRows, h->cfg.diagonal_covariance, h->dD);
  h->launches += 4;
  if (h->cfg.keep_population || h->has_bounds) {
    launch_feasibility(h->stream, h->dY, ld, nv, N, 0, h->dMean, h->dSc, h->has_bounds ? h->dLower : nullptr, h->dUpper,
                       h->has_bounds ? h->dInfeasible : nullptr, h->cfg.keep_population ? h->dX : nullptr, ld, h->dVioRows, h->num_sms);
    h->launches++;
  }
  return 0;
}

// updateConstraints (:347-385) + handleConstraints (:774-832)
int update_and_handle_constraints(kcma* h) {
  const int N = h->N, ld = h->ld, nc = (int)h->n_con;
  const int lambda = (int)h->cur_lambda;
  {
    PhaseTimer t(h, "constraints");
    if (evaluate_constraints(h, nullptr, lambda)) return 1;
    launch_constraint_count(h->stream, h->dG, h->ldg, lambda, nc, h->dBounds, (h->gen == 1 && h->is_viability) ? 1 : 0, h->dViol, h->dSc);
    h->launches += 1;
    h->scalars_fresh = false;
  }
  for (int iter = 0; iter < 100000; iter++) {
    if (pull_cached(h)) return 1;
    if (h->hSc->nonfinite) return fail(h, "Non finite value of constraint evaluation detected\n");
    if (h->hSc->max_violation_count == 0) break;
    int J, nv, aborted;
    {
      PhaseTimer t(h, "constraints");
      launch_constraint_events(h->stream, h->dViol, h->dIndicator, h->ldg, lambda, nc, h->cfg.max_covariance_matrix_corrections, h->dEvSample,
                               h->dEvCon, h->dVioRows, h->dCount, h->dSc);
      h->launches++;
      h->scalars_fresh = false;
      CUDA_OK(h, cudaMemcpyAsync(h->hCount, h->dCount, 2 * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
      if (pull_cached(h)) return 1;
      J = h->hCount[0]; nv = h->hCount[1]; aborted = h->hSc->adaptation_abort;
      int splits = 1;
      if (J > 0) {
        launch_constraint_normals(h->stream, h->dEvSample, h->dEvCon, h->dCount, h->dY, ld, h->dNormal, ld, h->normal_lr, h->dU, ld, N, nc);
        h->launches++;
        if (!aborted) {
          const int rows_padded = std::min(h->u_rows, round_up(J, 16) + 16);
          launch_constraint_scale(h->stream, h->dU, ld, N, h->dEvSample, h->dCount, h->dViol, h->cov_adaption_factor, rows_padded);
          splits = launch_syrk(h->stream, N, J, nullptr, h->dU, ld, h->u_rows, h->dWsplit, ld, J, h->num_sms, h->max_splits);
          h->launches += 2;
        }
      }
      if (aborted) {
        char buf[128];
        snprintf(buf, sizeof(buf), "Exiting adaption loop, max adaptions (%zu) reached.\n", (size_t)h->cfg.max_covariance_matrix_corrections);
        h->warn += buf;
        break;
      }
      launch_caux(h->stream, h->dC, h->dCaux, ld, h->dWsplit, ld, splits, N, h->dCount);
      h->launches++;
    }
    if (update_eigensystem(h, h->dCaux)) return 1;
    {
      PhaseTimer t(h, "constraints");
      if (resample_violators(h, nv)) return 1;
      // reEvaluateConstraints (:387-424)
      if (evaluate_constraints(h, h->dVioRows, nv)) return 1;
      launch_constraint_recount(h->stream, h->dG, h->ldg, nc, h->dBounds, h->dVioRows, h->dCount, nv, h->dViol, h->dIndicator);
      launch_constraint_max(h->stream, h->dViol, lambda, h->dCount, h->dSc);
      h->launches += 2;
      h->scalars_fresh = false;
    }
  }
  return 0;
}

int do_ask(kcma* h) {
  if (h->has_constraints && check_mean_and_set_regime(h)) return 1;
  if (update_eigensystem(h, h->dC)) return 1;
  if (sample_population(h)) return 1;
  if (h->has_constraints) return update_and_handle_constraints(h);
  return 0;
}

int do_eval(kcma* h) {
  h->model_evals += h->cur_lambda;  // ref :214
  const bool want_grad = h->cfg.use_gradient_information != 0;   // operation "Evaluate With Gradients" (:199-200, 226-228)
  if (want_grad && h->inj_f && !h->inj_grad)
    return fail(h, "Use Gradient Information: inject the gradients (KCMA_INJ_GRAD) together with the values of an external model");
  const bool have_grad = h->inj_grad;
  h->inj_grad = false;
  if (h->inj_f) { h->inj_f = false; return 0; }
  if (want_grad && h->host_obj_grad) {  // batched host conduit, model returns F and dF/dx
    PhaseTimer t(h, "host_objective");
    const size_t ls = eval_samples(h), N = h->N;
    h->hX.resize(ls * N); h->hF.resize(ls); h->hGrad.resize(ls * N);
    CUDA_OK(h, cudaMemcpy2DAsync(h->hX.data(), sizeof(double) * N, h->dX + eval_row0(h) * h->ld, sizeof(double) * h->ld, sizeof(double) * N, ls, cudaMemcpyDeviceToHost, h->stream));
    CUDA_OK(h, cudaStreamSynchronize(h->stream));
    h->host_obj_grad(h->host_obj_user, h->hX.data(), (uint64_t)ls, (uint64_t)N, h->hF.data(), h->hGrad.data());
    for (size_t i = 0; i < ls; i++)
      if (!std::isfinite(h->hF[i])) return fail(h, "Non finite value of function evaluation detected: %f\n", h->hF[i]);
    CUDA_OK(h, cudaMemcpyAsync(h->dF + h->eval_lo, h->hF.data(), sizeof(double) * ls, cudaMemcpyHostToDevice, h->stream));
    CUDA_OK(h, cudaMemcpy2DAsync(h->dGrad + eval_row0(h) * h->ld, sizeof(double) * h->ld, h->hGrad.data(), sizeof(double) * N, sizeof(double) * N, ls, cudaMemcpyHostToDevice, h->stream));
    CUDA_OK(h, cudaStreamSynchronize(h->stream));
    return 0;
  }
  if (want_grad && !have_grad && (h->host_obj || h->cfg.objective == KCMA_OBJ_EXTERNAL))
    return fail(h, "Use Gradient Information: the model must return gradients (kcma_set_host_objective_grad or KCMA_INJ_GRAD)");
  if (h->dev_obj) {   // user objective on the device: one call for the whole shard, X and F never leave HBM
    PhaseTimer t(h, "device_objective");
    const long long ls = (long long)eval_samples(h);
    h->dev_obj(h->dev_obj_user, h->dX + eval_row0(h) * h->ld, (uint64_t)ls, (uint64_t)h->N, (uint64_t)h->ld, h->dF + h->eval_lo, (void*)h->stream);
    launch_check_finite(h->stream, h->dF + h->eval_lo, ls, h->dSc);
    h->launches++;
    h->scalars_fresh = false;
    return 0;
  }
  if (h->host_obj) {  // batched host conduit
    PhaseTimer t(h, "host_objective");
    const size_t ls = eval_samples(h), N = h->N;
    h->hX.resize(ls * N); h->hF.resize(ls);
    CUDA_OK(h, cudaMemcpy2DAsync(h->hX.data(), sizeof(double) * N, h->dX + eval_row0(h) * h->ld, sizeof(double) * h->ld, sizeof(double) * N, ls, cudaMemcpyDeviceToHost, h->stream));
    CUDA_OK(h, cudaStreamSynchronize(h->stream));
    h->host_obj(h->host_obj_user, h->hX.data(), (uint64_t)ls, (uint64_t)N, h->hF.data());
    for (size_t i = 0; i < ls; i++)  // ref: optimization.cpp.base:32-33
      if (!std::isfinite(h->hF[i])) {
        if (h->cfg.nranks == 1) return fail(h, "Non finite value of function evaluation detected: %f\n", h->hF[i]);
        if (pull_cached(h)) return 1;      // several ranks: fail collectively at the end of the generation (flag in the all-reduce)
        h->hSc->nonfinite = 1;
        if (push_scalars(h)) return 1;
        h->hF[i] = -1e300;
      }
    CUDA_OK(h, cudaMemcpyAsync(h->dF + h->eval_lo, h->hF.data(), sizeof(double) * ls, cudaMemcpyHostToDevice, h->stream));
    return 0;
  }
  if (h->cfg.objective == KCMA_OBJ_EXTERNAL) return fail(h, "objective is External: inject the Value Vector with kcma_inject(KCMA_INJ_F) or set a host objective before eval");
  PhaseTimer t(h, "objective");
  const long long ls = (long long)eval_samples(h);
  double* f_local = h->dF + h->eval_lo;
  const double* src = (h->inj_x ? h->dX : h->dY) + eval_row0(h) * h->ld;
  if (launch_objective(h->stream, h->cfg.objective, src, h->ld, ls, h->N, h->cfg.mirrored_sampling, h->inj_x ? 1 : 0, h->dMean,
                       h->dSc, h->dCoef, f_local, h->num_sms))
    return fail(h, "unknown objective id %d", h->cfg.objective);
  h->launches++;
  if (want_grad && !have_grad) {
    launch_objective_gradient(h->stream, h->cfg.objective, src, h->ld, ls, h->N, h->cfg.mirrored_sampling, h->inj_x ? 1 : 0, h->dMean,
                              h->dSc, h->dCoef, h->dGrad + eval_row0(h) * h->ld, h->ld, h->num_sms);
    h->launches++;
  }
  h->scalars_fresh = false;
  return 0;
}

int do_tell(kcma* h) {
  const int N = h->N, ld = h->ld;
  const int lambda = (int)h->cur_lambda, mu = (int)h->cur_mu;
  const int multi = h->cfg.nranks > 1 && !h->repl;   // repl: every rank holds the whole population, nothing to reduce
  const int from_x = h->inj_x ? 1 : 0;
  const double* rows_src = from_x ? h->dX : h->dY;
  if (h->cfg.nranks > 1) {
    if (!h->comm) return fail(h, "nranks > 1 but kcma_comm_init was not called");
    PhaseTimer t(h, "collectives");
    if (nccl_check(h, g_nccl.AllGather(h->dF + h->eval_lo, h->dF, eval_samples(h), ncclFloat64, h->comm, h->stream), "all-gather(F)")) return 1;
    if (h->repl) {   // a non-finite F(x) of ANY rank fails the generation on EVERY rank (end_of_generation reads the flag)
      launch_check_finite(h->stream, h->dF, (long long)h->cur_lambda, h->dSc);
      h->launches++;
    }
  }
  {
    PhaseTimer t(h, "sort");
    h->launches += launch_sort_index(h->stream, h->dF, lambda, h->dSortWs, h->dIdx, h->num_sms);
    const int best_is_first = (!h->has_constraints || h->is_viability) ? 1 : 0;
    launch_rank_bookkeeping(h->stream, h->dF, h->dIdx, lambda, mu, best_is_first ? nullptr : h->dViol, best_is_first, h->dSc);
    h->launches++;
    if (h->cfg.mu_type == KCMA_MU_PROPORTIONAL) { launch_proportional_weights(h->stream, h->dF, h->dIdx, mu, h->dW); h->launches++; }
  }
  int max_count;
  {
    PhaseTimer t(h, "gather_mean");
    launch_select_local(h->stream, h->dIdx, h->dW, mu, (unsigned)h->shard_lo, (unsigned)h->shard_hi, h->dSelS, h->dSelW, h->dCount);
    max_count = (int)std::min<uint64_t>(mu, local_samples(h));
    launch_gather_mean(h->stream, rows_src, ld, h->cfg.mirrored_sampling, from_x, h->dSelS, h->dSelW, h->dCount, max_count, h->rows_per_cta,
                       N, ld, h->dMean, h->dSc, h->dS, ld, h->s_rows_padded, h->dPartial);
    double* mean_new = h->dRed + (size_t)N * ld;
    double* best_x = mean_new + ld;
    launch_mean_reduce(h->stream, h->dPartial, h->dCount, h->rows_per_cta, N, ld, mean_new, rows_src, ld, h->cfg.mirrored_sampling, from_x,
                       h->dMean, h->dSc, (unsigned)h->shard_lo, (unsigned)h->shard_hi, best_x);
    h->launches += 4;
    if (h->cfg.use_gradient_information) {   // :611-621, on this rank's share of the weighted sum
      launch_gradient_mean(h->stream, h->dGrad, ld, h->dSelS, h->dSelW, h->dCount, N, h->cfg.gradient_step_size, mean_new);
      h->launches++;
    }
  }
  int splits;
  {
    PhaseTimer t(h, "rank_mu");
    if (h->cfg.mu_type == KCMA_MU_PROPORTIONAL && !h->cfg.diagonal_covariance) {
      splits = 1;   // signed weights: see signed_rank_mu_kernel
      launch_signed_rank_mu(h->stream, h->dS, ld, h->dCount, h->dSelW, N, h->dWsplit, ld);
    } else if (h->cfg.diagonal_covariance) {
      splits = std::max(1, (max_count + h->rows_per_cta * 8 - 1) / (h->rows_per_cta * 8));
      if (splits > h->max_splits) splits = h->max_splits;
      const int rows_per = (max_count + splits - 1) / splits;
      launch_diag_rank_mu(h->stream, h->dS, ld, h->dCount, max_count, rows_per > 0 ? rows_per : 1, N, h->dWsplit, ld, splits);
    } else {
      // the number of selected samples this rank owns is only known on the device (dCount); size the split-K for its
      // expectation mu * local / lambda and let the kernel read the exact row count
      const int expect = (int)std::min<uint64_t>(max_count, (uint64_t)mu * local_samples(h) / h->cur_lambda + 1);
      splits = launch_syrk(h->stream, N, max_count, h->dCount, h->dS, ld, h->s_rows_padded, h->dWsplit, ld, expect, h->num_sms, h->max_splits);
    }
    h->launches++;
    if (multi) { launch_reduce_splits(h->stream, h->dWsplit, ld, splits, N, h->dRed); h->launches++; }
  }
  if (multi) {
    PhaseTimer t(h, "collectives");
    // the error flag rides along, so that a non-finite F(x) on ONE rank fails the generation on EVERY rank instead of leaving the
    // others blocked in the next collective
    const size_t cnt = (size_t)N * ld + 2 * (size_t)ld + 1;
    fold_error_flag_kernel<<<1, 1, 0, h->stream>>>(h->dRed + cnt - 1, h->dSc, 0);
    if (nccl_check(h, g_nccl.AllReduce(h->dRed, h->dRed, cnt, ncclFloat64, ncclSum, h->comm, h->stream), "all-reduce(P|mean|best)")) return 1;
    fold_error_flag_kernel<<<1, 1, 0, h->stream>>>(h->dRed + cnt - 1, h->dSc, 1);
    h->launches += 2;
  }
  {
    PhaseTimer t(h, "paths");
    double* mean_new = h->dRed + (size_t)N * ld;
    double* best_x = mean_new + ld;
    launch_best_update(h->stream, best_x, N, gen_arg(h), h->dCurBest, h->dBestEver, h->dSc, h->has_constraints ? h->dG : nullptr, h->ldg,
                       (int)h->n_con, h->dBestCon);
    launch_paths(h->stream, mean_new, h->dMean, h->dMeanOld, h->dMeanUpd, h->dT, h->dPs, h->dPc, h->dB, ld, h->dD, N,
                 h->cfg.diagonal_covariance, h->cs, h->cc, h->mueff, h->chi_n, gen_arg(h), h->dSc);
    const double c1 = 2.0 / (pow(N + 1.3, 2) + h->mueff);
    const double cmu = std::min(1.0 - c1, 2.0 * (h->mueff - 2. + 1. / h->mueff) / (pow(N + 2.0, 2) + h->mueff));
    if (multi) launch_adapt_c(h->stream, h->dC, ld, h->dRed, ld, 1, N, h->dPc, c1, cmu, h->cc, h->cfg.diagonal_covariance, h->dSc);
    else launch_adapt_c(h->stream, h->dC, ld, h->dWsplit, ld, splits, N, h->dPc, c1, cmu, h->cc, h->cfg.diagonal_covariance, h->dSc);
    if (h->has_discrete) {   // updateDiscreteMutationMatrix (:668): new C, sigma of before updateSigma
      launch_discrete_matrix(h->stream, h->dC, ld, N, h->dGran, h->dPs, h->cs, (double)h->cfg.population_size, h->dMask, h->dMaskSigma, h->dSc);
      h->launches++;
    }
    const int viab = (h->has_constraints && h->is_viability) ? 1 : 0;
    if (viab) { launch_viability_boundaries(h->stream, h->dG, h->ldg, (int)h->n_con, h->dIdx, mu, h->dBounds); h->launches++; }
    launch_sigma(h->stream, h->dC, ld, N, h->dMinSd, h->any_min_sd ? 1 : 0, h->cs, h->damp, h->chi_n, h->trace, h->cfg.is_sigma_bounded,
                 h->cfg.mu_value > 1 ? 1 : 0, viab, h->cfg.global_success_learning_rate, h->cfg.target_success_rate, h->has_discrete ? 1 : 0,
                 h->dSc);
    h->launches += 7;
  }
  h->inj_x = false;
  h->sampled_pending = false;
  h->scalars_fresh = false;
  h->gen++;
  return 0;
}

int end_of_generation(kcma* h) {
  if (pull_cached(h)) return 1;
  if (h->timing) resolve_timers(h);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(h, "CUDA error after generation: %s", cudaGetErrorString(e));
  if (h->hSc->nonfinite) {
    h->hSc->nonfinite = 0;
    push_scalars(h);
    return fail(h, "Non finite value of function evaluation detected: nan\n");
  }
  if (h->hSc->warn_no_valid) {
    h->warn += "No sample without constraint violations in this generation: using the best-ranked sample (the reference reads out of bounds here).\n";
    h->hSc->warn_no_valid = 0;
    if (push_scalars(h)) return 1;
  }
  if (h->hSc->eig_rejected) h->warn += "Min Eigenvalue smaller or equal 0.0 after Eigen decomp (no update possible).\n";
  if (h->hSc->warn_flat) { h->warn += "Sigma increased due to equal function values.\n"; }
  if (h->hSc->warn_minsd) { h->warn += "Sigma increased due to minimal standard deviation.\n"; }
  if (h->hSc->warn_flat || h->hSc->warn_minsd) {
    h->hSc->warn_flat = h->hSc->warn_minsd = 0;
    if (push_scalars(h)) return 1;
  }
  if (h->warn.size() > 3000) h->warn.erase(0, h->warn.size() - 3000);
  return 0;
}

}  // namespace

// =================================================== C ABI ===================================================
extern "C" {

void kcma_cfg_defaults(kcma_cfg* c) {
  memset(c, 0, sizeof(*c));
  c->abi_version = KCMA_ABI_VERSION;
  c->mu_type = KCMA_MU_LOGARITHMIC;
  c->initial_sigma_cumulation_factor = -1.0;
  c->initial_damp_factor = -1.0;
  c->initial_cumulative_covariance = -1.0;
  c->viability_population_size = 2;
  c->max_covariance_matrix_corrections = 1000000;
  c->target_success_rate = 0.1818;
  c->covariance_matrix_adaption_strength = 0.1;
  c->normal_vector_learning_rate = -1.0;
  c->global_success_learning_rate = 0.2;
  c->nranks = 1;
  c->use_gradient_information = 0;
  c->gradient_step_size = 0.01;
}

void kcma_shard_range(uint64_t population, int mirrored, int rank, int nranks, uint64_t* begin, uint64_t* end) {
  // contiguous equal shards in units of samples (pairs when mirrored); remainder units go to the low ranks
  const uint64_t unit = mirrored ? 2 : 1;
  const uint64_t units = population / unit;
  const uint64_t base = units / (uint64_t)nranks, rem = units % (uint64_t)nranks;
  const uint64_t r = (uint64_t)rank;
  const uint64_t b = r * base + std::min(r, rem);
  const uint64_t e = b + base + (r < rem ? 1 : 0);
  *begin = b * unit;
  *end = e * unit;
}

const char* kcma_last_error(const kcma_t* h) { return h ? h->err.c_str() : kcma::create_err; }

const char* kcma_take_warnings(kcma_t* h) {
  strncpy(h->warn_out, h->warn.c_str(), sizeof(h->warn_out) - 1);
  h->warn_out[sizeof(h->warn_out) - 1] = 0;
  h->warn.clear();
  return h->warn_out;
}

namespace { void invalidate_graph(kcma* h); }

kcma::~kcma() {
  cudaSetDevice(device);
  cudaStreamSynchronize(stream);
  invalidate_graph(this);
  if (cap_stream) cudaStreamDestroy(cap_stream);
  if (comm && g_nccl.CommDestroy) g_nccl.CommDestroy(comm);
  kc::tridiag_ws_destroy(tri);
  for (auto& p : pending) { cudaEventDestroy(p.a); cudaEventDestroy(p.b); }
  for (auto e : event_pool) cudaEventDestroy(e);
}

void kcma_destroy(kcma_t* h) { delete h; }

int kcma_create(const kcma_cfg* cfg, kcma_t** out) {
  *out = nullptr;
  kcma::create_err[0] = 0;
  if (!cfg || cfg->abi_version != KCMA_ABI_VERSION) return fail<kcma>(nullptr, "kcma_cfg ABI version mismatch");
  if (cfg->n == 0) return fail<kcma>(nullptr, "Optimization Evaluation problems require at least one variable.\n");
  if (cfg->n > 32768) return fail<kcma>(nullptr, "Variable Count %zu exceeds the supported maximum (32768)", (size_t)cfg->n);
  if (open_device<kcma>(cfg->device)) return 1;
  kcma* h = new kcma();
  h->cfg = *cfg;
  h->device = cfg->device;
  cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, h->device);
  const int N = h->N = (int)cfg->n;
  const int ld = h->ld = round_up(N, 16);
  auto copyv = [&](const double* p, size_t n, double fill) { std::vector<double> v(n, fill); if (p) std::copy(p, p + n, v.begin()); return v; };
  h->lower = copyv(cfg->lower_bound, N, -INFINITY);
  h->upper = copyv(cfg->upper_bound, N, INFINITY);
  h->init_val = copyv(cfg->initial_value, N, NAN);
  h->init_sd = copyv(cfg->initial_stddev, N, NAN);
  h->min_sd = copyv(cfg->min_stddev_update, N, 0.0);
  h->cfg.gradient_step_size = (double)(float)cfg->gradient_step_size;   // SURVEY Q9: _gradientStepSize is a float (CMAES.hpp:61)
  h->gran = copyv(cfg->granularity, N, 0.0);
  h->cfg.granularity = nullptr;
  for (int i = 0; i < N; i++) {   // CMAES.cpp.base:44-50
    if (h->gran[i] < 0.0) return create_fail(h, "Negative granularity for variable %d.\n", i);
    if (h->gran[i] > 0.0) h->has_discrete = true;
  }
  if (h->has_discrete) {
    if (cfg->n_constraints > 0) return create_fail(h, "discrete variables together with constraints are not supported");
    if (cfg->max_infeasible_resamplings != 0) return create_fail(h, "discrete variables with resampling rounds (Max Infeasible Resamplings > 0) are not supported");
    h->cfg.keep_population = 1;   // after the discrete mutations X is no longer mean + sigma * y: it is materialised
  }
  h->coef.resize(N);
  for (int i = 0; i < N; i++) h->coef[i] = cfg->objective_coef ? cfg->objective_coef[i] : (N > 1 ? pow(10.0, 6.0 * (double)i / (double)(N - 1)) : 1.0);
  h->n_con = (cfg->constraint_family == KCMA_CON_NONE && !cfg->n_constraints) ? 0 : cfg->n_constraints;
  h->con_shift = copyv(cfg->constraint_shift, h->n_con, 0.0);
  h->cfg.lower_bound = h->cfg.upper_bound = h->cfg.initial_value = h->cfg.initial_stddev = h->cfg.min_stddev_update = nullptr;
  h->cfg.objective_coef = h->cfg.constraint_shift = nullptr;
  for (int i = 0; i < N; i++) {
    if (std::isfinite(h->lower[i]) || std::isfinite(h->upper[i])) h->has_bounds = true;
    if (h->min_sd[i] > 0.0) h->any_min_sd = true;
  }
  // ref :26-31
  uint64_t lambda = cfg->population_size, mu = cfg->mu_value, vlambda = cfg->viability_population_size, vmu = cfg->viability_mu_value;
  if (cfg->use_gradient_information && cfg->gradient_step_size <= 0.)   // CMAES.cpp.base:86
    return create_fail(h, "Gradient Step Size must be larger than 0.0 (is %f)", cfg->gradient_step_size);
  if (lambda <= 1) return create_fail(h, "'Population Size' must be larger 1.");
  if (mu == 0) mu = lambda / 2;
  if (vmu == 0) vmu = vlambda / 2;
  if (mu > lambda) return create_fail(h, "'Mu Value' (%zu) must not exceed 'Population Size' (%zu).", (size_t)mu, (size_t)lambda);
  h->lambda = lambda; h->mu = mu; h->vlambda = vlambda; h->vmu = vmu;
  h->cfg.mu_value = mu; h->cfg.viability_mu_value = vmu;
  h->has_constraints = h->n_con > 0;
  h->s_max = std::max(lambda, h->has_constraints ? vlambda : lambda);
  h->mu_max = std::max(mu, h->has_constraints ? vmu : mu);
  if (h->s_max >= (1ull << 31)) return create_fail(h, "'Population Size' too large");
  h->chi_n = sqrt((double)N) * (1. - 1. / (4. * N) + 1. / (21. * N * N));
  h->is_viability = h->has_constraints;
  if (cfg->mirrored_sampling) {  // ref :89-93
    if (lambda % 2 == 1) return create_fail(h, "Mirrored Sampling can only be applied with an even Sample Population (is %zu)", (size_t)lambda);
    if (h->has_constraints) return create_fail(h, "Mirrored Sampling not applicable to problems with constraints");
  }
  if (cfg->nranks < 1 || cfg->rank < 0 || cfg->rank >= cfg->nranks) return create_fail(h, "invalid rank %d of %d", cfg->rank, cfg->nranks);
  if (cfg->nranks > 1) {
    const uint64_t unit = (cfg->mirrored_sampling ? 2 : 1) * (uint64_t)cfg->nranks;
    if (lambda % unit || (h->has_constraints && vlambda % unit))
      return create_fail(h, "population size must be divisible by %zu to shard it across %d GPUs", (size_t)unit, cfg->nranks);
  }
  for (int i = 0; i < N; ++i) {  // ref :111-126
    if (!std::isfinite(h->init_val[i])) {
      if (!std::isfinite(h->lower[i])) return create_fail(h, "'Initial Value' of variable 'X%d' not defined, and cannot be inferred because variable lower bound is not finite.\n", i);
      if (!std::isfinite(h->upper[i])) return create_fail(h, "'Initial Value' of variable 'X%d' not defined, and cannot be inferred because variable upper bound is not finite.\n", i);
      h->init_val[i] = (h->upper[i] + h->lower[i]) * 0.5;
    }
    if (!std::isfinite(h->init_sd[i])) {
      if (!std::isfinite(h->lower[i])) return create_fail(h, "Initial (Mean) Value of variable 'X%d' not defined, and cannot be inferred because variable lower bound is not finite.\n", i);
      if (!std::isfinite(h->upper[i])) return create_fail(h, "Initial Standard Deviation 'X%d' not defined, and cannot be inferred because variable upper bound is not finite.\n", i);
      h->init_sd[i] = (h->upper[i] - h->lower[i]) * 0.3;
    }
  }
  if (h->has_constraints) {
    if ((cfg->global_success_learning_rate <= 0.0) || (cfg->global_success_learning_rate > 1.0)) return create_fail(h, "Invalid Global Success Learning Rate (%f), must be greater than 0.0 and less than 1.0\n", cfg->global_success_learning_rate);
    if ((cfg->target_success_rate <= 0.0) || (cfg->target_success_rate > 1.0)) return create_fail(h, "Invalid Target Success Rate (%f), must be greater than 0.0 and less than 1.0\n", cfg->target_success_rate);
    if (cfg->covariance_matrix_adaption_strength <= 0.0) return create_fail(h, "Invalid Adaption Size (%f), must be greater than 0.0\n", cfg->covariance_matrix_adaption_strength);
  }
  h->repl = h->has_constraints && cfg->nranks > 1;
  set_population(h, h->is_viability ? vlambda : lambda, h->is_viability ? vmu : mu);
  {
    uint64_t lo, hi;
    kcma_shard_range(h->s_max, cfg->mirrored_sampling, cfg->rank, cfg->nranks, &lo, &hi);
    h->max_local = hi - lo;
    if (h->has_constraints) h->max_local = h->repl ? h->s_max + 1 : (h->s_max + cfg->nranks - 1) / cfg->nranks + 1;
    h->max_zrows = cfg->mirrored_sampling ? h->max_local / 2 : h->max_local;
  }
  const size_t nn = (size_t)N * ld;
  Allocations& m = h->mem;
  CREATE_OK(h, alloc(m, &h->dC, nn)); CREATE_OK(h, alloc(m, &h->dB, nn)); CREATE_OK(h, alloc(m, &h->dA, nn));
  CREATE_OK(h, alloc(m, &h->dVT, nn)); CREATE_OK(h, alloc(m, &h->dVTw, nn)); CREATE_OK(h, alloc(m, &h->dGT, nn));
  CREATE_OK(h, alloc(m, &h->dD, ld)); CREATE_OK(h, alloc(m, &h->dEv, ld)); CREATE_OK(h, alloc(m, &h->dPerm, ld));
  CREATE_OK(h, alloc(m, &h->dMean, ld)); CREATE_OK(h, alloc(m, &h->dMeanOld, ld)); CREATE_OK(h, alloc(m, &h->dMeanUpd, ld));
  CREATE_OK(h, alloc(m, &h->dT, ld)); CREATE_OK(h, alloc(m, &h->dPs, ld)); CREATE_OK(h, alloc(m, &h->dPc, ld));
  CREATE_OK(h, alloc(m, &h->dBestEver, ld)); CREATE_OK(h, alloc(m, &h->dCurBest, ld));
  CREATE_OK(h, alloc(m, &h->dZ, h->max_zrows * ld)); CREATE_OK(h, alloc(m, &h->dY, h->max_zrows * ld));
  CREATE_OK(h, alloc(m, &h->dX, (h->cfg.keep_population ? h->max_local : 1) * (size_t)ld));
  if (cfg->use_gradient_information) CREATE_OK(h, alloc(m, &h->dGrad, h->max_local * (size_t)ld));
  if (h->has_discrete) {
    CREATE_OK(h, alloc(m, &h->dGran, ld)); CREATE_OK(h, alloc(m, &h->dMask, ld)); CREATE_OK(h, alloc(m, &h->dMaskSigma, ld));
    CREATE_OK(h, alloc(m, &h->dDiscMut, h->max_local * (size_t)ld));
    CREATE_OK(h, cudaMemcpy(h->dGran, h->gran.data(), sizeof(double) * N, cudaMemcpyHostToDevice));
  }
  CREATE_OK(h, alloc(m, &h->dF, h->s_max)); CREATE_OK(h, alloc(m, &h->dIdx, h->s_max));
  CREATE_OK(h, alloc(m, &h->dSortWs, sort_workspace_bytes((int)h->s_max)));
  CREATE_OK(h, alloc(m, &h->dW, h->mu_max));
  const uint64_t max_sel = std::max<uint64_t>(std::min(h->mu_max, h->max_local), h->max_zrows);
  CREATE_OK(h, alloc(m, &h->dSelW, max_sel + 16)); CREATE_OK(h, alloc(m, &h->dSelS, max_sel + 16)); CREATE_OK(h, alloc(m, &h->dCount, 4));
  h->s_rows_padded = round_up((int)std::min(h->mu_max, h->max_local), 16) + 16;
  CREATE_OK(h, alloc(m, &h->dS, (size_t)h->s_rows_padded * ld));
  CREATE_OK(h, alloc(m, &h->dPartial, ((size_t)h->s_rows_padded / h->rows_per_cta + 2) * ld));
  CREATE_OK(h, alloc(m, &h->dWsplit, (size_t)h->max_splits * nn));
  CREATE_OK(h, alloc(m, &h->dRed, nn + 2 * (size_t)ld + 16));
  CREATE_OK(h, alloc(m, &h->dLower, ld)); CREATE_OK(h, alloc(m, &h->dUpper, ld)); CREATE_OK(h, alloc(m, &h->dMinSd, ld));
  CREATE_OK(h, alloc(m, &h->dCoef, ld)); CREATE_OK(h, alloc(m, &h->dShift, h->n_con + 1));
  CREATE_OK(h, alloc(m, &h->dSigmaSampling, 2)); CREATE_OK(h, alloc(m, &h->dInfeasible, h->max_local + 16));
  CREATE_OK(h, alloc(m, &h->dSc, 1));
  CREATE_OK(h, alloc(m, &h->dAttempt, h->max_zrows + 16));
  if (h->has_constraints) {
    if (cfg->constraint_family != KCMA_CON_HALFSPACE && cfg->constraint_family != KCMA_CON_EXTERNAL) return create_fail(h, "unknown constraint family %d", cfg->constraint_family);
    if (cfg->nranks > 1 && cfg->use_gradient_information) return create_fail(h, "Use Gradient Information together with constraints runs on one GPU (nranks must be 1)");
    h->ldg = (long long)h->s_max;
    h->u_rows = round_up((int)std::min<uint64_t>(h->n_con * h->s_max, 1u << 22), 16) + 32;
    CREATE_OK(h, alloc(m, &h->dG, h->n_con * h->s_max)); CREATE_OK(h, alloc(m, &h->dBounds, h->n_con)); CREATE_OK(h, alloc(m, &h->dNormal, h->n_con * ld));
    CREATE_OK(h, alloc(m, &h->dCaux, nn)); CREATE_OK(h, alloc(m, &h->dBestCon, h->n_con)); CREATE_OK(h, alloc(m, &h->dU, (size_t)h->u_rows * ld));
    CREATE_OK(h, alloc(m, &h->dViol, h->s_max)); CREATE_OK(h, alloc(m, &h->dIndicator, h->n_con * h->s_max));
    CREATE_OK(h, alloc(m, &h->dEvSample, h->n_con * h->s_max + 16)); CREATE_OK(h, alloc(m, &h->dEvCon, h->n_con * h->s_max + 16));
    CREATE_OK(h, alloc(m, &h->dVioRows, h->s_max + 16));
    h->normal_lr = 1.0 / (2.0 + N);                                           // ref :154
    h->cov_adaption_factor = cfg->covariance_matrix_adaption_strength / (N + 2.);  // ref :155
  }
  CREATE_OK(h, alloc_host(m, &h->hSc, 1));
  CREATE_OK(h, alloc_host(m, &h->hCount, 4));
  CREATE_OK(h, alloc_host(m, &h->hRound, 2));
  CREATE_OK(h, alloc(m, &h->dRound, 2)); CREATE_OK(h, alloc(m, &h->dFresh, h->max_local + 16));
  CREATE_OK(h, alloc(m, &h->dRoundV, (size_t)(h->cfg.nranks > 0 ? h->cfg.nranks : 1)));
  CREATE_OK(h, cudaMemcpy(h->dLower, h->lower.data(), sizeof(double) * N, cudaMemcpyHostToDevice));
  CREATE_OK(h, cudaMemcpy(h->dUpper, h->upper.data(), sizeof(double) * N, cudaMemcpyHostToDevice));
  CREATE_OK(h, cudaMemcpy(h->dMinSd, h->min_sd.data(), sizeof(double) * N, cudaMemcpyHostToDevice));
  CREATE_OK(h, cudaMemcpy(h->dCoef, h->coef.data(), sizeof(double) * N, cudaMemcpyHostToDevice));
  if (h->n_con) CREATE_OK(h, cudaMemcpy(h->dShift, h->con_shift.data(), sizeof(double) * h->n_con, cudaMemcpyHostToDevice));
  // ref :20-24, :138/159, :175-183
  DevScalars s; memset(&s, 0, sizeof(s));
  s.best_ever_value = s.previous_best_ever_value = s.previous_best_value = s.current_best_value = -INFINITY;
  s.cur_min_sd = INFINITY; s.cur_max_sd = -INFINITY;
  s.chi_dm = sqrt((double)N) * (1. - 1. / (4. * N) + 1. / (21. * (double)N * N));   // ref :34
  s.global_success_rate = h->has_constraints ? 0.5 : -1.0;
  s.best_valid_sample = h->has_constraints ? ~0ull : 0ull;
  *h->hSc = s;
  CREATE_OK(h, cudaMemcpy(h->dSc, h->hSc, sizeof(DevScalars), cudaMemcpyHostToDevice));
  h->h_weights.assign(h->mu_max, 0.0);
  if (init_mu_weights(h, h->is_viability ? vmu : mu)) return create_fail(h, "%s", h->err.c_str());
  init_covariance(h);
  CREATE_OK(h, cudaMemcpy(h->dMean, h->init_val.data(), sizeof(double) * N, cudaMemcpyHostToDevice));
  CREATE_OK(h, cudaMemcpy(h->dMeanOld, h->init_val.data(), sizeof(double) * N, cudaMemcpyHostToDevice));
  CREATE_OK(h, cudaDeviceSynchronize());
  *out = h;
  return 0;
}

int kcma_set_host_objective(kcma_t* h, kcma_host_objective_fn fn, void* user) {
  if (!h) return fail(h, "null solver handle");
  invalidate_graph(h);
  if (fn && !h->cfg.keep_population) return fail(h, "a host objective needs keep_population = 1 (X is copied to the host every generation)");
  h->host_obj = fn; h->host_obj_user = user;
  return 0;
}
int kcma_set_host_objective_grad(kcma_t* h, kcma_host_objective_grad_fn fn, void* user) {
  if (!h) return fail(h, "null solver handle");
  invalidate_graph(h);
  if (fn && !h->cfg.use_gradient_information) return fail(h, "a gradient-returning host objective needs Use Gradient Information");
  if (fn && !h->cfg.keep_population) return fail(h, "a host objective needs keep_population = 1 (X is copied to the host every generation)");
  h->host_obj_grad = fn; h->host_obj_user = user;
  return 0;
}
int kcma_set_device_objective(kcma_t* h, kcma_device_objective_fn fn, void* user) {
  if (!h) return fail(h, "null solver handle");
  invalidate_graph(h);
  if (fn && !h->cfg.keep_population) return fail(h, "a device objective needs keep_population = 1 (it reads the materialised X)");
  if (fn && h->cfg.use_gradient_information) return fail(h, "a device objective cannot return gradients: use kcma_set_host_objective_grad");
  h->dev_obj = fn; h->dev_obj_user = user;
  return 0;
}
int kcma_set_host_constraints(kcma_t* h, kcma_host_constraints_fn fn, void* user) {
  if (!h) return fail(h, "null solver handle");
  invalidate_graph(h);
  if (!h->has_constraints) return fail(h, "the problem has no constraints (n_constraints = 0)");
  if (fn && !h->cfg.keep_population) return fail(h, "host constraints need keep_population = 1 (X is copied to the host)");
  h->host_con = fn; h->host_con_user = user;
  return 0;
}

int kcma_comm_unique_id(uint8_t id_out[128]) {
  std::string err;
  if (!g_nccl.load(err)) return fail<kcma>(nullptr, "%s", err.c_str());
  ncclUniqueId id;
  if (g_nccl.GetUniqueId(&id) != ncclSuccess) return fail<kcma>(nullptr, "ncclGetUniqueId failed");
  memcpy(id_out, id.internal, 128);
  return 0;
}

int kcma_comm_init(kcma_t* h, const uint8_t id_in[128]) {
  if (!h) return fail(h, "null solver handle");
  std::string err;
  if (!g_nccl.load(err)) return fail(h, "%s", err.c_str());
  CUDA_OK(h, cudaSetDevice(h->device));
  ncclUniqueId id;
  memcpy(id.internal, id_in, 128);
  return nccl_check(h, g_nccl.CommInitRank(&h->comm, h->cfg.nranks, id, h->cfg.rank), "ncclCommInitRank");
}

// All ranks of ONE process (one handle per device, rank r = handles[r]): the communicator is built inside an NCCL group.
int kcma_comm_init_all(kcma_t** handles, int count) {
  if (!handles || count < 1) return fail<kcma>(nullptr, "kcma_comm_init_all: no handles");
  std::string err;
  if (!g_nccl.load(err)) return fail(handles[0], "%s", err.c_str());
  for (int r = 0; r < count; r++) {
    if (!handles[r]) return fail(handles[r], "null solver handle");
    if (handles[r]->cfg.nranks != count || handles[r]->cfg.rank != r)
      return fail(handles[r], "kcma_comm_init_all: handle %d was created as rank %d of %d, expected rank %d of %d", r, handles[r]->cfg.rank,
                  handles[r]->cfg.nranks, r, count);
  }
  ncclUniqueId id;
  if (g_nccl.GetUniqueId(&id) != ncclSuccess) return fail(handles[0], "ncclGetUniqueId failed");
  if (nccl_check(handles[0], g_nccl.GroupStart(), "ncclGroupStart")) return 1;
  int rc = 0;
  for (int r = 0; r < count && !rc; r++) {
    if (cudaSetDevice(handles[r]->device) != cudaSuccess) { rc = fail(handles[r], "cudaSetDevice(%d) failed", handles[r]->device); break; }
    rc = nccl_check(handles[r], g_nccl.CommInitRank(&handles[r]->comm, count, id, r), "ncclCommInitRank");
  }
  const ncclResult_t ge = g_nccl.GroupEnd();
  if (!rc) rc = nccl_check(handles[0], ge, "ncclGroupEnd");
  for (int r = 0; r < count; r++) handles[r]->comm_in_process = true;
  return rc;
}

int kcma_ask(kcma_t* h) {
  if (!h) return fail(h, "null solver handle");
  CUDA_OK(h, cudaSetDevice(h->device));
  return do_ask(h);
}

int kcma_eval(kcma_t* h) {
  if (!h) return fail(h, "null solver handle");
  CUDA_OK(h, cudaSetDevice(h->device));
  if (do_eval(h)) return 1;
  if (pull_cached(h)) return 1;
  if (h->hSc->nonfinite) {
    h->hSc->nonfinite = 0;
    push_scalars(h);
    return fail(h, "Non finite value of function evaluation detected: nan\n");
  }
  return 0;
}

int kcma_tell(kcma_t* h) {
  if (!h) return fail(h, "null solver handle");
  CUDA_OK(h, cudaSetDevice(h->device));
  if (do_tell(h)) return 1;
  return end_of_generation(h);
}

namespace {

__global__ void set_gen_kernel(DevScalars* sc, unsigned long long gen) { sc->gen = gen; }
__global__ void inc_gen_kernel(DevScalars* sc) { sc->gen += 1; }

void invalidate_graph(kcma* h) {
  if (h->gexec) { cudaGraphExecDestroy(h->gexec); h->gexec = nullptr; }
}

// A whole generation can be replayed as ONE CUDA graph when it is a fixed sequence of launches: built-in
// objective, no constraint path (its loops are host-driven), no resampling rounds, no pending injection, no phase timers,
// eigensolver = one launch (N <= 1184 or diagonal). Small configurations are launch-latency bound (44-47 launches of a few
// microseconds each per generation, SURVEY 8d): the graph removes the per-launch host cost. KCMA_GRAPH=0 disables it.
bool graph_eligible(const kcma* h) {
  static const int on = getenv("KCMA_GRAPH") ? atoi(getenv("KCMA_GRAPH")) : 1;
  // several ranks: the two collectives of a generation are captured with it (NCCL records them as graph nodes); every rank replays
  // the same sequence, and a rank that falls back to eager launches still issues the same collectives in the same order
  static const int multi_on = getenv("KCMA_GRAPH_MULTI") ? atoi(getenv("KCMA_GRAPH_MULTI")) : 1;
  // (one process per rank: 119.8 -> 121.6 generations/s on two GPUs. With the ranks as threads of ONE process the replay of graphs that
  // hold collectives measured slower than eager launches — 111 against 124 generations/s through Engine().run(e) — so that mode stays eager;
  // profiles/r02_bench_2gpu_graph_ab.log)
  if (h->cfg.nranks > 1 && (!multi_on || !h->comm || h->comm_in_process)) return false;
  if (!on || h->graph_failed || h->timing || h->host_obj || h->host_obj_grad || h->dev_obj || h->host_con || h->has_constraints) return false;
  if (h->cfg.objective == KCMA_OBJ_EXTERNAL || h->has_discrete) return false;
  if (h->has_bounds && h->cfg.max_infeasible_resamplings != 0) return false;
  if (h->inj_z || h->inj_bd || h->inj_y || h->inj_x || h->inj_f || h->inj_grad || h->sampled_pending || !h->vt_valid) return false;
  if (!h->cfg.diagonal_covariance && ((h->N + 3) / 4 + 1) / 2 > h->num_sms) return false;   // eigensolver with a host loop
  return h->gen >= 3;   // the first generations run eagerly (lazy one-time initialisations happen there)
}

// Capture ask + eval + tell of the NEXT generation; the capture pass only records, so the host-side bookkeeping it did is
// rolled back and re-applied per replay. Returns false (and never tries again) when anything in the sequence cannot be captured.
bool build_graph(kcma* h) {
  if (!h->cap_stream && cudaStreamCreateWithFlags(&h->cap_stream, cudaStreamNonBlocking) != cudaSuccess) { h->graph_failed = true; return false; }
  set_gen_kernel<<<1, 1, 0, h->stream>>>(h->dSc, h->gen - 1);
  h->dev_gen = h->gen - 1;
  const uint64_t gen0 = h->gen, launches0 = h->launches, evals0 = h->model_evals;
  const cudaStream_t saved = h->stream;
  h->capturing = true;
  h->stream = h->cap_stream;
  cudaGraph_t graph = nullptr;
  int rc = 1;
  if (cudaStreamBeginCapture(h->cap_stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
    inc_gen_kernel<<<1, 1, 0, h->stream>>>(h->dSc);
    h->launches++;
    rc = do_ask(h) || do_eval(h) || do_tell(h);
    if (cudaStreamEndCapture(h->cap_stream, &graph) != cudaSuccess) rc = 1;
  }
  h->stream = saved;
  h->capturing = false;
  h->g_launches = h->launches - launches0;
  h->g_evals = h->model_evals - evals0;
  h->gen = gen0; h->launches = launches0; h->model_evals = evals0;
  h->sampled_pending = false;
  h->scalars_fresh = false;
  if (!rc && cudaGraphInstantiate(&h->gexec, graph, 0) != cudaSuccess) rc = 1;
  if (graph) cudaGraphDestroy(graph);
  if (rc) {
    cudaGetLastError();
    h->gexec = nullptr;
    h->graph_failed = true;
    h->err.clear();
    return false;
  }
  return true;
}

}  // namespace

int kcma_run_generation(kcma_t* h) {
  if (!h) return fail(h, "null solver handle");
  CUDA_OK(h, cudaSetDevice(h->device));
  if (graph_eligible(h) && (h->gexec || build_graph(h))) {
    // The replay takes the generation from DevScalars::gen (inc_gen_kernel is its first node). Eager generations in between
    // (kcma_ask/eval/tell, or kcma_timing_enable) advance only the host counter: re-seed the device copy when it is behind.
    if (h->dev_gen != h->gen - 1) { set_gen_kernel<<<1, 1, 0, h->stream>>>(h->dSc, h->gen - 1); h->launches++; }
    CUDA_OK(h, cudaGraphLaunch(h->gexec, h->stream));
    h->gen++;
    h->dev_gen = h->gen - 1;
    h->launches += h->g_launches;
    h->model_evals += h->g_evals;
    h->scalars_fresh = false;
    return end_of_generation(h);
  }
  PhaseTimer* t = h->timing ? new PhaseTimer(h, "generation") : nullptr;
  int rc = do_ask(h) || do_eval(h) || do_tell(h);
  delete t;
  if (rc) return 1;
  return end_of_generation(h);
}

int kcma_check_termination(kcma_t* h, int* finished, const char** reason) {
  if (!h) return fail(h, "null solver handle");
  if (pull_cached(h)) return 1;
  const DevScalars& s = *h->hSc;
  int fin = 0;
  h->reason.clear();
  const uint64_t gen = h->gen, maxres = h->cfg.max_infeasible_resamplings;
  if (gen > 1 && ((maxres > 0) && (s.infeasible_sample_count >= maxres))) { h->reason += "CMAES['Max Infeasible Resamplings'];"; fin = 1; }
  if (gen > 1 && (s.max_eig >= h->tc_max_condition * s.min_eig)) { h->reason += "CMAES['Max Condition Covariance Matrix'];"; fin = 1; }
  if (gen > 1 && (s.cur_min_sd <= h->tc_min_sd)) { h->reason += "CMAES['Min Standard Deviation'];"; fin = 1; }
  if (gen > 1 && (s.cur_max_sd >= h->tc_max_sd)) { h->reason += "CMAES['Max Standard Deviation'];"; fin = 1; }
  if (!fin) {
    if (gen > 1 && (+s.best_ever_value > h->tc_max_value)) { h->reason += "optimizer['Max Value'];"; fin = 1; }
    // SURVEY Q1: the base-class _previousBestValue is never written and stays 0.0
    if (gen > 1 && (fabs(s.current_best_value - 0.0) < h->tc_min_value_diff)) { h->reason += "optimizer['Min Value Difference Threshold'];"; fin = 1; }
    if (!fin) {
      if (h->tc_max_model_evaluations <= (double)h->model_evals) { h->reason += "solver['Max Model Evaluations'];"; fin = 1; }
      if ((double)gen > h->tc_max_generations) { h->reason += "solver['Max Generations'];"; fin = 1; }
    }
  }
  *finished = fin;
  if (reason) *reason = h->reason.c_str();
  return 0;
}

int kcma_run(kcma_t* h, uint64_t max_generations, uint64_t* done) {
  return run(h, max_generations, done, kcma_check_termination, kcma_run_generation);
}

// ---- injection ---------------------------------------------------------------------------------------------
static int upload_rows(kcma* h, double* dst, const double* src, size_t rows) {
  CUDA_OK(h, cudaMemcpy2DAsync(dst, sizeof(double) * h->ld, src, sizeof(double) * h->N, sizeof(double) * h->N, rows,
                               cudaMemcpyHostToDevice, h->stream));
  CUDA_OK(h, cudaStreamSynchronize(h->stream));
  return 0;
}

int kcma_inject(kcma_t* h, int kind, const double* src, size_t count) {
  if (!h) return fail(h, "null solver handle");
  invalidate_graph(h);
  CUDA_OK(h, cudaSetDevice(h->device));
  const size_t N = h->N;
  const size_t zunit = h->cfg.mirrored_sampling ? 2 : 1;
  switch (kind) {
    case KCMA_INJ_Z: {
      if (count != h->cur_lambda / zunit * N) return fail(h, "inject Z: expected %zu values", (size_t)(h->cur_lambda / zunit * N));
      if (upload_rows(h, h->dZ, src + (h->shard_lo / zunit) * N, local_zrows(h))) return 1;
      h->inj_z = true;
      return 0;
    }
    case KCMA_INJ_BDZ: {
      if (count != h->cur_lambda * N) return fail(h, "inject BDZ: expected %zu values", (size_t)(h->cur_lambda * N));
      if (zunit == 1) { if (upload_rows(h, h->dY, src + h->shard_lo * N, local_samples(h))) return 1; }
      else {  // even members carry +y
        CUDA_OK(h, cudaMemcpy2DAsync(h->dY, sizeof(double) * h->ld, src + h->shard_lo * N, sizeof(double) * 2 * N, sizeof(double) * N,
                                     local_zrows(h), cudaMemcpyHostToDevice, h->stream));
        CUDA_OK(h, cudaStreamSynchronize(h->stream));
      }
      h->inj_y = true;
      return 0;
    }
    case KCMA_INJ_X: {
      if (count != h->cur_lambda * N) return fail(h, "inject X: expected %zu values", (size_t)(h->cur_lambda * N));
      if (!h->cfg.keep_population) return fail(h, "inject X needs keep_population = 1 (the Sample Population buffer)");
      if (upload_rows(h, h->dX, src + h->shard_lo * N, local_samples(h))) return 1;
      h->inj_x = true;
      return 0;
    }
    case KCMA_INJ_F: {
      if (count != h->cur_lambda) return fail(h, "inject F: expected %zu values", (size_t)h->cur_lambda);
      for (size_t i = 0; i < count; i++)
        if (!std::isfinite(src[i])) return fail(h, "Non finite value of function evaluation detected: %f\n", src[i]);
      CUDA_OK(h, cudaMemcpyAsync(h->dF, src, sizeof(double) * count, cudaMemcpyHostToDevice, h->stream));
      CUDA_OK(h, cudaStreamSynchronize(h->stream));
      h->inj_f = true;
      return 0;
    }
    case KCMA_INJ_GRAD: {
      if (!h->cfg.use_gradient_information) return fail(h, "inject Gradients: Use Gradient Information is off");
      if (count != h->cur_lambda * N) return fail(h, "inject Gradients: expected %zu values", (size_t)(h->cur_lambda * N));
      if (upload_rows(h, h->dGrad, src + h->shard_lo * N, local_samples(h))) return 1;
      h->inj_grad = true;
      return 0;
    }
    case KCMA_INJ_BD: {
      if (count != N * N + N) return fail(h, "inject BD: expected N*N+N values");
      if (upload_rows(h, h->dB, src, N)) return 1;
      CUDA_OK(h, cudaMemcpy(h->dD, src + N * N, sizeof(double) * N, cudaMemcpyHostToDevice));
      if (pull_cached(h)) return 1;
      double mn = INFINITY, mx = -INFINITY;
      for (size_t d = 0; d < N; d++) { const double ev = src[N * N + d] * src[N * N + d]; mn = std::min(mn, ev); mx = std::max(mx, ev); }
      h->hSc->min_eig = mn; h->hSc->max_eig = mx;
      if (push_scalars(h)) return 1;
      h->vt_valid = false;
      h->inj_bd = true;
      return 0;
    }
  }
  return fail(h, "unknown injection kind %d", kind);
}

// ---- state access ---------------------------------------------------------------------------------------------
namespace {
bool find_array(kcma* h, const char* key, Array* r) {
  const size_t N = h->N, ld = h->ld;
#define A(K, ARR) if (!strcmp(key, K)) { *r = ARR; return true; }
  A("Covariance Matrix", pitched(h->dC, N, N, ld))
  A("Covariance Eigenvector Matrix", pitched(h->dB, N, N, ld))
  A("Axis Lengths", dense(h->dD, N))
  A("Current Mean", dense(h->dMean, N))
  A("Previous Mean", dense(h->dMeanOld, N))
  A("Mean Update", dense(h->dMeanUpd, N))
  A("Evolution Path", dense(h->dPc, N))
  A("Conjugate Evolution Path", dense(h->dPs, N))
  A("Auxiliar BDZ Matrix", dense(h->dT, N))
  A("Mu Weights", dense(h->dW, h->cur_mu))
  A("Value Vector", dense(h->dF, h->cur_lambda))
  A("Best Ever Variables", dense(h->dBestEver, N))
  A("Current Best Variables", dense(h->dCurBest, N))
  A("Objective Coefficients", dense(h->dCoef, N))
  if (h->has_constraints) {
    A("Viability Boundaries", dense(h->dBounds, h->n_con))
    A("Normal Constraint Approximation", pitched(h->dNormal, h->n_con, N, ld))
    A("Best Constraint Evaluations", dense(h->dBestCon, h->n_con))
    A("Constraint Evaluations", pitched(h->dG, h->n_con, h->s_max, h->s_max))
    A("Auxiliar Covariance Matrix", pitched(h->dCaux, N, N, ld))
  }
#undef A
  return false;
}
}  // namespace

int kcma_get_array(kcma_t* h, const char* key, double* out, size_t cap, size_t* count) {
  if (!h) return fail(h, "null solver handle");
  CUDA_OK(h, cudaSetDevice(h->device));
  const size_t N = h->N;
  if (!strcmp(key, "BDZ Matrix") || !strcmp(key, "Sample Population")) {
    // LOCAL shard rows [shard_lo, shard_hi) of the population
    const size_t ls = local_samples(h), n = ls * N;
    if (count) *count = n;
    if (!out) return 0;
    if (cap < n) return fail(h, "buffer too small for '%s'", key);
    if (strcmp(key, "BDZ Matrix") && !h->cfg.keep_population)
      return fail(h, "'Sample Population' is not materialised: create the handle with keep_population = 1");
    Allocations scratch;
    double* tmp = nullptr;
    CUDA_OK(h, alloc(scratch, &tmp, n));
    if (strcmp(key, "BDZ Matrix"))
      cudaMemcpy2DAsync(tmp, sizeof(double) * N, h->dX, sizeof(double) * h->ld, sizeof(double) * N, ls, cudaMemcpyDeviceToDevice, h->stream);
    else if (h->cfg.mirrored_sampling)
      expand_mirrored_kernel<<<h->num_sms * 4, 256, 0, h->stream>>>(h->dY, tmp, h->ld, (long long)ls, (int)N);
    else
      cudaMemcpy2DAsync(tmp, sizeof(double) * N, h->dY, sizeof(double) * h->ld, sizeof(double) * N, ls, cudaMemcpyDeviceToDevice, h->stream);
    cudaError_t e = cudaMemcpyAsync(out, tmp, sizeof(double) * n, cudaMemcpyDeviceToHost, h->stream);
    cudaStreamSynchronize(h->stream);
    CUDA_OK(h, e);
    return 0;
  }
  Array r;
  if (!strcmp(key, "Gradients") && h->dGrad) r = pitched(h->dGrad, local_samples(h), N, h->ld);   // LOCAL shard rows, like "Sample Population"
  else if (!strcmp(key, "Discrete Mutations") && h->dDiscMut) r = pitched(h->dDiscMut, local_samples(h), N, h->ld);
  else if (!strcmp(key, "Masking Matrix") && h->dMask) r = dense(h->dMask, N);
  else if (!strcmp(key, "Masking Matrix Sigma") && h->dMaskSigma) r = dense(h->dMaskSigma, N);
  else if (!find_array(h, key, &r)) return fail(h, "unknown array key '%s'", key);
  return copy_out(h, key, r, out, cap, count, "buffer too small for '%s' (%zu < %zu)");
}

int kcma_set_array(kcma_t* h, const char* key, const double* in, size_t count) {
  if (!h) return fail(h, "null solver handle");
  invalidate_graph(h);
  CUDA_OK(h, cudaSetDevice(h->device));
  Array r;
  if (!find_array(h, key, &r)) return fail(h, "unknown array key '%s'", key);
  if (copy_in(h, key, r, in, count)) return 1;
  if (!strcmp(key, "Covariance Eigenvector Matrix") || !strcmp(key, "Axis Lengths")) h->vt_valid = false;
  if (!strcmp(key, "Mu Weights")) std::copy(in, in + count, h->h_weights.begin());
  return 0;
}

int kcma_get_index_array(kcma_t* h, const char* key, uint64_t* out, size_t cap, size_t* count) {
  if (!h) return fail(h, "null solver handle");
  CUDA_OK(h, cudaSetDevice(h->device));
  const size_t n = h->cur_lambda;
  Array r;
  if (!strcmp(key, "Sample Constraint Violation Counts")) r = dense(h->dViol, h->has_constraints ? n : 0, Elem::u64);
  else if (!strcmp(key, "Sorting Index")) r = dense(h->dIdx, n, Elem::u32);
  else return fail(h, "unknown index key '%s'", key);
  return copy_out(h, key, r, out, cap, count, "buffer too small for '%s'");
}

namespace {
double* find_dev_scalar(kcma* h, const char* key) {
  DevScalars* s = h->hSc;
#define S(K, F) if (!strcmp(key, K)) return &s->F;
  S("Sigma", sigma) S("Conjugate Evolution Path L2 Norm", ps_l2norm)
  S("Best Ever Value", best_ever_value) S("Previous Best Ever Value", previous_best_ever_value)
  S("Previous Best Value", previous_best_value) S("Current Best Value", current_best_value)
  S("Maximum Diagonal Covariance Matrix Element", max_diag_c) S("Minimum Diagonal Covariance Matrix Element", min_diag_c)
  S("Maximum Covariance Eigenvalue", max_eig) S("Minimum Covariance Eigenvalue", min_eig)
  S("Current Min Standard Deviation", cur_min_sd) S("Current Max Standard Deviation", cur_max_sd)
  S("Global Success Rate", global_success_rate) S("Chi Square Number Discrete Mutations", chi_dm)
#undef S
  return nullptr;
}
const HostScalar<kcma> kHostScalars[] = {
    {"Trace", &kcma::trace, true},
    {"Effective Mu", &kcma::mueff, true},
    {"Sigma Cumulation Factor", &kcma::cs, true},
    {"Damp Factor", &kcma::damp, true},
    {"Cumulative Covariance", &kcma::cc, true},
    {"Chi Square Number", &kcma::chi_n, true},
    {"Termination Criteria/Max Condition Covariance Matrix", &kcma::tc_max_condition, true},
    {"Termination Criteria/Min Standard Deviation", &kcma::tc_min_sd, true},
    {"Termination Criteria/Max Standard Deviation", &kcma::tc_max_sd, true},
    {"Termination Criteria/Max Value", &kcma::tc_max_value, true},
    {"Termination Criteria/Min Value Difference Threshold", &kcma::tc_min_value_diff, true},
    {"Termination Criteria/Max Model Evaluations", &kcma::tc_max_model_evaluations, true},
    {"Termination Criteria/Max Generations", &kcma::tc_max_generations, true},
};
}  // namespace

int kcma_get_scalar(kcma_t* h, const char* key, double* out) {
  if (!h) return fail(h, "null solver handle");
  CUDA_OK(h, cudaSetDevice(h->device));
  if (double* p = host_scalar(h, kHostScalars, key, false)) { *out = *p; return 0; }
  if (pull_cached(h)) return 1;
  if (double* p = find_dev_scalar(h, key)) { *out = *p; return 0; }
#define U(K, V) if (!strcmp(key, K)) { *out = (double)(V); return 0; }
  U("Current Generation", h->gen - 1) U("Model Evaluation Count", h->model_evals) U("Variable Count", h->N)
  U("Current Population Size", h->cur_lambda) U("Current Mu Value", h->cur_mu)
  U("Infeasible Sample Count", h->hSc->infeasible_sample_count)
  U("Number Of Discrete Mutations", h->hSc->n_disc_mut) U("Number Masking Matrix Entries", h->hSc->n_mask)
  U("Resampled Parameter Count", h->hSc->resampled_parameter_count)
  U("Covariance Matrix Adaptation Count", h->hSc->cov_adaptation_count)
  U("Max Constraint Violation Count", h->hSc->max_violation_count)
  U("Constraint Evaluation Count", h->hSc->constraint_evaluation_count)
  U("Covariance Matrix Adaption Factor", h->cov_adaption_factor) U("Normal Vector Learning Rate", h->normal_lr)
  U("Is Viability Regime", h->is_viability) U("Has Constraints", h->has_constraints)
  U("Best Valid Sample", (long long)h->hSc->best_valid_sample)
  U("Termination Criteria/Max Infeasible Resamplings", h->cfg.max_infeasible_resamplings)
  U("Shard Begin", h->eval_lo) U("Shard End", h->eval_hi)   // the samples this rank evaluates
#undef U
  return fail(h, "unknown scalar key '%s'", key);
}

int kcma_set_scalar(kcma_t* h, const char* key, double v) {
  if (!h) return fail(h, "null solver handle");
  invalidate_graph(h);
  CUDA_OK(h, cudaSetDevice(h->device));
  if (double* p = host_scalar(h, kHostScalars, key, true)) { *p = v; return 0; }
  if (pull_cached(h)) return 1;
  if (double* p = find_dev_scalar(h, key)) { *p = v; return push_scalars(h); }
#define U(K, STMT) if (!strcmp(key, K)) { STMT; return 0; }
  U("Current Generation", h->gen = (uint64_t)v + 1)
  U("Model Evaluation Count", h->model_evals = (uint64_t)v)
  U("Termination Criteria/Max Infeasible Resamplings", h->cfg.max_infeasible_resamplings = (uint64_t)v)
#undef U
  if (!strcmp(key, "Infeasible Sample Count")) { h->hSc->infeasible_sample_count = (unsigned long long)v; return push_scalars(h); }
  // counters of the constraint path (restored by loadState: CMAES.cpp:1042-1560 reads every internal setting back)
#define C(K, F) if (!strcmp(key, K)) { h->hSc->F = (unsigned long long)(long long)v; return push_scalars(h); }
  C("Resampled Parameter Count", resampled_parameter_count) C("Covariance Matrix Adaptation Count", cov_adaptation_count)
  C("Max Constraint Violation Count", max_violation_count) C("Constraint Evaluation Count", constraint_evaluation_count)
  C("Best Valid Sample", best_valid_sample)
#undef C
  if (!strcmp(key, "Is Viability Regime")) {
    // the regime decides population size, mu and the weights (:52-62, :336-344); unlike checkMeanAndSetRegime this restores a
    // saved regime and therefore must NOT re-initialise C, sigma and the boundaries
    if (!h->has_constraints) return (v != 0.0) ? fail(h, "'Is Viability Regime' needs a constrained problem") : 0;
    h->is_viability = v != 0.0 ? 1 : 0;
    set_population(h, h->is_viability ? h->vlambda : h->lambda, h->is_viability ? h->vmu : h->mu);
    return init_mu_weights(h, h->cur_mu);
  }
  return fail(h, "unknown scalar key '%s'", key);
}

// ---- measurement ------------------------------------------------------------------------------------------
// debug hook (not part of include/kcma.h): phase timestamps of the Gram Jacobi kernel, 32 steps x 8 slots
extern "C" int kcma_debug_jacobi_timestamps(long long* out3584) {
  if (!kc::g_jacobi_dbg) return 1;
  return cudaMemcpy(out3584, kc::g_jacobi_dbg, sizeof(long long) * 3584, cudaMemcpyDeviceToHost) != cudaSuccess;
}
int kcma_timing_enable(kcma_t* h, int on) { if (!h) return fail(h, "null solver handle"); h->timing = on != 0; return 0; }   // the graph path is skipped while timing
int kcma_timing_get(kcma_t* h, const char* phase, double* ms, uint64_t* calls) {
  if (!h) return fail(h, "null solver handle");
  resolve_timers(h);
  auto it = h->phases.find(phase);
  if (ms) *ms = it == h->phases.end() ? 0.0 : it->second.ms;
  if (calls) *calls = it == h->phases.end() ? 0 : it->second.calls;
  if (calls && !strcmp(phase, "eigen_sweeps")) {   // persistent kernel: counted on the device; per-step path: counted by the host loop
    h->scalars_fresh = false;
    if (pull_cached(h)) return 1;
    *calls += h->hSc->jacobi_sweeps_total - h->sweeps_base;
  }
  return 0;
}
int kcma_timing_reset(kcma_t* h) {
  if (!h) return fail(h, "null solver handle");
  resolve_timers(h);
  h->phases.clear();
  h->scalars_fresh = false;
  if (pull_cached(h)) return 1;
  h->sweeps_base = h->hSc->jacobi_sweeps_total;
  return 0;
}
uint64_t kcma_launch_count(const kcma_t* h) { return h ? h->launches : 0; }
int kcma_flush_l2(kcma_t* h) {
  if (!h) return fail(h, "null solver handle");
  CUDA_OK(h, cudaSetDevice(h->device));
  if (!h->dFlush) { h->flush_bytes = 256ull << 20; CUDA_OK(h, alloc(h->mem, &h->dFlush, h->flush_bytes / sizeof(double))); }
  flush_kernel<<<h->num_sms * 8, 256, 0, h->stream>>>(h->dFlush, h->flush_bytes / sizeof(double));
  return 0;
}

// ---- single kernels on host buffers -----------------------------------------------------------------------
// They have no handle: failures are reported through kcma_last_error(NULL), and each call's buffers are freed on every return.
static kcma* const kNoHandle = nullptr;

int kcma_k_sort_index(int device, const double* f, uint64_t n, uint64_t* index_out) {
  if (n == 0) return 0;
  CUDA_OK(kNoHandle, cudaSetDevice(device));
  int sms; cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  Allocations scratch;
  double* df; unsigned* di; unsigned char* ws;
  CUDA_OK(kNoHandle, alloc(scratch, &df, n)); CUDA_OK(kNoHandle, alloc(scratch, &di, n));
  CUDA_OK(kNoHandle, alloc(scratch, &ws, sort_workspace_bytes((int)n)));
  CUDA_OK(kNoHandle, cudaMemcpy(df, f, sizeof(double) * n, cudaMemcpyHostToDevice));
  launch_sort_index(0, df, (int)n, ws, di, sms);
  std::vector<unsigned> tmp(n);
  CUDA_OK(kNoHandle, cudaMemcpy(tmp.data(), di, sizeof(unsigned) * n, cudaMemcpyDeviceToHost));
  for (uint64_t i = 0; i < n; i++) index_out[i] = tmp[i];
  return 0;
}

int kcma_k_sample(int device, uint64_t n, uint64_t rows, const double* z, const double* b, const double* d, const double* mean,
                  double sigma, double* y_out, double* x_out) {
  CUDA_OK(kNoHandle, cudaSetDevice(device));
  const int N = (int)n, ld = round_up(N, 16);
  Allocations scratch;
  double *dZ, *dB, *dA, *dD, *dY;
  CUDA_OK(kNoHandle, alloc(scratch, &dZ, rows * ld)); CUDA_OK(kNoHandle, alloc(scratch, &dY, rows * ld));
  CUDA_OK(kNoHandle, alloc(scratch, &dB, (size_t)N * ld)); CUDA_OK(kNoHandle, alloc(scratch, &dA, (size_t)N * ld));
  CUDA_OK(kNoHandle, alloc(scratch, &dD, ld));
  CUDA_OK(kNoHandle, cudaMemcpy2D(dZ, sizeof(double) * ld, z, sizeof(double) * N, sizeof(double) * N, rows, cudaMemcpyHostToDevice));
  CUDA_OK(kNoHandle, cudaMemcpy2D(dB, sizeof(double) * ld, b, sizeof(double) * N, sizeof(double) * N, N, cudaMemcpyHostToDevice));
  CUDA_OK(kNoHandle, cudaMemcpy(dD, d, sizeof(double) * N, cudaMemcpyHostToDevice));
  launch_scale_bd(0, dB, ld, dD, dA, ld, N);
  launch_gemm_tn(0, (int)rows, N, N, dZ, ld, dA, ld, dY, ld);
  CUDA_OK(kNoHandle, cudaMemcpy2D(y_out, sizeof(double) * N, dY, sizeof(double) * ld, sizeof(double) * N, rows, cudaMemcpyDeviceToHost));
  if (x_out)
    for (uint64_t i = 0; i < rows; i++)
      for (int k = 0; k < N; k++) x_out[i * N + k] = mean[k] + sigma * y_out[i * N + k];
  CUDA_OK(kNoHandle, cudaGetLastError());
  return 0;
}

int kcma_k_rank_mu(int device, uint64_t n, uint64_t rows, const double* t, const double* w, double* p_out) {
  CUDA_OK(kNoHandle, cudaSetDevice(device));
  int sms; cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  const int N = (int)n, ld = round_up(N, 16);
  const size_t rp = round_up((int)rows, 16) + 16;
  std::vector<double> s(rows * N);
  for (uint64_t k = 0; k < rows; k++) {
    const double rw = sqrt(w[k]);
    for (int d = 0; d < N; d++) s[k * N + d] = rw * t[k * N + d];
  }
  Allocations scratch;
  double *dS, *dW, *dP;
  CUDA_OK(kNoHandle, alloc(scratch, &dS, rp * ld));
  CUDA_OK(kNoHandle, alloc(scratch, &dW, (size_t)16 * N * ld)); CUDA_OK(kNoHandle, alloc(scratch, &dP, (size_t)N * ld));
  CUDA_OK(kNoHandle, cudaMemcpy2D(dS, sizeof(double) * ld, s.data(), sizeof(double) * N, sizeof(double) * N, rows, cudaMemcpyHostToDevice));
  const int splits = launch_syrk(0, N, (int)rows, nullptr, dS, ld, (long long)rp, dW, ld, (int)rows, sms, 16);
  launch_reduce_splits(0, dW, ld, splits, N, dP);
  std::vector<double> p((size_t)N * N);
  CUDA_OK(kNoHandle, cudaMemcpy2D(p.data(), sizeof(double) * N, dP, sizeof(double) * ld, sizeof(double) * N, N, cudaMemcpyDeviceToHost));
  for (int d = 0; d < N; d++)
    for (int e = 0; e <= d; e++) p_out[(size_t)d * N + e] = p_out[(size_t)e * N + d] = p[(size_t)d * N + e];
  CUDA_OK(kNoHandle, cudaGetLastError());
  return 0;
}

int kcma_k_philox_normal(int device, uint64_t seed, uint64_t generation, uint64_t row_begin, uint64_t rows, uint64_t n, double* z_out) {
  CUDA_OK(kNoHandle, cudaSetDevice(device));
  int sms; cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  const int N = (int)n, ld = round_up(N, 16);
  Allocations scratch;
  double* dZ;
  CUDA_OK(kNoHandle, alloc(scratch, &dZ, rows * ld));
  launch_philox_normal(0, dZ, ld, (long long)rows, N, seed, (unsigned)generation, row_begin, nullptr, nullptr, sms);
  CUDA_OK(kNoHandle, cudaMemcpy2D(z_out, sizeof(double) * N, dZ, sizeof(double) * ld, sizeof(double) * N, rows, cudaMemcpyDeviceToHost));
  CUDA_OK(kNoHandle, cudaGetLastError());
  return 0;
}

int kcma_k_philox_raw(int device, const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
  CUDA_OK(kNoHandle, cudaSetDevice(device));
  uint32_t in[6] = {ctr[0], ctr[1], ctr[2], ctr[3], key[0], key[1]};
  Allocations scratch;
  uint32_t *din, *dout;
  CUDA_OK(kNoHandle, alloc(scratch, &din, 6)); CUDA_OK(kNoHandle, alloc(scratch, &dout, 4));
  CUDA_OK(kNoHandle, cudaMemcpy(din, in, sizeof(in), cudaMemcpyHostToDevice));
  launch_philox_raw(0, din, dout);
  CUDA_OK(kNoHandle, cudaMemcpy(out, dout, 16, cudaMemcpyDeviceToHost));
  return 0;
}

int kcma_k_objective(int device, int objective, uint64_t n, uint64_t rows, const double* x, const double* coef, double* f_out) {
  CUDA_OK(kNoHandle, cudaSetDevice(device));
  int sms; cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  const int N = (int)n, ld = round_up(N, 16);
  Allocations scratch;
  double *dX, *dCoef, *dF; DevScalars* dSc;
  CUDA_OK(kNoHandle, alloc(scratch, &dX, rows * ld)); CUDA_OK(kNoHandle, alloc(scratch, &dCoef, ld));
  CUDA_OK(kNoHandle, alloc(scratch, &dF, rows)); CUDA_OK(kNoHandle, alloc(scratch, &dSc, 1));
  CUDA_OK(kNoHandle, cudaMemcpy2D(dX, sizeof(double) * ld, x, sizeof(double) * N, sizeof(double) * N, rows, cudaMemcpyHostToDevice));
  std::vector<double> c(N);
  for (int i = 0; i < N; i++) c[i] = coef ? coef[i] : (N > 1 ? pow(10.0, 6.0 * (double)i / (double)(N - 1)) : 1.0);
  CUDA_OK(kNoHandle, cudaMemcpy(dCoef, c.data(), sizeof(double) * N, cudaMemcpyHostToDevice));
  if (launch_objective(0, objective, dX, ld, (long long)rows, N, 0, 1, dCoef, dSc, dCoef, dF, sms)) return fail(kNoHandle, "unknown objective id %d", objective);
  CUDA_OK(kNoHandle, cudaMemcpy(f_out, dF, sizeof(double) * rows, cudaMemcpyDeviceToHost));
  CUDA_OK(kNoHandle, cudaGetLastError());
  return 0;
}

int kcma_k_eigen(int device, uint64_t n, const double* c, double* eigenvalues, double* q) {
  kcma_cfg cfg;
  kcma_cfg_defaults(&cfg);
  cfg.n = n; cfg.population_size = 4; cfg.device = device; cfg.objective = KCMA_OBJ_EXTERNAL;
  std::vector<double> zero(n, 0.0), one(n, 1.0);
  cfg.initial_value = zero.data(); cfg.initial_stddev = one.data();
  kcma_t* h = nullptr;
  if (kcma_create(&cfg, &h)) return 1;
  int rc = kcma_set_array(h, "Covariance Matrix", c, n * n);
  if (!rc) rc = update_eigensystem(h, h->dC);
  if (!rc) rc = pull_cached(h);
  if (!rc) { cudaError_t e = cudaGetLastError(); if (e != cudaSuccess) rc = fail(kNoHandle, "CUDA error in the eigensolver: %s", cudaGetErrorString(e)); }
  if (!rc && h->hSc->eig_rejected) {  // report the raw spectrum anyway (unsorted acceptance is the caller's business)
    rc = fail(kNoHandle, "matrix is not positive definite: eigensystem rejected (CMAES.cpp.base:876-880)");
  }
  if (!rc) rc = kcma_get_array(h, "Covariance Eigenvector Matrix", q, n * n, nullptr);
  if (!rc) {
    rc = kcma_get_array(h, "Axis Lengths", eigenvalues, n, nullptr);
    for (uint64_t i = 0; i < n; i++) eigenvalues[i] *= eigenvalues[i];
  } else if (h->err.size()) fail(kNoHandle, "%s", h->err.c_str());
  kcma_destroy(h);
  return rc;
}


// Stages of the tridiagonalisation-based eigensolver on host buffers (parity tests only).
// mode 0: C (n x n) -> d, e, tau, reflector rows vr (n x n); mode 1: (d, e) -> eigenvalues lam, eigenvectors as rows zt (n x n).
int kcma_k_tridiag_stage(int device, int mode, uint64_t n, const double* c, double* d, double* e, double* tau, double* vr,
                         double* lam, double* zt) {
  if (cudaSetDevice(device) != cudaSuccess) return fail(kNoHandle, "no CUDA device %d (libkcma has no CPU fallback)", device);
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  const int N = (int)n, ld = round_up(N, 16);
  char msg[512] = "";
  TridiagWs* ws = tridiag_ws_create(N, ld, prop.multiProcessorCount, msg, sizeof(msg));
  if (!ws) return fail(kNoHandle, "%s", msg);
  int rc = 0, l = 0;
  if (mode == 0) {
    Allocations scratch;
    double* dM = nullptr;
    alloc(scratch, &dM, (size_t)N * ld);
    cudaMemcpy2D(dM, sizeof(double) * ld, c, sizeof(double) * N, sizeof(double) * N, N, cudaMemcpyHostToDevice);
    if (!tridiag_stage_sytrd(0, ws, dM)) rc = fail(kNoHandle, "sytrd launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    if (!rc && cudaDeviceSynchronize() != cudaSuccess) rc = fail(kNoHandle, "sytrd failed: %s", cudaGetErrorString(cudaGetLastError()));
    if (!rc) { tridiag_get_tridiagonal(ws, d, e, tau, vr); tridiag_dump_prof(ws); }
  } else {
    tridiag_set_tridiagonal(ws, d, e);
    if (!tridiag_stage_dc(0, ws, &l)) rc = fail(kNoHandle, "divide & conquer launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    if (!rc && cudaDeviceSynchronize() != cudaSuccess) rc = fail(kNoHandle, "divide & conquer failed: %s", cudaGetErrorString(cudaGetLastError()));
    if (!rc) {
      cudaMemcpy(lam, tridiag_result_values(ws), sizeof(double) * N, cudaMemcpyDeviceToHost);
      cudaMemcpy2D(zt, sizeof(double) * N, tridiag_result_vectors(ws), sizeof(double) * ld, sizeof(double) * N, N, cudaMemcpyDeviceToHost);
    }
  }
  tridiag_ws_destroy(ws);
  return rc;
}

}  // extern "C"
