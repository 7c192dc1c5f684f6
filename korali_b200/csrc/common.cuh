// common.cuh — shared device helpers for libkcma (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace kc {

// FP64 tensor-core tile: D(8x8) += A(8x4, row) * B(4x8, col). SASS: DMMA.8x8x4 (the only native
// FP64 MMA shape on sm_100a; m16n8k{4,8,16} decompose into it — checked with cuobjdump).
// Fragment layout (g = lane>>2, t = lane&3): a = A[g][t], b = B[t][g], c0 = C[g][2t], c1 = C[g][2t+1].
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

// 16-byte async copy global -> shared (SASS: LDGSTS). src_bytes = 0 zero-fills the destination.
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem, int src_bytes) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(s), "l"(gmem), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N));
}

__device__ __forceinline__ double warp_sum_butterfly(double v) {
  // xor butterfly 16,8,4,2,1: every lane ends with the same bits (fp add is commutative);
  // the CPU oracle uses the identical tree (oracle/okcma.c butterfly32).
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) v = __dadd_rn(v, __shfl_xor_sync(0xffffffffu, v, off));
  return v;
}

__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, off));
  return v;
}
__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, off));
  return v;
}

// Device-resident scalars of the solver (one struct in HBM, mirrored to pinned host memory once per
// generation for the termination chain). Names follow CMAES.hpp members.
struct DevScalars {
  double sigma;
  double ps_l2norm;
  double hsig;
  double current_best_value, previous_best_value, best_ever_value, previous_best_ever_value;
  double max_diag_c, min_diag_c, max_eig, min_eig, cur_min_sd, cur_max_sd;
  double global_success_rate;
  double value_at_mu;        // _valueVector[_sortingIndex[mu-1]]
  double weight_sum;         // sum of proportional weights (Mu Type Proportional)
  unsigned long long infeasible_sample_count;
  unsigned long long infeasible_this_round;
  unsigned long long best_valid_sample;
  unsigned long long violating_samples;
  unsigned long long max_violation_count;
  unsigned long long cov_adaptation_count;        // _covarianceMatrixAdaptationCount
  unsigned long long resampled_parameter_count;   // _resampledParameterCount
  unsigned long long constraint_evaluation_count; // _constraintEvaluationCount
  unsigned long long jacobi_max_rel_bits;         // largest |cos| rotated away in the last sweep (double bits)
  int jacobi_sweeps;         // sweeps the persistent Jacobi kernel ran
  int warn_no_valid;         // no sample without constraint violations in a non-viability generation
  int n_events;              // rank-1 corrections applied in this handleConstraints iteration
  int adaptation_abort;      // "Exiting adaption loop, max adaptions reached" (CMAES.cpp.base:789-793)
  int mean_feasible;         // checkMeanAndSetRegime: all g_c(mean) <= 0
  int pad2;
  int nonfinite;             // a non-finite F(x) / constraint value was produced
  int eig_rejected;          // min eigenvalue <= 0: previous B, D kept (CMAES.cpp.base:876-880)
  int warn_flat;             // "Sigma increased due to equal function values."
  int warn_minsd;            // "Sigma increased due to minimal standard deviation."
  int best_updated;          // best-ever was replaced this generation
  int jacobi_rotations;      // rotations applied in the last Jacobi sweep
  // discrete variables (CMAES.cpp.base:834-860): set by discrete_matrix_kernel after the covariance update
  double chi_dm;             // _chiSquareNumberDiscreteMutations
  double disc_path_l2;       // sum_d maskingMatrixSigma[d] * ps[d]^2 (:733)
  int n_mask;                // _numberMaskingMatrixEntries
  int n_disc_mut;            // _numberOfDiscreteMutations
  unsigned long long jacobi_sweeps_total;   // sweeps of the persistent Jacobi kernel since creation (read once by the timers)
  unsigned long long gen;    // generation counter for CUDA-graph replays (kernels launched with generation == kGenFromDevice read it)
  unsigned long long post_err;   // Bayesian problems: ~(sample << 3 | code) of the first bad log-likelihood (atomicMax), 0 = none
};

// Sentinel for the by-value `generation` kernel argument: take the counter from DevScalars::gen instead. A captured CUDA graph
// bakes its kernel arguments, so the replayed generation loop keeps the one argument that changes per generation on the device.
constexpr unsigned kGenFromDevice = 0xffffffffu;

// Codes of DevScalars::post_err beyond the model-output codes of bayes.cuh (kRefNonFinite, kRefParameter, kRefPoissonMean)
enum { kPostNaN = 3, kPostPosInf = 4 };

// The priors of a Bayesian problem on the device (kcma_set_priors): per variable its KCMA_PRIOR_* type, parameters and
// prior_const(type, a, b)
struct PriorCols {
  const int* type;
  const double* a;
  const double* b;
  const double* c;
};

}  // namespace kc
