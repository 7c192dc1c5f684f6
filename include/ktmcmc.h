/*
 * ktmcmc.h — C ABI of the B200-native transitional Markov chain Monte Carlo sampler (TMCMC; Ching & Chen 2007) behind
 * "Solver": {"Type": "Sampler/TMCMC"} with "Problem": {"Type": "Bayesian/Custom"}. Same conventions as kcma.h / kdea.h / kmocma.h:
 * extern "C", plain pointers and sizes, caller-owned host buffers that the library copies, non-zero return + ktmcmc_last_error on
 * failure, one caller thread per handle, no CPU fallback. DESIGN.md section 14 states the algorithm; oracle/otmcmc.c restates it.
 *
 * Notation: lambda = "Population Size", N variables, l_i = log-likelihood, p_i = log-prior, rho = annealing exponent.
 *
 * Generation 1: lambda samples from the priors; l and p of every sample; rho = 0, LogEvidence = 0.
 * Generation j > 1 (while rho < "Target Annealing Exponent"):
 *   1. annealing: l_max = max of the finite l_i, w_i(D) = exp(D (l_i - l_max)), CoV(D) = std(w) / mean(w) (divisor lambda), computed
 *      as sqrt(max(0, lambda S2 / S1^2 - 1)) with S1 = sum w, S2 = sum w^2. D = 1 - rho if CoV(1 - rho) <= target, otherwise 64
 *      bisection steps on [0, 1 - rho] (mid = (lo + hi) / 2; CoV(mid) > target -> hi = mid, else lo = mid; D = lo). D is clamped into
 *      [Min, Max Annealing Exponent Update]; rho <- rho + D, or 1 when D >= 1 - rho (then D = 1 - rho). l = -inf has weight 0;
 *      a NaN l, or every l = -inf, is an error.
 *   2. w~ = w / S1; LogEvidence += log(S1 / lambda) + D l_max.
 *   3. mean = sum w~_i x_i; Sigma = s sum w~_i (x_i - mean)(x_i - mean)^T (the stream-K SYRK over rows sqrt(w~_i)(x_i - mean)),
 *      s = "Covariance Scaling"; Sigma = B D^2 B^T by the CMA-ES path's eigensolvers (N <= 24: the single-CTA Jacobi solver,
 *      which keeps the previous factor when its smallest eigenvalue is <= 0; above: tridiagonalisation + divide & conquer, with
 *      eigenvalues below 0 clamped to 0). The proposal factor is A = B D.
 *   4. resampling: u_k (k < lambda) picks leader i = first index with cumsum(w~)_i >= u_k (the last index of positive weight when
 *      roundoff leaves cumsum below u_k); counts c_i; every leader with c_i > 0, in ascending i, gives ceil(c_i / L) chains of
 *      length L = "Max Chain Length", the last one c_i - (ceil(c_i / L) - 1) L. Chains start at their leader's (x, l, p).
 *   5. MCMC: chain k runs b + L_k steps (b = "Per Generation Burn In"[j] when that list has an entry j, else
 *      "Default Burn In"). Step t, for every chain at once: x' = x + A z (one GEMM), p(x'); p(x') = -inf is rejected without an
 *      evaluation; the other proposals are evaluated in one batched call and accepted iff log u < rho (l' - l) + (p' - p). From
 *      step b on, the chain's state is appended to the database (chain order, then step order): exactly lambda rows, which become
 *      the next population.
 * Termination: rho >= "Target Annealing Exponent", "Max Generations" (Current Generation > max), "Max Model Evaluations"
 * (model evaluations = lambda + in-support proposals).
 *
 * Summation orders (restated by the oracle): S1, S2 — thread t < 1024 sums w_i for i = t, t + 1024, ... ascending, then an xor
 * butterfly inside each warp (16, 8, 4, 2, 1) and the same butterfly over the 32 warp sums. cumsum(w~) — contiguous chunks of
 * ceil(lambda / 1024) entries per thread, sequential inside a chunk; chunk totals prefix-summed in order; cumsum_i = prefix + local.
 * Weighted mean — 64 contiguous row chunks of ceil(lambda / 64) rows, sequential inside a chunk, chunk sums added in order.
 * Log-prior — 32 lane-strided partial sums over the variables, then the xor butterfly (the order of the built-in models).
 *
 * Random numbers: Philox4x32-10, key = { seed_lo, seed_hi ^ "TMCM" }, two 52-bit uniforms per block, u = (bits >> 12) 2^-52 + 2^-53:
 *   prior draw of sample i, variables 2p and 2p+1 : ctr { 2^20 + p, i, 0, 0 }; Uniform uses the first / second uniform of the block,
 *                                                   Normal the Box-Muller pair (rad cos, rad sin) as in kcma.h;
 *   resampling uniform of draw k                  : ctr { 0, k, 0, generation }, first uniform;
 *   accept uniform of chain k at step t           : ctr { 1, k, t, generation }, first uniform;
 *   z of chain k at step t, components 2p, 2p+1   : ctr { 2^20 + p, k, t, generation } -> Box-Muller pair.
 *
 * Bayesian/Reference (ktmcmc_set_reference): the log-likelihood of an evaluated row is reduced on the device from M model outputs.
 * d_j = reference datum j (j < M), g_j = the computational model's prediction, p_j = its per-point parameter, r_j = d_j - g_j:
 *   KTMCMC_LIK_NORMAL           p = sigma ("Standard Deviation") > 0:  t_j = -log(2 pi)/2 - log sigma - (r / sigma)^2 / 2
 *   KTMCMC_LIK_POSITIVE_NORMAL  p = sigma > 0, the normal truncated to d >= 0:  t_j = the Normal term - log Phi(g / sigma), with
 *                               log Phi(u) = log(erfc(-u / sqrt 2) / 2) for u >= -1, else log(erfcx(-u / sqrt 2) / 2) - u^2 / 2
 *                               (finite for every finite u); a term that rounds to NaN (only when |g / sigma| overflows) is -inf
 *   KTMCMC_LIK_STUDENT_T        p = nu ("Degrees Of Freedom") > 0, the standard t of the residual:
 *                               t_j = lgamma((nu + 1) / 2) - lgamma(nu / 2) - log(nu pi) / 2 - (nu + 1) / 2 log1p(r^2 / nu); for nu >= 50
 *                               the first three terms are evaluated as their asymptotic series in x = nu / 2,
 *                               -log(2 pi) / 2 + (1 / x)(-1/8 + y (1/192 + y (-1/640 + y 17/14336))), y = 1 / x^2 (exact to double
 *                               precision there; the difference of two lgamma values would cancel)
 *   KTMCMC_LIK_POISSON          no parameter, g = the mean >= 0:  t_j = d log g - g - lgamma(d + 1) (lgamma(d + 1) computed once on the
 *                               host from the data); t_j = -g when d = 0 and -inf when g = 0 < d
 * l = sum_j t_j: lane k of one warp per row sums j = k, k + 32, ... ascending, then the xor butterfly (the order of the log-prior).
 * Errors (reported after the step with the evaluation row): a non-finite g, a parameter <= 0 or non-finite, a Poisson mean < 0.
 * A finite model output can give l = -inf (weight 0), never +inf or NaN.
 */
#ifndef KTMCMC_H
#define KTMCMC_H
#include <stddef.h>
#include <stdint.h>

#include "kcma.h"

#ifdef __cplusplus
extern "C" {
#endif

#define KTMCMC_ABI_VERSION 1u

enum { KTMCMC_PRIOR_UNIFORM = KCMA_PRIOR_UNIFORM, KTMCMC_PRIOR_NORMAL = KCMA_PRIOR_NORMAL };

/* Log-likelihood models: the built-in CMA-ES device objectives read as log-likelihoods (KCMA_OBJ_*, e.g. KCMA_OBJ_NEG_SPHERE gives
 * -1/2 sum x^2), or KCMA_OBJ_EXTERNAL: the host conduit, a device callback or ktmcmc_inject_loglik. */
typedef struct ktmcmc ktmcmc_t;

/* TMCMC.config "Configuration Settings" and their defaults (ktmcmc_cfg_defaults). */
typedef struct ktmcmc_cfg {
  uint32_t abi_version, reserved0;
  uint64_t n;                             /* variables */
  uint64_t population_size;               /* "Population Size" (lambda >= 2) */
  uint64_t max_chain_length;              /* "Max Chain Length" (1) */
  uint64_t default_burn_in;               /* "Default Burn In" (0) */
  uint64_t burn_in_count;                 /* entries of per_generation_burn_in */
  const uint64_t* per_generation_burn_in; /* "Per Generation Burn In": entry j applies to generation j */
  double target_cov;                      /* "Target Coefficient Of Variation" (1.0) */
  double covariance_scaling;              /* "Covariance Scaling" (0.04) */
  double min_annealing_update;            /* "Min Annealing Exponent Update" (1e-5) */
  double max_annealing_update;            /* "Max Annealing Exponent Update" (1.0) */
  uint64_t seed;
  int32_t loglik;                         /* KCMA_OBJ_* */
  int32_t device;
  const int32_t* prior_type;              /* n: KTMCMC_PRIOR_* */
  const double* prior_a;                  /* n: Minimum (Uniform) / Mean (Normal) */
  const double* prior_b;                  /* n: Maximum (Uniform) / Standard Deviation (Normal) */
  const double* loglik_coef;              /* n or NULL: coefficients of KCMA_OBJ_NEG_ELLIPSOID (NULL: 10^(6 i / (n - 1))) */
} ktmcmc_cfg;

/* batched host conduit: l[rows] from X[rows x n] (row-major, packed), once per evaluation */
typedef void (*ktmcmc_host_loglik_fn)(void* user, const double* x, uint64_t rows, uint64_t n, double* l_out);

void ktmcmc_cfg_defaults(ktmcmc_cfg* cfg);
int ktmcmc_create(const ktmcmc_cfg* cfg, ktmcmc_t** out);
void ktmcmc_destroy(ktmcmc_t* h);
const char* ktmcmc_last_error(const ktmcmc_t* h);

int ktmcmc_run_generation(ktmcmc_t* h);
/* Stage entry points. Generation 1 is propose (prior draws) + eval + accept (the draws become the population). A later generation
 * is anneal (steps 1-3) + resample (step 4) + (propose + eval + accept) once per MCMC step; the accept of the last step makes the
 * database the population. */
int ktmcmc_anneal(ktmcmc_t* h);
int ktmcmc_resample(ktmcmc_t* h);
int ktmcmc_propose(ktmcmc_t* h);
int ktmcmc_eval(ktmcmc_t* h);
int ktmcmc_accept(ktmcmc_t* h);
/* The log-likelihoods of the rows the next ktmcmc_eval evaluates ("Evaluation Rows": lambda prior draws in generation 1, else the
 * in-support proposals of active chains in chain order); count must equal their number. */
int ktmcmc_inject_loglik(ktmcmc_t* h, const double* l, size_t count);
/* Replaces the proposal factor A = B D (n x n, row-major) computed by the last ktmcmc_anneal (parity tests). */
int ktmcmc_inject_factor(ktmcmc_t* h, const double* a, size_t count);
int ktmcmc_set_host_loglik(ktmcmc_t* h, ktmcmc_host_loglik_fn fn, void* user);
int ktmcmc_set_device_loglik(ktmcmc_t* h, kcma_device_objective_fn fn, void* user);

/* Bayesian/Reference: the log-likelihood is reduced on the device from the outputs of a computational model (definitions above). */
enum { KTMCMC_LIK_NORMAL = KCMA_LIK_NORMAL, KTMCMC_LIK_POSITIVE_NORMAL = KCMA_LIK_POSITIVE_NORMAL, KTMCMC_LIK_STUDENT_T = KCMA_LIK_STUDENT_T,
       KTMCMC_LIK_POISSON = KCMA_LIK_POISSON };
/* Once, after create and before generation 1; cfg.loglik must be KCMA_OBJ_EXTERNAL. Copies data[m]. Allocates the model outputs
 * (lambda x m, and as many per-point parameters unless the likelihood has none); an allocation failure names the GiB needed. */
int ktmcmc_set_reference(ktmcmc_t* h, int32_t likelihood, const double* data, uint64_t m);
/* the computational models of kcma.h (kcma_host_reference_fn, kcma_device_reference_fn) */
typedef kcma_host_reference_fn ktmcmc_host_reference_fn;
typedef kcma_device_reference_fn ktmcmc_device_reference_fn;
int ktmcmc_set_host_reference_model(ktmcmc_t* h, ktmcmc_host_reference_fn fn, void* user);
int ktmcmc_set_device_reference_model(ktmcmc_t* h, ktmcmc_device_reference_fn fn, void* user);
/* The model outputs of the rows the next ktmcmc_eval evaluates (parity tests); count = rows * m; p is NULL for Poisson. */
int ktmcmc_inject_reference(ktmcmc_t* h, const double* g, const double* p, size_t count);

int ktmcmc_check_termination(ktmcmc_t* h, int* finished, const char** reason);
int ktmcmc_run(ktmcmc_t* h, uint64_t max_generations, uint64_t* done);

/* State by Korali key name. Arrays: "Sample Database" (lambda x n), "Sample LogLikelihood Database", "Sample LogPrior Database",
 * "Covariance Matrix" (n x n), "Proposal Factor" (A = B D, n x n), "Mean Theta" (n), "Weights" (w~), "Selection Counts" (c_i),
 * "Chain Leaders", "Chain Lengths" (chain count each), "Evaluation Rows" (rows of the next evaluation, packed),
 * "Proposal Support" (per chain: 1 = the last proposal was inside the priors' support), "Accept Flags" (per chain, last step),
 * "Evaluation LogLikelihoods" (the log-likelihoods the last ktmcmc_eval produced, packed like "Evaluation Rows"; read it before the
 * next ktmcmc_propose).
 * Scalars: "Annealing Exponent", "Previous Annealing Exponent", "Annealing Exponent Update", "Coefficient Of Variation",
 * "LogEvidence", "Max Loglikelihood", "Chain Count", "Max Chain Steps", "Current Step", "Proposals Acceptance Rate",
 * "Selection Acceptance Rate", "Model Evaluation Count", "Current Generation", "Population Size", "Burn In",
 * "Termination Criteria/<name>". */
int ktmcmc_get_array(ktmcmc_t* h, const char* key, double* out, size_t capacity, size_t* count);
int ktmcmc_get_scalar(ktmcmc_t* h, const char* key, double* out);
int ktmcmc_set_scalar(ktmcmc_t* h, const char* key, double value);
uint64_t ktmcmc_launch_count(const ktmcmc_t* h);

#ifdef __cplusplus
}
#endif
#endif
