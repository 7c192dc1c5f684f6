/*
 * kcma.h — C ABI of the B200-native CMA-ES generation loop (libkcma.so).
 *
 * This is the drop-in boundary for ONE hot path of Korali: the generation loop of
 * source/modules/solver/optimizer/CMAES (reference file:line cited per entry point).
 * Plain C types only: pointers + sizes, no torch / CUDA types in any signature.
 * All `double*` / `uint64_t*` arguments are HOST pointers owned by the caller; the
 * library copies and never retains them. Every function returns 0 on success and a
 * non-zero code on failure, with the Korali-style message in kcma_last_error()
 * (the host shim rethrows it as std::runtime_error, mirroring KORALI_LOG_ERROR,
 * source/auxiliar/logger.cpp:83-99).
 *
 * A handle is NOT thread-safe: one caller thread, like the reference solver
 * (single host thread inside the experiment coroutine, experiment.cpp.base:171).
 *
 * The same kcma_cfg / key names are implemented by the CPU oracle (oracle/okcma.h,
 * test infrastructure only) so parity tests drive both through one vocabulary.
 */
#ifndef KCMA_H
#define KCMA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KCMA_ABI_VERSION 3

/* "Mu Type" (CMAES.cpp.base:236-245). */
enum { KCMA_MU_LINEAR = 0, KCMA_MU_EQUAL = 1, KCMA_MU_LOGARITHMIC = 2, KCMA_MU_PROPORTIONAL = 3 };

/* Built-in batched device objectives (maximised, F4). They replace the per-sample
 * Conduit dispatch runGeneration() does at CMAES.cpp.base:205-224.
 * Definitions follow examples/optimization/stochastic/_model/model.py. */
enum {
  KCMA_OBJ_NEG_SPHERE = 0,    /* F = -0.5 * sum x_i^2                                   model.py:10-20 */
  KCMA_OBJ_NEG_ROSENBROCK = 1,/* F = -sum_{i<N-1} 100 (x_{i+1}-x_i^2)^2 + (1-x_i)^2      model.py:23-34 */
  KCMA_OBJ_NEG_ACKLEY = 2,    /* F = 20 exp(-0.2 sqrt(sum x^2/N)) + exp(sum cos(2 pi x)/N) - 20 - e   model.py:37-63 */
  KCMA_OBJ_NEG_ELLIPSOID = 3, /* F = -sum_i coef_i x_i^2, coef_i = 10^(6 i/(N-1)) by default  (SURVEY 8d config 3) */
  KCMA_OBJ_NEG_SUMSQ = 4,     /* F = -sum x_i^2   (the objective behind tests/python/plot/cmaes/gen*.json) */
  KCMA_OBJ_NEG_SPHERE_SIN2 = 5,/* F = -sum (x_i^2 + sin(x_i)^2)   ccmaes/helpers/helpers.py:5-9 generalised to N-D */
  KCMA_OBJ_EXTERNAL = 100     /* no device objective: caller injects F with kcma_inject(KCMA_INJ_F) */
};

/* Built-in constraint families g_c(x) <= 0 feasible (CMAES.cpp.base:333-334). */
enum {
  KCMA_CON_NONE = 0,
  KCMA_CON_HALFSPACE = 1,     /* g_c(x) = -(x_{c} - shift_c), c < n_constraints <= N  (helpers.py:20-37 activeMax*) */
  KCMA_CON_EXTERNAL = 100     /* constraints evaluated by kcma_set_host_constraints() */
};

/* What kcma_inject overwrites (parity hooks: "injecting the reference's own z draws and fitness values"). */
enum {
  KCMA_INJ_Z = 0,   /* lambda_z x N standard normals used instead of Philox for the NEXT ask   */
  KCMA_INJ_BDZ = 1, /* lambda x N "BDZ Matrix" (y_i); X is recomputed as m + sigma*y            */
  KCMA_INJ_X = 2,   /* lambda x N "Sample Population" overriding the sampled X                  */
  KCMA_INJ_F = 3,   /* lambda "Value Vector"; taken as F as it is (on a Bayesian handle: as the log-posterior, no prior added) */
  KCMA_INJ_GRAD = 5, /* lambda*N gradients dF/dx of the current population ("Gradients", row-major); with KCMA_INJ_F */
  KCMA_INJ_BD = 4   /* N*N eigenvectors (row-major, columns = vectors) followed by N axis lengths; skips the eigensolver for the NEXT ask */
};

/* Solver configuration. Field names follow CMAES.config:11-107 "Configuration Settings"
 * and optimizer.config:45-82 "Variables Configuration". Defaults (0 / -1 meaning "auto")
 * are the reference's own (CMAES.config:485-538). */
typedef struct kcma_cfg {
  uint32_t abi_version;                 /* = KCMA_ABI_VERSION */
  uint32_t reserved0;
  uint64_t n;                           /* "Variable Count" = number of experiment variables      */
  uint64_t population_size;             /* "Population Size"                                      */
  uint64_t mu_value;                    /* "Mu Value"; 0 -> population/2 (CMAES.cpp.base:27)      */
  int32_t mu_type;                      /* KCMA_MU_*                                              */
  int32_t diagonal_covariance;          /* "Diagonal Covariance"                                  */
  int32_t mirrored_sampling;            /* "Mirrored Sampling"                                    */
  int32_t is_sigma_bounded;             /* "Is Sigma Bounded"                                     */
  double initial_sigma_cumulation_factor; /* <=0 or >=1 -> auto (CMAES.cpp.base:267-278)         */
  double initial_damp_factor;           /* <=0 -> auto (:281-283)                                 */
  double initial_cumulative_covariance; /* <=0 or >1 -> auto (:261-264)                           */
  uint64_t viability_population_size;   /* "Viability Population Size" (default 2)                */
  uint64_t viability_mu_value;          /* "Viability Mu Value"; 0 -> viability population/2      */
  uint64_t max_covariance_matrix_corrections; /* default 1000000                                 */
  double target_success_rate;           /* 0.1818                                                 */
  double covariance_matrix_adaption_strength; /* 0.1                                             */
  double normal_vector_learning_rate;   /* overwritten with 1/(N+2) when constrained (:154)       */
  double global_success_learning_rate;  /* 0.2                                                    */
  uint64_t max_infeasible_resamplings;  /* Termination Criteria key also used as a loop bound (:459);
                                           reference default = size_t(Infinity) = 0 in release builds (SURVEY Q2) */
  uint64_t seed;                        /* "Random Seed" of the Normal Generator                  */
  /* batched device conduit */
  int32_t objective;                    /* KCMA_OBJ_*                                             */
  int32_t constraint_family;            /* KCMA_CON_*                                             */
  uint64_t n_constraints;               /* number of constraint functions                         */
  const double* objective_coef;         /* N doubles or NULL (ellipsoid weights)                  */
  const double* constraint_shift;       /* n_constraints doubles or NULL (zeros)                  */
  /* per-variable arrays, length n, caller-owned */
  const double* lower_bound;            /* "Lower Bound"  (NULL = -inf)                           */
  const double* upper_bound;            /* "Upper Bound"  (NULL = +inf)                           */
  const double* initial_value;          /* "Initial Value" (NULL/NaN -> mid-domain, :111-118)     */
  const double* initial_stddev;         /* "Initial Standard Deviation" (NULL/NaN -> 0.3*width)   */
  const double* min_stddev_update;      /* "Minimum Standard Deviation Update" (NULL = 0)         */
  /* placement */
  int32_t device;                       /* CUDA device ordinal                                    */
  int32_t rank;                         /* population shard owner, 0 <= rank < nranks             */
  int32_t nranks;                       /* 1 = single GPU                                         */
  int32_t keep_population;              /* 1: materialise "Sample Population" (X) every generation */
  /* "Use Gradient Information" / "Gradient Step Size" (CMAES.config:43-52, CMAES.cpp.base:82-86,199-200,226-228,611-621):
     the model also returns dF/dx per sample and the new mean takes a step along the weighted gradients */
  int32_t use_gradient_information;     /* default 0                                              */
  int32_t reserved1;
  double gradient_step_size;            /* default 0.01; must be > 0 when gradients are used      */
  /* discrete variables (optimizer.config "Granularity"; CMAES.cpp.base:44-50, 515-544, 668, 730-734, 834-867, after Hansen 2011,
     "A CMA-ES for Mixed-Integer Nonlinear Optimization"): length n or NULL (all continuous); 0 = continuous, < 0 is an error */
  const double* granularity;
} kcma_cfg;

typedef struct kcma kcma_t;

/* Fill cfg with the reference defaults (CMAES.config:485-538). */
void kcma_cfg_defaults(kcma_cfg* cfg);

/* ---- lifecycle --------------------------------------------------------------------- */
/* CMAES::setInitialConfiguration (CMAES.cpp.base:14-184): validation, allocation on the
 * device, initMuWeights (:233-284), initCovariance (:286-313). */
int kcma_create(const kcma_cfg* cfg, kcma_t** out);
void kcma_destroy(kcma_t* h);
/* Last KORALI_LOG_ERROR-style message ("" if none). h may be NULL for create() errors. */
const char* kcma_last_error(const kcma_t* h);
/* Warnings the reference sends to stderr via logWarning("Detailed", ...) since the last call. */
const char* kcma_take_warnings(kcma_t* h);

/* ---- multi-GPU (population sharded across ranks, SURVEY 8e) ------------------------ */
/* NCCL bootstrap: rank 0 makes an id, the launcher broadcasts the 128 bytes, every rank calls comm_init. */
int kcma_comm_unique_id(uint8_t id_out[128]);
int kcma_comm_init(kcma_t* h, const uint8_t id[128]);
/* One process driving several devices (the Engine's k["Conduit"]["Devices"] = G; the reference analogue selects its Distributed
 * conduit purely from k["Conduit"], distributed.cpp.base:13-90, engine.cpp:69-128): handles[r] was created with rank = r,
 * nranks = count on its own device; builds the communicator of all of them. Afterwards kcma_run_generation must be called for every
 * handle of a generation from its own host thread (the calls meet in the collectives). */
int kcma_comm_init_all(kcma_t** handles, int count);
/* Shard arithmetic used by every rank (pairs stay together when mirrored). Pure host code. */
void kcma_shard_range(uint64_t population, int mirrored, int rank, int nranks, uint64_t* begin, uint64_t* end);

/* ---- the generation loop ------------------------------------------------------------ */
/* CMAES::runGeneration (CMAES.cpp.base:186-231) = ask + eval + tell. Increments "Current Generation". */
int kcma_run_generation(kcma_t* h);
/* checkMeanAndSetRegime (:315-345) + prepareGeneration (:439-492) [+ updateConstraints (:347-385)
 * + handleConstraints (:774-832)]: eigendecomposition, Philox z, sampling GEMM, feasibility. */
int kcma_ask(kcma_t* h);
/* Batched device conduit: replaces the KORALI_START / KORALI_WAITALL loop (:205-224) and
 * Optimization::evaluate (optimization.cpp.base:26-34; non-finite F(x) is an error). */
int kcma_eval(kcma_t* h);
/* CMAES::updateDistribution (:547-688): sort_index, best bookkeeping, mean, paths, adaptC, updateSigma. */
int kcma_tell(kcma_t* h);
/* Generated CMAES/Optimizer/Solver::checkTermination chain (CMAES.cpp:1903-1933, optimizer.cpp:188-206,
 * solver.cpp:92-110) evaluated on the criteria set with kcma_set_scalar("Termination Criteria/<name>").
 * *finished = 1 and reason (static string, ';'-separated criteria names) when any fires. */
int kcma_check_termination(kcma_t* h, int* finished, const char** reason);
/* Experiment::run loop (experiment.cpp.base:57-100): while (!checkTermination) runGeneration.
 * Runs at most max_generations more generations; *done = number actually run. */
int kcma_run(kcma_t* h, uint64_t max_generations, uint64_t* done);

/* ---- batched HOST conduit (user-supplied Python / C++ models) -------------------------
 * The reference ships every sample to the user model as a JSON message (Conduit::runSample, conduit.cpp.base:29-88,
 * Optimization::evaluate / evaluateConstraints, optimization.cpp.base:11-34). Here the whole population crosses the
 * boundary once per generation: X is copied to the host, the callback fills F (or G), the values go back to HBM.
 * This is a conduit for models that only exist on the host, not a compute fallback: sampling, ranking and the
 * distribution update stay on the device. x is row-major rows x n; g_out is [n_constraints][rows]. */
typedef void (*kcma_host_objective_fn)(void* user, const double* x, uint64_t rows, uint64_t n, double* f_out);
typedef void (*kcma_host_constraints_fn)(void* user, const double* x, uint64_t rows, uint64_t n, double* g_out,
                                         uint64_t n_constraints);
int kcma_set_host_objective(kcma_t* h, kcma_host_objective_fn fn, void* user);
/* operation "Evaluate With Gradients" (CMAES.cpp.base:199-200,226-228): the model fills F and the rows x n gradients */
typedef void (*kcma_host_objective_grad_fn)(void* user, const double* x, uint64_t rows, uint64_t n, double* f_out, double* grad_out);
int kcma_set_host_objective_grad(kcma_t* h, kcma_host_objective_grad_fn fn, void* user);
int kcma_set_host_constraints(kcma_t* h, kcma_host_constraints_fn fn, void* user);
/* User objective that stays on the device (SURVEY 8f-3: the whole population in ONE call instead of the reference's lambda
 * per-sample Sample trips, conduit.cpp.base:29-88): the callback receives the device pointer of this rank's samples
 * (rows x n, leading dimension ldx doubles, row-major) and writes F(x) for every row to f_dev. It must enqueue its work on
 * `stream` (the handle's stream) or synchronise before it returns. Needs keep_population = 1; non-finite values are an error
 * like everywhere else (optimization.cpp.base:32-33). */
typedef void (*kcma_device_objective_fn)(void* user, const double* x_dev, uint64_t rows, uint64_t n, uint64_t ldx, double* f_dev, void* stream);
int kcma_set_device_objective(kcma_t* h, kcma_device_objective_fn fn, void* user);

/* ---- Bayesian problems: F(x) is the log-posterior and CMA-ES returns the maximum a posteriori estimate -----------------
 * For a sample x with log-prior p = sum_d prior_d(x_d) and log-likelihood l:
 *   p = -inf (x outside the prior's support): F = -inf. The model is still called on the whole batch; its output for that row is
 *            ignored and is never an error.
 *   p finite: l = -inf gives F = -inf, a finite l gives F = p + l, l = NaN or +inf is an error naming the sample. On Bayesian/Reference
 *            problems the model-output errors of include/ktmcmc.h (a non-finite prediction, a per-point parameter <= 0 or non-finite, a
 *            Poisson mean < 0) apply to these rows only.
 * F = -inf ranks last (ties by ascending index); a generation in which every F is -inf completes. Optimization problems are unchanged:
 * there every non-finite F, -inf included, is an error.
 * The log-prior is summed like TMCMC's (include/ktmcmc.h): lane d % 32 of one warp sums its variables ascending, then the xor butterfly.
 * Uniform(a, b): -log(b - a) on [a, b], -inf outside; Normal(a = mean, b = standard deviation): -((x - a) / b)^2 / 2 - log b - log(2 pi) / 2.
 * The prior enters only through F: it does not set the bounds. Not defined on Bayesian problems (rejected by kcma_set_priors):
 * Mu Type Proportional (its weights are computed from F), Use Gradient Information, constraints.
 * Built-in device objectives (KCMA_OBJ_*) are read as log-likelihoods; the log-prior is reduced in the same pass over the samples. */
enum { KCMA_PRIOR_UNIFORM = 0, KCMA_PRIOR_NORMAL = 1 };
/* Bayesian/Reference likelihoods (definitions in include/ktmcmc.h) */
enum { KCMA_LIK_NORMAL = 1, KCMA_LIK_POSITIVE_NORMAL = 2, KCMA_LIK_STUDENT_T = 3, KCMA_LIK_POISSON = 4 };
/* Once, after create and before the first ask: type[n] (KCMA_PRIOR_*), a[n] = Minimum / Mean, b[n] = Maximum / Standard Deviation.
 * From then on F is the log-posterior. */
int kcma_set_priors(kcma_t* h, const int32_t* type, const double* a, const double* b);
/* Bayesian/Reference: once, after kcma_set_priors and before the first ask; needs objective = KCMA_OBJ_EXTERNAL and keep_population = 1.
 * Copies data[m] and allocates the model outputs of this rank's samples (rows x m, and as many per-point parameters unless the
 * likelihood has none). The computational model is set with one of the two setters below. */
int kcma_set_reference(kcma_t* h, int32_t likelihood, const double* data, uint64_t m);
/* g_out / p_out: rows x m, row-major, packed; p_out is NULL for a likelihood without a per-point parameter (Poisson) */
typedef void (*kcma_host_reference_fn)(void* user, const double* x, uint64_t rows, uint64_t n, double* g_out, double* p_out, uint64_t m);
/* x_dev: rows x n with leading dimension ldx; g_dev / p_dev: rows x m with leading dimension ldm (p_dev NULL as above); the model
 * writes them on `stream` (a cudaStream_t) */
typedef void (*kcma_device_reference_fn)(void* user, const double* x_dev, uint64_t rows, uint64_t n, uint64_t ldx, double* g_dev,
                                         double* p_dev, uint64_t m, uint64_t ldm, void* stream);
/* Both need kcma_set_reference first. Like the objective setters they may be called between generations; the model set last is the
 * one the next evaluation calls (the device model when both are set). */
int kcma_set_host_reference_model(kcma_t* h, kcma_host_reference_fn fn, void* user);
int kcma_set_device_reference_model(kcma_t* h, kcma_device_reference_fn fn, void* user);

/* ---- parity hooks ------------------------------------------------------------------- */
int kcma_inject(kcma_t* h, int kind, const double* host, size_t count);

/* ---- state access by Korali "Internal Settings" key (CMAES.config:137-483) ----------
 * Arrays: "Covariance Matrix", "Covariance Eigenvector Matrix", "Axis Lengths", "Current Mean",
 * "Previous Mean", "Mean Update", "Evolution Path", "Conjugate Evolution Path", "Mu Weights",
 * "Value Vector", "BDZ Matrix", "Sample Population", "Best Ever Variables", "Current Best Variables",
 * "Viability Boundaries", "Constraint Evaluations", "Normal Constraint Approximation", ...
 * Scalars: "Sigma", "Effective Mu", "Current Generation", "Best Ever Value", ... and
 * "Termination Criteria/<name>". Index arrays: "Sorting Index", "Sample Constraint Violation Counts". */
int kcma_get_array(kcma_t* h, const char* key, double* out, size_t capacity, size_t* count);
int kcma_set_array(kcma_t* h, const char* key, const double* in, size_t count);
int kcma_get_index_array(kcma_t* h, const char* key, uint64_t* out, size_t capacity, size_t* count);
int kcma_get_scalar(kcma_t* h, const char* key, double* out);
int kcma_set_scalar(kcma_t* h, const char* key, double value);

/* ---- measurement -------------------------------------------------------------------- */
/* Accumulated CUDA-event time (ms) and call count of a phase since the last reset. Phases:
 * "eigen", "rng", "sample_gemm", "objective", "sort", "gather_mean", "rank_mu", "paths", "collectives", "generation";
 * Bayesian problems with a host / device model add "posterior" (the log-posterior kernel) and "reference_model" (the computational
 * model's call). */
int kcma_timing_enable(kcma_t* h, int on);
int kcma_timing_get(kcma_t* h, const char* phase, double* ms, uint64_t* calls);
int kcma_timing_reset(kcma_t* h);
/* Number of kernels this library launched since the handle was created. */
uint64_t kcma_launch_count(const kcma_t* h);
/* Overwrite C with a never-written L2-sized scratch buffer (bench hygiene). */
int kcma_flush_l2(kcma_t* h);

/* ---- single kernels on HOST buffers (unit parity tests; each copies in, launches, copies out) ---- */
/* sort_index (CMAES.cpp.base:940-950): descending in f, ascending index among equal values. */
int kcma_k_sort_index(int device, const double* f, uint64_t n, uint64_t* index_out);
/* eigen (CMAES.cpp.base:896-938): symmetric N x N (row-major) -> eigenvalues ascending,
 * eigenvectors as COLUMNS of Q (row-major). */
int kcma_k_eigen(int device, uint64_t n, const double* c, double* eigenvalues, double* q);
/* Stages of the tridiagonalisation-based eigensolver (the Householder + QL halves of gsl_eigen_symmv, CMAES.cpp.base:917-936).
 * mode 0: C (n x n) -> tridiagonal d[n], e[n-1 used of n], reflector scalars tau[n], reflector rows vr (n x n);
 * mode 1: (d, e) -> eigenvalues lam ascending, eigenvectors of the tridiagonal as ROWS of zt (n x n). Unused pointers may be NULL. */
int kcma_k_tridiag_stage(int device, int mode, uint64_t n, const double* c, double* d, double* e, double* tau, double* vr,
                         double* lam, double* zt);
/* sampleSingle (CMAES.cpp.base:494-513) for a batch: Y = Z (B diag(D))^T, X = m + sigma Y. */
int kcma_k_sample(int device, uint64_t n, uint64_t rows, const double* z, const double* b, const double* d,
                  const double* mean, double sigma, double* y_out, double* x_out);
/* rank-mu sum of adaptC (CMAES.cpp.base:703-704): P = sum_k w_k t_k t_k^T with t_k = x_k - mean_old. */
int kcma_k_rank_mu(int device, uint64_t n, uint64_t rows, const double* t, const double* w, double* p_out);
/* Philox4x32-10 normals as the device generates them (counter layout in DESIGN.md). */
int kcma_k_philox_normal(int device, uint64_t seed, uint64_t generation, uint64_t row_begin, uint64_t rows,
                         uint64_t n, double* z_out);
/* One raw Philox4x32-10 block (known-answer tests against the Random123 vectors). */
int kcma_k_philox_raw(int device, const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);
/* Batched objective (device conduit) on host X. */
int kcma_k_objective(int device, int objective, uint64_t n, uint64_t rows, const double* x,
                     const double* coef, double* f_out);

#ifdef __cplusplus
}
#endif
#endif /* KCMA_H */
