/*
 * otmcmc_reference.c — CPU restatement of Bayesian/Reference for the TMCMC oracle (include/ktmcmc.h). TEST INFRASTRUCTURE ONLY.
 *
 * Builds on oracle/otmcmc.c unchanged: this file includes it, keeps its Bayesian/Custom algorithm, and adds what ktmcmc_set_reference
 * adds on the device: reference data, a host computational model or injected outputs (G, P), and the per-point likelihood terms of
 * include/ktmcmc.h summed in the order of tm_reference_loglik_kernel (lane k of a warp sums j = k, k + 32, ... ascending, then the
 * xor butterfly), compiled like the oracle with -ffp-contract=off. The entry points whose behaviour changes (eval, run_generation,
 * run, get_array, destroy) are renamed in the included source and restated here; the reference state of a handle lives in a side
 * table, because the oracle's handle struct is left as it is. glibc has no erfcx, so otmcmc_erfcx restates it.
 * Exported under the prefix "otmcmc_" like the oracle; tests/tmcmc_reference_oracle.py links it with oracle/okcma.c.
 */
#define otmcmc_eval otmcmc_base_eval
#define otmcmc_run_generation otmcmc_base_run_generation
#define otmcmc_run otmcmc_base_run
#define otmcmc_get_array otmcmc_base_get_array
#define otmcmc_destroy otmcmc_base_destroy
#include "../../oracle/otmcmc.c"
#undef otmcmc_eval
#undef otmcmc_run_generation
#undef otmcmc_run
#undef otmcmc_get_array
#undef otmcmc_destroy

/* ---- the per-point terms, in the operation order of tm_reference_loglik_kernel */
static const double kInvSqrt2 = 0.70710678118654752440;
static const double kPi = 3.14159265358979323846;
/* erfcx(x) = exp(x^2) erfc(x): in long double while erfcl does not underflow, then the asymptotic series
 * 1 / (x sqrt pi) sum_k (-1)^k (2k - 1)!! / (2 x^2)^k (10 terms reach long double precision for x >= 50) */
double otmcmc_erfcx(double x) {
  if (x < 50.0) return (double)(expl((long double)x * x) * erfcl(x));
  const long double y = 1.0L / (2.0L * (long double)x * x);
  long double term = 1.0L, sum = 1.0L;
  for (int k = 1; k <= 10; k++) { term *= -(2 * k - 1) * y; sum += term; }
  return (double)(sum / ((long double)x * 1.77245385090551602729816748334114518L));
}
double otmcmc_log_ndtr(double u) {
  if (u >= -1.0) return log(0.5 * erfc(-u * kInvSqrt2));
  return log(0.5 * otmcmc_erfcx(-u * kInvSqrt2)) - 0.5 * (u * u);
}
static double student_t_const(double nu) {
  if (nu < 50.0) return lgamma(0.5 * (nu + 1.0)) - lgamma(0.5 * nu) - 0.5 * log(nu * kPi);
  const double ix = 1.0 / (0.5 * nu), y = ix * ix;
  return ix * (-0.125 + y * (1.0 / 192.0 + y * (-1.0 / 640.0 + y * (17.0 / 14336.0)))) - kHalfLog2Pi;
}
/* t_j of datum d, prediction g, parameter p (ignored by Poisson); dc = lgamma(d + 1). *bad: 0 non-finite g, 1 bad parameter,
 * 2 negative Poisson mean, left as it is for a valid point. */
static double reference_term(int lik, double d, double dc, double g, double p, int* bad) {
  if (!isfinite(g)) { *bad = 0; return NAN; }
  if (lik == KTMCMC_LIK_POISSON) {
    if (g < 0.0) { *bad = 2; return NAN; }
    return d == 0.0 ? -g : (g == 0.0 ? -INFINITY : d * log(g) - g - dc);
  }
  if (!(p > 0.0) || !isfinite(p)) { *bad = 1; return NAN; }
  const double r = d - g;
  if (lik == KTMCMC_LIK_STUDENT_T) return student_t_const(p) - 0.5 * (p + 1.0) * log1p(r * r / p);
  const double z = r / p;
  double t = -kHalfLog2Pi - log(p) - 0.5 * (z * z);
  if (lik == KTMCMC_LIK_POSITIVE_NORMAL) { t = t - otmcmc_log_ndtr(g / p); if (t != t) t = -INFINITY; }
  return t;
}
/* one term, for the tests against scipy */
double otmcmc_reference_term(int32_t lik, double d, double g, double p) {
  int bad = -1;
  return reference_term(lik, d, lik == KTMCMC_LIK_POISSON ? lgamma(d + 1.0) : 0.0, g, p, &bad);
}
static const char* param_key(int lik) { return lik == KTMCMC_LIK_STUDENT_T ? "Degrees Of Freedom" : "Standard Deviation"; }

/* ---- the reference state of a handle (lik = 0: Bayesian/Custom) */
typedef struct ref_state {
  const otmcmc_t* h;
  int lik, have_inj, ef_rows;
  uint64_t m;
  double *data, *dc, *G, *P;    /* data, lgamma(data + 1); model outputs G and parameters P (lambda x m, packed) */
  ktmcmc_host_reference_fn fn;
  void* user;
  struct ref_state* next;
} ref_state;
static ref_state* g_states;

static ref_state* state_of(const otmcmc_t* h, int create) {
  for (ref_state* s = g_states; s; s = s->next)
    if (s->h == h) return s;
  if (!create) return NULL;
  ref_state* s = (ref_state*)calloc(1, sizeof(ref_state));
  s->h = h; s->next = g_states; g_states = s;
  return s;
}

void otmcmc_destroy(otmcmc_t* h) {
  for (ref_state** p = &g_states; *p; p = &(*p)->next)
    if ((*p)->h == h) {
      ref_state* s = *p;
      *p = s->next;
      free(s->data); free(s->dc); free(s->G); free(s->P); free(s);
      break;
    }
  otmcmc_base_destroy(h);
}

int otmcmc_set_reference(otmcmc_t* h, int32_t likelihood, const double* data, uint64_t m) {
  ref_state* s = state_of(h, 1);
  if (s->lik) return fail(h, "set_reference: the reference data are already set");
  if (h->gen != 1 || h->proposed) return fail(h, "set_reference: call it before generation 1");
  if (h->cfg.loglik != KCMA_OBJ_EXTERNAL) return fail(h, "set_reference: the log-likelihood must be External (KCMA_OBJ_EXTERNAL)");
  if (likelihood < KTMCMC_LIK_NORMAL || likelihood > KTMCMC_LIK_POISSON) return fail(h, "set_reference: unknown likelihood %d", likelihood);
  if (!data || m < 1) return fail(h, "set_reference: need at least one reference datum");
  for (uint64_t j = 0; j < m; j++) {
    const double d = data[j];
    if (!isfinite(d)) return fail(h, "Bayesian/Reference: 'Reference Data' %zu is not finite\n", (size_t)j);
    if (likelihood == KTMCMC_LIK_POISSON && (d < 0.0 || d != floor(d)))
      return fail(h, "Bayesian/Reference: 'Reference Data' %zu (%g) must be a non-negative integer for the Poisson likelihood\n", (size_t)j, d);
    if (likelihood == KTMCMC_LIK_POSITIVE_NORMAL && d < 0.0)
      return fail(h, "Bayesian/Reference: 'Reference Data' %zu (%g) must be >= 0 for the Positive Normal likelihood\n", (size_t)j, d);
  }
  s->data = (double*)malloc(sizeof(double) * m);
  s->dc = (double*)calloc(m, sizeof(double));
  memcpy(s->data, data, sizeof(double) * m);
  if (likelihood == KTMCMC_LIK_POISSON)
    for (uint64_t j = 0; j < m; j++) s->dc[j] = lgamma(data[j] + 1.0);
  s->G = (double*)calloc((size_t)h->lambda * m, sizeof(double));
  s->P = (double*)calloc((size_t)h->lambda * m, sizeof(double));
  s->lik = likelihood; s->m = m;
  return 0;
}
int otmcmc_set_host_reference_model(otmcmc_t* h, ktmcmc_host_reference_fn fn, void* user) {
  ref_state* s = state_of(h, 1);
  s->fn = fn; s->user = user;
  return 0;
}
int otmcmc_inject_reference(otmcmc_t* h, const double* g, const double* p, size_t count) {
  ref_state* s = state_of(h, 0);
  if (!s || !s->lik) return fail(h, "inject_reference: no reference data (otmcmc_set_reference)");
  if (!h->proposed || h->evaluated) return fail(h, "inject_reference: no proposals waiting for an evaluation");
  if (!g || (s->lik != KTMCMC_LIK_POISSON) != (p != NULL)) return fail(h, "inject_reference: need g, and p exactly when the likelihood has a parameter");
  if (count != (size_t)h->eval_rows * s->m) return fail(h, "inject_reference: %zu values for %d evaluation rows x %zu", count, h->eval_rows, (size_t)s->m);
  memcpy(s->G, g, sizeof(double) * count);
  if (p) memcpy(s->P, p, sizeof(double) * count);
  s->have_inj = 1;
  return 0;
}

/* l of the evaluated rows: lane k sums j = k, k + 32, ... ascending, then the xor butterfly; the first bad row is an error */
static int reference_loglik(otmcmc_t* h, ref_state* s, int rows) {
  const size_t m = s->m;
  for (int i = 0; i < rows; i++) {
    double p[32] = {0};
    int bad = 3;
    for (size_t j = 0; j < m; j++) {
      int b = 3;
      const double t = reference_term(s->lik, s->data[j], s->dc[j], s->G[i * m + j], s->P[i * m + j], &b);
      if (b < bad) bad = b;
      p[j & 31] = p[j & 31] + t;
    }
    if (bad == 0) return fail(h, "Bayesian/Reference: 'Reference Evaluations' of sample %d contains a non-finite value\n", i);
    if (bad == 1) return fail(h, "Bayesian/Reference: '%s' of sample %d contains a value that is not positive and finite\n", param_key(s->lik), i);
    if (bad == 2) return fail(h, "Bayesian/Reference: 'Reference Evaluations' of sample %d contains a negative Poisson mean\n", i);
    h->EF[i] = butterfly32(p);
  }
  return 0;
}

int otmcmc_eval(otmcmc_t* h) {
  ref_state* s = state_of(h, 1);
  if (!s->lik || h->have_inj) {     /* Bayesian/Custom, or injected log-likelihoods: the oracle as it is */
    const int rows = h->eval_rows;
    if (otmcmc_base_eval(h)) return 1;
    s->ef_rows = rows;
    return 0;
  }
  if (!h->proposed || h->evaluated) return fail(h, "eval: call otmcmc_propose first");
  if (s->have_inj) s->have_inj = 0;
  else if (s->fn) { if (h->eval_rows) s->fn(s->user, h->EX, h->eval_rows, h->N, s->G, s->lik == KTMCMC_LIK_POISSON ? NULL : s->P, s->m); }
  else if (h->eval_rows) return fail(h, "Bayesian/Reference: inject the model outputs or set a host computational model before eval");
  if (reference_loglik(h, s, h->eval_rows)) return 1;
  s->ef_rows = h->eval_rows;
  h->evaluated = 1;
  return 0;
}

int otmcmc_run_generation(otmcmc_t* h) {
  if (h->gen == 1) return otmcmc_propose(h) || otmcmc_eval(h) || otmcmc_accept(h);
  if (otmcmc_anneal(h) || otmcmc_resample(h)) return 1;
  while (h->in_generation)
    if (otmcmc_propose(h) || otmcmc_eval(h) || otmcmc_accept(h)) return 1;
  return 0;
}

int otmcmc_run(otmcmc_t* h, uint64_t max_generations, uint64_t* done) {
  uint64_t g = 0;
  for (; g < max_generations; g++) {
    int fin;
    const char* why;
    otmcmc_check_termination(h, &fin, &why);
    if (fin) break;
    if (otmcmc_run_generation(h)) return 1;
  }
  if (done) *done = g;
  return 0;
}

/* "Evaluation LogLikelihoods" (the log-likelihoods of the last eval, packed like "Evaluation Rows"), else the oracle's keys */
int otmcmc_get_array(otmcmc_t* h, const char* key, double* out, size_t cap, size_t* count) {
  if (strcmp(key, "Evaluation LogLikelihoods")) return otmcmc_base_get_array(h, key, out, cap, count);
  const ref_state* s = state_of(h, 0);
  const size_t n = s ? (size_t)s->ef_rows : 0;
  if (count) *count = n;
  if (!out) return 0;
  if (cap < n) return fail(h, "get_array(%s): capacity %zu < %zu", key, cap, n);
  memcpy(out, h->EF, sizeof(double) * n);
  return 0;
}
