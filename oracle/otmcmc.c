/*
 * otmcmc.c — CPU ORACLE for the transitional MCMC sampler (include/ktmcmc.h). TEST INFRASTRUCTURE ONLY.
 *
 * A plain-C restatement of the algorithm stated in include/ktmcmc.h and DESIGN.md section 14, on the same Philox streams and in
 * the same summation orders as korali_b200/csrc/tmcmc.cu (compiled with -ffp-contract=off). Where the device sums in its own order
 * (the proposal GEMM x' = x + A z, the covariance SYRK) this file sums sequentially in ascending index; the eigendecomposition is
 * okcma_eigen (Householder + QL, ascending |eigenvalue|), with eigenvalues below 0 clamped to 0. Exported under the prefix
 * "otmcmc_" with the signatures of the ktmcmc_ entry points, so that korali_b200/_tmcmc.py drives both; oracle/otmcmc.py links it
 * with okcma.c (Philox, built-in objectives, eigensolver) into libotmcmc.so.
 */
#define _GNU_SOURCE
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../include/ktmcmc.h"

void okcma_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);
void okcma_objective(int objective, uint64_t n, uint64_t rows, const double* x, const double* coef, double* f_out);
int okcma_eigen(uint64_t n64, const double* c, double* w, double* q);

#define T_THREADS 1024
#define T_MEAN_CHUNKS 64
#define T_KEY_TAG 0x544d434du /* "TMCM" */
static const double kHalfLog2Pi = 0.91893853320467274178;

typedef struct otmcmc {
  ktmcmc_cfg cfg;
  int N, lambda, L;
  uint64_t gen, init_evals, evals, accepted, proposals;
  uint64_t* burn_in;
  int32_t* type;
  double *pa, *pb, *coef;
  double *X, *LL, *LP, *DX, *DLL, *DLP, *CX, *CLL, *CLP, *XP, *LPP, *EX, *EF;
  double *W, *Cum, *mean, *cov, *A;
  int *counts, *leader, *len, *dbstart, *flag, *slot, *acc;
  double rho, rho_prev, delta, covv, logev, llmax;
  int chains, steps, step, burn, eval_rows, leaders, last_pos, in_generation, proposed, evaluated, have_inj;
  double tc_target, tc_max_generations, tc_max_model_evaluations;
  ktmcmc_host_loglik_fn host_fn;
  void* host_user;
  char err[512], reason[256];
} otmcmc_t;

static char g_err[512];
static int fail(otmcmc_t* h, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(h ? h->err : g_err, 512, fmt, ap);
  va_end(ap);
  return 1;
}

static void philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint64_t seed, uint32_t r[4]) {
  uint32_t ctr[4] = {c0, c1, c2, c3};
  uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32) ^ T_KEY_TAG};
  okcma_philox4x32_10(ctr, key, r);
}
static double unit(uint32_t lo, uint32_t hi) {
  uint64_t v = ((uint64_t)hi << 32) | lo;
  return (double)(v >> 12) * 0x1.0p-52 + 0x1.0p-53;
}
static void box_muller(const uint32_t r[4], double* z0, double* z1) {
  double u1 = unit(r[0], r[1]), u2 = unit(r[2], r[3]);
  double rad = sqrt(-2.0 * log(u1));
  double s, c;
  sincos(2.0 * M_PI * u2, &s, &c);
  *z0 = rad * c;
  *z1 = rad * s;
}
static double butterfly32(double p[32]) {
  for (int off = 16; off >= 1; off >>= 1) {
    double q[32];
    for (int l = 0; l < 32; l++) q[l] = p[l] + p[l ^ off];
    memcpy(p, q, sizeof(q));
  }
  return p[0];
}
static double prior_term(int type, double a, double b, double x) {
  if (type == KTMCMC_PRIOR_UNIFORM) return (x >= a && x <= b) ? -log(b - a) : -INFINITY;
  double z = (x - a) / b;
  return -0.5 * (z * z) - log(b) - kHalfLog2Pi;
}
static double log_prior(const otmcmc_t* h, const double* x) {
  double p[32] = {0};
  for (int d = 0; d < h->N; d++) p[d & 31] = p[d & 31] + prior_term(h->type[d], h->pa[d], h->pb[d], x[d]);
  return butterfly32(p);
}
/* the device's block sum: thread t < 1024 sums v[t], v[t + 1024], ...; butterfly per warp; butterfly over the 32 warp sums */
static double block_sum(const double* part) {
  double ws[32];
  for (int w = 0; w < 32; w++) {
    double p[32];
    memcpy(p, part + 32 * w, sizeof(p));
    ws[w] = butterfly32(p);
  }
  return butterfly32(ws);
}
static double weight(double l, double D, double llmax) { return l == -INFINITY ? 0.0 : exp(D * (l - llmax)); }
static double cov_of(const otmcmc_t* h, double D, double llmax, double* s1) {
  static double p1[T_THREADS], p2[T_THREADS];
  for (int t = 0; t < T_THREADS; t++) {
    double a = 0.0, b = 0.0;
    for (int i = t; i < h->lambda; i += T_THREADS) { double w = weight(h->LL[i], D, llmax); a = a + w; b = b + w * w; }
    p1[t] = a; p2[t] = b;
  }
  *s1 = block_sum(p1);
  double s2 = block_sum(p2);
  return sqrt(fmax(0.0, (double)h->lambda * s2 / (*s1 * *s1) - 1.0));
}

void otmcmc_cfg_defaults(ktmcmc_cfg* c) {
  memset(c, 0, sizeof(*c));
  c->abi_version = KTMCMC_ABI_VERSION;
  c->max_chain_length = 1;
  c->target_cov = 1.0;
  c->covariance_scaling = 0.04;
  c->min_annealing_update = 1e-5;
  c->max_annealing_update = 1.0;
  c->loglik = KCMA_OBJ_EXTERNAL;
}
const char* otmcmc_last_error(const otmcmc_t* h) { return h ? h->err : g_err; }

void otmcmc_destroy(otmcmc_t* h) {
  if (!h) return;
  void* p[] = {h->burn_in, h->type, h->pa, h->pb, h->coef, h->X, h->LL, h->LP, h->DX, h->DLL, h->DLP, h->CX, h->CLL, h->CLP, h->XP, h->LPP,
               h->EX, h->EF, h->W, h->Cum, h->mean, h->cov, h->A, h->counts, h->leader, h->len, h->dbstart, h->flag, h->slot, h->acc};
  for (size_t i = 0; i < sizeof(p) / sizeof(p[0]); i++) free(p[i]);
  free(h);
}

int otmcmc_create(const ktmcmc_cfg* cfg, otmcmc_t** out) {
  if (!cfg || !out) return fail(NULL, "null argument");
  if (cfg->abi_version != KTMCMC_ABI_VERSION) return fail(NULL, "ktmcmc_cfg ABI version mismatch");
  if (cfg->n < 1 || cfg->population_size < 2 || cfg->max_chain_length < 1) return fail(NULL, "invalid sizes");
  if (!cfg->prior_type || !cfg->prior_a || !cfg->prior_b) return fail(NULL, "every variable needs a prior distribution");
  otmcmc_t* h = (otmcmc_t*)calloc(1, sizeof(otmcmc_t));
  h->cfg = *cfg;
  const int N = h->N = (int)cfg->n, lam = h->lambda = (int)cfg->population_size;
  h->L = (int)(cfg->max_chain_length < cfg->population_size ? cfg->max_chain_length : cfg->population_size);
  h->gen = 1;
  h->tc_target = 1.0; h->tc_max_generations = 1e10; h->tc_max_model_evaluations = 1e9;
  h->burn_in = (uint64_t*)calloc(cfg->burn_in_count + 1, sizeof(uint64_t));
  if (cfg->per_generation_burn_in) memcpy(h->burn_in, cfg->per_generation_burn_in, sizeof(uint64_t) * cfg->burn_in_count);
  else h->cfg.burn_in_count = 0;
  h->type = (int32_t*)malloc(sizeof(int32_t) * N);
  memcpy(h->type, cfg->prior_type, sizeof(int32_t) * N);
  h->pa = (double*)malloc(sizeof(double) * N); memcpy(h->pa, cfg->prior_a, sizeof(double) * N);
  h->pb = (double*)malloc(sizeof(double) * N); memcpy(h->pb, cfg->prior_b, sizeof(double) * N);
  h->coef = (double*)malloc(sizeof(double) * N);
  for (int d = 0; d < N; d++) h->coef[d] = cfg->loglik_coef ? cfg->loglik_coef[d] : pow(10.0, 6.0 * d / (double)(N > 1 ? N - 1 : 1));
  double** rowsN[] = {&h->X, &h->DX, &h->CX, &h->XP, &h->EX};
  for (size_t i = 0; i < 5; i++) *rowsN[i] = (double*)calloc((size_t)lam * N, sizeof(double));
  double** rows1[] = {&h->LL, &h->LP, &h->DLL, &h->DLP, &h->CLL, &h->CLP, &h->LPP, &h->EF, &h->W, &h->Cum};
  for (size_t i = 0; i < 10; i++) *rows1[i] = (double*)calloc(lam, sizeof(double));
  int** ints[] = {&h->counts, &h->leader, &h->len, &h->dbstart, &h->flag, &h->slot, &h->acc};
  for (size_t i = 0; i < 7; i++) *ints[i] = (int*)calloc(lam, sizeof(int));
  h->mean = (double*)calloc(N, sizeof(double));
  h->cov = (double*)calloc((size_t)N * N, sizeof(double));
  h->A = (double*)calloc((size_t)N * N, sizeof(double));
  h->cfg.per_generation_burn_in = NULL; h->cfg.prior_type = NULL; h->cfg.prior_a = h->cfg.prior_b = h->cfg.loglik_coef = NULL;
  *out = h;
  return 0;
}

int otmcmc_set_host_loglik(otmcmc_t* h, ktmcmc_host_loglik_fn fn, void* user) { h->host_fn = fn; h->host_user = user; return 0; }

int otmcmc_anneal(otmcmc_t* h) {
  if (h->gen < 2 || h->in_generation) return fail(h, "anneal: expected the start of a generation after the first");
  const int N = h->N, lam = h->lambda;
  double llmax = -INFINITY;
  int nan = 0, fin = 0;
  for (int i = 0; i < lam; i++) {
    double l = h->LL[i];
    if (l != l) nan = 1;
    else if (l != -INFINITY) { fin = 1; llmax = fmax(llmax, l); }
  }
  if (nan) return fail(h, "A NaN log-likelihood was produced by the likelihood model\n");
  if (!fin) return fail(h, "Every sample of the population has a log-likelihood of -inf: the annealing step is undefined\n");
  const double rho = h->rho, rem = 1.0 - rho;
  double s1, D = rem;
  if (cov_of(h, rem, llmax, &s1) > h->cfg.target_cov) {
    double lo = 0.0, hi = rem;
    for (int it = 0; it < 64; it++) {
      double mid = 0.5 * (lo + hi);
      if (cov_of(h, mid, llmax, &s1) > h->cfg.target_cov) hi = mid; else lo = mid;
    }
    D = lo;
  }
  D = fmin(fmax(D, h->cfg.min_annealing_update), h->cfg.max_annealing_update);
  double rho_new;
  if (D >= rem) { D = rem; rho_new = 1.0; } else rho_new = rho + D;
  h->covv = cov_of(h, D, llmax, &s1);
  for (int i = 0; i < lam; i++) h->W[i] = weight(h->LL[i], D, llmax) / s1;
  /* cumsum: contiguous chunks */
  const int chunk = (lam + T_THREADS - 1) / T_THREADS;
  double pre = 0.0;
  h->last_pos = -1;
  for (int t = 0; t < T_THREADS; t++) {
    int b0 = t * chunk < lam ? t * chunk : lam, b1 = b0 + chunk < lam ? b0 + chunk : lam;
    double loc = 0.0;
    for (int i = b0; i < b1; i++) { loc = loc + h->W[i]; h->Cum[i] = pre + loc; if (h->W[i] > 0.0) h->last_pos = i; }
    pre = pre + loc;
  }
  h->rho_prev = rho; h->rho = rho_new; h->delta = D; h->llmax = llmax;
  h->logev = h->logev + (log(s1 / (double)lam) + D * llmax);
  /* weighted mean: 64 row chunks */
  const int rows = (lam + T_MEAN_CHUNKS - 1) / T_MEAN_CHUNKS;
  for (int d = 0; d < N; d++) {
    double m = 0.0;
    for (int c = 0; c < T_MEAN_CHUNKS; c++) {
      int r0 = c * rows < lam ? c * rows : lam, r1 = r0 + rows < lam ? r0 + rows : lam;
      double p = 0.0;
      for (int i = r0; i < r1; i++) p = p + h->W[i] * h->X[(size_t)i * N + d];
      m = m + p;
    }
    h->mean[d] = m;
  }
  /* Sigma = s sum_i S_i S_i^T with S_i = sqrt(w~_i)(x_i - mean), rows summed in ascending i */
  double* S = (double*)malloc(sizeof(double) * (size_t)lam * N);
  for (int i = 0; i < lam; i++)
    for (int d = 0; d < N; d++) S[(size_t)i * N + d] = sqrt(h->W[i]) * (h->X[(size_t)i * N + d] - h->mean[d]);
  for (int d = 0; d < N; d++)
    for (int e = 0; e <= d; e++) {
      double p = 0.0;
      for (int i = 0; i < lam; i++) p = p + S[(size_t)i * N + d] * S[(size_t)i * N + e];
      h->cov[(size_t)d * N + e] = h->cov[(size_t)e * N + d] = h->cfg.covariance_scaling * p;
    }
  free(S);
  double* w = (double*)malloc(sizeof(double) * N);
  double* q = (double*)malloc(sizeof(double) * (size_t)N * N);
  okcma_eigen(N, h->cov, w, q);
  for (int d = 0; d < N; d++)
    for (int e = 0; e < N; e++) h->A[(size_t)d * N + e] = q[(size_t)d * N + e] * sqrt(fmax(w[e], 0.0));
  free(w); free(q);
  h->in_generation = 1;
  h->chains = 0;
  return 0;
}

int otmcmc_resample(otmcmc_t* h) {
  if (!h->in_generation || h->chains) return fail(h, "resample: call otmcmc_anneal first");
  const int lam = h->lambda, L = h->L;
  memset(h->counts, 0, sizeof(int) * lam);
  for (int k = 0; k < lam; k++) {
    uint32_t r[4];
    philox(0u, (uint32_t)k, 0u, (uint32_t)h->gen, h->cfg.seed, r);
    double u = unit(r[0], r[1]);
    int lo = 0, hi = lam;
    while (lo < hi) { int mid = (lo + hi) >> 1; if (h->Cum[mid] >= u) hi = mid; else lo = mid + 1; }
    if (lo >= lam) lo = h->last_pos;
    h->counts[lo]++;
  }
  int k = 0, db = 0, mc = 0;
  h->leaders = 0;
  for (int i = 0; i < lam; i++) {
    int c = h->counts[i];
    if (c > mc) mc = c;
    h->leaders += c > 0;
    for (int j = 0; j * L < c; j++) { h->leader[k] = i; h->len[k] = c - j * L < L ? c - j * L : L; h->dbstart[k] = db + j * L; k++; }
    db += c;
  }
  h->chains = k;
  const int N = h->N;
  for (int c = 0; c < k; c++) {
    memcpy(h->CX + (size_t)c * N, h->X + (size_t)h->leader[c] * N, sizeof(double) * N);
    h->CLL[c] = h->LL[h->leader[c]]; h->CLP[c] = h->LP[h->leader[c]];
  }
  h->burn = (int)(h->gen < h->cfg.burn_in_count ? h->burn_in[h->gen] : h->cfg.default_burn_in);
  h->steps = h->burn + (mc < L ? mc : L);
  h->step = 0;
  h->accepted = h->proposals = 0;
  h->proposed = h->evaluated = 0;
  return 0;
}

int otmcmc_propose(otmcmc_t* h) {
  const int N = h->N;
  if (h->gen == 1) {
    if (h->proposed) return fail(h, "propose: the prior draws of generation 1 are waiting for eval / accept");
    for (int i = 0; i < h->lambda; i++) {
      double* x = h->EX + (size_t)i * N;
      for (int p = 0; 2 * p < N; p++) {
        uint32_t r[4];
        philox((1u << 20) + (uint32_t)p, (uint32_t)i, 0u, 0u, h->cfg.seed, r);
        double z[2], u[2] = {unit(r[0], r[1]), unit(r[2], r[3])};
        box_muller(r, &z[0], &z[1]);
        for (int s = 0; s < 2 && 2 * p + s < N; s++) {
          int d = 2 * p + s;
          x[d] = h->type[d] == KTMCMC_PRIOR_UNIFORM ? h->pa[d] + (h->pb[d] - h->pa[d]) * u[s] : h->pa[d] + h->pb[d] * z[s];
        }
      }
      h->LP[i] = log_prior(h, x);
    }
    h->eval_rows = h->lambda;
  } else {
    if (!h->in_generation || !h->chains || h->step >= h->steps || h->proposed) return fail(h, "propose: no MCMC step pending (anneal and resample first)");
    double* z = (double*)malloc(sizeof(double) * (N + 1));
    int rows = 0;
    for (int k = 0; k < h->chains; k++) {
      const int active = h->step < h->burn + h->len[k];
      if (!active) { h->LPP[k] = -INFINITY; h->flag[k] = -1; h->slot[k] = -1; continue; }
      for (int p = 0; 2 * p < N; p++) {
        uint32_t r[4];
        philox((1u << 20) + (uint32_t)p, (uint32_t)k, (uint32_t)h->step, (uint32_t)h->gen, h->cfg.seed, r);
        box_muller(r, &z[2 * p], &z[2 * p + 1]);
      }
      double* xp = h->XP + (size_t)k * N;
      for (int d = 0; d < N; d++) {
        double y = 0.0;
        for (int e = 0; e < N; e++) y = y + h->A[(size_t)d * N + e] * z[e];
        xp[d] = h->CX[(size_t)k * N + d] + y;
      }
      h->LPP[k] = log_prior(h, xp);
      h->flag[k] = h->LPP[k] != -INFINITY ? 1 : 0;
      h->slot[k] = h->flag[k] == 1 ? rows : -1;
      if (h->flag[k] == 1) memcpy(h->EX + (size_t)rows++ * N, xp, sizeof(double) * N);
      h->proposals++;
    }
    free(z);
    h->eval_rows = rows;
    h->evals += (uint64_t)rows;
  }
  h->proposed = 1;
  h->evaluated = 0;
  return 0;
}

int otmcmc_inject_loglik(otmcmc_t* h, const double* l, size_t count) {
  if (!h->proposed || h->evaluated) return fail(h, "inject_loglik: no proposals waiting for an evaluation");
  if (count != (size_t)h->eval_rows) return fail(h, "inject_loglik: %zu values for %d evaluation rows", count, h->eval_rows);
  memcpy(h->EF, l, sizeof(double) * count);
  h->have_inj = 1;
  return 0;
}
int otmcmc_inject_factor(otmcmc_t* h, const double* a, size_t count) {
  if (count != (size_t)h->N * h->N) return fail(h, "inject_factor: %zu values", count);
  memcpy(h->A, a, sizeof(double) * count);
  return 0;
}

int otmcmc_eval(otmcmc_t* h) {
  if (!h->proposed || h->evaluated) return fail(h, "eval: call otmcmc_propose first");
  if (h->have_inj) h->have_inj = 0;
  else if (h->cfg.loglik != KCMA_OBJ_EXTERNAL) okcma_objective(h->cfg.loglik, h->N, h->eval_rows, h->EX, h->coef, h->EF);
  else if (h->host_fn) { if (h->eval_rows) h->host_fn(h->host_user, h->EX, h->eval_rows, h->N, h->EF); }
  else return fail(h, "the log-likelihood is External: inject the values or set a host model before eval");
  h->evaluated = 1;
  return 0;
}

int otmcmc_accept(otmcmc_t* h) {
  if (!h->evaluated) return fail(h, "accept: call otmcmc_eval first");
  const int N = h->N, lam = h->lambda;
  h->proposed = h->evaluated = 0;
  if (h->gen == 1) {
    memcpy(h->X, h->EX, sizeof(double) * (size_t)lam * N);
    memcpy(h->LL, h->EF, sizeof(double) * lam);
    h->init_evals = lam;
    for (int i = 0; i < lam; i++) if (h->LL[i] != h->LL[i]) return fail(h, "A NaN log-likelihood was produced by the likelihood model\n");
    h->gen = 2;
    return 0;
  }
  for (int k = 0; k < h->chains; k++) {
    if (h->step >= h->burn + h->len[k]) continue;
    int acc = 0;
    if (h->slot[k] >= 0) {
      double l = h->EF[h->slot[k]];
      if (l != l) return fail(h, "A NaN log-likelihood was produced by the likelihood model\n");
      uint32_t r[4];
      philox(1u, (uint32_t)k, (uint32_t)h->step, (uint32_t)h->gen, h->cfg.seed, r);
      double u = unit(r[0], r[1]);
      acc = log(u) < h->rho * (l - h->CLL[k]) + (h->LPP[k] - h->CLP[k]);
      if (acc) {
        h->CLL[k] = l; h->CLP[k] = h->LPP[k]; h->accepted++;
        memcpy(h->CX + (size_t)k * N, h->XP + (size_t)k * N, sizeof(double) * N);
      }
    }
    h->acc[k] = acc;
    if (h->step >= h->burn) {
      int row = h->dbstart[k] + h->step - h->burn;
      memcpy(h->DX + (size_t)row * N, h->CX + (size_t)k * N, sizeof(double) * N);
      h->DLL[row] = h->CLL[k]; h->DLP[row] = h->CLP[k];
    }
  }
  if (++h->step < h->steps) return 0;
  double* t;
  t = h->X; h->X = h->DX; h->DX = t;
  t = h->LL; h->LL = h->DLL; h->DLL = t;
  t = h->LP; h->LP = h->DLP; h->DLP = t;
  h->in_generation = 0;
  h->gen++;
  return 0;
}

int otmcmc_run_generation(otmcmc_t* h) {
  if (h->gen == 1) return otmcmc_propose(h) || otmcmc_eval(h) || otmcmc_accept(h);
  if (otmcmc_anneal(h) || otmcmc_resample(h)) return 1;
  while (h->in_generation)
    if (otmcmc_propose(h) || otmcmc_eval(h) || otmcmc_accept(h)) return 1;
  return 0;
}

int otmcmc_check_termination(otmcmc_t* h, int* finished, const char** reason) {
  h->reason[0] = 0;
  int fin = 0;
  if (h->gen > 1 && h->rho >= h->tc_target) { strcat(h->reason, "Target Annealing Exponent;"); fin = 1; }
  if (h->tc_max_model_evaluations <= (double)(h->init_evals + h->evals)) { strcat(h->reason, "solver['Max Model Evaluations'];"); fin = 1; }
  if ((double)h->gen > h->tc_max_generations) { strcat(h->reason, "solver['Max Generations'];"); fin = 1; }
  *finished = fin;
  if (reason) *reason = h->reason;
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

int otmcmc_get_array(otmcmc_t* h, const char* key, double* out, size_t cap, size_t* count) {
  const size_t N = h->N, lam = h->lambda;
  const double* src = NULL;
  const int* isrc = NULL;
  size_t n = 0;
  if (!strcmp(key, "Sample Database")) { src = h->X; n = lam * N; }
  else if (!strcmp(key, "Sample LogLikelihood Database")) { src = h->LL; n = lam; }
  else if (!strcmp(key, "Sample LogPrior Database")) { src = h->LP; n = lam; }
  else if (!strcmp(key, "Covariance Matrix")) { src = h->cov; n = N * N; }
  else if (!strcmp(key, "Proposal Factor")) { src = h->A; n = N * N; }
  else if (!strcmp(key, "Mean Theta")) { src = h->mean; n = N; }
  else if (!strcmp(key, "Weights")) { src = h->W; n = lam; }
  else if (!strcmp(key, "Selection Counts")) { isrc = h->counts; n = lam; }
  else if (!strcmp(key, "Chain Leaders")) { isrc = h->leader; n = h->chains; }
  else if (!strcmp(key, "Chain Lengths")) { isrc = h->len; n = h->chains; }
  else if (!strcmp(key, "Proposal Support")) { isrc = h->flag; n = h->chains; }
  else if (!strcmp(key, "Accept Flags")) { isrc = h->acc; n = h->chains; }
  else if (!strcmp(key, "Evaluation Rows")) { src = h->EX; n = h->proposed ? (size_t)h->eval_rows * N : 0; }
  else return fail(h, "unknown array key '%s'", key);
  if (count) *count = n;
  if (!out) return 0;
  if (cap < n) return fail(h, "get_array(%s): capacity %zu < %zu", key, cap, n);
  for (size_t i = 0; i < n; i++) out[i] = src ? src[i] : (double)isrc[i];
  return 0;
}

int otmcmc_get_scalar(otmcmc_t* h, const char* key, double* out) {
  if (!strcmp(key, "Annealing Exponent")) *out = h->rho;
  else if (!strcmp(key, "Previous Annealing Exponent")) *out = h->rho_prev;
  else if (!strcmp(key, "Annealing Exponent Update")) *out = h->delta;
  else if (!strcmp(key, "Coefficient Of Variation")) *out = h->covv;
  else if (!strcmp(key, "LogEvidence")) *out = h->logev;
  else if (!strcmp(key, "Max Loglikelihood")) *out = h->llmax;
  else if (!strcmp(key, "Chain Count")) *out = h->chains;
  else if (!strcmp(key, "Max Chain Steps")) *out = h->steps;
  else if (!strcmp(key, "Current Step")) *out = h->step;
  else if (!strcmp(key, "Proposals Acceptance Rate")) *out = h->proposals ? (double)h->accepted / (double)h->proposals : 0.0;
  else if (!strcmp(key, "Selection Acceptance Rate")) *out = (double)h->leaders / (double)h->lambda;
  else if (!strcmp(key, "Model Evaluation Count")) *out = (double)(h->init_evals + h->evals);
  else if (!strcmp(key, "Current Generation")) *out = (double)h->gen;
  else if (!strcmp(key, "Population Size")) *out = h->lambda;
  else if (!strcmp(key, "Burn In")) *out = h->burn;
  else if (!strcmp(key, "Termination Criteria/Target Annealing Exponent")) *out = h->tc_target;
  else if (!strcmp(key, "Termination Criteria/Max Generations")) *out = h->tc_max_generations;
  else if (!strcmp(key, "Termination Criteria/Max Model Evaluations")) *out = h->tc_max_model_evaluations;
  else return fail(h, "unknown scalar key '%s'", key);
  return 0;
}

int otmcmc_set_scalar(otmcmc_t* h, const char* key, double v) {
  if (!strcmp(key, "Termination Criteria/Target Annealing Exponent")) h->tc_target = v;
  else if (!strcmp(key, "Termination Criteria/Max Generations")) h->tc_max_generations = v;
  else if (!strcmp(key, "Termination Criteria/Max Model Evaluations")) h->tc_max_model_evaluations = v;
  else return fail(h, "unknown scalar key '%s'", key);
  return 0;
}

uint64_t otmcmc_launch_count(const otmcmc_t* h) { (void)h; return 0; }
