// kernels.h — host-side launchers of the libkcma CUDA kernels (internal; the public surface is include/kcma.h).
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <stddef.h>
#include <stdint.h>

namespace kc {

// True exactly once per device of this process. Function attributes (dynamic shared-memory limits) are per device, and one
// process may drive several devices (Engine: k["Conduit"]["Devices"], one host thread per device).
inline bool first_call_on_device(std::atomic<unsigned long long>& mask) {
  int d = 0;
  cudaGetDevice(&d);
  const unsigned long long bit = 1ull << (d & 63);
  return !(mask.fetch_or(bit) & bit);
}
struct DevScalars;

// gemm.cu
size_t gemm_tn_smem_bytes();
size_t syrk_tt_smem_bytes();
void launch_gemm_tn(cudaStream_t st, int M, int Nc, int K, const double* A, int lda, const double* B, int ldb, double* C, int ldc);
int syrk_tiles(int n);
int syrk_pick_splits(int n, int K, int num_sms, int max_splits);
void launch_syrk_tt(cudaStream_t st, int n, int K, const int* kptr, const double* S, int lds, long long s_rows, double* W, int ldw,
                    int splits);

int launch_syrk(cudaStream_t st, int n, int K, const int* kptr, const double* S, int lds, long long s_rows, double* W, int ldw,
                int expect_rows, int num_sms, int max_splits);
// gemm_tma.cu (TMA + mbarrier staging; return false when the tensor maps cannot be built)
int launch_syrk_sk_tma(cudaStream_t st, int n, int K, const int* kptr, const double* S, int lds, long long s_rows, double* W, int ldw,
                       int num_sms, int max_splits);
bool launch_gemm_tn_tma(cudaStream_t st, int M, int Nc, int K, const double* A, int lda, const double* B, int ldb, double* C, int ldc);
bool launch_syrk_tt_tma(cudaStream_t st, int n, int K, const int* kptr, const double* S, int lds, long long s_rows, double* W, int ldw,
                        int splits);

// gemm_batched.cu (descriptor-driven batched GEMM of the tridiagonalisation-based eigensolver)
struct GemmDesc {
  const double* A; const double* B; double* C;   // C[M x Nc] = beta*C + alpha * A[M x K] * B[Nc x K]^T
  int M, Nc, K, lda, ldb, ldc;
  double alpha, beta;
  int krule;            // 0: full k-range; 1 / 2: A / B is block diagonal with first block n1 x n1 (tile-wise k-range) unless *mixed
  int n1;
  const int* mixed;
  int splits;           // > 1: split-K, slab s stored (not accumulated) at C + s*split_stride
  long long split_stride;
};
size_t gemm_batched_smem_bytes();
void launch_gemm_batched(cudaStream_t st, const GemmDesc* d_descs, int batch, int max_m, int max_nc, int max_splits);
void launch_reduce_slabs(cudaStream_t st, const double* slabs, long long stride, int splits, int rows, int cols, int ld, double* out,
                         int num_sms);

// tridiag.cu + dc.cu: Householder tridiagonalisation, divide & conquer, compact-WY back-transform (DESIGN.md section 6)
struct TridiagWs;
TridiagWs* tridiag_ws_create(int n, int ld, int num_sms, char* err, size_t errlen);
void tridiag_ws_destroy(TridiagWs* ws);
// eigenvectors of the symmetric M as the ROWS of *VT_out (n x ld, owned by the workspace), ascending eigenvalues in *ev_out;
// false when a launch failed
bool launch_eigen_tridiag(cudaStream_t st, TridiagWs* ws, const double* M, double** VT_out, double** ev_out, int* launches);
// stage entry points for the parity tests (kcma_k_sytrd / kcma_k_stedc)
bool tridiag_stage_sytrd(cudaStream_t st, TridiagWs* ws, const double* M);
bool tridiag_stage_dc(cudaStream_t st, TridiagWs* ws, int* launches);
bool tridiag_stage_back_fork(cudaStream_t st, TridiagWs* ws, int* launches);   // Q accumulation on the side stream (before stage 2)
bool tridiag_stage_back_join(cudaStream_t st, TridiagWs* ws, int* launches);   // X^T = Z^T Q^T (after stage 2)
const double* tridiag_result_vectors(const TridiagWs* ws);
const double* tridiag_result_values(const TridiagWs* ws);
void tridiag_get_tridiagonal(TridiagWs* ws, double* d, double* e, double* tau, double* vr /* n x n row-major reflectors */);
void tridiag_set_tridiagonal(TridiagWs* ws, const double* d, const double* e);
void tridiag_dump_prof(TridiagWs* ws);   // KCMA_SYTRD_PROF=step0[,cta]: prints the phase stamps of sytrd_kernel to stderr
void launch_eig_sign(cudaStream_t st, const double* VT, int ld, int n, double* sign);
// The size policy of the symmetric eigensolvers, one rule for CMA-ES (api.cu) and TMCMC (tmcmc.cu): eigen_use_small (eigen.cu),
// else the tridiagonal solver while its shared-memory vectors fit.
bool eigen_tridiag_fits(int n);

// rng.cu
void launch_philox_normal(cudaStream_t st, double* Z, int ldz, long long rows, int n, unsigned long long seed, unsigned generation,
                          unsigned long long row_begin, const unsigned* attempt, const int* row_list, int num_sms,
                          const DevScalars* gen_src = nullptr /* read when generation == kGenFromDevice */);
void launch_philox_raw(cudaStream_t st, const uint32_t* in6, uint32_t* out4);

// objective.cu
int launch_objective(cudaStream_t st, int objective, const double* Y, int ldy, long long samples, int n, int mirrored, int from_x,
                     const double* mean, DevScalars* sc, const double* coef, double* f, int num_sms);
void launch_feasibility(cudaStream_t st, const double* Y, int ldy, long long samples, int n, int mirrored, const double* mean,
                        const DevScalars* sc, const double* lower, const double* upper, unsigned char* infeasible, double* X,
                        int ldx, const int* row_list, int num_sms);
void launch_constraints_halfspace(cudaStream_t st, const double* Y, int ldy, long long samples, int n, const double* mean,
                                  DevScalars* sc, const double* shift, int n_con, double* G, long long ldg, const int* row_list,
                                  int num_sms);

// sort.cu
size_t sort_workspace_bytes(int n);
int launch_sort_index(cudaStream_t st, const double* f, int n, void* workspace, unsigned* sorted_idx, int num_sms);

// update.cu
void launch_scale_bd(cudaStream_t st, const double* B, int ldb, const double* D, double* A, int lda, int n);
void launch_rank_bookkeeping(cudaStream_t st, const double* f, const unsigned* idx, int lambda, int mu,
                             const unsigned long long* viol, int best_is_first, DevScalars* sc);
void launch_proportional_weights(cudaStream_t st, const double* f, const unsigned* idx, int mu, double* w);
void launch_select_local(cudaStream_t st, const unsigned* idx, const double* w, int mu, unsigned lo, unsigned hi, int* sel_sample,
                         double* sel_weight, int* count_out);
void launch_gather_mean(cudaStream_t st, const double* Y, int ldy, int mirrored, int from_x, const int* sel_sample,
                        const double* sel_weight, const int* count_ptr, int max_count, int rows_per_cta, int n, int ld,
                        const double* mean, const DevScalars* sc, double* S, int lds, int rows_padded, double* partial);
void launch_mean_reduce(cudaStream_t st, const double* partial, const int* count_ptr, int rows_per_cta, int n, int ld,
                        double* mean_out, const double* Y, int ldy, int mirrored, int from_x, const double* mean,
                        const DevScalars* sc, unsigned lo, unsigned hi, double* best_x);
void launch_objective_gradient(cudaStream_t st, int objective, const double* Y, int ldy, long long samples, int n, int mirrored, int from_x,
                               const double* mean, const DevScalars* sc, const double* coef, double* G, int ldg, int num_sms);
void launch_gradient_mean(cudaStream_t st, const double* G, int ldg, const int* sel_sample, const double* sel_weight, const int* count_ptr,
                          int n, double step, double* mean_new);
void launch_best_update(cudaStream_t st, const double* best_x, int n, unsigned generation, double* cur_best_vars,
                        double* best_ever_vars, DevScalars* sc, const double* con_evals, long long ldg, int n_con,
                        double* best_con_evals);
void launch_paths(cudaStream_t st, const double* mean_new, double* mean, double* mean_old, double* y, double* tvec, double* ps,
                  double* pc, const double* B, int ldb, const double* D, int n, int diagonal, double cs, double cc, double mueff,
                  double chi_n, unsigned generation, DevScalars* sc);
void launch_adapt_c(cudaStream_t st, double* C, int ldc, const double* W, int ldw, int splits, int n, const double* pc, double c1,
                    double cmu, double cc, int diagonal, const DevScalars* sc);
void launch_reduce_splits(cudaStream_t st, const double* W, int ldw, int splits, int n, double* P);
void launch_diag_rank_mu(cudaStream_t st, const double* S, int lds, const int* count_ptr, int max_count, int rows_per_cta, int n,
                         double* W, int ldw, int slabs);
void launch_signed_rank_mu(cudaStream_t st, const double* S, int lds, const int* count_ptr, const double* sel_weight, int n, double* W,
                           int ldw);
void launch_sigma(cudaStream_t st, const double* C, int ldc, int n, const double* min_sd_update, int any_min_sd, double cs,
                  double damp, double chi_n, double trace, int is_sigma_bounded, int mu_value_gt1, int viability_regime,
                  double global_success_lr, double target_success_rate, int has_discrete, DevScalars* sc);
void launch_discrete_mutation(cudaStream_t st, double* X, int ldx, long long samples, int n, unsigned long long sample_begin, int mirrored,
                              const DevScalars* sc, const double* mask, const double* gran, const double* best_ever, unsigned long long seed,
                              unsigned generation, const unsigned* attempt, double* disc_mut);
void launch_discrete_matrix(cudaStream_t st, const double* C, int ldc, int n, const double* gran, const double* ps, double cs,
                            double population_size, double* mask, double* mask_sigma, DevScalars* sc);
void launch_feasibility_x(cudaStream_t st, const double* X, int ldx, long long samples, int n, const double* lower, const double* upper,
                          unsigned char* infeasible, int num_sms);
void launch_viability_boundaries(cudaStream_t st, const double* G, long long ldg, int n_con, const unsigned* idx, int mu,
                                 double* bounds);

// eigen.cu
void launch_set_identity(cudaStream_t st, double* M, int ld, int n);
bool eigen_use_small(int n);   // N <= 24: launch_eigen_small, the whole solver in one CTA
void launch_eigen_small(cudaStream_t st, const double* C, int ld, int n, double* VT, double* GT, double* B, double* A, double* D,
                        double tol, int max_sweeps, DevScalars* sc);
bool launch_jacobi_persistent(cudaStream_t st, double* GT, double* VT, int ld, int n, double tol, int max_sweeps, DevScalars* sc,
                              int num_sms, unsigned* ready);
void launch_jacobi_block_sweep(cudaStream_t st, double* GT, double* VT, int ld, int n, double tol, DevScalars* sc, int* launches);
void launch_jacobi_block_flush(cudaStream_t st, double* GT, double* VT, int ld, int n, double tol, DevScalars* sc, int* launches);
void launch_rayleigh(cudaStream_t st, const double* GT, const double* VT, int ld, int n, double* ev, double* sign);
void launch_eig_order(cudaStream_t st, const double* ev, int n, int* perm, DevScalars* sc);
void launch_eig_commit(cudaStream_t st, const double* VTw, int ld, int n, const int* perm, const double* ev, const double* sign,
                       double* B, double* A, double* D, double* VT, const DevScalars* sc);
void launch_eig_diagonal(cudaStream_t st, const double* C, int ldc, int n, double* D, DevScalars* sc);

// constraints.cu
void launch_constraints_mean(cudaStream_t st, const double* mean, const double* shift, int n, int n_con, DevScalars* sc);
void launch_constraint_count(cudaStream_t st, const double* G, long long ldg, int lambda, int n_con, double* bounds, int set_bounds,
                             unsigned long long* viol, DevScalars* sc);
void launch_constraint_events(cudaStream_t st, const unsigned long long* viol, const unsigned char* indicator, long long ldg, int lambda,
                              int n_con, unsigned long long max_corrections, int* ev_sample, int* ev_con, int* vio_rows, int* counts_out,
                              DevScalars* sc);
void launch_constraint_normals(cudaStream_t st, const int* ev_sample, const int* ev_con, const int* counts, const double* Y, int ldy,
                               double* normal, int ldn, double lr, double* U, int ldu, int n, int n_con);
void launch_constraint_scale(cudaStream_t st, double* U, int ldu, int n, const int* ev_sample, const int* counts,
                             const unsigned long long* viol, double beta, int rows_padded);
void launch_caux(cudaStream_t st, const double* C, double* Caux, int ldc, const double* W, int ldw, int splits, int n, const int* counts);
void launch_constraint_recount(cudaStream_t st, const double* G, long long ldg, int n_con, const double* bounds, const int* rows,
                               const int* counts, int max_rows, unsigned long long* viol, unsigned char* indicator);
void launch_constraint_max(cudaStream_t st, const unsigned long long* viol, int lambda, const int* counts, DevScalars* sc);
void launch_add_resampled(cudaStream_t st, DevScalars* sc, const int* counts);

}  // namespace kc
