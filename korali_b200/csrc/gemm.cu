// gemm.cu — FP64 tensor-core (DMMA.8x8x4) GEMM kernels of the CMA-ES generation loop.
//
//  K2  gemm_tn : Y[M x Nc] = Z[M x K] * A[Nc x K]^T          (sampling product, CMAES.cpp.base:507-513:
//                y_i = B * (D o z_i) for all lambda samples at once; A = B*diag(D), both operands K-contiguous)
//  K6  syrk_tt : P[n x n]  = S^T S, S[K x n] n-contiguous     (rank-mu sum of adaptC, CMAES.cpp.base:703-704;
//                lower-triangular tiles only, split-K with a deterministic second-stage reduction)
//
// Version 1 staging: 16-byte cp.async (LDGSTS) into padded shared-memory tiles whose row stride is
// == 32 B (mod 128 B), which makes every LDS.64 fragment read of a half-warp hit 16 distinct bank pairs.

#include "common.cuh"
#include "kernels.h"

namespace kc {

namespace {
constexpr int BM = 128, BN = 128, BK = 16;
constexpr int THREADS = 256;
constexpr int STAGES = 4;
constexpr int PADK = BK + 4;   // TN tiles: [rows][PADK] doubles, 160 B stride
constexpr int PADN = BM + 4;   // TT tiles: [BK][PADN] doubles, 1056 B stride

__device__ __forceinline__ void store_pair(double* p, bool ok0, bool ok1, double c0, double c1) {
  if (ok1) {
    *reinterpret_cast<double2*>(p) = make_double2(c0, c1);
  } else if (ok0) {
    p[0] = c0;
  }
}
}  // namespace

// ------------------------------------------------------------------------------------------------
// C[M x Nc] = A[M x K] * B[Nc x K]^T ; lda/ldb/ldc even (16-byte aligned rows); pads must be zero.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(THREADS, 1)
gemm_tn_kernel(int M, int Nc, int K, const double* __restrict__ A, int lda, const double* __restrict__ B, int ldb,
               double* __restrict__ C, int ldc) {
  extern __shared__ __align__(16) double smem[];
  double* As = smem;                          // [STAGES][BM][PADK]
  double* Bs = smem + STAGES * BM * PADK;     // [STAGES][BN][PADK]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int wm = warp >> 2, wn = warp & 3;    // 2 x 4 warps, warp tile 64 x 32
  const int row0 = blockIdx.y * BM, col0 = blockIdx.x * BN;
  const int nk = (K + BK - 1) / BK;

  auto load_stage = [&](int stage, int kt) {
    const int k0 = kt * BK;
    double* as = As + stage * BM * PADK;
    double* bs = Bs + stage * BN * PADK;
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const int idx = tid + i * THREADS;
      const int r = idx >> 3, ch = idx & 7;
      const int gk = k0 + 2 * ch;
      {
        const int gr = row0 + r;
        const bool ok = (gr < M) && (gk < K);
        const double* src = ok ? (A + (size_t)gr * lda + gk) : A;
        cp_async16(as + r * PADK + 2 * ch, src, ok ? 16 : 0);
      }
      {
        const int gr = col0 + r;
        const bool ok = (gr < Nc) && (gk < K);
        const double* src = ok ? (B + (size_t)gr * ldb + gk) : B;
        cp_async16(bs + r * PADK + 2 * ch, src, ok ? 16 : 0);
      }
    }
  };

  double acc[8][4][2];
#pragma unroll
  for (int i = 0; i < 8; i++)
#pragma unroll
    for (int j = 0; j < 4; j++) acc[i][j][0] = acc[i][j][1] = 0.0;

#pragma unroll
  for (int s = 0; s < STAGES - 1; s++) {
    if (s < nk) load_stage(s, s);
    cp_async_commit();
  }

  for (int kt = 0; kt < nk; kt++) {
    cp_async_wait<STAGES - 2>();
    __syncthreads();
    {
      const int nxt = kt + STAGES - 1;
      if (nxt < nk) load_stage(nxt % STAGES, nxt);
      cp_async_commit();
    }
    const double* as = As + (kt % STAGES) * BM * PADK + (wm * 64 + g) * PADK + t;
    const double* bs = Bs + (kt % STAGES) * BN * PADK + (wn * 32 + g) * PADK + t;
#pragma unroll
    for (int kk = 0; kk < BK / 4; kk++) {
      double a[8], b[4];
#pragma unroll
      for (int i = 0; i < 8; i++) a[i] = as[i * 8 * PADK + kk * 4];
#pragma unroll
      for (int j = 0; j < 4; j++) b[j] = bs[j * 8 * PADK + kk * 4];
#pragma unroll
      for (int i = 0; i < 8; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
    }
  }
  cp_async_wait<0>();

#pragma unroll
  for (int i = 0; i < 8; i++) {
    const int row = row0 + wm * 64 + i * 8 + g;
    if (row >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const int col = col0 + wn * 32 + j * 8 + 2 * t;
      store_pair(C + (size_t)row * ldc + col, col < Nc, col + 1 < Nc, acc[i][j][0], acc[i][j][1]);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// W[split][n x ldw] (lower-triangular 128x128 tiles) = sum over this split's k-range of S[k][d]*S[k][e].
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(THREADS, 1)
syrk_tt_kernel(int n, int K, const int* __restrict__ kptr, const double* __restrict__ S, int lds, double* __restrict__ W, int ldw) {
  if (kptr) K = min(K, *kptr);   // actual number of operand rows, known only on the device (selected samples of this rank)
  extern __shared__ __align__(16) double smem[];
  double* Sa = smem;                          // [STAGES][BK][PADN]
  double* Sb = smem + STAGES * BK * PADN;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int wm = warp >> 2, wn = warp & 3;
  // linear lower-triangular tile id -> (bi >= bj)
  int bi = (int)((sqrt(8.0 * (double)blockIdx.x + 1.0) - 1.0) * 0.5);
  while ((bi + 1) * (bi + 2) / 2 <= (int)blockIdx.x) bi++;
  while (bi * (bi + 1) / 2 > (int)blockIdx.x) bi--;
  const int bj = blockIdx.x - bi * (bi + 1) / 2;
  const bool diag = (bi == bj);
  const int d0 = bi * BM, e0 = bj * BN;
  const int nk_total = (K + BK - 1) / BK;
  const int ktiles_per_split = (nk_total + (int)gridDim.y - 1) / (int)gridDim.y;
  const int kt_begin = blockIdx.y * ktiles_per_split;
  const int kt_end = min(nk_total, kt_begin + ktiles_per_split);
  const int nk = max(0, kt_end - kt_begin);

  auto load_stage = [&](int stage, int kt) {
    const int k0 = (kt_begin + kt) * BK;
    double* sa = Sa + stage * BK * PADN;
    double* sb = Sb + stage * BK * PADN;
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const int idx = tid + i * THREADS;
      const int r = idx >> 6, ch = idx & 63;
      const int gk = k0 + r;
      {
        const int gc = d0 + 2 * ch;
        const bool ok = (gk < K) && (gc < n);
        const double* src = ok ? (S + (size_t)gk * lds + gc) : S;
        cp_async16(sa + r * PADN + 2 * ch, src, ok ? 16 : 0);
      }
      if (!diag) {
        const int gc = e0 + 2 * ch;
        const bool ok = (gk < K) && (gc < n);
        const double* src = ok ? (S + (size_t)gk * lds + gc) : S;
        cp_async16(sb + r * PADN + 2 * ch, src, ok ? 16 : 0);
      }
    }
  };

  double acc[8][4][2];
#pragma unroll
  for (int i = 0; i < 8; i++)
#pragma unroll
    for (int j = 0; j < 4; j++) acc[i][j][0] = acc[i][j][1] = 0.0;

#pragma unroll
  for (int s = 0; s < STAGES - 1; s++) {
    if (s < nk) load_stage(s, s);
    cp_async_commit();
  }
  for (int kt = 0; kt < nk; kt++) {
    cp_async_wait<STAGES - 2>();
    __syncthreads();
    {
      const int nxt = kt + STAGES - 1;
      if (nxt < nk) load_stage(nxt % STAGES, nxt);
      cp_async_commit();
    }
    const double* sa = Sa + (kt % STAGES) * BK * PADN + t * PADN + wm * 64 + g;
    const double* sb = (diag ? Sa : Sb) + (kt % STAGES) * BK * PADN + t * PADN + wn * 32 + g;
#pragma unroll
    for (int kk = 0; kk < BK / 4; kk++) {
      double a[8], b[4];
#pragma unroll
      for (int i = 0; i < 8; i++) a[i] = sa[kk * 4 * PADN + i * 8];
#pragma unroll
      for (int j = 0; j < 4; j++) b[j] = sb[kk * 4 * PADN + j * 8];
#pragma unroll
      for (int i = 0; i < 8; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
    }
  }
  cp_async_wait<0>();

  double* Wp = W + (size_t)blockIdx.y * n * ldw;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    const int row = d0 + wm * 64 + i * 8 + g;
    if (row >= n) continue;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const int col = e0 + wn * 32 + j * 8 + 2 * t;
      store_pair(Wp + (size_t)row * ldw + col, col < n, col + 1 < n, acc[i][j][0], acc[i][j][1]);
    }
  }
}

// ---- host launchers ------------------------------------------------------------------------------
static std::atomic<unsigned long long> g_attr_set{0};
static void ensure_attrs() {
  if (!first_call_on_device(g_attr_set)) return;
  cudaFuncSetAttribute(gemm_tn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gemm_tn_smem_bytes());
  cudaFuncSetAttribute(syrk_tt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)syrk_tt_smem_bytes());
}

size_t gemm_tn_smem_bytes() { return sizeof(double) * STAGES * (BM + BN) * PADK; }
size_t syrk_tt_smem_bytes() { return sizeof(double) * STAGES * 2 * BK * PADN; }

void launch_gemm_tn(cudaStream_t st, int M, int Nc, int K, const double* A, int lda, const double* B, int ldb,
                    double* C, int ldc) {
  if (M <= 0 || Nc <= 0) return;
  if (launch_gemm_tn_tma(st, M, Nc, K, A, lda, B, ldb, C, ldc)) return;   // the cp.async kernel when no tensor map can be built
  ensure_attrs();
  dim3 grid((Nc + BN - 1) / BN, (M + BM - 1) / BM);
  gemm_tn_kernel<<<grid, THREADS, gemm_tn_smem_bytes(), st>>>(M, Nc, K, A, lda, B, ldb, C, ldc);
}

int syrk_tiles(int n) {
  const int nb = (n + BM - 1) / BM;
  return nb * (nb + 1) / 2;
}

int syrk_pick_splits(int n, int K, int num_sms, int max_splits) {
  // one CTA per SM: minimise (waves of CTAs) x (k-tiles per CTA); ties -> fewer splits (less reduction traffic)
  const int tiles = syrk_tiles(n);
  const int nk = (K + BK - 1) / BK;
  int best = 1;
  long long best_cost = -1;
  for (int s = 1; s <= max_splits && s <= (nk > 0 ? nk : 1); s++) {
    const long long waves = ((long long)tiles * s + num_sms - 1) / num_sms;
    const long long per = (nk + s - 1) / s;
    const long long cost = waves * (per + 6);  // +6: pipeline fill / epilogue of a CTA in k-tile units
    if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = s; }
  }
  return best;
}

void launch_syrk_tt(cudaStream_t st, int n, int K, const int* kptr, const double* S, int lds, long long s_rows, double* W, int ldw,
                    int splits) {
  if (launch_syrk_tt_tma(st, n, K, kptr, S, lds, s_rows, W, ldw, splits)) return;
  ensure_attrs();
  dim3 grid(syrk_tiles(n), splits);
  syrk_tt_kernel<<<grid, THREADS, syrk_tt_smem_bytes(), st>>>(n, K, kptr, S, lds, W, ldw);
}

// The rank-mu product with the scheduling chosen here: stream-K over the triangular tiles (gemm_tma.cu), or the split-K kernels when
// the TMA path is unavailable. Returns the number of slabs of W to sum.
int launch_syrk(cudaStream_t st, int n, int K, const int* kptr, const double* S, int lds, long long s_rows, double* W, int ldw,
                int expect_rows, int num_sms, int max_splits) {
  const int parts = launch_syrk_sk_tma(st, n, K, kptr, S, lds, s_rows, W, ldw, num_sms, max_splits);
  if (parts > 0) return parts;
  const int splits = syrk_pick_splits(n, expect_rows, num_sms, max_splits);
  launch_syrk_tt(st, n, K, kptr, S, lds, s_rows, W, ldw, splits);
  return splits;
}

}  // namespace kc
