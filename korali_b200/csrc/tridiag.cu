// tridiag.cu — K8b: symmetric eigendecomposition by Householder tridiagonalisation + divide & conquer + compact-WY
// back-transform (the default eigensolver above N = 24). Replaces eigen() (CMAES.cpp.base:896-938: gsl_eigen_symmv is the same
// three stages with a QL iteration in the middle); DESIGN.md section 6.
//
//   stage 1  sytrd_kernel     C = Q T Q^T. ONE persistent cooperative launch, one CTA per SM; CTA b owns the columns
//                             b, b+G, b+2G, ... of the (symmetric) trailing matrix — in SHARED MEMORY up to N ~ 1600 — and
//                             the N-1 dependent Householder steps cost ONE all-to-all exchange each:
//                               receive  p = A v (every CTA's slice) and the next column (from its owner)
//                               every CTA redundantly: w = tau p - (tau^2 p.v / 2) v, the column's own rank-2 update, the
//                                         next reflector (v', tau')            [bitwise identical on all CTAs]
//                               one pass over the CTA's columns: A -= v w^T + w v^T, then p' = A v'; publish.
//                             The exchange is an LL protocol (value + step tag in one 16-byte store/load, double-buffered by
//                             step parity): no fence, no flag, no grid barrier.
//   stage 2  dc_solve         T = Z diag(lam) Z^T (dc.cu)
//   stage 3  back-transform   X^T = Z^T H_{N-3} ... H_0 with compact-WY panels (I - V T V^T) of nb reflectors: the panel
//                             factors T_p and T_p V_p^T come from three batched launches that do not depend on Z; each
//                             panel is then two tensor-core GEMMs, W = X^T (T_p V_p^T)^T (split-K) and X^T -= W V_p^T.
// NumPy statement of all three stages: profiles/microbench/tridiag_dc_proto.py.
#include <algorithm>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "tridiag.h"

namespace kc {

void launch_transpose(cudaStream_t st, const double* in, double* out, int ld, int n);   // dc.cu

namespace {

constexpr int SY_NT = 256;
constexpr int SY_NW = SY_NT / 32;
constexpr size_t kSmemCap = 227 * 1024 - 1024;

struct __align__(16) LL { double v; unsigned long long tag; };
#ifdef KC_LL_GPU_SCOPE
#define KC_LL_ST "st.relaxed.gpu.global"
#define KC_LL_LD "ld.relaxed.gpu.global"
#else
#define KC_LL_ST "st.volatile.global"
#define KC_LL_LD "ld.volatile.global"
#endif

__device__ __forceinline__ void ll_store(LL* p, double v, unsigned long long tag) {
  asm volatile(KC_LL_ST ".v2.u64 [%0], {%1, %2};" ::"l"(p), "l"((unsigned long long)__double_as_longlong(v)), "l"(tag) : "memory");
}
__device__ __forceinline__ double ll_wait(const LL* p, unsigned long long tag) {
  unsigned long long a, b;
  do {
    asm volatile(KC_LL_LD ".v2.u64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "l"(p) : "memory");
  } while (b != tag);
  return __longlong_as_double((long long)a);
}

__device__ __forceinline__ void ll_load(const LL* p, unsigned long long& a, unsigned long long& b) {
  asm volatile(KC_LL_LD ".v2.u64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "l"(p) : "memory");
}

// Sum over the block, identical bits in every thread (and in every CTA: same thread count, same order). ONE barrier: `slot`
// (SY_NW doubles) must not be rewritten before every thread has read it — the caller alternates four slots (2 sums x step parity),
// so a slot is reused two steps (six barriers) later.
__device__ __forceinline__ double block_sum(double v, double* slot) {
  v = warp_sum_butterfly(v);
  if ((threadIdx.x & 31) == 0) slot[threadIdx.x >> 5] = v;
  __syncthreads();
  double s = 0.0;
#pragma unroll
  for (int k = 0; k < SY_NW; k++) s += slot[k];
  return s;
}

// The two element formulas of a step, with explicit roundings: they are evaluated per row by the row's thread AND for rows i, i+1
// by every thread (scalars), and both must give the same bits.
__device__ __forceinline__ double w_of(double tau, double p, double alpha, double v) { return __fma_rn(tau, p, __dmul_rn(alpha, v)); }
__device__ __forceinline__ double col_upd(double c, double v, double wi, double w, double vi) {
  return __dsub_rn(c, __fma_rn(v, wi, __dmul_rn(w, vi)));
}

// One column of the trailing matrix in the pass of a step: rank-2 update of the previous step, product with the new reflector,
// optional publication (LL stores) of the updated column. Two rows per lane and access (16-byte shared / global accesses), PU
// independent accesses in flight per lane; rows [rs, ne) with rs = (i+1) rounded down to even (row i is dead data: it is updated
// along, its reflector entry is zero) and ne = n rounded up to even (zero pads). The same code and summation order for the
// shared-memory and the global-memory variant: their results are bitwise equal.
constexpr int PU = 8;
template <bool PUB>
__device__ __forceinline__ double pass_column(double* __restrict__ col, const double* __restrict__ vold, const double* __restrict__ wv,
                                              const double* __restrict__ vnew, double wc, double vc, int i, int ne, int n, int lane,
                                              LL* __restrict__ Cout, unsigned long long otag) {
  double dot[PU];
#pragma unroll
  for (int u = 0; u < PU; u++) dot[u] = 0.0;
  int r = ((i + 1) & ~1) + 2 * lane;
  for (; r + 64 * (PU - 1) < ne; r += 64 * PU) {
    double2 a[PU];
#pragma unroll
    for (int u = 0; u < PU; u++) a[u] = *reinterpret_cast<const double2*>(col + r + 64 * u);
#pragma unroll
    for (int u = 0; u < PU; u++) {
      const double2 vo = *reinterpret_cast<const double2*>(vold + r + 64 * u);
      const double2 w2 = *reinterpret_cast<const double2*>(wv + r + 64 * u);
      const double2 vn = *reinterpret_cast<const double2*>(vnew + r + 64 * u);
      a[u].x -= vo.x * wc + w2.x * vc;
      a[u].y -= vo.y * wc + w2.y * vc;
      *reinterpret_cast<double2*>(col + r + 64 * u) = a[u];
      dot[u] += a[u].x * vn.x;
      dot[u] += a[u].y * vn.y;
      if (PUB) {
        if (r + 64 * u > i) ll_store(Cout + r + 64 * u, a[u].x, otag);
        if (r + 64 * u + 1 < n) ll_store(Cout + r + 64 * u + 1, a[u].y, otag);
      }
    }
  }
#pragma unroll
  for (int u = 0; u < PU; u++) {
    const int q = r + 64 * u;
    if (q < ne) {
      double2 a = *reinterpret_cast<const double2*>(col + q);
      const double2 vo = *reinterpret_cast<const double2*>(vold + q);
      const double2 w2 = *reinterpret_cast<const double2*>(wv + q);
      const double2 vn = *reinterpret_cast<const double2*>(vnew + q);
      a.x -= vo.x * wc + w2.x * vc;
      a.y -= vo.y * wc + w2.y * vc;
      *reinterpret_cast<double2*>(col + q) = a;
      dot[u] += a.x * vn.x;
      dot[u] += a.y * vn.y;
      if (PUB) {
        if (q > i) ll_store(Cout + q, a.x, otag);
        if (q + 1 < n) ll_store(Cout + q + 1, a.y, otag);
      }
    }
  }
  return ((dot[0] + dot[1]) + (dot[2] + dot[3])) + ((dot[4] + dot[5]) + (dot[6] + dot[7]));
}

// A step of thread t works on the rows r = t (mod SY_NT), r >= i, in every phase, so the received column (cs), the received
// product (ps) and the reflector entries are thread-private although they live in shared memory: three block-wide barriers per
// step (the two sums and the one in front of the pass over the columns).
__global__ void __launch_bounds__(SY_NT, 1)
sytrd_kernel(const double* __restrict__ M, double* __restrict__ Awork, int ld, int n, int ns /* smem vector stride */,
             LL* __restrict__ xP, LL* __restrict__ xC, double* __restrict__ dT, double* __restrict__ eT, double* __restrict__ tauv,
             double* __restrict__ VR, long long* __restrict__ prof, int prof_step0, int prof_cta) {
  extern __shared__ __align__(16) double sm[];
  const int G = gridDim.x, b = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  double* vold = sm;
  double* vnew = sm + ns;
  double* wv = sm + 2 * ns;
  double* ps = sm + 3 * ns;
  double* cs = sm + 4 * ns;
  double* red = sm + 5 * ns;       // 4 slots x SY_NW doubles
  double* bc = red + 32;           // 2 parities x {c_i, p_i, c_{i+1}, p_{i+1}}
  const int nloc = b < n ? (n - b + G - 1) / G : 0;
  for (int r = tid; r < ns; r += SY_NT) { vold[r] = 0.0; vnew[r] = 0.0; wv[r] = 0.0; ps[r] = 0.0; }
  if (b == 0) {   // owner of column 0 publishes it for step 0
    const double* src = M;
    for (int r = tid; r < n; r += SY_NT) ll_store(xC + r, src[r], 1ull);
  }
  __syncthreads();
  double tau_old = 0.0;
  for (int i = 0; i < n; i++) {
    const int par = i & 1;
    const unsigned long long tag = (unsigned long long)i + 1ull;
    const LL* Pin = xP + (size_t)par * n;
    const LL* Cin = xC + (size_t)par * n;
    const bool have_p = i > 0;
    const bool pr = prof && b == prof_cta && tid == 0 && i >= prof_step0 && i < prof_step0 + 32;
    if (pr) prof[(i - prof_step0) * 8 + 0] = clock64();
    const int r0 = i + ((tid - i) & (SY_NT - 1));   // first row >= i of this thread
    // ---- receive column i and p = A v_{i-1}. One lane per warp spins on ONE slot first (148 CTAs x 256 threads x 8 slots of
    // back-to-back polling saturate the L2 and delay the very stores they wait for); then up to 8 slots are polled together, so
    // that their L2 round trips overlap — nearly always a single round.
    if (have_p) {
      if (lane == 0 && r0 < n) (void)ll_wait(Pin + r0, tag);
      __syncwarp();
    }
    for (int rb = r0; rb < n; rb += 4 * SY_NT) {
      unsigned long long va[8], ta[8];
      unsigned pend = 0;
#pragma unroll
      for (int k = 0; k < 4; k++)
        if (rb + k * SY_NT < n) pend |= (1u << k) | (have_p ? (16u << k) : 0u);
      const unsigned want = pend;
      while (pend) {
#pragma unroll
        for (int k = 0; k < 4; k++) {
          if (pend & (1u << k)) ll_load(Cin + rb + k * SY_NT, va[k], ta[k]);
          if (pend & (16u << k)) ll_load(Pin + rb + k * SY_NT, va[4 + k], ta[4 + k]);
        }
#pragma unroll
        for (int k = 0; k < 8; k++)
          if ((pend >> k & 1u) && ta[k] == tag) pend &= ~(1u << k);
      }
#pragma unroll
      for (int k = 0; k < 4; k++) {
        if (want & (1u << k)) cs[rb + k * SY_NT] = __longlong_as_double((long long)va[k]);
        if (want & (16u << k)) ps[rb + k * SY_NT] = __longlong_as_double((long long)va[4 + k]);
      }
    }
    if (pr) prof[(i - prof_step0) * 8 + 1] = clock64();
    // ---- p.v (own rows), the four scalars every thread needs
    double part = 0.0;
    if (have_p)
      for (int r = r0; r < n; r += SY_NT) part = __fma_rn(ps[r], vold[r], part);
    double* bcp = bc + par * 4;
    if (tid == (i & (SY_NT - 1))) { bcp[0] = cs[i]; bcp[1] = ps[i]; }
    if (i + 1 < n && tid == ((i + 1) & (SY_NT - 1))) { bcp[2] = cs[i + 1]; bcp[3] = ps[i + 1]; }
    const double pv = block_sum(part, red + (par * 2 + 0) * SY_NW);
    const double alpha = -0.5 * tau_old * (tau_old * pv);
    const double vi = vold[i];
    const double wi = w_of(tau_old, bcp[1], alpha, vi);
    // ---- w = tau p + alpha v and the column's own rank-2 update, own rows
    double xpart = 0.0;
    for (int r = r0; r < n; r += SY_NT) {
      const double v = vold[r];
      const double w = w_of(tau_old, ps[r], alpha, v);
      wv[r] = w;
      const double c = col_upd(cs[r], v, wi, w, vi);
      cs[r] = c;
      if (r >= i + 2) xpart = __fma_rn(c, c, xpart);
    }
    const double di = col_upd(bcp[0], vi, wi, wi, vi);
    if (i == n - 1) {
      if (b == 0 && tid == 0) dT[i] = di;
      break;
    }
    const double vi1 = vold[i + 1];
    const double alph = col_upd(bcp[2], vi1, wi, w_of(tau_old, bcp[3], alpha, vi1), vi);
    const double xn2 = block_sum(xpart, red + (par * 2 + 1) * SY_NW);
    double tau = 0.0, scale = 0.0, ei = alph;
    if (xn2 > 0.0) {
      const double beta = -copysign(sqrt(alph * alph + xn2), alph);
      tau = (beta - alph) / beta;
      scale = 1.0 / (alph - beta);
      ei = beta;
    }
    if (r0 == i) vnew[i] = 0.0;   // row i rides along in the pass when i+1 is odd (16-byte accesses): it must not enter the product
    for (int r = (r0 > i ? r0 : r0 + SY_NT); r < n; r += SY_NT) vnew[r] = (r == i + 1) ? 1.0 : cs[r] * scale;
    if (b == i % G && tid == 0) { dT[i] = di; eT[i] = ei; tauv[i] = tau; }   // the owner of the retired column records the step
    __syncthreads();
    if (pr) prof[(i - prof_step0) * 8 + 2] = clock64();
    // one pass over this CTA's columns c >= i+1: rank-2 update of step i-1, then p = A v_new; the owner of column i+1 publishes it
    LL* Pout = xP + (size_t)(par ^ 1) * n;
    LL* Cout = xC + (size_t)(par ^ 1) * n;
    const unsigned long long otag = tag + 1ull;
    const int s0 = (i + 1 > b) ? (i + 1 - b + G - 1) / G : 0;
    for (int s = s0 + warp; s < nloc; s += SY_NW) {
      const int c = b + s * G;
      double* col = Awork + (size_t)c * ld;
      const double wc = wv[c], vc = vold[c];
      double dot = (c == i + 1) ? pass_column<true>(col, vold, wv, vnew, wc, vc, i, ns, n, lane, Cout, otag)
                                : pass_column<false>(col, vold, wv, vnew, wc, vc, i, ns, n, lane, Cout, otag);
      dot = warp_sum_butterfly(dot);
      if (lane == 0) ll_store(Pout + c, dot, otag);
    }
    if (pr) prof[(i - prof_step0) * 8 + 3] = clock64();
    if (b == i % G) {   // reflector i for the back-transform: off the critical path (the other CTAs' products are in flight meanwhile)
      double* vr = VR + (size_t)i * ld;       // entries r <= i and r >= n stay zero from the allocation: no step ever writes them
      for (int r = i + 1 + tid; r < n; r += SY_NT) vr[r] = vnew[r];
    }
    double* t = vold; vold = vnew; vnew = t;
    tau_old = tau;
    // no barrier here: the pass reads vold / vnew / wv only; the next step writes its thread-private cs / ps rows first and reaches
    // wv and the other v buffer only behind the barrier of its first sum, which every warp passes after leaving this loop
  }
}

// ---- register-resident variant (N <= 1536) -----------------------------------------------------------------------------------
// The 148 register files hold 37 MB: the trailing matrix lives in REGISTERS. Thread t owns the row pairs (2u, 2u+1), u = t + 256 k
// (k < KU), in every phase: it receives their entries of the column and of p = A v (one 256-bit load per pair of LL slots), keeps
// their entries of the reflectors and of w, and holds the entries A[r][c] of all NC columns of its CTA for its rows. A pass over
// the columns is then register arithmetic (the shared-memory variant moved 250 KB per step through the 128 B/clk shared-memory
// pipe); shared memory only carries what is looked up by COLUMN index (w[c], v[c]) and the per-thread partial products.
__device__ __forceinline__ void ll_load2(const LL* p, unsigned long long (&q)[4]) {
  asm volatile(KC_LL_LD ".v4.u64 {%0, %1, %2, %3}, [%4];" : "=l"(q[0]), "=l"(q[1]), "=l"(q[2]), "=l"(q[3]) : "l"(p) : "memory");
}

template <int KU, int NC>
__global__ void __launch_bounds__(SY_NT, 1)
sytrd_reg_kernel(const double* __restrict__ M, int ld, int n, int ns /* n rounded up to even: LL stride per parity, vector stride */,
                 LL* __restrict__ xP, LL* __restrict__ xC, double* __restrict__ dT, double* __restrict__ eT, double* __restrict__ tauv,
                 double* __restrict__ VR, long long* __restrict__ prof, int prof_step0, int prof_cta, int opt, int copies) {
  extern __shared__ __align__(16) double sm[];
  const int G = gridDim.x, b = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  double* vs_old = sm;             // reflector v_{i-1} by index (lookups v[c], v[i+1])
  double* vs_new = sm + ns;
  double* wsm = sm + 2 * ns;       // w_{i-1} by index (lookups w[c])
  double* red = sm + 3 * ns;       // 4 slots x SY_NW
  double* bc = red + 64;           // 2 parities x {c_i, p_i, c_{i+1}, p_{i+1}}
  double* pp = red + 80;           // NC x SY_NT partial products of the pass
  const int nloc = b < n ? (n - b + G - 1) / G : 0;
  double A[KU][NC][2], v[2 * KU], w[2 * KU], vnw[2 * KU];
#pragma unroll
  for (int k = 0; k < KU; k++) {
    const int r = 2 * (tid + SY_NT * k);
#pragma unroll
    for (int s = 0; s < NC; s++) {
      const double* src = M + (size_t)(b + s * G) * ld;   // column c of a symmetric matrix = its row c
      A[k][s][0] = (s < nloc && r < n) ? src[r] : 0.0;
      A[k][s][1] = (s < nloc && r + 1 < n) ? src[r + 1] : 0.0;
    }
    v[2 * k] = v[2 * k + 1] = w[2 * k] = w[2 * k + 1] = vnw[2 * k] = vnw[2 * k + 1] = 0.0;
  }
  for (int r = tid; r < ns; r += SY_NT) { vs_old[r] = 0.0; vs_new[r] = 0.0; wsm[r] = 0.0; }
  // Every slot exists `copies` times (stride cstride): all CTAs poll the same 2 n slots, and 148 requests per 128-byte line and
  // polling round serialise in the L2 slice that owns the line; CTA b reads copy b % copies, the producers write all copies.
  const size_t cstride = 4 * (size_t)ns;
  // (`copies` packs two counts: bits 0-7 for the column slots, bits 8-15 for the product slots when they differ — the column costs its
  // owner n stores per copy, a product entry one)
  const int ccop = copies & 255, pcop = (copies >> 8) ? (copies >> 8) : ccop;
  const size_t my_copy = (size_t)(b % ccop) * cstride, my_copy_p = (size_t)(b % pcop) * cstride;
  if (b == 0)   // owner of column 0 publishes it for step 0
    for (int r = tid; r < n; r += SY_NT)
      for (int q = 0; q < ccop; q++) ll_store(xC + q * cstride + r, M[r], 1ull);
  __syncthreads();
  double tau_old = 0.0;
  for (int i = 0; i < n; i++) {
    const int par = i & 1;
    const unsigned long long tag = (unsigned long long)i + 1ull;
    const LL* Pin = xP + my_copy_p + (size_t)par * ns;
    const LL* Cin = xC + my_copy + (size_t)par * ns;
    const bool have_p = i > 0;
    const bool pr = prof && b == prof_cta && tid == 0 && i >= prof_step0 && i < prof_step0 + 32;
    if (pr) prof[(i - prof_step0) * 8 + 0] = clock64();
    // ---- receive column i and p = A v_{i-1} for this thread's rows >= i
    double cv[2 * KU], pq[2 * KU];
    unsigned need = 0;
#pragma unroll
    for (int j = 0; j < 2 * KU; j++) {
      const int r = 2 * (tid + SY_NT * (j >> 1)) + (j & 1);
      if (r >= i && r < n) need |= 1u << j;
      cv[j] = 0.0; pq[j] = 0.0;
    }
    if (have_p && (opt & 4)) {
      // Gate: a few lanes spin on ONE slot per producer — the products of the last G columns (every CTA that still owns a column
      // publishes exactly one of them), plus the last row of the column when it travels in this step — and only then does the
      // block read its 2 x 16 KB of slots, once. A round of everybody polling everything is ~1000 cycles of L2 traffic
      // (148 CTAs x 32 KB) that the late producers' stores queue behind (profiles/r02_pf_stamps.log).
      const int lo = max(i, n - G) & ~1;
      const int npairs = (ns - lo) >> 1;
      if (tid < npairs) {
        const int r0 = lo + 2 * tid;
        const bool n0 = r0 >= i && r0 < n, n1 = r0 + 1 < n;
        unsigned long long q[4];
        do { ll_load2(Pin + r0, q); } while ((n0 && q[1] != tag) || (n1 && q[3] != tag));
      } else if (tid == SY_NT - 1) {
        unsigned long long q[4];
        const bool n0 = ns - 2 >= i, n1 = ns - 1 < n;
        do { ll_load2(Cin + ns - 2, q); } while ((n0 && q[1] != tag) || (n1 && q[3] != tag));
      }
      __syncthreads();
    } else if (have_p && (opt & 1)) {   // one lane per warp spins on one slot first: 148 x 256 threads polling everything back to back saturate the L2
      if (lane == 0 && need) {
        const int j0 = __ffs(need) - 1;
        (void)ll_wait(Pin + 2 * (tid + SY_NT * (j0 >> 1)) + (j0 & 1), tag);
      }
      __syncwarp();
    }
    unsigned pc = need, ppn = have_p ? need : 0u;
    while (pc | ppn) {
      unsigned long long qc[KU][4], qp[KU][4];
#pragma unroll
      for (int k = 0; k < KU; k++) {
        if ((pc >> (2 * k)) & 3u) ll_load2(Cin + 2 * (tid + SY_NT * k), qc[k]);
        if ((ppn >> (2 * k)) & 3u) ll_load2(Pin + 2 * (tid + SY_NT * k), qp[k]);
      }
#pragma unroll
      for (int k = 0; k < KU; k++)
#pragma unroll
        for (int h = 0; h < 2; h++) {
          const unsigned bit = 1u << (2 * k + h);
          if ((pc & bit) && qc[k][2 * h + 1] == tag) { cv[2 * k + h] = __longlong_as_double((long long)qc[k][2 * h]); pc &= ~bit; }
          if ((ppn & bit) && qp[k][2 * h + 1] == tag) { pq[2 * k + h] = __longlong_as_double((long long)qp[k][2 * h]); ppn &= ~bit; }
        }
    }
    if (pr) prof[(i - prof_step0) * 8 + 1] = clock64();
    // ---- p.v over the own rows; the four scalars every thread needs
    double part = 0.0;
    double* bcp = bc + par * 4;
#pragma unroll
    for (int j = 0; j < 2 * KU; j++) {
      const int r = 2 * (tid + SY_NT * (j >> 1)) + (j & 1);
      if (need & (1u << j)) part = __fma_rn(pq[j], v[j], part);
      if (r == i) { bcp[0] = cv[j]; bcp[1] = pq[j]; }
      if (r == i + 1 && r < n) { bcp[2] = cv[j]; bcp[3] = pq[j]; }
    }
    const double pv = block_sum(part, red + (par * 2 + 0) * SY_NW);
    const double alpha = -0.5 * tau_old * (tau_old * pv);
    const double vi = vs_old[i];
    const double wi = w_of(tau_old, bcp[1], alpha, vi);
    double xpart = 0.0;
#pragma unroll
    for (int j = 0; j < 2 * KU; j++) {
      const int r = 2 * (tid + SY_NT * (j >> 1)) + (j & 1);
      if (need & (1u << j)) {
        w[j] = w_of(tau_old, pq[j], alpha, v[j]);
        wsm[r] = w[j];
        cv[j] = col_upd(cv[j], v[j], wi, w[j], vi);
        if (r >= i + 2) xpart = __fma_rn(cv[j], cv[j], xpart);
      } else {
        w[j] = 0.0;
      }
    }
    const double di = col_upd(bcp[0], vi, wi, wi, vi);
    if (i == n - 1) {
      if (b == 0 && tid == 0) dT[i] = di;
      break;
    }
    const double vi1 = vs_old[i + 1];
    const double alph = col_upd(bcp[2], vi1, wi, w_of(tau_old, bcp[3], alpha, vi1), vi);
    const double xn2 = block_sum(xpart, red + (par * 2 + 1) * SY_NW);
    double tau = 0.0, scale = 0.0, ei = alph;
    if (xn2 > 0.0) {
      const double beta = -copysign(sqrt(alph * alph + xn2), alph);
      tau = (beta - alph) / beta;
      scale = 1.0 / (alph - beta);
      ei = beta;
    }
#pragma unroll
    for (int j = 0; j < 2 * KU; j++) {
      const int r = 2 * (tid + SY_NT * (j >> 1)) + (j & 1);
      vnw[j] = (r == i + 1) ? 1.0 : ((r >= i + 2 && r < n) ? cv[j] * scale : 0.0);
      if (r < ns) vs_new[r] = vnw[j];
    }
    if (b == i % G && tid == 0) { dT[i] = di; eT[i] = ei; tauv[i] = tau; }   // the owner of the retired column records the step
    // no barrier here: wsm (read by column index in the pass) was written in front of the second block sum's barrier, and vs_new
    // is first read — as vs_old — behind the first block sum's barrier of the next step
    if (pr) prof[(i - prof_step0) * 8 + 2] = clock64();
    // ---- pass over this CTA's columns c >= i+1 (registers): rank-2 update of step i-1, partial p = A v_i, publication of column i+1
    LL* Pout = xP + (size_t)(par ^ 1) * ns;
    LL* Cout = xC + (size_t)(par ^ 1) * ns;
    const unsigned long long otag = tag + 1ull;
    const int s0 = (i + 1 > b) ? (i + 1 - b + G - 1) / G : 0;
#pragma unroll
    for (int s = 0; s < NC; s++) {
      if (s >= s0 && s < nloc) {
        const int c = b + s * G;
        const double wc = wsm[c], vc = vs_old[c];
        double dot = 0.0;
#pragma unroll
        for (int k = 0; k < KU; k++) {
          double a0 = A[k][s][0], a1 = A[k][s][1];
          a0 = __fma_rn(-w[2 * k], vc, __fma_rn(-v[2 * k], wc, a0));              // two dependent DFMA instead of DMUL, DFMA, DADD
          a1 = __fma_rn(-w[2 * k + 1], vc, __fma_rn(-v[2 * k + 1], wc, a1));
          A[k][s][0] = a0; A[k][s][1] = a1;
          dot = __fma_rn(a0, vnw[2 * k], dot);
          dot = __fma_rn(a1, vnw[2 * k + 1], dot);
          if (c == i + 1) {
            const int r = 2 * (tid + SY_NT * k);
            for (int q = 0; q < ccop; q++) {
              if (r > i && r < n) ll_store(Cout + q * cstride + r, a0, otag);
              if (r + 1 > i && r + 1 < n) ll_store(Cout + q * cstride + r + 1, a1, otag);
            }
          }
        }
        pp[s * SY_NT + tid] = dot;
      }
    }
    __syncthreads();
    for (int s = warp; s < NC; s += SY_NW)   // a warp finishes column s: 256 partials in a fixed order
      if (s >= s0 && s < nloc) {
        double x = 0.0;
#pragma unroll
        for (int j = 0; j < SY_NW; j++) x += pp[s * SY_NT + lane + 32 * j];
        x = warp_sum_butterfly(x);
        if (lane < pcop) ll_store(Pout + lane * cstride + b + s * G, x, otag);
      }
    if (pr) prof[(i - prof_step0) * 8 + 3] = clock64();
    if (b == i % G) {   // reflector i for the back-transform (entries r <= i and r >= n stay zero from the allocation)
      double* vr = VR + (size_t)i * ld;
#pragma unroll
      for (int j = 0; j < 2 * KU; j++) {
        const int r = 2 * (tid + SY_NT * (j >> 1)) + (j & 1);
        if (r > i && r < n) vr[r] = vnw[j];
      }
    }
#pragma unroll
    for (int j = 0; j < 2 * KU; j++) v[j] = vnw[j];
    double* t = vs_old; vs_old = vs_new; vs_new = t;
    tau_old = tau;
  }
}

// (A single-CTA variant for N <= 128 — the whole matrix in the registers of one CTA, no exchange, four block barriers per step — was
// built and measured at N = 100: 0.338 ms against 0.294 ms for the 25-CTA exchange kernel (profiles/r02_eigen_ab13.log); not kept.)
// ---- compact-WY panel factor (dlarft, forward / columnwise): T upper triangular, nb x nb, from G = V^T V and tau ------------
// T is the inverse of the upper triangular S = striu(G) + diag(1 / tau) (the column recurrence of dlarft,
// T[0:p, p] = -tau_p T[0:p, 0:p] G[0:p, p], is the column-by-column inverse of S), so column j follows from S t_j = e_j by back
// substitution on its own:
//   t_jj = tau_j,   t_ij = -tau_i sum_{k = i+1 .. j} G_ik t_kj   (i = j-1 .. 0).
// One WARP per column (lane l keeps t_k for k = l mod 32), rows of G prefetched four steps ahead: nb dependent steps of one shuffle
// reduction each. (The column recurrence with one CTA per panel, nb block-wide steps of two barriers each, took 0.20 ms instead of
// ~0.02 ms per decomposition at N = 1000.)
// tau_j = 0 (H_j = I) gives a zero row and column like the recurrence does. Needs nb <= 128, nb % 32 == 0.
__global__ void __launch_bounds__(256)
larft_cols_kernel(const double* __restrict__ Gbuf, const double* __restrict__ tauv, int n_refl, int nb, double* __restrict__ Tbuf) {
  const int panel = blockIdx.y, lane = threadIdx.x & 31;
  const int j = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (j >= nb) return;
  const int p0 = panel * nb, kb = min(nb, n_refl - p0);
  const double* __restrict__ G = Gbuf + (size_t)panel * nb * nb;
  double* __restrict__ T = Tbuf + (size_t)panel * nb * nb;
  double t[4] = {0.0, 0.0, 0.0, 0.0};
  if (j < kb) {
    constexpr int PF = 4;
    double g[PF][4];
    auto load = [&](int i, double (&row)[4]) {
#pragma unroll
      for (int q = 0; q < 4; q++) { const int k = lane + 32 * q; row[q] = (i >= 0 && k > i && k <= j) ? G[(size_t)i * nb + k] : 0.0; }
    };
#pragma unroll
    for (int a = 0; a < PF; a++) load(j - 1 - a, g[a]);
    if (lane == (j & 31)) t[j >> 5] = tauv[p0 + j];
    for (int i0 = j - 1; i0 >= 0; i0 -= PF) {
#pragma unroll
      for (int a = 0; a < PF; a++) {
        const int i = i0 - a;
        if (i < 0) break;     // warp-uniform
        double acc = 0.0;
#pragma unroll
        for (int q = 0; q < 4; q++) acc = __fma_rn(g[a][q], t[q], acc);
        acc = warp_sum_butterfly(acc);
        const double ti = -tauv[p0 + i] * acc;
#pragma unroll
        for (int q = 0; q < 4; q++) if ((i >> 5) == q && lane == (i & 31)) t[q] = ti;
      }
#pragma unroll
      for (int a = 0; a < PF; a++) load(i0 - PF - a, g[a]);
    }
  }
#pragma unroll
  for (int q = 0; q < 4; q++) { const int i = lane + 32 * q; if (i < nb) T[(size_t)i * nb + j] = (i <= j) ? t[q] : 0.0; }
}

// sign[i] = -1 if the component of largest magnitude of row i (first on ties) is negative — the convention of rayleigh_kernel
__global__ void __launch_bounds__(256)
eig_sign_kernel(const double* __restrict__ VT, int ld, int n, double* __restrict__ sign) {
  const int lane = threadIdx.x & 31;
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (i >= n) return;
  double best = -1.0, bval = 0.0;
  int bidx = 0x7fffffff;
  for (int k = lane; k < n; k += 32) {
    const double v = VT[(size_t)i * ld + k];
    if (fabs(v) > best) { best = fabs(v); bval = v; bidx = k; }
  }
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    const double ob = __shfl_xor_sync(0xffffffffu, best, off), ov = __shfl_xor_sync(0xffffffffu, bval, off);
    const int oi = __shfl_xor_sync(0xffffffffu, bidx, off);
    if (ob > best || (ob == best && oi < bidx)) { best = ob; bval = ov; bidx = oi; }
  }
  if (lane == 0) sign[i] = bval < 0.0 ? -1.0 : 1.0;
}

template <typename T>
bool ws_alloc(TridiagWs* ws, T** p, size_t count) {
  if (cudaMalloc((void**)p, sizeof(T) * (count ? count : 1)) != cudaSuccess) return false;
  cudaMemset(*p, 0, sizeof(T) * (count ? count : 1));
  ws->allocs.push_back(*p);
  return true;
}

int round_even(double x) { return 2 * (int)(x / 2.0 + 0.5); }

}  // namespace

void launch_eig_sign(cudaStream_t st, const double* VT, int ld, int n, double* sign) {
  eig_sign_kernel<<<(n * 32 + 255) / 256, 256, 0, st>>>(VT, ld, n, sign);
}

bool eigen_tridiag_fits(int n) { return n >= 4 && (size_t)n * 5 * sizeof(double) + 4096 <= 226 * 1024; }

TridiagWs* tridiag_ws_create(int n, int ld, int num_sms, char* err, size_t errlen) {
  TridiagWs* ws = new TridiagWs();
  ws->n = n; ws->ld = ld; ws->num_sms = num_sms;
  auto fail = [&](const char* what) { if (err) snprintf(err, errlen, "tridiagonal eigensolver workspace: %s", what); tridiag_ws_destroy(ws); return (TridiagWs*)nullptr; };
  const size_t mat = (size_t)n * ld;
  // ---- stage 1 geometry
  const int ns = (n + 1) & ~1;
  int grid = num_sms < 1 ? 1 : num_sms;
  if (grid > (n + 3) / 4) grid = (n + 3) / 4;        // at least ~4 columns per CTA: fewer slices to collect per step at small N
  if (grid < 1) grid = 1;
  const int nloc_max = (n + grid - 1) / grid;
  const size_t vec_bytes = sizeof(double) * (5 * (size_t)ns + 48);
  if (vec_bytes > kSmemCap) return fail("N too large for the shared-memory vectors of sytrd_kernel");
  // register-resident instantiations <KU, NC>: row pairs per thread x columns per CTA
  const char* force = getenv("KCMA_SYTRD_RESIDENT");
  const int units = ns / 2;
  ws->reg_variant = 0;
  if (!(force && atoi(force) == 0)) {
    if (units <= SY_NT && nloc_max <= 4) ws->reg_variant = 1;
    else if (units <= 2 * SY_NT && nloc_max <= 7) ws->reg_variant = 2;
    else if (units <= 2 * SY_NT && nloc_max <= 14) ws->reg_variant = 4;
    else if (units <= 3 * SY_NT && nloc_max <= 11) ws->reg_variant = 3;
  }
  // (74 CTAs x 512 threads, <KU, NC> = <1, 14>, was measured and dropped: 6.1 instead of 4.3 ms, profiles/r02_eigen_ab10.log)
  ws->resident = ws->reg_variant != 0;
  ws->sy_grid = grid;
  static const int kNC[5] = {0, 4, 7, 11, 14};
  ws->sy_smem = ws->resident ? sizeof(double) * (3 * (size_t)ns + 80 + (size_t)kNC[ws->reg_variant] * SY_NT) : vec_bytes;
  // (thread-block clusters of 2 or 4 CTAs for <2, 7>, whose leader polled the slots and pushed the entries into its peers' shared
  // memory, were measured and dropped: config 3, sytrd 4.30 ms without, 4.44 / 4.30 ms with, profiles/r02_eigen_ab9_cluster.log)
  bool ok = true;
  if (!ws->resident) ok = ok && ws_alloc(ws, &ws->Awork, mat);
  ok = ok && ws_alloc(ws, &ws->dT, n) && ws_alloc(ws, &ws->eT, n) && ws_alloc(ws, &ws->tau, n) && ws_alloc(ws, &ws->VR, mat) &&
       ws_alloc(ws, &ws->VC, mat);
  LL* xb = nullptr;
  ws->ll_copies = 2;
  // product slots: four copies at large N (a copy costs a producer one more 16-byte store per entry; 37 pollers per line instead of 74:
  // sytrd 4.17 -> 4.05 ms at N = 1000; three, six or eight copies, or more than two copies of the COLUMN slots, lose again:
  // profiles/r02_eigen_ab15.log, r02_eigen_ab16.log)
  ws->ll_pcopies = n > 512 ? 4 : ws->ll_copies;
  ok = ok && ws_alloc(ws, &xb, (size_t)std::max(ws->ll_copies, ws->ll_pcopies) * 4 * (size_t)ns);
  ws->xbuf = xb;
  if (const char* pe = getenv("KCMA_SYTRD_PROF")) {   // "step0[,cta]": clock64 stamps of 32 steps of one CTA (tridiag_dump_prof)
    ws->prof_step0 = atoi(pe);
    if (const char* comma = strchr(pe, ',')) ws->prof_cta = atoi(comma + 1);
    ok = ok && ws_alloc(ws, &ws->prof, 32 * 8);
  }
  // ---- stage 2 tree: uniform depth, even leaf boundaries, leaves of 2..32 rows
  int levels = 0;
  // largest leaf: 12 rows. Smaller leaves = cheaper Jacobi leaves, more merge levels: at N = 100 the
  // stage takes 0.38 ms with leaves of 25 rows, 0.25 with 6; at N = 1000 0.79 ms with 16 rows, 0.75 with 8 (profiles/r02_eigen_ab12.log)
  const int leaf_rows = 12;
  if (n > 32)
    while ((n + (1 << levels) - 1) / (1 << levels) > leaf_rows) levels++;
  const int leaves = 1 << levels;
  ws->bounds.resize(leaves + 1);
  for (int k = 0; k <= leaves; k++) ws->bounds[k] = (k == leaves) ? n : round_even((double)k * n / leaves);
  for (int k = 0; k < leaves; k++) {
    const int m = ws->bounds[k + 1] - ws->bounds[k];
    if (m > 32 || (leaves > 1 && m < 2)) return fail("could not build the divide & conquer tree");
  }
  ws->levels = levels; ws->leaf_count = leaves;
  std::vector<DcNode> all_nodes;
  std::vector<int> row2node((size_t)std::max(levels, 1) * n, 0);
  for (int l = 1; l <= levels; l++) {
    std::vector<DcNode> v;
    const int span = 1 << l;
    ws->lvl_node_begin.push_back((int)all_nodes.size());
    for (int k = 0; k < leaves; k += span) {
      DcNode nd;
      nd.off = ws->bounds[k];
      nd.n1 = ws->bounds[k + span / 2] - nd.off;
      nd.n = ws->bounds[k + span] - nd.off;
      for (int r = nd.off; r < nd.off + nd.n; r++) row2node[(size_t)(l - 1) * n + r] = (int)all_nodes.size();
      v.push_back(nd);
      all_nodes.push_back(nd);
    }
    ws->lvl.push_back(v);
  }
  const size_t nn = all_nodes.size() ? all_nodes.size() : 1;
  ok = ok && ws_alloc(ws, &ws->d_nodes, nn) && ws_alloc(ws, &ws->d_bounds, leaves + 1) && ws_alloc(ws, &ws->d_row2node, row2node.size());
  ok = ok && ws_alloc(ws, &ws->dA, n) && ws_alloc(ws, &ws->dB, n) && ws_alloc(ws, &ws->Qa, mat) && ws_alloc(ws, &ws->XT, mat);
  if (levels > 0) {
    ok = ok && ws_alloc(ws, &ws->UT, mat) && ws_alloc(ws, &ws->DELTA, mat);
    if (levels > 1) ok = ok && ws_alloc(ws, &ws->Qb, mat);
    ok = ok && ws_alloc(ws, &ws->dl, n) && ws_alloc(ws, &ws->w, n) && ws_alloc(ws, &ws->what, n) && ws_alloc(ws, &ws->lam, n) &&
         ws_alloc(ws, &ws->defl_val, n) && ws_alloc(ws, &ws->col2k, n) && ws_alloc(ws, &ws->nd_col, n) && ws_alloc(ws, &ws->defl_col, n) &&
         ws_alloc(ws, &ws->rho, nn) && ws_alloc(ws, &ws->Kcnt, nn) && ws_alloc(ws, &ws->mixed, nn) && ws_alloc(ws, &ws->rot_c, n) &&
         ws_alloc(ws, &ws->rot_s, n) && ws_alloc(ws, &ws->rot_p, n) && ws_alloc(ws, &ws->rot_q, n);
  }
  if (!ok) return fail("out of device memory");
  if (!all_nodes.empty()) cudaMemcpy(ws->d_nodes, all_nodes.data(), sizeof(DcNode) * all_nodes.size(), cudaMemcpyHostToDevice);
  cudaMemcpy(ws->d_bounds, ws->bounds.data(), sizeof(int) * (leaves + 1), cudaMemcpyHostToDevice);
  cudaMemcpy(ws->d_row2node, row2node.data(), sizeof(int) * row2node.size(), cudaMemcpyHostToDevice);
  // ---- stage 3 geometry
  const int n_refl = n - 1;     // reflectors 0 .. n-2 (the last one is the identity, tau = 0)
  ws->nb = 128;
  ws->nbld = ws->nb;
  ws->npanels = n_refl > 0 ? (n_refl + ws->nb - 1) / ws->nb : 0;
  const int row_tiles = (n + 127) / 128;
  ws->split1 = std::max(1, std::min(16, (num_sms + row_tiles - 1) / row_tiles));
  if (ws->npanels > 0) {
    ws->gsplits = std::max(1, std::min(8, num_sms / std::max(1, ws->npanels)));
    ok = ok && ws_alloc(ws, &ws->Gbuf, (size_t)ws->gsplits * ws->npanels * ws->nb * ws->nb) && ws_alloc(ws, &ws->Tbuf, (size_t)ws->npanels * ws->nb * ws->nb) &&
         ws_alloc(ws, &ws->Gred, (size_t)ws->npanels * ws->nb * ws->nb) &&
         ws_alloc(ws, &ws->VtilR, mat) && ws_alloc(ws, &ws->W2, (size_t)n * ws->nbld) &&
         ws_alloc(ws, &ws->slabs, (size_t)ws->split1 * n * ws->nbld) && ws_alloc(ws, &ws->QT, mat) && ws_alloc(ws, &ws->QF, mat) &&
         ws_alloc(ws, &ws->XF, mat);
    const int tiles = row_tiles * row_tiles;
    ws->splitF = std::max(1, std::min(8, num_sms / std::max(1, tiles)));
    // merges below the top: a level of 2 (4, 8) products of 500 (250, 125) rows is 32 (16, 8) CTAs at N = 1000; split-K fills the SMs
    // (the slabs are summed over the diagonal blocks only, dc_reduce_blocks_kernel). Bounded by 256 MB of slabs.
    ws->lvl_split.assign(std::max(levels, 1), 1);
    int max_split = ws->splitF;
    for (int l = 1; l < levels; l++) {
      int nmax = 0;
      for (const DcNode& nd : ws->lvl[l - 1]) nmax = std::max(nmax, nd.n);
      const int t = (nmax + 127) / 128, ctas = (int)ws->lvl[l - 1].size() * t * t;
      int sp = std::min(std::min(8, num_sms / std::max(1, ctas)), nmax / 64);
      while (sp > 1 && (size_t)sp * mat * sizeof(double) > ((size_t)256 << 20)) sp--;
      if (sp >= 2 && nmax >= 100) { ws->lvl_split[l - 1] = sp; max_split = std::max(max_split, sp); }
    }
    if (max_split > 1) ok = ok && ws_alloc(ws, &ws->slabsF, (size_t)max_split * mat);
    ws->split_top = (levels > 0 && ws->splitF > 1) ? std::min(ws->splitF, 2) : 1;
    if (!ok) return fail("out of device memory");
    if (cudaStreamCreateWithFlags(&ws->st2, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&ws->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&ws->ev_join, cudaEventDisableTiming) != cudaSuccess)
      return fail("could not create the side stream of the back-transform");
  }
  // ---- static GEMM descriptors
  std::vector<GemmDesc> descs;
  for (int l = 1; l <= levels; l++) {
    ws->desc_level_begin.push_back((int)descs.size());
    const bool src_a = (l & 1) == 1;                 // leaves write Qa; level 1 reads Qa and writes Qb; ...
    double* src = src_a ? ws->Qa : ws->Qb;
    double* dst = src_a ? ws->Qb : ws->Qa;
    const int node0 = ws->lvl_node_begin[l - 1];
    for (size_t k = 0; k < ws->lvl[l - 1].size(); k++) {
      const DcNode& nd = ws->lvl[l - 1][k];
      GemmDesc g;
      memset(&g, 0, sizeof(g));
      const size_t o = (size_t)nd.off * ld + nd.off;
      g.K = nd.n; g.alpha = 1.0; g.beta = 0.0; g.n1 = nd.n1; g.mixed = ws->mixed + node0 + k; g.splits = 1; g.split_stride = 0;
      g.lda = g.ldb = g.ldc = ld;
      if (l < levels) {          // Q_new[r][c] = sum_k Q[r][k] U^T[c][k]
        g.A = src + o; g.B = ws->UT + o; g.C = dst + o; g.M = nd.n; g.Nc = nd.n; g.krule = 1;
        if (ws->npanels > 0 && ws->lvl_split[l - 1] > 1) { g.C = ws->slabsF + o; g.splits = ws->lvl_split[l - 1]; g.split_stride = (long long)mat; }
      } else {                   // last merge, transposed: X^T[r][c] = sum_k U^T[r][k] Q[c][k]
        g.A = ws->UT + o; g.B = src + o; g.C = ws->XT + o; g.M = nd.n; g.Nc = nd.n; g.krule = 2;
        if (ws->split_top > 1) { g.C = ws->slabsF; g.splits = ws->split_top; g.split_stride = (long long)mat; }
      }
      descs.push_back(g);
    }
  }
  const int nb = ws->nb;
  ws->desc_g = (int)descs.size();
  for (int p = 0; p < ws->npanels; p++) {      // G_p = V_p^T V_p  (rows of VR)
    const int p0 = p * nb, kb = std::min(nb, n_refl - p0);
    GemmDesc g; memset(&g, 0, sizeof(g));
    g.A = ws->VR + (size_t)p0 * ld + p0; g.B = g.A; g.C = ws->Gbuf + (size_t)p * nb * nb;
    g.M = kb; g.Nc = kb; g.K = n - p0; g.lda = g.ldb = ld; g.ldc = nb; g.alpha = 1.0; g.splits = ws->gsplits;
    g.split_stride = (long long)ws->npanels * nb * nb;
    descs.push_back(g);
  }
  ws->desc_vtil = (int)descs.size();
  for (int p = 0; p < ws->npanels; p++) {      // VtilR_p[q][c] = sum_k T_p[q][k] V[c][p0 + k]
    const int p0 = p * nb, kb = std::min(nb, n_refl - p0);
    GemmDesc g; memset(&g, 0, sizeof(g));
    g.A = ws->Tbuf + (size_t)p * nb * nb; g.B = ws->VC + (size_t)p0 * ld + p0; g.C = ws->VtilR + (size_t)p0 * ld + p0;
    g.M = kb; g.Nc = n - p0; g.K = kb; g.lda = nb; g.ldb = ld; g.ldc = ld; g.alpha = 1.0; g.splits = 1;
    descs.push_back(g);
  }
  ws->desc_gemm1 = (int)descs.size();
  // Q^T = H_{n-2} ... H_0 is accumulated from the identity, last panel first; before panel p is applied Q^T differs from the
  // identity only in rows / columns > p0 + nb, and V_p has no rows <= p0: only the block [p0, n) x [p0, n) takes part.
  for (int p = 0; p < ws->npanels; p++) {      // slabs: W[r][q] = sum_c Q^T[r][c] VtilR_p[q][c], r, c >= p0
    const int p0 = p * nb, kb = std::min(nb, n_refl - p0);
    GemmDesc g; memset(&g, 0, sizeof(g));
    g.A = ws->QT + (size_t)p0 * ld + p0; g.B = ws->VtilR + (size_t)p0 * ld + p0; g.C = ws->slabs;
    g.M = n - p0; g.Nc = kb; g.K = n - p0; g.lda = ld; g.ldb = ld; g.ldc = ws->nbld; g.alpha = 1.0; g.splits = ws->split1;
    g.split_stride = (long long)n * ws->nbld;
    descs.push_back(g);
  }
  ws->desc_gemm2 = (int)descs.size();
  for (int p = 0; p < ws->npanels; p++) {      // Q^T[r][c] -= sum_q W[r][q] V[c][p0 + q], r, c >= p0
    const int p0 = p * nb, kb = std::min(nb, n_refl - p0);
    GemmDesc g; memset(&g, 0, sizeof(g));
    g.A = ws->W2; g.B = ws->VC + (size_t)p0 * ld + p0; g.C = ws->QT + (size_t)p0 * ld + p0;
    g.M = n - p0; g.Nc = n - p0; g.K = kb; g.lda = ws->nbld; g.ldb = ld; g.ldc = ld; g.alpha = -1.0; g.beta = 1.0; g.splits = 1;
    descs.push_back(g);
  }
  ws->desc_final = (int)descs.size();
  if (ws->npanels > 0) {                       // X^T[r][c] = sum_k Z^T[r][k] Q[c][k]   (Z^T = the last merge's output in XT, Q = (Q^T)^T in QF)
    GemmDesc g; memset(&g, 0, sizeof(g));
    g.A = ws->XT; g.B = ws->QF; g.C = ws->splitF > 1 ? ws->slabsF : ws->XF;
    g.M = n; g.Nc = n; g.K = n; g.lda = g.ldb = g.ldc = ld; g.alpha = 1.0; g.splits = ws->splitF; g.split_stride = (long long)mat;
    descs.push_back(g);
  }
  if (!ws_alloc(ws, &ws->d_desc, descs.size() ? descs.size() : 1)) return fail("out of device memory");
  if (!descs.empty()) cudaMemcpy(ws->d_desc, descs.data(), sizeof(GemmDesc) * descs.size(), cudaMemcpyHostToDevice);
  // kernel attributes
  cudaError_t e1 = cudaFuncSetAttribute(sytrd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemCap);
  cudaError_t e2 = cudaFuncSetAttribute(sytrd_reg_kernel<3, 11>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
  if (e2 == cudaSuccess) e2 = cudaFuncSetAttribute(sytrd_reg_kernel<2, 14>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
  if (e1 != cudaSuccess || e2 != cudaSuccess) return fail("cudaFuncSetAttribute failed");
  if (cudaDeviceSynchronize() != cudaSuccess) return fail("CUDA error while building the workspace");
  return ws;
}

void tridiag_ws_destroy(TridiagWs* ws) {
  if (!ws) return;
  if (ws->st2) { cudaStreamSynchronize(ws->st2); cudaStreamDestroy(ws->st2); }
  if (ws->ev_fork) cudaEventDestroy(ws->ev_fork);
  if (ws->ev_join) cudaEventDestroy(ws->ev_join);
  for (void* p : ws->allocs) cudaFree(p);
  delete ws;
}

bool tridiag_stage_sytrd(cudaStream_t st, TridiagWs* ws, const double* M) {
  int n = ws->n, ld = ws->ld, ns = (n + 1) & ~1;
  LL* xP = (LL*)ws->xbuf;
  LL* xC = xP + 2 * (size_t)(ws->resident ? ns : n);   // per-parity stride: ns (32-byte aligned slot pairs) in the register variant
  cudaMemsetAsync(ws->xbuf, 0, sizeof(LL) * 4 * (size_t)ns * (ws->resident ? std::max(ws->ll_copies, ws->ll_pcopies) : 1), st);
  double* Awork = ws->Awork;
  if (!ws->resident) cudaMemcpyAsync(Awork, M, sizeof(double) * (size_t)n * ld, cudaMemcpyDeviceToDevice, st);
  double *dT = ws->dT, *eT = ws->eT, *tau = ws->tau, *VR = ws->VR;
  long long* prof = ws->prof;
  int prof_step0 = ws->prof_step0, prof_cta = ws->prof_cta;
  void* args[] = {&M, &Awork, &ld, &n, &ns, &xP, &xC, &dT, &eT, &tau, &VR, &prof, &prof_step0, &prof_cta};
  // exchange: 1 = one lane per warp spins on one slot before the block polls everything; 4 = a gate on one slot per producer first
  // (same time at N = 1000, 0.33 -> 0.28 ms at N = 100 where a step is short: profiles/r02_sytrd_exchange_ab.log)
  int opt = n <= 512 ? 4 : 1;
  int copies = ws->ll_copies | (ws->ll_pcopies != ws->ll_copies ? ws->ll_pcopies << 8 : 0);
  void* rargs[] = {&M, &ld, &n, &ns, &xP, &xC, &dT, &eT, &tau, &VR, &prof, &prof_step0, &prof_cta, &opt, &copies};
  const void* fn = ws->reg_variant == 1 ? (const void*)sytrd_reg_kernel<1, 4> : ws->reg_variant == 2 ? (const void*)sytrd_reg_kernel<2, 7>
                   : ws->reg_variant == 3 ? (const void*)sytrd_reg_kernel<3, 11> : ws->reg_variant == 4 ? (const void*)sytrd_reg_kernel<2, 14>
                   : (const void*)sytrd_kernel;
  // (column prefetch, where column c travels one step early and the exchange a step waits for is p = A v alone, was measured and
  // dropped: config 3, sytrd 4.67 against 4.30 ms — the column's loads come back late inside the pass, profiles/r02_sytrd_exchange_ab.log)
  if (cudaLaunchCooperativeKernel(fn, dim3(ws->sy_grid), dim3(SY_NT), ws->resident ? rargs : args, ws->sy_smem, st) != cudaSuccess) return false;
  // row n-1 of VR (no reflector) and tau[n-1] stay zero from the allocation; VC = VR^T
  launch_transpose(st, ws->VR, ws->VC, ld, n);
  return cudaGetLastError() == cudaSuccess;
}

bool tridiag_stage_dc(cudaStream_t st, TridiagWs* ws, int* launches) {
  const bool ok = dc_solve(st, ws, launches);
  ws->result = ws->XT;
  return ok;
}

// Stage 3 runs in two parts. fork: Q^T = H_{n-2} ... H_0 from the reflectors alone (panel factors, then two GEMMs per panel),
// on the workspace's side stream — it does not depend on the tridiagonal eigenvectors, so it runs NEXT TO the divide & conquer
// stage, whose kernels leave most SMs idle. join: X^T = Z^T Q^T, one GEMM on the caller's stream.
bool tridiag_stage_back_fork(cudaStream_t st, TridiagWs* ws, int* launches) {
  const int n = ws->n, nb = ws->nb, n_refl = n - 1, ld = ws->ld;
  if (ws->npanels == 0) return true;
  cudaStream_t s2 = ws->st2;
  cudaEventRecord(ws->ev_fork, st);
  cudaStreamWaitEvent(s2, ws->ev_fork, 0);
  launch_set_identity(s2, ws->QT, ld, n);
  launch_gemm_batched(s2, ws->d_desc + ws->desc_g, ws->npanels, nb, nb, ws->gsplits);
  const double* G = ws->Gbuf;
  if (ws->gsplits > 1) {   // sum the split-K slabs once (fixed order)
    launch_reduce_slabs(s2, ws->Gbuf, (long long)ws->npanels * nb * nb, ws->gsplits, ws->npanels * nb, nb, nb, ws->Gred, ws->num_sms);
    G = ws->Gred;
    *launches += 1;
  }
  larft_cols_kernel<<<dim3((nb + 7) / 8, ws->npanels), 256, 0, s2>>>(G, ws->tau, n_refl, nb, ws->Tbuf);
  launch_gemm_batched(s2, ws->d_desc + ws->desc_vtil, ws->npanels, nb, n, 1);
  *launches += 4;
  for (int p = ws->npanels - 1; p >= 0; p--) {
    const int p0 = p * nb, kb = std::min(nb, n_refl - p0);
    launch_gemm_batched(s2, ws->d_desc + ws->desc_gemm1 + p, 1, n - p0, kb, ws->split1);
    launch_reduce_slabs(s2, ws->slabs, (long long)n * ws->nbld, ws->split1, n - p0, kb, ws->nbld, ws->W2, ws->num_sms);
    launch_gemm_batched(s2, ws->d_desc + ws->desc_gemm2 + p, 1, n - p0, n - p0, 1);
    *launches += 3;
  }
  launch_transpose(s2, ws->QT, ws->QF, ld, n);
  *launches += 1;
  cudaEventRecord(ws->ev_join, s2);
  return cudaGetLastError() == cudaSuccess;
}

bool tridiag_stage_back_join(cudaStream_t st, TridiagWs* ws, int* launches) {
  const int n = ws->n;
  if (ws->npanels == 0) return true;
  cudaStreamWaitEvent(st, ws->ev_join, 0);
  launch_gemm_batched(st, ws->d_desc + ws->desc_final, 1, n, n, ws->splitF);
  *launches += 1;
  if (ws->splitF > 1) {
    launch_reduce_slabs(st, ws->slabsF, (long long)n * ws->ld, ws->splitF, n, n, ws->ld, ws->XF, ws->num_sms);
    *launches += 1;
  }
  ws->result = ws->XF;
  return cudaGetLastError() == cudaSuccess;
}

bool launch_eigen_tridiag(cudaStream_t st, TridiagWs* ws, const double* M, double** VT_out, double** ev_out, int* launches) {
  if (!tridiag_stage_sytrd(st, ws, M)) return false;
  *launches += 4;
  if (!tridiag_stage_back_fork(st, ws, launches)) return false;
  if (!tridiag_stage_dc(st, ws, launches)) return false;
  if (!tridiag_stage_back_join(st, ws, launches)) return false;
  *VT_out = ws->result;
  *ev_out = ws->ev_final;
  return true;
}

const double* tridiag_result_vectors(const TridiagWs* ws) { return ws->result; }
const double* tridiag_result_values(const TridiagWs* ws) { return ws->ev_final; }

void tridiag_get_tridiagonal(TridiagWs* ws, double* d, double* e, double* tau, double* vr) {
  const int n = ws->n;
  cudaMemcpy(d, ws->dT, sizeof(double) * n, cudaMemcpyDeviceToHost);
  cudaMemcpy(e, ws->eT, sizeof(double) * n, cudaMemcpyDeviceToHost);
  cudaMemcpy(tau, ws->tau, sizeof(double) * n, cudaMemcpyDeviceToHost);
  if (vr) cudaMemcpy2D(vr, sizeof(double) * n, ws->VR, sizeof(double) * ws->ld, sizeof(double) * n, n, cudaMemcpyDeviceToHost);
}

void tridiag_dump_prof(TridiagWs* ws) {
  if (!ws->prof) return;
  long long h[32 * 8];
  cudaMemcpy(h, ws->prof, sizeof(h), cudaMemcpyDeviceToHost);
  fprintf(stderr, "sytrd_kernel phase stamps (clock64 cycles), CTA %d, n = %d, grid %d, %s:\n  step   receive   vectors      pass   to-next-step\n",
          ws->prof_cta, ws->n, ws->sy_grid, ws->resident ? "register resident" : "global working copy");
  for (int k = 0; k < 32; k++) {
    const long long* r = h + k * 8;
    if (!r[0] || !r[3]) continue;
    fprintf(stderr, "  %4d  %8lld  %8lld  %8lld  %8lld\n", ws->prof_step0 + k, r[1] - r[0], r[2] - r[1], r[3] - r[2], k < 31 && h[(k + 1) * 8] ? h[(k + 1) * 8] - r[3] : 0ll);
  }
}

void tridiag_set_tridiagonal(TridiagWs* ws, const double* d, const double* e) {
  const int n = ws->n;
  cudaMemcpy(ws->dT, d, sizeof(double) * n, cudaMemcpyHostToDevice);
  cudaMemset(ws->eT, 0, sizeof(double) * n);
  if (n > 1) cudaMemcpy(ws->eT, e, sizeof(double) * (n - 1), cudaMemcpyHostToDevice);
}

}  // namespace kc
