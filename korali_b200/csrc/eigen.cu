// eigen.cu — K8: symmetric eigendecomposition of the covariance matrix, once per generation.
// Replaces eigen() (CMAES.cpp.base:896-938: gsl_eigen_symmv + sort ABS_ASC) — the one step of the loop that
// is not population-parallel; timed separately ("eigen" phase).
//
// Method: WARM-STARTED one-sided (Hestenes) Jacobi. With V0 = the eigenvectors of the previous generation (C changes by
// ~c1+cmu per generation), form G = C V0 with the FP64 tensor-core GEMM and orthogonalise the columns of G by plane
// rotations accumulated into V. At convergence C V = G has orthogonal columns: V holds the eigenvectors and
// lambda_i = v_i . g_i (Rayleigh quotient, signed). Vectors are stored as ROWS (VT, GT) so rotations touch contiguous memory.
// Kernels: eigen_small_kernel (tiny N, everything in one launch), jacobi_pipe_kernel (24 < N <= 1184: persistent cooperative,
// warp-specialised Gram-update steps on the DMMA pipe, 4-row blocks), jacobi_big_step_kernel (larger N: one launch per
// tournament step, 16-row blocks, V updated one launch late).
// DESIGN.md section 6.
#include <cooperative_groups.h>
#include <stdlib.h>

#include "common.cuh"
#include "jacobi_inner.cuh"
#include "kernels.h"

namespace cg = cooperative_groups;

namespace kc {

__global__ void reset_rotations_kernel(DevScalars* sc) { sc->jacobi_rotations = 0; sc->jacobi_max_rel_bits = 0ull; }


// (rr_pair / ring_pair: the tournament schedules, jacobi_inner.cuh)
template <int ORDER>
__device__ __forceinline__ void tournament_pair(int np, int step, int k, int& p, int& q) {
  if (ORDER >= 1) ring_pair(np, step, k, p, q); else rr_pair(np, step, k, p, q);
}

// 256-bit global accesses (SASS LDG.E.ENL2.256 / STG.E.ENL2.256, sm_100+): a lane moves 4 consecutive doubles, so the four
// t-lanes of a row cover one full 128-byte line per request instead of half of it (the LSU wavefront count per byte halves).
struct double4x { double a, b, c, d; };
__device__ __forceinline__ double4x ldcg_256(const double* p) {
  double4x v;
  asm volatile("ld.global.cg.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(v.a), "=d"(v.b), "=d"(v.c), "=d"(v.d) : "l"(p));
  return v;
}
__device__ __forceinline__ void stcg_256(double* p, double a, double b, double c, double d) {
  asm volatile("st.global.cg.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(p), "d"(a), "d"(b), "d"(c), "d"(d) : "memory");
}

// ------------------------------------------------------------------------------------------------------
// GRAM-UPDATE one-sided Jacobi, persistent + cooperative. A CTA owns the block pair (I, J) = 8 rows per step:
//   (i)   Gamma = G8 G8^T (8x8) in ONE pass over the 8 rows with DMMA.8x8x4 (fragment a == b);
//   (ii)  the step's plane rotations are carried out on Gamma alone (Gamma <- J Gamma J^T is exact algebra: the dot products
//         of the rotated rows ARE the entries of the updated Gamma), accumulating R (8x8);
//   (iii) rows <- R rows for G and V as DMMAs, written back once.
// Steps are ordered by point-to-point ready flags (each block is produced by one CTA and consumed by one), a grid barrier
// only once per sweep. The pairing of a step comes from tournament_pair<ORDER>: the ring order (ORDER = 1, power-of-two block
// count, the default whenever its phantom blocks cost <= 1/8 more steps) or the round-robin order (ORDER = 0). The kernel is WARP-SPECIALISED around what the phase timestamps of the first, uniform version showed
// (profiles/microbench/jacobi_phases.py; 18-20k cycles per step): 40 % of a step were the 4 rotation rounds on Gamma in
// shared memory (LDS/STS round trips queue behind the step's own global loads in the MIO pipe), 30 % the loads (G fetched
// twice, in the Gram and in the apply layout, plus V), 20 % apply + stores of G AND V, 10 % the flag handshake. Here:
//   * G group (warps 0..NWG-1) runs the critical path: flag -> G load (once: Gram fragments straight from the registers,
//     staged to shared memory for the apply layout) -> Gram (DMMA) -> rotations on Gamma held in REGISTERS by warp 0
//     (jacobi_inner.cuh) -> apply G (DMMA) -> store -> flag;
//   * V group (the last NWV warps, none on warp 0's scheduler) applies the same R to the V rows behind it, decoupled:
//     R travels through a small ring in shared memory, V blocks have their own ready flags, nothing on the G path waits for V.
// ------------------------------------------------------------------------------------------------------
template <int NT, int ORDER /* 0: round-robin, 1: ring (nb = power of two) */>
__global__ void __launch_bounds__(NT, 1)
jacobi_pipe_kernel(double* GT, double* VT, int ld, int n, int nb, double tol, int max_sweeps, DevScalars* sc, unsigned* readyG,
                   unsigned* readyV, long long* dbg /* nullable: phase timestamps (profiles/microbench/jacobi_phases.py) */, int dbg_sweep, int dbg_step0) {
  cg::grid_group grid = cg::this_grid();
#define KCMA_TS(slot) do { if (dbg && blockIdx.x == 1 && tid == 0 && sweep == dbg_sweep && step >= dbg_step0 && step < dbg_step0 + 32) dbg[(step - dbg_step0) * 16 + (slot)] = clock64(); } while (0)
#define KCMA_TSV(slot) do { if (dbg && blockIdx.x == 1 && tid == NWG * 32 && sweep == dbg_sweep && step >= dbg_step0 && step < dbg_step0 + 32) dbg[(step - dbg_step0) * 16 + (slot)] = clock64(); } while (0)
  constexpr int NW = NT / 32;                       // 8: warp 0 | data warps 1..4 | V warps 5..7
  constexpr int NWV = 3;                            // V warps on schedulers 1, 2, 3 (none shares the FP64 pipe of warp 0)
  constexpr int NWG = NW - NWV;                     // G group: warp 0 (flags, rotations) + NWD data warps
  constexpr int NWD = NWG - 1;                      // 4 data warps, one per scheduler: the DMMA pipe (one 8x8x4 per 16 cycles
                                                    // per scheduler) is saturated by one warp with two accumulator chains
  static_assert(NWD == 4, "partial tiles are read back as two double2 per entry");
  constexpr int BG = 16;                            // 16-column spans per data warp and batch (loads in flight: BG x 1 KB per warp)
  constexpr int RING = 4;
  extern __shared__ __align__(16) double dyn_smem[];
  // Columns are handled in SPANS of 16 (one 128-byte line per row): lane (g,t) owns columns 4t..4t+3 of the span in row g.
  // The Gram sum does not care which column sits in which k-slot; for the apply, N-tile A takes columns 4q + {0,1} and
  // N-tile B columns 4q + {2,3} (q = 0..3), so that a lane's two D fragments are again 4 consecutive doubles.
  const int S = ld + 2;                             // row stride = 2 mod 16 doubles: STS.128 / LDS.64 fragments conflict-free
  double* Gs = dyn_smem;                            // [8][S] rows of G of this step
  double* Vs = dyn_smem + 8 * S;                    // [8][S] rows of V of the step the V group works on
  __shared__ double2 part[64][NWD / 2];             // partial Gram tiles, entry-major: one shared-memory round trip for warp 0
  __shared__ double Rring[RING][64];                // rows_new = R rows_old, one entry per step in flight
  __shared__ int rot_ring[RING];
  __shared__ volatile unsigned g_head, v_tail;      // steps whose R is posted / whose V rows are done
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int nspans = ld >> 4;
  const double tol2 = tol * tol;
  unsigned epoch = 0;                               // steps completed by this group of this CTA
  if (tid == 0) { g_head = 0; v_tail = 0; }
  __syncthreads();

  for (int sweep = 0; sweep < max_sweeps; sweep++) {
    if (blockIdx.x == 0 && tid == 0) {
      sc->jacobi_rotations = 0; sc->jacobi_max_rel_bits = 0ull; sc->jacobi_sweeps = sweep + 1;
      sc->jacobi_sweeps_total += 1;
    }
    int sweep_rot = 0, sweep_big = 0;
    grid.sync();
    if (warp < NWG) {
      // =========================== G group: the critical path ===========================
      for (int step = 0; step < nb - 1; step++) {
        int I, J;
        tournament_pair<ORDER>(nb, step, blockIdx.x, I, J);
        const int slot = epoch & (RING - 1);
        KCMA_TS(0);
        if (dbg && blockIdx.x == 1 && tid == 0 && sweep == dbg_sweep && step < 1024) dbg[512 + step] = clock64();
        if (warp == 0) {   // lanes 0 and 1 each watch one flag (acquire loads: no fence, no serialised round trips)
          if (lane < 2) {
            const unsigned* f = readyG + (lane == 0 ? I : J);
            unsigned v;
            do { asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory"); } while (v < epoch);
          }
          __syncwarp();
        }
        asm volatile("bar.sync 1, %0;" ::"n"(NWG * 32));
        KCMA_TS(1);
        const int rowg = (g < 4 ? I * 4 + g : J * 4 + (g - 4));
        const bool rvalid = rowg < n;
        if (warp != 0) {
          // ---- Gram: lane (g,t) feeds x = G[row g][8 grp + 2t (+1)] as both A and B fragment; the same registers are staged ----
          const int dw = warp - 1;
          const double* grow = GT + (size_t)rowg * ld;
          double c0 = 0.0, c1 = 0.0, c2 = 0.0, c3 = 0.0;
          for (int kb = 0; dw + kb * NWD < nspans; kb += BG) {
            double4x xs[BG];   // all loads of the batch in flight before its first DMMA
#pragma unroll
            for (int k = 0; k < BG; k++) {
              const int h = dw + (kb + k) * NWD;
              xs[k].a = xs[k].b = xs[k].c = xs[k].d = 0.0;
              if (rvalid && h < nspans) xs[k] = ldcg_256(grow + 16 * h + 4 * t);
            }
#pragma unroll
            for (int k = 0; k < BG; k++) {   // two independent accumulator chains
              const int h = dw + (kb + k) * NWD;
              if (h < nspans) {
                double* dst = Gs + g * S + 16 * h + 4 * t;
                *reinterpret_cast<double2*>(dst) = make_double2(xs[k].a, xs[k].b);
                *reinterpret_cast<double2*>(dst + 2) = make_double2(xs[k].c, xs[k].d);
              }
              dmma884(c0, c1, xs[k].a, xs[k].a);
              dmma884(c2, c3, xs[k].b, xs[k].b);
              dmma884(c0, c1, xs[k].c, xs[k].c);
              dmma884(c2, c3, xs[k].d, xs[k].d);
            }
          }
          double* pw = reinterpret_cast<double*>(&part[0][0]) + dw;   // part[e][dw]
          pw[(g * 8 + 2 * t) * NWD] = c0 + c2;
          pw[(g * 8 + 2 * t + 1) * NWD] = c1 + c3;
        }
        KCMA_TS(2);
        asm volatile("bar.sync 1, %0;" ::"n"(NWG * 32));
        KCMA_TS(3);
        // ---- warp 0: sum the partial tiles into registers, then the step's rotations on Gamma ----
        if (warp == 0) {
          Inner8 m;
#pragma unroll
          for (int a = 0; a < 8; a++) {
#pragma unroll
            for (int b = a; b < 8; b++) {
              const double2 p0 = part[a * 8 + b][0], p1 = part[a * 8 + b][1];
              m.g[a][b] = (p0.x + p0.y) + (p1.x + p1.y);
            }
          }
#pragma unroll
          for (int a = 0; a < 8; a++) m.rc[a] = (a == (lane & 7)) ? 1.0 : 0.0;
          m.rotations = 0; m.big = 0;
          KCMA_TS(14);
          if (step == 0) inner_full(m, tol2); else inner_cross(m, tol2);
          KCMA_TS(8);
          while (epoch - v_tail >= RING) { }        // ring slot still in use by the V group (it lags by < RING steps)
          if (lane < 8) {
#pragma unroll
            for (int a = 0; a < 8; a++) Rring[slot][a * 8 + lane] = m.rc[a];
          }
          if (lane == 0) { rot_ring[slot] = m.rotations; sweep_rot += m.rotations; sweep_big |= m.big; }
        }
        asm volatile("bar.sync 1, %0;" ::"n"(NWG * 32));
        KCMA_TS(4);
        // ---- rows of G <- R rows (skipped when nothing rotated) ----
        const int rot = rot_ring[slot];
        if (rot != 0 && warp != 0) {
          const int dw = warp - 1;
          const double a_lo = Rring[slot][g * 8 + t], a_hi = Rring[slot][g * 8 + 4 + t];
          double* gout = GT + (size_t)rowg * ld;
          const int cA = 4 * (g >> 1) + (g & 1);              // column of N-index g inside the span, tile A (tile B: + 2)
          for (int h0 = dw; h0 < nspans; h0 += NWD * 8) {     // 8 spans (32 operand loads) in flight per warp
            double bA0[8], bA1[8], bB0[8], bB1[8];
#pragma unroll
            for (int k = 0; k < 8; k++) {
              const int h = h0 + k * NWD;
              const double* src = Gs + t * S + 16 * h + cA;
              const bool ok = h < nspans;
              bA0[k] = ok ? src[0] : 0.0;         bB0[k] = ok ? src[2] : 0.0;
              bA1[k] = ok ? src[4 * S] : 0.0;     bB1[k] = ok ? src[4 * S + 2] : 0.0;
            }
#pragma unroll
            for (int k = 0; k < 8; k++) {
              const int h = h0 + k * NWD;
              double d0 = 0.0, d1 = 0.0, e0 = 0.0, e1 = 0.0;
              dmma884(d0, d1, a_lo, bA0[k]); dmma884(e0, e1, a_lo, bB0[k]);
              dmma884(d0, d1, a_hi, bA1[k]); dmma884(e0, e1, a_hi, bB1[k]);
              if (h < nspans && rvalid) stcg_256(gout + 16 * h + 4 * t, d0, d1, e0, e1);
            }
          }
        }
        KCMA_TS(5);
        asm volatile("bar.sync 1, %0;" ::"n"(NWG * 32));
        if (tid == 0) {
          __threadfence();                          // gpu scope: the G rows; also orders Rring before g_head for the V group
          volatile unsigned* rg = readyG;
          rg[I] = epoch + 1;
          rg[J] = epoch + 1;
          g_head = epoch + 1;
        }
        KCMA_TS(6);
        epoch++;
      }
    } else {
      // =========================== V group: rows of V <- R rows, behind the G group ===========================
      const int vtid = tid - NWG * 32, vw = warp - NWG;
      for (int step = 0; step < nb - 1; step++) {
        int I, J;
        tournament_pair<ORDER>(nb, step, blockIdx.x, I, J);
        const int slot = epoch & (RING - 1);
        KCMA_TSV(9);
        if (dbg && blockIdx.x == 1 && tid == NWG * 32 && sweep == dbg_sweep && step < 1024) dbg[512 + 1024 + step] = clock64();
        if (vtid == 0) {
          while (g_head <= epoch) { }
          __threadfence_block();
        }
        asm volatile("bar.sync 2, %0;" ::"n"(NWV * 32));
        KCMA_TSV(10);
        const int rot = rot_ring[slot];
        if (vtid < 2) {   // the previous owners are done with these V blocks (also when nothing rotates here:
          const unsigned* f = readyV + (vtid == 0 ? I : J);   // publishing them early would let the next owner overtake a pending update)
          unsigned v;
          do { asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory"); } while (v < epoch);
        }
        __syncwarp();
        if (rot != 0) {
          asm volatile("bar.sync 2, %0;" ::"n"(NWV * 32));
          const int chunks = ld >> 1;   // 16-byte chunks per row
#pragma unroll
          for (int r = 0; r < 8; r++) {
            const int row = (r < 4 ? I * 4 + r : J * 4 + (r - 4));
            const bool ok = row < n;
            const double* src = VT + (ok ? (size_t)row * ld : 0);
            for (int c = vtid; c < chunks; c += NWV * 32) cp_async16(Vs + r * S + 2 * c, src + (ok ? 2 * c : 0), ok ? 16 : 0);
          }
          cp_async_commit();
          KCMA_TSV(11);
          const int prow = (g < 4 ? I * 4 + g : J * 4 + (g - 4));
          const double a_lo = Rring[slot][g * 8 + t], a_hi = Rring[slot][g * 8 + 4 + t];
          double* vout = VT + (size_t)prow * ld;
          cp_async_wait<0>();
          asm volatile("bar.sync 2, %0;" ::"n"(NWV * 32));
          KCMA_TSV(12);
          const int cA = 4 * (g >> 1) + (g & 1);
          for (int h0 = vw; h0 < nspans; h0 += NWV * 8) {     // 8 spans (32 operand loads) in flight per warp
            double bA0[8], bA1[8], bB0[8], bB1[8];
#pragma unroll
            for (int k = 0; k < 8; k++) {
              const int h = h0 + k * NWV;
              const double* src = Vs + t * S + 16 * h + cA;
              const bool ok = h < nspans;
              bA0[k] = ok ? src[0] : 0.0;         bB0[k] = ok ? src[2] : 0.0;
              bA1[k] = ok ? src[4 * S] : 0.0;     bB1[k] = ok ? src[4 * S + 2] : 0.0;
            }
#pragma unroll
            for (int k = 0; k < 8; k++) {
              const int h = h0 + k * NWV;
              double d0 = 0.0, d1 = 0.0, e0 = 0.0, e1 = 0.0;
              dmma884(d0, d1, a_lo, bA0[k]); dmma884(e0, e1, a_lo, bB0[k]);
              dmma884(d0, d1, a_hi, bA1[k]); dmma884(e0, e1, a_hi, bB1[k]);
              if (h < nspans && prow < n) stcg_256(vout + 16 * h + 4 * t, d0, d1, e0, e1);
            }
          }
        }
        KCMA_TSV(13);
        asm volatile("bar.sync 2, %0;" ::"n"(NWV * 32));
        if (vtid == 0) {
          __threadfence();   // release: our stores, and (when nothing rotated here) the previous owners' rows we acquired above
          volatile unsigned* rv = readyV;
          rv[I] = epoch + 1;
          rv[J] = epoch + 1;
          v_tail = epoch + 1;
        }
        KCMA_TSV(15);
        epoch++;
      }
    }
    if (tid == 0 && sweep_rot) {
      atomicAdd(&sc->jacobi_rotations, sweep_rot);
      if (sweep_big) atomicMax(&sc->jacobi_max_rel_bits, 0x3ff0000000000000ull);   // "max cos^2" collapsed to {0, 1.0}
    }
    grid.sync();
    const int total = *reinterpret_cast<volatile int*>(&sc->jacobi_rotations);
    const unsigned long long mb = *reinterpret_cast<volatile unsigned long long*>(&sc->jacobi_max_rel_bits);
    grid.sync();
    if (total == 0 || __longlong_as_double((long long)mb) < 1e-20) break;
  }
#undef KCMA_TS
#undef KCMA_TSV
}

// ------------------------------------------------------------------------------------------------------
// Version 2b: the WHOLE eigensolver in one launch for small N (N <= 116: G and V fit the 227 KB of one SM):
// G = V C, cyclic one-sided Jacobi sweeps until no rotation fires, Rayleigh quotients, sign convention, ascending
// |lambda| order, acceptance test and the commit of B, A = B D, D, VT. One warp per row pair.
// ------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024, 1)
eigen_small_kernel(const double* __restrict__ GT, int ld, int n, double* __restrict__ VT, double* __restrict__ B, double* __restrict__ A,
                   double* __restrict__ D, double tol, int max_sweeps, DevScalars* __restrict__ sc) {
  extern __shared__ __align__(16) double sm[];
  const int np = (n + 1) & ~1;           // players of the round-robin (dummy when n is odd)
  const int rs = n | 1;                  // odd row stride: conflict-free column access in the commit phase
  double* Gs = sm;                       // [n][rs]
  double* Vs = sm + (size_t)n * rs;      // [n][rs]
  double* ev = Vs + (size_t)n * rs;      // [n]
  double* sg = ev + n;                   // [n]
  int* perm = reinterpret_cast<int*>(sg + n);  // [n]
  __shared__ int rotations, rejected;
  __shared__ double smin[32], smax[32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  // G = V C was formed by the tensor-core GEMM just before this launch
  for (int i = tid; i < n * n; i += blockDim.x) {
    Vs[(i / n) * rs + (i % n)] = VT[(size_t)(i / n) * ld + (i % n)];
    Gs[(i / n) * rs + (i % n)] = GT[(size_t)(i / n) * ld + (i % n)];
  }
  __syncthreads();
  for (int sweep = 0; sweep < max_sweeps; sweep++) {
    if (tid == 0) rotations = 0;
    int my_rot = 0;          // per-warp count, published once per sweep (one shared atomic per round per pair serialises)
    __syncthreads();
    for (int step = 0; step < np - 1; step++) {
      for (int k = warp; k < np / 2; k += nwarps) {
        int p, q;
        rr_pair(np, step, k, p, q);
        if (q >= n) continue;
        double* gp = Gs + (size_t)p * rs; double* gq = Gs + (size_t)q * rs;
        double a = 0, b = 0, g = 0;
        for (int c = lane; c < n; c += 32) { const double x = gp[c], y = gq[c]; a += x * x; b += y * y; g += x * y; }
        a = warp_sum_butterfly(a); b = warp_sum_butterfly(b); g = warp_sum_butterfly(g);
        if (g * g > tol * tol * a * b) {
          double c, s;
          if (!jacobi_cs_fast(a, b, g, c, s)) jacobi_cs_scaled(a, b, g, c, s);
          my_rot++;
          double* vp = Vs + (size_t)p * rs; double* vq = Vs + (size_t)q * rs;
          for (int cidx = lane; cidx < n; cidx += 32) {
            const double x = gp[cidx], y = gq[cidx];
            gp[cidx] = c * x - s * y; gq[cidx] = s * x + c * y;
            const double u = vp[cidx], v = vq[cidx];
            vp[cidx] = c * u - s * v; vq[cidx] = s * u + c * v;
          }
        }
      }
      __syncthreads();
    }
    if (lane == 0 && my_rot) atomicAdd(&rotations, my_rot);
    __syncthreads();
    const int done = (rotations == 0);
    __syncthreads();
    if (done) break;
  }
  // Rayleigh quotients + sign convention
  for (int i = warp; i < n; i += nwarps) {
    double a = 0.0, nv = 0.0, best = -1.0, bval = 0.0;
    int bidx = 0x7fffffff;
    for (int k = lane; k < n; k += 32) {
      const double v = Vs[(size_t)i * rs + k];
      a += v * Gs[(size_t)i * rs + k]; nv += v * v;
      if (fabs(v) > best) { best = fabs(v); bval = v; bidx = k; }
    }
    a = warp_sum_butterfly(a); nv = warp_sum_butterfly(nv);
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
      const double ob = __shfl_xor_sync(0xffffffffu, best, off), ov = __shfl_xor_sync(0xffffffffu, bval, off);
      const int oi = __shfl_xor_sync(0xffffffffu, bidx, off);
      if (ob > best || (ob == best && oi < bidx)) { best = ob; bval = ov; bidx = oi; }
    }
    if (lane == 0) { ev[i] = a / nv; sg[i] = bval < 0.0 ? -1.0 : 1.0; }
  }
  __syncthreads();
  double mn = INFINITY, mx = -INFINITY;
  for (int i = tid; i < n; i += blockDim.x) {
    const double a = fabs(ev[i]);
    int r = 0;
    for (int jx = 0; jx < n; jx++) { const double b = fabs(ev[jx]); r += (b < a) || (b == a && jx < i); }
    perm[r] = i;
    mn = fmin(mn, ev[i]); mx = fmax(mx, ev[i]);
  }
  mn = warp_min(mn); mx = warp_max(mx);
  if (lane == 0) { smin[warp] = mn; smax[warp] = mx; }
  __syncthreads();
  if (tid == 0) {
    for (int w = 0; w < nwarps; w++) { mn = fmin(mn, smin[w]); mx = fmax(mx, smax[w]); }
    rejected = (mn <= 0.0 || !(mn == mn));
    sc->eig_rejected = rejected;
    if (!rejected) { sc->min_eig = mn; sc->max_eig = mx; }
  }
  __syncthreads();
  if (rejected) return;
  for (int i = tid; i < n * n; i += blockDim.x) {
    const int e = i / n, d = i % n;      // VT[e][d] = sign * V[perm[e]][d]
    VT[(size_t)e * ld + d] = sg[perm[e]] * Vs[(size_t)perm[e] * rs + d];
  }
  for (int i = tid; i < n * n; i += blockDim.x) {
    const int d = i / n, e = i % n;      // B[d][e] = VT[e][d]
    const double v = sg[perm[e]] * Vs[(size_t)perm[e] * rs + d];
    const double dd = sqrt(ev[perm[e]]);
    B[(size_t)d * ld + e] = v;
    A[(size_t)d * ld + e] = v * dd;
    if (d == 0) D[e] = dd;
  }
}

// ev[i] = v_i . g_i ; sign[i] = -1 if the component of largest magnitude (first on ties) is negative
// (sign convention shared with the CPU oracle). One warp per vector.
__global__ void __launch_bounds__(256)
rayleigh_kernel(const double* __restrict__ GT, const double* __restrict__ VT, int ld, int n, double* __restrict__ ev,
                double* __restrict__ sign) {
  const int lane = threadIdx.x & 31;
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (i >= n) return;
  double a = 0.0, nv = 0.0, best = -1.0, bval = 0.0;
  int bidx = 0x7fffffff;
  for (int k = lane; k < n; k += 32) {
    const double v = VT[(size_t)i * ld + k];
    a += v * GT[(size_t)i * ld + k];
    nv += v * v;
    if (fabs(v) > best) { best = fabs(v); bval = v; bidx = k; }
  }
  a = warp_sum_butterfly(a); nv = warp_sum_butterfly(nv);
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    const double ob = __shfl_xor_sync(0xffffffffu, best, off), ov = __shfl_xor_sync(0xffffffffu, bval, off);
    const int oi = __shfl_xor_sync(0xffffffffu, bidx, off);
    if (ob > best || (ob == best && oi < bidx)) { best = ob; bval = ov; bidx = oi; }
  }
  if (lane == 0) { ev[i] = a / nv; sign[i] = bval < 0.0 ? -1.0 : 1.0; }
}

// perm = ascending order of |ev| (GSL_EIGEN_SORT_ABS_ASC; ties by index): rank by counting, one thread per eigenvalue, any n.
__global__ void __launch_bounds__(128)
eig_rank_kernel(const double* __restrict__ ev, int n, int* __restrict__ perm) {
  __shared__ double chunk[128];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const double a = i < n ? fabs(ev[i]) : 0.0;
  int r = 0;
  for (int j0 = 0; j0 < n; j0 += 128) {
    __syncthreads();
    chunk[threadIdx.x] = (j0 + threadIdx.x < n) ? fabs(ev[j0 + threadIdx.x]) : INFINITY;
    __syncthreads();
    const int lim = min(128, n - j0);
    for (int k = 0; k < lim; k++) {
      const double bv = chunk[k];
      r += (bv < a) || (bv == a && j0 + k < i);
    }
  }
  if (i < n) perm[r] = i;
}

// min / max eigenvalue and the acceptance test (min <= 0 keeps the previous B, D: CMAES.cpp.base:876-880). A non-finite eigenvalue
// rejects the decomposition as well: fmin / fmax drop NaN operands, so non-finiteness is tracked explicitly.
__global__ void __launch_bounds__(1024)
eig_accept_kernel(const double* __restrict__ ev, int n, DevScalars* __restrict__ sc) {
  __shared__ double smin[32], smax[32];
  __shared__ int sbad;
  if (threadIdx.x == 0) sbad = 0;
  __syncthreads();
  double mn = INFINITY, mx = -INFINITY;
  int bad = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const double v = ev[i];
    bad |= !isfinite(v);
    mn = fmin(mn, v); mx = fmax(mx, v);
  }
  if (bad) atomicOr(&sbad, 1);
  mn = warp_min(mn); mx = warp_max(mx);
  if ((threadIdx.x & 31) == 0) { smin[threadIdx.x >> 5] = mn; smax[threadIdx.x >> 5] = mx; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) { mn = fmin(mn, smin[w]); mx = fmax(mx, smax[w]); }
    if (sbad || mn <= 0.0 || !(mn == mn)) {
      sc->eig_rejected = 1;
    } else {
      sc->eig_rejected = 0;
      sc->min_eig = mn;
      sc->max_eig = mx;
    }
  }
}

// On acceptance: B[d][e] = VTw[perm[e]][d], D[e] = sqrt(ev[perm[e]]), A[d][e] = B[d][e]*D[e], VT <- VTw (permuted).
// 32x32 smem transpose tiles. On rejection nothing is written.
__global__ void __launch_bounds__(256)
eig_commit_kernel(const double* __restrict__ VTw, int ld, int n, const int* __restrict__ perm, const double* __restrict__ ev,
                  const double* __restrict__ sign, double* __restrict__ B, double* __restrict__ A, double* __restrict__ D, double* __restrict__ VT,
                  const DevScalars* __restrict__ sc) {
  if (sc->eig_rejected) return;
  __shared__ double tile[32][33];
  const int e0 = blockIdx.x * 32, d0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int r = ty; r < 32; r += 8) {
    const int e = e0 + r, d = d0 + tx;
    double v = 0.0;
    if (e < n && d < n) {
      v = sign[perm[e]] * VTw[(size_t)perm[e] * ld + d];
      VT[(size_t)e * ld + d] = v;
    }
    tile[r][tx] = v;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int d = d0 + r, e = e0 + tx;
    if (d < n && e < n) {
      const double v = tile[tx][r];
      const double dd = sqrt(ev[perm[e]]);
      B[(size_t)d * ld + e] = v;
      A[(size_t)d * ld + e] = v * dd;
      if (d == 0) D[e] = dd;
    }
  }
}

// Diagonal Covariance mode (:898-903): Q = I, eigenvalues = diag(C) UNSORTED (SURVEY Q7).
__global__ void __launch_bounds__(256)
eig_diagonal_kernel(const double* __restrict__ C, int ldc, int n, double* __restrict__ D, DevScalars* __restrict__ sc) {
  __shared__ double smin[8], smax[8];
  __shared__ int rej, sbad;
  if (threadIdx.x == 0) sbad = 0;
  __syncthreads();
  double mn = INFINITY, mx = -INFINITY;
  int bad = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) { const double v = C[(size_t)i * ldc + i]; bad |= !isfinite(v); mn = fmin(mn, v); mx = fmax(mx, v); }
  if (bad) atomicOr(&sbad, 1);   // fmin / fmax drop NaN operands: non-finiteness is tracked explicitly
  mn = warp_min(mn); mx = warp_max(mx);
  if ((threadIdx.x & 31) == 0) { smin[threadIdx.x >> 5] = mn; smax[threadIdx.x >> 5] = mx; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 0; w < 8; w++) { mn = fmin(mn, smin[w]); mx = fmax(mx, smax[w]); }
    rej = (sbad || mn <= 0.0 || !(mn == mn));
    sc->eig_rejected = rej;
    if (!rej) { sc->min_eig = mn; sc->max_eig = mx; }
  }
  __syncthreads();
  if (rej) return;
  for (int i = threadIdx.x; i < n; i += blockDim.x) D[i] = sqrt(C[(size_t)i * ldc + i]);
}

__global__ void __launch_bounds__(256) set_identity_kernel(double* __restrict__ M, int ld, int n) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
  if (j < ld) M[(size_t)i * ld + j] = (i == j && j < n) ? 1.0 : 0.0;
}

void launch_set_identity(cudaStream_t st, double* M, int ld, int n) {
  dim3 grid((ld + 255) / 256, n);
  set_identity_kernel<<<grid, 256, 0, st>>>(M, ld, n);
}

constexpr size_t kMaxDynSmem = 227 * 1024 - 2048;  // leave room for the kernels' static shared memory
constexpr int kEigenSmallMax = 24;                 // largest N for eigen_small_kernel
size_t eigen_small_smem_bytes(int n) { return sizeof(double) * (2 * (size_t)n * (n | 1) + 2 * n) + sizeof(int) * n + 16; }
bool eigen_use_small(int n) { return n <= kEigenSmallMax && eigen_small_smem_bytes(n) <= kMaxDynSmem; }
void launch_eigen_small(cudaStream_t st, const double* C, int ld, int n, double* VT, double* GT, double* B, double* A, double* D,
                        double tol, int max_sweeps, DevScalars* sc) {
  launch_gemm_tn(st, n, n, n, VT, ld, C, ld, GT, ld);   // GT[i][j] = sum_k VT[i][k] C[j][k]
  static std::atomic<unsigned long long> attr{0};
  if (first_call_on_device(attr)) cudaFuncSetAttribute(eigen_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxDynSmem);
  eigen_small_kernel<<<1, 1024, eigen_small_smem_bytes(n), st>>>(GT, ld, n, VT, B, A, D, tol, max_sweeps, sc);
}

long long* g_jacobi_dbg = nullptr;   // device buffer of phase timestamps (KCMA_JACOBI_DEBUG=1)

// All sweeps in one cooperative launch: one CTA per pair of 4-row blocks, so the whole tournament round must be
// co-resident. Returns false when it is not (N > 8*num_sms, or rows longer than the kernel's register tile covers) or when the
// cooperative launch fails; the caller then launches one jacobi_big_step_kernel per tournament step.
bool launch_jacobi_persistent(cudaStream_t st, double* GT, double* VT, int ld, int n, double tol, int max_sweeps, DevScalars* sc,
                              int num_sms, unsigned* ready) {
  int nb = ((n + 3) / 4 + 1) & ~1;
  if (nb / 2 > num_sms || ld > 1280) return false;
  // Tournament order: the ring order needs a power-of-two block count; it is used when the phantom blocks that pads in cost less
  // than the sweep it saves (<= 1/8 more steps) and the padded round is still co-resident; otherwise the round-robin order.
  // Measured on config 3 (same box, profiles/r01_jacobi_order_ab.log): 7.80 instead of 8.65 sweeps per decomposition, 13.2
  // instead of 14.6 ms. (Keeping the ring order's first block of a slot resident in shared memory was measured and dropped: 14.30
  // instead of 13.23 ms, profiles/r02_jacobi_anchor_ab.log.)
  int nb_ring = 2;
  while (nb_ring < nb) nb_ring <<= 1;
  const bool ring = nb_ring / 2 <= num_sms && (nb_ring - nb) * 8 <= nb && 2 * nb_ring <= ld;
  if (ring) nb = nb_ring;
  static int coop = -1;
  static std::atomic<unsigned long long> attr{0};
  if (first_call_on_device(attr)) {
    int dev = 0, c = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&c, cudaDevAttrCooperativeLaunch, dev);
    if (c && (cudaFuncSetAttribute(jacobi_pipe_kernel<256, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxDynSmem - 16 * 1024) != cudaSuccess ||
              cudaFuncSetAttribute(jacobi_pipe_kernel<256, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxDynSmem - 16 * 1024) != cudaSuccess))
      c = 0;
    if (coop != 0) coop = c;
  }
  if (coop <= 0) return false;
  static long long* dbg = nullptr;   // phase timestamps, only with KCMA_JACOBI_DEBUG=<sweep to trace>
  const char* de = getenv("KCMA_JACOBI_DEBUG");
  if (de && !dbg) {
    cudaMalloc(&dbg, sizeof(long long) * 3584);
    cudaMemset(dbg, 0, sizeof(long long) * 3584);
    g_jacobi_dbg = dbg;
  }
  int dbg_sweep = de ? atoi(de) : -1;
  int dbg_step0 = getenv("KCMA_JACOBI_DEBUG_STEP0") ? atoi(getenv("KCMA_JACOBI_DEBUG_STEP0")) : 8;
  const size_t smem = sizeof(double) * 16 * (size_t)(ld + 2);   // 8 rows of G + 8 rows of V, stride ld + 2
  cudaMemsetAsync(ready, 0, sizeof(unsigned) * 2 * nb, st);
  unsigned* ready_v = ready + nb;
  void* args[] = {&GT, &VT, &ld, &n, &nb, &tol, &max_sweeps, &sc, &ready, &ready_v, &dbg, &dbg_sweep, &dbg_step0};
  const void* fn = ring ? (const void*)jacobi_pipe_kernel<256, 1> : (const void*)jacobi_pipe_kernel<256, 0>;
  if (cudaLaunchCooperativeKernel(fn, dim3(nb / 2), dim3(256), args, smem, st) == cudaSuccess) return true;
  cudaGetLastError();
  return false;
}

// ------------------------------------------------------------------------------------------------------
// Large N (G and V no longer fit L2: N = 4096 -> 2 x 134 MB): one launch per tournament step, but with 16-ROW blocks.
// A step with 4-row blocks streams all of G and V through HBM for 16 rotations per 8 rows (1.5 flop/byte; N/4 - 1 steps per
// sweep: 1.28 s per decomposition at N = 4096). The algebra does not care about the block size: a CTA that owns the block pair
// (I, J) = 32 rows forms Gamma = G32 G32^T (32 x 32, ten symmetric 8x8 DMMA tiles) in ONE pass over the rows, carries out all
// 16 rounds x 16 rotations of the step on Gamma in shared memory (one warp-slot per rotation pair, R accumulating), and applies
// R (32 x 32) to the rows of G and V in one more pass: 4x fewer steps and 4x less HBM traffic per sweep, ~6 flop/byte, so a
// step costs about what its 670 MB of HBM traffic and its DMMAs cost (both ~90 us at N = 4096).
// ------------------------------------------------------------------------------------------------------
constexpr int BIG_B = 16;             // rows per block
constexpr int BIG_R = 2 * BIG_B;      // rows per CTA
constexpr int BIG_TILES = 10;         // upper-triangular 8x8 tiles of the 32 x 32 Gamma
constexpr int BIG_LDS = BIG_R + 1;    // padded leading dimension of Gamma and R in shared memory

__device__ __forceinline__ int big_row(int I, int J, int i) { return i < BIG_B ? I * BIG_B + i : J * BIG_B + (i - BIG_B); }

constexpr int BIG_RLOG = BIG_R * BIG_R + 8;   // doubles per pair in the R log: R (row-major 32 x 32) + rotation count

// rows <- R rows for the 32 rows of the block pair (I, J) of M (G or V), on the spans w0, w0 + nw, ... Rs = R in shared memory.
// Per 16-column span 4 M-tiles x 2 N-tiles x 8 k-steps. N-tile A takes the columns 4q, 4q+2 and N-tile B the columns 4q+1, 4q+3
// of the span (q = 0..3), so that lane g loads ONE 16-byte operand per k-row (columns 2g, 2g+1) and lane t stores 4 consecutive
// doubles (columns 4t..4t+3). Every warp owns whole spans and reads all 32 rows of a span before writing it: in place is safe.
__device__ __forceinline__ void big_apply(double* M, int ld, int n, int I, int J, const double* Rs, int w0, int nw, int lane, int nspans) {
  const int g = lane >> 2, t = lane & 3;
  size_t soff[8];   // operand offsets: k-row 4 ks + t, columns 2g, 2g+1 of the span
  bool sok[8];
#pragma unroll
  for (int ks = 0; ks < 8; ks++) {
    const int row = big_row(I, J, 4 * ks + t);
    sok[ks] = row < n;
    soff[ks] = (size_t)(sok[ks] ? row : 0) * ld + 2 * g;
  }
  int orow[4];
#pragma unroll
  for (int m = 0; m < 4; m++) orow[m] = big_row(I, J, 8 * m + g);
  constexpr int SP = 4;   // spans in flight per lane (32 x 16-byte operand loads = 16 KB per warp): HBM latency x bandwidth
  for (int h0 = w0; h0 < nspans; h0 += SP * nw) {
    double2 b[SP][8];
#pragma unroll
    for (int u = 0; u < SP; u++) {
      const int h = h0 + u * nw;
#pragma unroll
      for (int ks = 0; ks < 8; ks++) {
        b[u][ks] = make_double2(0.0, 0.0);
        if (h < nspans && sok[ks]) b[u][ks] = __ldcg(reinterpret_cast<const double2*>(M + soff[ks] + 16 * h));
      }
    }
    __syncwarp();
#pragma unroll
    for (int m = 0; m < 4; m++) {
      double af[8];   // A fragments of M-tile m: R[8m + g][4 ks + t]
#pragma unroll
      for (int ks = 0; ks < 8; ks++) af[ks] = Rs[(8 * m + g) * BIG_LDS + 4 * ks + t];
#pragma unroll
      for (int u = 0; u < SP; u++) {
        const int h = h0 + u * nw;
        double d0 = 0.0, d1 = 0.0, e0 = 0.0, e1 = 0.0;
#pragma unroll
        for (int ks = 0; ks < 8; ks++) {
          dmma884(d0, d1, af[ks], b[u][ks].x);   // tile A: columns 4q, 4q+2 -> lane t gets columns 4t, 4t+2
          dmma884(e0, e1, af[ks], b[u][ks].y);   // tile B: columns 4q+1, 4q+3 -> lane t gets columns 4t+1, 4t+3
        }
        if (h < nspans && orow[m] < n) stcg_256(M + (size_t)orow[m] * ld + 16 * h + 4 * t, d0, e0, d1, e1);
      }
    }
  }
}

// One tournament step. The V rows are updated ONE LAUNCH LATE: the launch of step s computes Gamma and the rotations of
// step s on the first NWG warps (HBM-bound Gram pass, then the rotation rounds, which leave the DMMA pipe idle) while the other
// warps apply the R of the PREVIOUS step (read back from the R log in global memory) to its V rows; then all warps apply
// the new R to the G rows. V never feeds the rotations, so the only ordering it needs is launch order.
// prev_step < 0: nothing pending; do_g == 0: flush launch (only the pending V update).
template <int NT>
__global__ void __launch_bounds__(NT, 1)
jacobi_big_step_kernel(double* GT, double* VT, int ld, int n, int nsb, int order /* 0: round-robin, 1: ring (nsb = 2^k) */, int step,
                       int prev_step, int do_g, double tol, DevScalars* sc, const double* __restrict__ rlog_prev, double* __restrict__ rlog_cur) {
  constexpr int NW = NT / 32, NWG = NW / 2, NWV = NW - NWG;
  constexpr int PPW = BIG_B / NWG;                       // rotation pairs per warp of the G group
  extern __shared__ __align__(16) double big_smem[];
  double* part = big_smem;                               // [NWG][BIG_TILES][64] partial Gram tiles
  double* Gam = part + NWG * BIG_TILES * 64;             // [32][33]
  double* Rm = Gam + BIG_R * BIG_LDS;                    // [32][33] this step, rows_new = R rows_old
  double* Rv = Rm + BIG_R * BIG_LDS;                     // [32][33] previous step (V update)
  __shared__ int s_rot, s_big;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int nspans = ld >> 4;
  if (tid == 0) { s_rot = 0; s_big = 0; }
  __syncthreads();
  int I = 0, J = 0;
  if (do_g) { if (order == 1) ring_pair(nsb, step, blockIdx.x, I, J); else rr_pair(nsb, step, blockIdx.x, I, J); }

  if (warp >= NWG) {
    // ================= V group: the pending update of the previous step =================
    if (prev_step >= 0) {
      int Ip, Jp;
      if (order == 1) ring_pair(nsb, prev_step, blockIdx.x, Ip, Jp); else rr_pair(nsb, prev_step, blockIdx.x, Ip, Jp);
      const double* src = rlog_prev + (size_t)blockIdx.x * BIG_RLOG;
      if (src[BIG_R * BIG_R] != 0.0) {
        const int vt = tid - NWG * 32;
        for (int e = vt; e < BIG_R * BIG_R; e += NWV * 32) Rv[(e >> 5) * BIG_LDS + (e & 31)] = src[e];
        asm volatile("bar.sync 2, %0;" ::"n"(NWV * 32));
        big_apply(VT, ld, n, Ip, Jp, Rv, warp - NWG, NWV, lane, nspans);
      }
    }
  } else if (do_g) {
    // ================= G group: Gamma, then the step's rotations =================
    const int gt = tid;   // 0 .. NWG*32-1
    {
      // (i) Gamma: lane (g,t) holds columns 4t..4t+3 of a 16-column span for the four 8-row groups
      double acc[BIG_TILES][2];
#pragma unroll
      for (int q = 0; q < BIG_TILES; q++) acc[q][0] = acc[q][1] = 0.0;
      const double* rowp[4];
      bool rok[4];
#pragma unroll
      for (int r = 0; r < 4; r++) {
        const int row = big_row(I, J, 8 * r + g);
        rok[r] = row < n;
        rowp[r] = GT + (size_t)(rok[r] ? row : 0) * ld + 4 * t;
      }
      constexpr int SPG = 4;   // spans in flight per lane (16 x 256-bit loads = 16 KB per warp)
      for (int h0 = warp; h0 < nspans; h0 += SPG * NWG) {
        double4x x[SPG][4];
#pragma unroll
        for (int u = 0; u < SPG; u++) {
          const int h = h0 + u * NWG;
#pragma unroll
          for (int r = 0; r < 4; r++) {
            x[u][r].a = x[u][r].b = x[u][r].c = x[u][r].d = 0.0;
            if (h < nspans && rok[r]) x[u][r] = ldcg_256(rowp[r] + 16 * h);
          }
        }
#pragma unroll
        for (int u = 0; u < SPG; u++) {
          int q = 0;
#pragma unroll
          for (int r1 = 0; r1 < 4; r1++) {
#pragma unroll
            for (int r2 = r1; r2 < 4; r2++, q++) {   // tile (r1, r2): Gamma[8 r1 + m][8 r2 + n]
              dmma884(acc[q][0], acc[q][1], x[u][r1].a, x[u][r2].a);
              dmma884(acc[q][0], acc[q][1], x[u][r1].b, x[u][r2].b);
              dmma884(acc[q][0], acc[q][1], x[u][r1].c, x[u][r2].c);
              dmma884(acc[q][0], acc[q][1], x[u][r1].d, x[u][r2].d);
            }
          }
        }
      }
#pragma unroll
      for (int q = 0; q < BIG_TILES; q++) {
        part[(warp * BIG_TILES + q) * 64 + g * 8 + 2 * t] = acc[q][0];
        part[(warp * BIG_TILES + q) * 64 + g * 8 + 2 * t + 1] = acc[q][1];
      }
    }
    asm volatile("bar.sync 1, %0;" ::"n"(NWG * 32));
    for (int e = gt; e < BIG_TILES * 64; e += NWG * 32) {
      double a = 0.0;
#pragma unroll
      for (int w = 0; w < NWG; w++) a += part[w * BIG_TILES * 64 + e];
      const int q = e >> 6, m = (e >> 3) & 7, nn = e & 7;
      int r1 = 0, base = 0;   // tile index -> (r1, r2): rows of tiles start at 0, 4, 7, 9
      if (q >= 9) { r1 = 3; base = 9; } else if (q >= 7) { r1 = 2; base = 7; } else if (q >= 4) { r1 = 1; base = 4; }
      const int r2 = r1 + (q - base);
      const int i = 8 * r1 + m, j = 8 * r2 + nn;
      Gam[i * BIG_LDS + j] = a;
      if (r1 != r2) Gam[j * BIG_LDS + i] = a;
    }
    for (int e = gt; e < BIG_R * BIG_R; e += NWG * 32) Rm[(e >> 5) * BIG_LDS + (e & 31)] = ((e >> 5) == (e & 31)) ? 1.0 : 0.0;
    asm volatile("bar.sync 1, %0;" ::"n"(NWG * 32));
    // (ii) the step's rotations on Gamma: BIG_B disjoint pairs per round, PPW per warp, lane j = column index
    {
      const double tol2 = tol * tol;
      const int rounds = (step == 0) ? BIG_R - 1 : BIG_B;   // first step of a sweep: all pairs of the 32 rows
      int my_rot = 0, my_big = 0;
      for (int r = 0; r < rounds; r++) {
        double cc[PPW], ss[PPW];
        int pp[PPW], qq[PPW];
#pragma unroll
        for (int u = 0; u < PPW; u++) {   // rows p, q of Gamma and of R
          const int k = warp + u * NWG;
          int p, q;
          if (step == 0) rr_pair(BIG_R, r, k, p, q); else { p = k; q = BIG_B + ((k + r) & (BIG_B - 1)); }
          const double alpha = Gam[p * BIG_LDS + p], beta = Gam[q * BIG_LDS + q], gamma = Gam[p * BIG_LDS + q];
          const double g2 = gamma * gamma, ab = alpha * beta;
          const bool on = g2 > tol2 * ab;
          double c = 1.0, sn = 0.0;
          if (on) {
            if (!jacobi_cs_fast(alpha, beta, gamma, c, sn)) jacobi_cs_scaled(alpha, beta, gamma, c, sn);
            my_rot++;
            my_big |= (g2 > KC_QUAD_TAIL * ab) ? 1 : 0;
          }
          const double x = Gam[p * BIG_LDS + lane], y = Gam[q * BIG_LDS + lane];
          const double a = Rm[p * BIG_LDS + lane], b = Rm[q * BIG_LDS + lane];
          __syncwarp();
          Gam[p * BIG_LDS + lane] = c * x - sn * y; Gam[q * BIG_LDS + lane] = sn * x + c * y;
          Rm[p * BIG_LDS + lane] = c * a - sn * b;  Rm[q * BIG_LDS + lane] = sn * a + c * b;
          cc[u] = c; ss[u] = sn; pp[u] = p; qq[u] = q;
        }
        asm volatile("bar.sync 1, %0;" ::"n"(NWG * 32));
#pragma unroll
        for (int u = 0; u < PPW; u++) {   // columns p, q of Gamma
          const double x = Gam[lane * BIG_LDS + pp[u]], y = Gam[lane * BIG_LDS + qq[u]];
          Gam[lane * BIG_LDS + pp[u]] = cc[u] * x - ss[u] * y;
          Gam[lane * BIG_LDS + qq[u]] = ss[u] * x + cc[u] * y;
        }
        asm volatile("bar.sync 1, %0;" ::"n"(NWG * 32));
      }
      if (lane == 0 && my_rot) { atomicAdd(&s_rot, my_rot); if (my_big) atomicOr(&s_big, 1); }
    }
    asm volatile("bar.sync 1, %0;" ::"n"(NWG * 32));
    // R and the rotation count go to the log: the NEXT launch applies them to the V rows of this pair
    {
      double* dst = rlog_cur + (size_t)blockIdx.x * BIG_RLOG;
      const int rot = s_rot;
      if (rot) for (int e = gt; e < BIG_R * BIG_R; e += NWG * 32) dst[e] = Rm[(e >> 5) * BIG_LDS + (e & 31)];
      if (gt == 0) dst[BIG_R * BIG_R] = (double)rot;
    }
  }
  __syncthreads();
  // (iii) rows of G <- R rows, all warps
  if (do_g && s_rot != 0) {
    big_apply(GT, ld, n, I, J, Rm, warp, NW, lane, nspans);
    if (tid == 0) {
      atomicAdd(&sc->jacobi_rotations, s_rot);
      if (s_big) atomicMax(&sc->jacobi_max_rel_bits, 0x3ff0000000000000ull);
    }
  }
}

// One sweep of per-step launches (N too large for the persistent kernel); the host checks sc->jacobi_max_rel_bits between
// sweeps and calls launch_jacobi_block_flush once after the last sweep (the 16-row-block kernel updates V one launch late).
namespace {
constexpr int BIG_NT = 256;
// R log and launch bookkeeping, per device (one process normally drives one GPU, but kcma_cfg::device is free)
struct BigState {
  double* rlog = nullptr;      // 2 x (pairs x BIG_RLOG) doubles, double-buffered by launch parity
  size_t pairs = 0;
  unsigned launch = 0;         // parity of the next launch
  int pending = -1;            // step whose V update is still pending (-1: none)
};
BigState g_big[64];
BigState& big_state() {
  int dev = 0;
  cudaGetDevice(&dev);
  return g_big[dev & 63];
}
size_t big_smem_bytes() { return sizeof(double) * ((BIG_NT / 64) * BIG_TILES * 64 + 3 * BIG_R * BIG_LDS); }
// Block count and tournament order of the 16-row-block path: the ring order (jacobi_inner.cuh) when padding the block count
// to a power of two costs <= 1/8 more steps (N = 4096: 256 blocks, no padding), else round-robin.
int big_blocks(int n, int* order) {
  int nsb = ((n + BIG_B - 1) / BIG_B + 1) & ~1;
  int nsb_ring = 2;
  while (nsb_ring < nsb) nsb_ring <<= 1;
  const bool ring = (nsb_ring - nsb) * 8 <= nsb;
  *order = ring ? 1 : 0;
  return ring ? nsb_ring : nsb;
}
void big_launch(cudaStream_t st, double* GT, double* VT, int ld, int n, int nsb, int order, int step, int do_g, double tol, DevScalars* sc) {
  BigState& b = big_state();
  double* cur = b.rlog + (size_t)(b.launch & 1u) * b.pairs * BIG_RLOG;
  const double* prev = b.rlog + (size_t)((b.launch & 1u) ^ 1u) * b.pairs * BIG_RLOG;
  jacobi_big_step_kernel<BIG_NT><<<nsb / 2, BIG_NT, big_smem_bytes(), st>>>(GT, VT, ld, n, nsb, order, step, b.pending, do_g, tol, sc, prev, cur);
  b.launch++;
  b.pending = do_g ? step : -1;
}
}  // namespace

void launch_jacobi_block_sweep(cudaStream_t st, double* GT, double* VT, int ld, int n, double tol, DevScalars* sc, int* launches) {
  reset_rotations_kernel<<<1, 1, 0, st>>>(sc);
  int order = 0;
  const int nsb = big_blocks(n, &order);   // 16-row blocks: N/16 - 1 steps per sweep
  static std::atomic<unsigned long long> attr{0};
  if (first_call_on_device(attr)) cudaFuncSetAttribute(jacobi_big_step_kernel<BIG_NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)big_smem_bytes());
  BigState& b = big_state();
  if ((size_t)(nsb / 2) > b.pairs) {
    cudaStreamSynchronize(st);
    if (b.rlog) cudaFree(b.rlog);
    b.pairs = (size_t)(nsb / 2);
    cudaMalloc(&b.rlog, sizeof(double) * 2 * b.pairs * BIG_RLOG);
    b.pending = -1;
  }
  for (int step = 0; step < nsb - 1; step++) big_launch(st, GT, VT, ld, n, nsb, order, step, 1, tol, sc);
  if (launches) *launches += nsb;
}

// The V update of the last step is still pending after the last sweep.
void launch_jacobi_block_flush(cudaStream_t st, double* GT, double* VT, int ld, int n, double tol, DevScalars* sc, int* launches) {
  if (big_state().pending < 0) return;
  int order = 0;
  const int nsb = big_blocks(n, &order);
  big_launch(st, GT, VT, ld, n, nsb, order, 0, 0, tol, sc);
  if (launches) *launches += 1;
}

void launch_rayleigh(cudaStream_t st, const double* GT, const double* VT, int ld, int n, double* ev, double* sign) {
  rayleigh_kernel<<<(n + 7) / 8, 256, 0, st>>>(GT, VT, ld, n, ev, sign);
}
void launch_eig_order(cudaStream_t st, const double* ev, int n, int* perm, DevScalars* sc) {
  eig_rank_kernel<<<(n + 127) / 128, 128, 0, st>>>(ev, n, perm);
  eig_accept_kernel<<<1, 1024, 0, st>>>(ev, n, sc);
}
void launch_eig_commit(cudaStream_t st, const double* VTw, int ld, int n, const int* perm, const double* ev, const double* sign,
                       double* B, double* A, double* D, double* VT, const DevScalars* sc) {
  dim3 grid((n + 31) / 32, (n + 31) / 32);
  eig_commit_kernel<<<grid, 256, 0, st>>>(VTw, ld, n, perm, ev, sign, B, A, D, VT, sc);
}
void launch_eig_diagonal(cudaStream_t st, const double* C, int ldc, int n, double* D, DevScalars* sc) {
  eig_diagonal_kernel<<<1, 256, 0, st>>>(C, ldc, n, D, sc);
}

}  // namespace kc
