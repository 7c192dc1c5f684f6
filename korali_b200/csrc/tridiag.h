// tridiag.h — workspace of the tridiagonalisation-based eigensolver (internal; shared by tridiag.cu and dc.cu).
#pragma once
#include <vector>

#include "kernels.h"

namespace kc {

struct DcNode { int off, n1, n; };   // a merge: rows/columns [off, off + n), children [off, off + n1) and [off + n1, off + n)

struct TridiagWs {
  int n = 0, ld = 0, num_sms = 148;
  // ---- stage 1: Householder tridiagonalisation (sytrd_kernel)
  bool resident = false;       // this CTA's columns live in REGISTERS (N <= 1536: sytrd_reg_kernel), else in the global working copy
  int reg_variant = 0;         // 1, 2, 3, 4 = sytrd_reg_kernel<1,4>, <2,7>, <3,11>, <2,14>
  int sy_grid = 0; size_t sy_smem = 0;
  double* Awork = nullptr;     // n x ld working copy (global variant only)
  double *dT = nullptr, *eT = nullptr, *tau = nullptr;   // diagonal, off-diagonal, reflector scalars
  double *VR = nullptr;        // row i = reflector v_i (support i+1.., v_i[i+1] = 1)
  double *VC = nullptr;        // VR^T (column i = v_i)
  void* xbuf = nullptr;        // LL exchange slots: copies x [P | C] x 2 parities x n x 16 B
  int ll_copies = 2;           // replicas of every slot (spreads the polling of 148 CTAs over several L2 lines)
  int ll_pcopies = 2;          // copies of the product slots (four above N = 512, else ll_copies)
  long long* prof = nullptr; int prof_step0 = 0, prof_cta = 0;   // optional clock64 phase stamps of 32 steps (KCMA_SYTRD_PROF)
  // ---- stage 2: divide & conquer on (dT, eT)
  int levels = 0, leaf_count = 0;
  std::vector<int> bounds;                 // leaf boundaries (even), leaf_count + 1 entries
  std::vector<std::vector<DcNode>> lvl;    // lvl[l-1] = merges of level l = 1..levels
  std::vector<int> lvl_node_begin;         // index of the level's first node in d_nodes
  DcNode* d_nodes = nullptr;
  int* d_bounds = nullptr;
  int* d_row2node = nullptr;               // levels x n: global node index of the merge that owns row g at that level
  double *dA = nullptr, *dB = nullptr;     // eigenvalues of the current / next level (ping-pong), n each
  double *Qa = nullptr, *Qb = nullptr;     // eigenvector blocks (natural layout: columns = vectors), n x ld each (ping-pong)
  double *UT = nullptr, *DELTA = nullptr;  // secular eigenvectors (rows) and pole differences, n x ld each
  double *dl = nullptr, *w = nullptr, *what = nullptr, *lam = nullptr, *defl_val = nullptr;   // n each, indexed off + k
  int *col2k = nullptr, *nd_col = nullptr, *defl_col = nullptr;                              // n each
  double *rho = nullptr; int *Kcnt = nullptr, *mixed = nullptr, *nrot = nullptr;              // per node
  double *rot_c = nullptr, *rot_s = nullptr; int *rot_p = nullptr, *rot_q = nullptr;          // n each (per-node lists at off)
  double* XT = nullptr;                    // result: rows = eigenvectors (n x ld)
  double* ev_final = nullptr;              // points at dA or dB
  // ---- stage 3: compact-WY back-transform
  int nb = 128, npanels = 0, split1 = 1, nbld = 128, gsplits = 1;
  double *Gbuf = nullptr, *Tbuf = nullptr;   // (gsplits x) npanels x nb x nb
  double *Gred = nullptr;                    // G with the split-K slabs summed
  double *VtilR = nullptr;                   // rows p = (T V^T)[p][:] per panel, n x ld
  double *W2 = nullptr, *slabs = nullptr;    // n x nbld, split1 x n x nbld
  double *QT = nullptr, *QF = nullptr;       // Q^T = H_{n-2} ... H_0 accumulated from the identity (side stream), and its transpose Q
  double *XF = nullptr, *slabsF = nullptr;   // X^T = Z^T Q^T (final result), split-K slabs of that product
  int splitF = 1, desc_final = 0;
  int split_top = 1;                         // split-K of the top merge of stage 2 (slabs in slabsF, reduced into XT)
  std::vector<int> lvl_split;                // split-K of the merges below the top (few, small products: 16-32 CTAs without it)
  cudaStream_t st2 = nullptr;                // side stream: the Q accumulation runs next to the divide & conquer stage
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  double* result = nullptr;                  // rows = eigenvectors of the last stage run (XT after stage 2, XF after stage 3)
  // ---- descriptors (static: built once on the host)
  GemmDesc* d_desc = nullptr;
  std::vector<int> desc_level_begin;         // per merge level
  int desc_g = 0, desc_vtil = 0, desc_gemm1 = 0, desc_gemm2 = 0;
  std::vector<void*> allocs;
};

// dc.cu
bool dc_solve(cudaStream_t st, TridiagWs* ws, int* launches);

}  // namespace kc
