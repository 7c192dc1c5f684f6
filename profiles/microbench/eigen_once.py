"""One stand-alone eigendecomposition (kcma_k_eigen) of a CMA-ES-like covariance, for `ncu --metrics gpu__time_duration.sum`
launch lists of the tridiagonalisation path (sytrd_kernel, dc_*, gemm_tn_batched_kernel, larft_cols_kernel ...).

    python profiles/microbench/eigen_once.py [n] [repeats]
"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import numpy as np
from korali_b200 import _lib

n = int(sys.argv[1]) if len(sys.argv) > 1 else 1000
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 2
rng = np.random.default_rng(5)
e = rng.standard_normal((n, 2 * n))
c = 0.9 * np.eye(n) + 0.1 * (e @ e.T) / (2 * n)
c = 0.5 * (c + c.T)
for _ in range(reps):
    w, v = _lib.k_eigen(c)
print("n", n, "residual", np.abs(c @ v - v * w).max(), "orthonormality", np.abs(v.T @ v - np.eye(n)).max())
if os.environ.get("KCMA_SYTRD_PROF"):
    _lib.k_sytrd(c)
