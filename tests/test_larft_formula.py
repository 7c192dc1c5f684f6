"""The algebra behind larft_cols_kernel (korali_b200/csrc/tridiag.cu), stated in NumPy: the compact-WY factor T of a panel of
Householder reflectors H_0 H_1 ... H_{k-1} = I - V T V^T (dlarft, forward / columnwise) is the inverse of the upper triangular
S = striu(V^T V) + diag(1 / tau), so every column of T follows from a back substitution of its own,
    t_jj = tau_j,   t_ij = -tau_i sum_{k = i+1 .. j} G_ik t_kj   (i = j-1 .. 0),
which is what one warp per column computes on the device. Checked against the column recurrence of dlarft (what a
column-sequential kernel computes) and against the product of the reflectors; tau_j = 0 (H_j = I) gives a zero row and column in both."""
import numpy as np


def reflectors(n, k, rng, zero_tau=()):
    v = np.zeros((n, k))
    tau = np.zeros(k)
    for j in range(k):
        x = rng.standard_normal(n - j - 1)
        v[j + 1:, j] = x / x[0] if x.size else []
        if x.size:
            v[j + 1, j] = 1.0
            tau[j] = 2.0 / (v[:, j] @ v[:, j])
        if j in zero_tau:
            tau[j] = 0.0
    return v, tau


def larft_recurrence(g, tau):
    k = len(tau)
    t = np.zeros((k, k))
    for p in range(k):
        t[:p, p] = -tau[p] * (t[:p, :p] @ g[:p, p])
        t[p, p] = tau[p]
    return t


def larft_columns(g, tau):
    k = len(tau)
    t = np.zeros((k, k))
    for j in range(k):                      # every column on its own
        t[j, j] = tau[j]
        for i in range(j - 1, -1, -1):
            t[i, j] = -tau[i] * (g[i, i + 1:j + 1] @ t[i + 1:j + 1, j])
    return t


def test_back_substitution_gives_the_dlarft_factor():
    rng = np.random.default_rng(11)
    for n, k, zero in [(40, 12, ()), (200, 128, ()), (64, 32, (3, 17)), (130, 128, (0,))]:
        v, tau = reflectors(n, k, rng, zero)
        g = v.T @ v
        t1, t2 = larft_recurrence(g, tau), larft_columns(g, tau)
        assert np.abs(t1 - t2).max() <= 1e-13 * max(1.0, np.abs(t1).max())
        q = np.eye(n)
        for j in range(k):
            q = q @ (np.eye(n) - tau[j] * np.outer(v[:, j], v[:, j]))
        assert np.abs((np.eye(n) - v @ t2 @ v.T) - q).max() <= 1e-12
        for j in zero:
            assert not t2[j].any() and not t2[:, j].any()
        nz = [j for j in range(k) if tau[j] != 0.0]
        s = np.triu(g, 1)[np.ix_(nz, nz)] + np.diag(1.0 / tau[nz])
        assert np.abs(t2[np.ix_(nz, nz)] @ s - np.eye(len(nz))).max() <= 1e-11
