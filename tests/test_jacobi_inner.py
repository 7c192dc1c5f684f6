"""CPU tests of the register-resident 8x8 inner solver of the Jacobi eigensolver (korali_b200/csrc/jacobi_inner.cuh).

The header is host/device code; here it is built with g++ and checked against numpy: the accumulated R must be
orthonormal to FP64 precision, R Gamma R^T must equal the tracked Gamma, and one pass must annihilate the cross pairs the
way cyclic Jacobi does (quadratic reduction of the off-diagonal mass once it is small).
"""
import ctypes as C
import os
import subprocess
import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def inner(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("jinner") / "libjinner.so")
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-o", so,
                           os.path.join(HERE, "helpers", "jacobi_inner_host.cpp")])
    lib = C.CDLL(so)
    dp = C.POINTER(C.c_double)
    lib.jacobi_inner_host.argtypes = [dp, C.c_double, C.c_int, dp, dp, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.jacobi_cs_host.argtypes = [C.c_double, C.c_double, C.c_double, dp, dp, C.POINTER(C.c_int)]

    def run(gamma, tol, mode):
        g = np.ascontiguousarray(gamma, dtype=np.float64)
        R = np.zeros((8, 8)); go = np.zeros((8, 8)); rot = C.c_int(0); big = C.c_int(0)
        lib.jacobi_inner_host(g.ctypes.data_as(dp), tol, mode, R.ctypes.data_as(dp), go.ctypes.data_as(dp), C.byref(rot), C.byref(big))
        return R, go, rot.value, big.value

    def cs(a, b, g):
        c = C.c_double(); s = C.c_double(); safe = C.c_int()
        lib.jacobi_cs_host(a, b, g, C.byref(c), C.byref(s), C.byref(safe))
        return c.value, s.value, safe.value
    run.cs = cs
    run.lib = lib
    return run


def _gram(rng, cols=40, scale=None):
    X = rng.standard_normal((8, cols))
    if scale is not None:
        X *= np.asarray(scale)[:, None]
    return X, X @ X.T


def test_rotation_parameters_orthonormal_and_annihilating(inner):
    rng = np.random.default_rng(1)
    for _ in range(2000):
        X = rng.standard_normal((2, 12)) * 10.0 ** rng.uniform(-6, 6, size=(2, 1))
        a, b, g = X[0] @ X[0], X[1] @ X[1], X[0] @ X[1]
        c, s, safe = inner.cs(a, b, g)
        assert safe == 1
        assert abs(c * c + s * s - 1.0) < 7e-16
        p, q = c * X[0] - s * X[1], s * X[0] + c * X[1]
        # a 22-bit angle leaves |cos| <= ~1e-6 of the original one
        assert abs(p @ q) <= 2e-6 * abs(g) + 1e-15 * np.sqrt(a * b)
        assert abs(s) <= c * (1 + 1e-6)          # inner rotation: |theta| <= pi/4


def test_rotation_parameters_extreme_exponents(inner):
    for e in (-170.0, 170.0, -300.0, 300.0):
        sc = 10.0 ** e
        c, s, safe = inner.cs(2.0 * sc, 3.0 * sc, 0.5 * sc)
        c0, s0, _ = inner.cs(2.0, 3.0, 0.5)
        assert abs(c * c + s * s - 1.0) < 7e-16
        assert abs(c - c0) < 1e-6 and abs(s - s0) < 1e-6
    assert inner.cs(2e170, 3e170, 0.5e170)[2] == 0   # the scaled path was taken


@pytest.mark.parametrize("mode", [0, 1])
def test_inner_solver_tracks_gamma_and_reduces_offdiagonal(inner, mode):
    rng = np.random.default_rng(7 + mode)
    for trial in range(200):
        scale = 10.0 ** rng.uniform(-3, 3, size=8) if trial % 2 else None
        X, G = _gram(rng, scale=scale)
        if mode == 0:   # blocks internally orthogonal, as after the first step of a sweep
            for blk in (slice(0, 4), slice(4, 8)):
                q, r = np.linalg.qr(X[blk].T)
                X[blk] = (q * np.abs(np.diag(r))).T
            G = X @ X.T
        R, Go, rot, big = inner(G, 1e-14, mode)
        assert rot > 0 and big == 1
        assert np.abs(R @ R.T - np.eye(8)).max() < 2e-15
        ref = R @ G @ R.T
        nrm = np.sqrt(np.outer(np.diag(ref), np.diag(ref)))
        # the tracked Gamma uses closed forms for the pivot entries (22-bit angle): good to ~1e-6 of the rotated-away part
        assert (np.abs(ref - Go) / nrm).max() < 2e-6
        # the rows really rotated: Gram of R X equals the tracked Gamma
        Y = R @ X
        assert (np.abs(Y @ Y.T - ref) / nrm).max() < 1e-13
        cosb = np.abs(G / np.sqrt(np.outer(np.diag(G), np.diag(G))))
        cosa = np.abs(Go / nrm)
        sel = np.zeros((8, 8), bool)
        if mode == 0:
            sel[:4, 4:] = True
        else:
            sel[np.triu_indices(8, 1)] = True
        assert (cosa[sel] ** 2).sum() < (cosb[sel] ** 2).sum()


def test_inner_solver_quadratic_tail_and_noop(inner):
    rng = np.random.default_rng(3)
    d = np.array([1.0, 2.0, 3.5, 5.0, 7.0, 11.0, 13.0, 17.0])
    E = rng.standard_normal((8, 8)) * 1e-6
    G = np.diag(d) + E + E.T
    R, Go, rot, big = inner(G, 1e-14, 0)
    off = np.abs(Go[:4, 4:]).max()
    assert rot == 16 and big == 1 and off < 1e-10          # ~ (1e-6)^2 / gap, plus the 22-bit angle residual
    # below tolerance: nothing happens, R = I exactly, Gamma untouched
    G2 = np.diag(d) + (E + E.T) * 1e-12
    R2, Go2, rot2, big2 = inner(G2, 1e-14, 0)
    assert rot2 == 0 and big2 == 0 and np.array_equal(R2, np.eye(8)) and np.array_equal(Go2, G2)
    # rotated pairs already below 1e-10: counted, but not "big"
    G3 = np.diag(d) + (E + E.T) * 1e-6
    R3, Go3, rot3, big3 = inner(G3, 1e-14, 0)
    assert rot3 > 0 and big3 == 0
    # zero padding rows (alpha = 0) never rotate and never produce NaN
    G4 = G.copy(); G4[6:, :] = 0.0; G4[:, 6:] = 0.0
    R4, Go4, rot4, _ = inner(G4, 1e-14, 0)
    assert np.isfinite(R4).all() and np.isfinite(Go4).all() and np.array_equal(R4[6:, 6:], np.eye(2))


@pytest.mark.parametrize("order,sizes", [(0, [2, 4, 6, 8, 26, 250, 296]), (1, [2, 4, 8, 16, 32, 256])])
def test_tournament_schedules_are_one_factorisations(inner, order, sizes):
    """Both tournament orders of jacobi_pipe_kernel (rr_pair / ring_pair, the code the kernel runs): every step pairs every
    block exactly once, every pair of blocks meets exactly once per sweep, p < q. The ring order additionally keeps the
    first block of slot k in place for all but log2(np) - 1 of the step transitions."""
    so = inner.lib
    for nb in sizes:
        seen = set()
        prev_p, stays = None, 0
        for step in range(nb - 1):
            used, ps = [], []
            for k in range(nb // 2):
                p, q = C.c_int(-1), C.c_int(-1)
                so.jacobi_pair_host(order, nb, step, k, C.byref(p), C.byref(q))
                assert 0 <= p.value < q.value < nb
                used += [p.value, q.value]
                ps.append(p.value)
                assert (p.value, q.value) not in seen
                seen.add((p.value, q.value))
            assert sorted(used) == list(range(nb))
            if prev_p is not None:
                stays += sum(1 for a, b in zip(ps, prev_p) if a == b)
            prev_p = ps
        assert len(seen) == nb * (nb - 1) // 2
        if order == 1 and nb >= 8:
            # slot k changes its first block only when a sub-tournament hands it a block of the B half: at most once per level
            assert stays >= (nb - 2) * (nb // 2) - (nb // 2) * (int(np.log2(nb)) - 1)
