"""GPU parity tests proper: every call goes through the C ABI of korali_b200/libkcma.so and is compared with the
CPU oracle (oracle/okcma.c) or with the reference's own saved trajectory (tests/golden).

Bars (BASELINE.json north_star): ranking / selection indices bit-exact; mean, paths, sigma and C within a relative
1e-11 in FP64 (TOL below); polynomial objectives bit-exact; optimum within 1e-8.
"""

import numpy as np
import pytest
import torch
from conftest import relerr
from korali_b200 import _lib
from korali_b200._abi import INJ_BD, INJ_BDZ, INJ_F, INJ_GRAD, INJ_X, INJ_Z, KcmaError
from oracle import oracle as O

pytestmark = pytest.mark.gpu
TOL = 1e-11  # stated FP64 tolerance for mean, evolution paths, sigma and C

if not torch.cuda.is_available():
    pytest.skip("needs a CUDA device", allow_module_level=True)


# ---------------------------------------------------------------- K1 Philox ---------------------------------
def test_philox_known_answers_on_device():
    assert _lib.k_philox_raw([0, 0, 0, 0], [0, 0]) == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    assert _lib.k_philox_raw([0xffffffff] * 4, [0xffffffff] * 2) == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    assert _lib.k_philox_raw([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0]) == \
        [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]
    for ctr, key in [([1, 2, 3, 4], [5, 6]), ([123456, 7, 0, 99], [0xdeadbeef, 0x1337])]:
        assert _lib.k_philox_raw(ctr, key) == O.philox4x32_10(ctr, key)


@pytest.mark.parametrize("rows,n,row_begin,gen", [(64, 10, 0, 1), (33, 7, 1000, 5), (4096, 100, 0, 2), (512, 1000, 65000, 3)])
def test_philox_normals_match_oracle(rows, n, row_begin, gen):
    z = _lib.k_philox_normal(1337, gen, row_begin, rows, n)
    zo = O.philox_normal(1337, gen, row_begin, rows, n)
    # same integer stream; log / sincos differ by a few ulp between libdevice and glibc
    assert np.abs(z - zo).max() < 5e-15 * max(1.0, np.abs(zo).max())
    assert np.isfinite(z).all()


def test_philox_independent_of_sharding():
    a = _lib.k_philox_normal(7, 3, 0, 256, 50)
    b = np.concatenate([_lib.k_philox_normal(7, 3, 0, 100, 50), _lib.k_philox_normal(7, 3, 100, 156, 50)])
    assert np.array_equal(a, b)


# ---------------------------------------------------------------- K4 sort -----------------------------------
@pytest.mark.parametrize("n", [1, 2, 31, 32, 33, 255, 256, 257, 511, 512, 513, 2047, 2048, 2049, 4096, 8192, 16384, 16385, 65536, 100003, 1 << 20])
def test_sort_index_bit_exact(n):
    rng = np.random.default_rng(n)
    f = rng.standard_normal(n) * 10.0 ** rng.integers(-30, 30, n)
    assert np.array_equal(_lib.k_sort_index(f), O.sort_index(f))


def test_sort_index_ties_and_signed_zero():
    rng = np.random.default_rng(1)
    for n in (50000, 9000, 700):   # radix passes | rank-by-counting (n <= 16384), several candidate chunks | one chunk pair
        f = rng.integers(-3, 4, n).astype(np.float64)
        f[::7] = -0.0
        f[3::11] = 0.0
        got = _lib.k_sort_index(f)
        assert np.array_equal(got, O.sort_index(f))
        assert np.array_equal(got, np.argsort(-f, kind="stable").astype(np.uint64))
    const = np.full(5000, -2.5)
    assert np.array_equal(_lib.k_sort_index(const), np.arange(5000, dtype=np.uint64))
    ext = np.array([1e308, -1e308, 5e-324, -5e-324, 0.0, 1.0, -1.0, 2.2250738585072014e-308])
    assert np.array_equal(_lib.k_sort_index(ext), O.sort_index(ext))


# ---------------------------------------------------------------- K2 sampling GEMM --------------------------
@pytest.mark.parametrize("rows,n", [(32, 10), (100, 100), (257, 129), (300, 257), (1000, 1000), (130, 999)])
def test_sampling_gemm_matches_oracle(rows, n):
    rng = np.random.default_rng(rows * 1000 + n)
    z = rng.standard_normal((rows, n))
    q, _ = np.linalg.qr(rng.standard_normal((n, n)))
    d = 10.0 ** rng.uniform(-3, 1, n)
    mean = rng.standard_normal(n) * 3
    sigma = 0.37
    y, x = _lib.k_sample(z, q, d, mean, sigma)
    yo, xo = O.sample(z, q, d, mean, sigma)
    assert relerr(y, yo) < 2e-14
    assert relerr(x, xo) < 2e-14


# ---------------------------------------------------------------- K6 rank-mu SYRK ---------------------------
@pytest.mark.parametrize("rows,n", [(16, 10), (5, 10), (500, 100), (2048, 129), (777, 257), (4096, 1000), (33, 999)])
def test_rank_mu_matches_oracle(rows, n):
    rng = np.random.default_rng(rows + n)
    t = rng.standard_normal((rows, n)) * 10.0 ** rng.uniform(-2, 2, n)[None, :]
    w = np.log(rows + 0.5) - np.log(np.arange(rows) + 1.0)
    w /= w.sum()
    p = _lib.k_rank_mu(t, w)
    po = O.rank_mu(t, w)
    scale = np.sqrt(np.outer(np.diag(po), np.diag(po)))
    assert (np.abs(p - po) / scale).max() < 1e-13
    assert np.array_equal(p, p.T)


# ---------------------------------------------------------------- K3 objectives -----------------------------
@pytest.mark.parametrize("obj", ["NegSphere", "NegSumSq", "NegRosenbrock", "NegEllipsoid"])
@pytest.mark.parametrize("rows,n", [(32, 10), (100, 100), (64, 1000), (9, 33), (3, 1)])
def test_polynomial_objectives_bit_exact(obj, rows, n):
    x = np.random.default_rng(n).standard_normal((rows, n)) * 3
    coef = 10.0 ** (6.0 * np.arange(n) / max(n - 1, 1))   # same coefficient bits on both sides
    assert np.array_equal(_lib.k_objective(obj, x, coef), O.objective(obj, x, coef))


@pytest.mark.parametrize("obj", ["NegAckley", "NegSphereSin2"])
def test_transcendental_objectives(obj):
    x = np.random.default_rng(5).standard_normal((200, 100)) * 2
    assert relerr(_lib.k_objective(obj, x), O.objective(obj, x)) < 1e-14


# ---------------------------------------------------------------- K8 eigen ----------------------------------
@pytest.mark.parametrize("n,cond", [(2, 10.0), (10, 1e3), (33, 1e6), (100, 1e8), (257, 1e4), (1000, 1e6), (1300, 1e3)])
def test_eigen_residuals_and_eigenvalues(n, cond):
    rng = np.random.default_rng(n)
    q, _ = np.linalg.qr(rng.standard_normal((n, n)))
    lam = np.sort(10.0 ** rng.uniform(0, np.log10(cond), n))
    c = (q * lam) @ q.T
    c = 0.5 * (c + c.T)
    w, v = _lib.k_eigen(c)
    assert np.all(np.diff(w) >= 0)
    assert np.abs(v @ np.diag(w) @ v.T - c).max() < 1e-12 * np.abs(c).max()
    assert np.abs(v.T @ v - np.eye(n)).max() < 1e-12
    wo, _ = O.eigen(c)
    assert np.abs(w - wo).max() < 1e-12 * lam.max()


@pytest.mark.parametrize("n", [25, 26, 27, 31, 120, 1001, 1180, 1184, 1185])
def test_eigen_kernel_boundaries(n):
    """Sizes around the dispatch limits of the eigensolver: 24|25 single-CTA -> pipelined kernel, rows that do not fill the
    last 4-row block / the even number of blocks (zero padding rows), 1184 = one CTA per SM (148 block pairs), 1185 = first
    size on the one-launch-per-step path. Checked on the decomposition itself (residual, orthonormality, order)."""
    rng = np.random.default_rng(1000 + n)
    q, _ = np.linalg.qr(rng.standard_normal((n, n)))
    lam = np.sort(10.0 ** rng.uniform(0, 3, n))
    c = (q * lam) @ q.T
    c = 0.5 * (c + c.T)
    w, v = _lib.k_eigen(c)
    assert np.all(np.diff(w) >= 0)
    assert np.abs(v @ np.diag(w) @ v.T - c).max() < 1e-12 * np.abs(c).max()
    assert np.abs(v.T @ v - np.eye(n)).max() < 1e-12
    assert np.abs(w - lam).max() < 1e-11 * lam.max()


@pytest.mark.parametrize("n", [64, 300])
def test_eigen_clustered_and_repeated_spectrum(n):
    """C = I + 1e-6 E (every eigenvalue in one cluster) and an exactly repeated eigenvalue: any orthonormal basis of an
    eigenspace is acceptable, so the check is the reconstruction and the orthonormality, not the vectors."""
    rng = np.random.default_rng(n)
    e = rng.standard_normal((n, n))
    c = np.eye(n) + 1e-6 * 0.5 * (e + e.T)
    w, v = _lib.k_eigen(c)
    assert np.abs(v @ np.diag(w) @ v.T - c).max() < 1e-13
    assert np.abs(v.T @ v - np.eye(n)).max() < 1e-12
    assert np.abs(w - np.linalg.eigvalsh(c)).max() < 1e-13
    q, _ = np.linalg.qr(rng.standard_normal((n, n)))
    lam = np.concatenate([np.full(n // 2, 2.0), np.full(n - n // 2, 5.0)])
    c2 = (q * lam) @ q.T
    c2 = 0.5 * (c2 + c2.T)
    w2, v2 = _lib.k_eigen(c2)
    assert np.abs(w2 - lam).max() < 1e-12
    assert np.abs(v2 @ np.diag(w2) @ v2.T - c2).max() < 1e-12
    assert np.abs(v2.T @ v2 - np.eye(n)).max() < 1e-12


@pytest.mark.parametrize("n,order", [(31, "ring"), (120, "ring"), (1000, "ring"), (200, "rr"), (300, "rr"), (600, "rr")])
def test_eigen_tournament_orders(n, order, monkeypatch):
    """Both tournament orders of jacobi_pipe_kernel, each reached by size: the ring order when padding the block count to a power
    of two costs <= 1/8 more steps (8, 32 and 256 blocks), else round-robin (50, 76 and 150 blocks). KCMA_EIGEN=jacobi, because
    without constraints these sizes go to the tridiagonal solver. Same decomposition quality; the eigenvalues agree to round-off."""
    monkeypatch.setenv("KCMA_EIGEN", "jacobi")
    rng = np.random.default_rng(77 + n)
    q, _ = np.linalg.qr(rng.standard_normal((n, n)))
    lam = np.sort(10.0 ** rng.uniform(0, 3, n))
    c = (q * lam) @ q.T
    c = 0.5 * (c + c.T)
    w, v = _lib.k_eigen(c)
    assert np.all(np.diff(w) >= 0)
    assert np.abs(v @ np.diag(w) @ v.T - c).max() < 1e-12 * np.abs(c).max()
    assert np.abs(v.T @ v - np.eye(n)).max() < 1e-12
    assert np.abs(w - lam).max() < 1e-11 * lam.max()


@pytest.mark.parametrize("n,order", [(2000, "ring"), (1300, "rr")])
def test_eigen_tournament_orders_large_n_path(n, order, monkeypatch):
    """Rows longer than 1280 run on the one-launch-per-step path with 16-row blocks, in both orders by size: N = 2000 has 126
    blocks, 128 with the ring order's two phantom blocks; N = 1300 has 82 blocks and takes the round-robin order. KCMA_EIGEN=jacobi
    as above; both must deliver the decomposition of a clustered CMA-ES-like spectrum."""
    monkeypatch.setenv("KCMA_EIGEN", "jacobi")
    rng = np.random.default_rng(n)
    z = rng.standard_normal((2 * n, n))
    c = 0.965 * np.eye(n) + 0.035 * (z.T @ z) / (2 * n)
    c = 0.5 * (c + c.T)
    w, v = _lib.k_eigen(c)
    assert np.all(np.diff(w) >= 0)
    assert np.abs(v @ np.diag(w) @ v.T - c).max() < 1e-12 * np.abs(c).max()
    assert np.abs(v.T @ v - np.eye(n)).max() < 1e-12
    assert np.abs(w - np.linalg.eigvalsh(c)).max() < 1e-12 * np.abs(w).max()


def test_eigen_identity_and_rejection():
    w, v = _lib.k_eigen(np.eye(7) * 2.0)
    assert np.allclose(w, 2.0) and np.abs(v.T @ v - np.eye(7)).max() < 1e-14
    with pytest.raises(KcmaError, match="positive definite"):
        _lib.k_eigen(np.diag([1.0, -1.0, 2.0]))


# ---------------------------------------------------------------- golden trajectory on the GPU --------------
N, LAM = 10, 32
STATE_ARR = ["Covariance Matrix", "Current Mean", "Previous Mean", "Evolution Path", "Conjugate Evolution Path", "Best Ever Variables"]
STATE_SCA = ["Sigma", "Best Ever Value", "Current Best Value", "Previous Best Value", "Previous Best Ever Value"]


def make_gpu(golden, **kw):
    return _lib.Solver(n=N, population_size=LAM, objective="NegSphere", seed=int(golden["Normal Generator Seed"][0]),
                       lower_bound=golden["Lower Bound"], upper_bound=golden["Upper Bound"], keep_population=1,
                       initial_value=golden["Initial Value"], initial_stddev=golden["Initial Standard Deviation"], **kw)


def test_init_constants_bit_exact_on_gpu(golden):
    s = make_gpu(golden)
    assert np.array_equal(s.get("Mu Weights"), golden["Mu Weights"][1])
    for k in ["Effective Mu", "Sigma Cumulation Factor", "Damp Factor", "Cumulative Covariance", "Chi Square Number", "Trace"]:
        assert s.scalar(k) == golden[k][1], k
    assert s.scalar("Sigma") == np.sqrt(22.5)
    assert np.array_equal(s.get("Covariance Eigenvector Matrix").reshape(N, N), np.eye(N))
    assert np.array_equal(s.get("Covariance Matrix").reshape(N, N), np.eye(N))


def test_golden_trajectory_all_transitions_on_gpu(golden):
    """State(g-1) + the reference's own {B, D, X, F}(g) -> State(g), g = 1..100, against the reference's dumps."""
    worst = 0.0
    for g in range(1, 101):
        s = make_gpu(golden)
        if g > 1:
            for k in STATE_ARR:
                s.set(k, golden[k][g - 1])
            for k in STATE_SCA:
                s.set_scalar(k, golden[k][g - 1])
            s.set_scalar("Current Generation", g - 1)
            s.set_scalar("Model Evaluation Count", golden["Model Evaluation Count"][g - 1])
        s.inject(INJ_BD, np.concatenate([golden["Covariance Eigenvector Matrix"][g], golden["Axis Lengths"][g]]))
        s.inject(INJ_X, golden["Sample Population"][g])
        s.inject(INJ_F, golden["Value Vector"][g])
        s.run_generation()
        assert np.array_equal(s.get_index("Sorting Index"), golden["Sorting Index"][g].astype(np.uint64)), g
        for k in ["Current Mean", "Previous Mean", "Mean Update", "Evolution Path", "Conjugate Evolution Path", "Covariance Matrix",
                  "Best Ever Variables", "Current Best Variables"]:
            e = relerr(s.get(k), golden[k][g]); worst = max(worst, e)
            assert e < TOL, (g, k, e)
        for k in ["Sigma", "Conjugate Evolution Path L2 Norm", "Best Ever Value", "Current Best Value",
                  "Maximum Diagonal Covariance Matrix Element", "Minimum Diagonal Covariance Matrix Element",
                  "Current Min Standard Deviation", "Current Max Standard Deviation"]:
            a, b = s.scalar(k), golden[k][g]
            assert abs(a - b) <= TOL * abs(b), (g, k, a, b)
        assert s.scalar("Current Generation") == g
        assert s.scalar("Model Evaluation Count") == golden["Model Evaluation Count"][g]
        s.close()
    print("worst relative deviation from the reference dumps over 100 transitions: %.2e" % worst)


def test_golden_sampling_from_reference_z(golden):
    """Injecting the reference's own z draws (MT19937 stream) and its (B, D) reproduces its BDZ Matrix / Sample Population."""
    for g in (1, 2, 50):
        s = make_gpu(golden)
        if g > 1:
            for k in STATE_ARR:
                s.set(k, golden[k][g - 1])
            s.set_scalar("Sigma", golden["Sigma"][g - 1])
            s.set_scalar("Current Generation", g - 1)
        b = golden["Covariance Eigenvector Matrix"][g].reshape(N, N)
        d = golden["Axis Lengths"][g]
        # z = D^-1 B^T y of the reference's BDZ (exact for g=1 where B=I, D=1)
        z = (golden["BDZ Matrix"][g].reshape(LAM, N) @ b) / d
        s.inject(INJ_BD, np.concatenate([b.ravel(), d]))
        s.inject(INJ_Z, z)
        s.ask()
        assert relerr(s.get("BDZ Matrix"), golden["BDZ Matrix"][g]) < 1e-13
        assert relerr(s.get("Sample Population"), golden["Sample Population"][g]) < 1e-13
        s.close()


# ---------------------------------------------------------------- lockstep with the oracle ------------------
CASES = [
    dict(n=10, population_size=32, objective="NegRosenbrock", initial_value=0.3, initial_stddev=1.5),                   # config 1
    dict(n=100, population_size=4096, objective="NegAckley", initial_value=1.0, initial_stddev=3.0),                   # config 2
    dict(n=64, population_size=256, objective="NegSphere", mirrored_sampling=1, initial_value=1.0, initial_stddev=1.0),  # mirrored
    dict(n=50, population_size=128, objective="NegEllipsoid", diagonal_covariance=1, initial_value=3.0, initial_stddev=1.0),
    dict(n=33, population_size=40, mu_value=7, mu_type="Linear", objective="NegSumSq", initial_value=2.0, initial_stddev=0.5),
    dict(n=20, population_size=64, mu_type="Equal", objective="NegSphereSin2", initial_value=1.0, initial_stddev=2.0),
    dict(n=257, population_size=2048, objective="NegEllipsoid", initial_value=3.0, initial_stddev=1.0),
]


@pytest.mark.parametrize("case", CASES, ids=lambda c: "%s-N%d-l%d" % (c["objective"], c["n"], c["population_size"]))
def test_lockstep_generations_against_oracle(case):
    """Same (B, D, y) and F injected into both each generation; state must track within TOL for 15 generations."""
    o = O.Oracle(seed=11, **case)
    s = _lib.Solver(seed=11, keep_population=1, **case)
    o.set_scalar("Oracle/RNG Kind", 1)
    n, lam = case["n"], case["population_size"]
    exact_f = case["objective"] in ("NegRosenbrock", "NegSphere", "NegEllipsoid", "NegSumSq")
    for g in range(15):
        o.ask()
        bd = np.concatenate([o.get("Covariance Eigenvector Matrix"), o.get("Axis Lengths")])
        s.inject(INJ_BD, bd)
        s.inject(INJ_BDZ, o.get("BDZ Matrix"))
        s.ask()
        # x = m + sigma*y recomputed on the device from the injected y; m and sigma carry the device's own rounding
        # history (<= TOL), so compare with a tolerance, then pin X for a strict lockstep of the ranking
        assert relerr(s.get("Sample Population"), o.get("Sample Population")) < 1e-13, g
        if g == 0:
            assert np.array_equal(s.get("Sample Population"), o.get("Sample Population"))
        s.inject(INJ_X, o.get("Sample Population"))
        o.eval()
        fo = o.get("Value Vector")
        if exact_f:
            s.eval()
            assert np.array_equal(s.get("Value Vector"), fo), g   # device objective bit-identical
        else:
            s.eval()
            assert relerr(s.get("Value Vector"), fo) < 1e-13
            s.inject(INJ_F, fo)   # keep the ranking in lockstep
            s.set_scalar("Model Evaluation Count", s.scalar("Model Evaluation Count") - lam)
            s.eval()
        o.tell(); s.tell()
        assert np.array_equal(s.get_index("Sorting Index"), o.get_index("Sorting Index")), g
        for k in ["Current Mean", "Mean Update", "Evolution Path", "Conjugate Evolution Path", "Covariance Matrix",
                  "Best Ever Variables", "Current Best Variables"]:
            assert relerr(s.get(k), o.get(k)) < TOL, (g, k, relerr(s.get(k), o.get(k)))
        for k in ["Sigma", "Conjugate Evolution Path L2 Norm", "Best Ever Value", "Current Best Value",
                  "Current Min Standard Deviation", "Current Max Standard Deviation"]:
            a, b = s.scalar(k), o.scalar(k)
            assert abs(a - b) <= TOL * max(abs(b), 1e-300), (g, k, a, b)


def test_device_eigensystem_reproduces_covariance_each_generation():
    """Free-running (own Philox draws, own eigensolver): B D^2 B^T == C and B orthogonal at every generation."""
    s = _lib.Solver(n=40, population_size=200, objective="NegEllipsoid", seed=3, initial_value=3.0, initial_stddev=1.0)
    for g in range(30):
        c = s.get("Covariance Matrix").reshape(40, 40)
        s.ask()
        b = s.get("Covariance Eigenvector Matrix").reshape(40, 40)
        d = s.get("Axis Lengths")
        assert np.abs((b * d**2) @ b.T - c).max() < 1e-12 * np.abs(c).max(), g
        assert np.abs(b.T @ b - np.eye(40)).max() < 1e-12
        assert np.all(np.diff(d) >= 0)
        s.eval(); s.tell()


# ---------------------------------------------------------------- convergence -------------------------------
CONV = [
    ("config1: 10-D Rosenbrock, lambda 32", dict(n=10, population_size=32, objective="NegRosenbrock", initial_value=0.0, initial_stddev=0.5), 6000),
    ("config2: 100-D Ackley, lambda 4096", dict(n=100, population_size=4096, objective="NegAckley", initial_value=1.0, initial_stddev=3.0), 1500),
    ("config3 (reduced): 200-D ellipsoid, lambda 2048", dict(n=200, population_size=2048, objective="NegEllipsoid", initial_value=3.0, initial_stddev=1.0), 2500),
    ("config4 (reduced): 256-D sphere mirrored", dict(n=256, population_size=4096, objective="NegSphere", mirrored_sampling=1, initial_value=1.0, initial_stddev=1.0), 800),
    ("diagonal covariance: 100-D sphere", dict(n=100, population_size=256, objective="NegSphere", diagonal_covariance=1, initial_value=1.0, initial_stddev=1.0), 1500),
]


@pytest.mark.parametrize("name,case,max_gens", CONV, ids=[c[0].split(":")[0] for c in CONV])
def test_converges_to_the_optimum_within_1e8(name, case, max_gens):
    s = _lib.Solver(seed=1337, **case)
    s.set_scalar("Termination Criteria/Max Value", -1e-9)
    s.set_scalar("Termination Criteria/Max Generations", max_gens)
    s.set_scalar("Termination Criteria/Max Model Evaluations", 1e15)
    done = s.run(max_gens + 1)
    best = s.scalar("Best Ever Value")
    fin, reason = s.check_termination()
    print("%s: best %.3e after %d generations (%s)" % (name, best, done, reason))
    assert fin and abs(best) < 1e-8, (name, best, done, reason)
    xb = s.get("Best Ever Variables")
    target = 1.0 if case["objective"] == "NegRosenbrock" else 0.0
    assert np.abs(xb - target).max() < 1e-3


# ---------------------------------------------------------------- free-running (no injection) ---------------
def _track(s, o, gens, tol, int_keys=(), label=""):
    for g in range(gens):
        s.run_generation(); o.run_generation()
        for k in int_keys:
            assert s.scalar(k) == o.scalar(k), (label, g, k, s.scalar(k), o.scalar(k))
        assert np.array_equal(s.get_index("Sorting Index"), o.get_index("Sorting Index")), (label, g)
        for k in ["Current Mean", "Evolution Path", "Conjugate Evolution Path", "Covariance Matrix"]:
            e = relerr(s.get(k), o.get(k))
            assert e < tol, (label, g, k, e)
        assert abs(s.scalar("Sigma") - o.scalar("Sigma")) < tol * o.scalar("Sigma"), (label, g)


def test_free_running_matches_oracle_philox_stream():
    """No injection at all: device Philox + device eigensolver vs the oracle's restatement of both (same counters,
    same eigenvector sign convention). Looser tolerance: eigenvectors of two different solvers agree to ~eps*|C|/gap."""
    case = dict(n=16, population_size=48, objective="NegRosenbrock", initial_value=0.1, initial_stddev=0.7, seed=99)
    s = _lib.Solver(**case); o = O.Oracle(**case); o.set_scalar("Oracle/RNG Kind", 1)
    _track(s, o, 25, 1e-8, label="rosenbrock")


@pytest.mark.parametrize("case", [
    dict(n=10, population_size=32, objective="NegRosenbrock", initial_value=0.0, initial_stddev=0.5, seed=7),                       # single-CTA eigensolver
    dict(n=100, population_size=512, objective="NegAckley", initial_value=1.0, initial_stddev=3.0, seed=8),                           # pipelined eigensolver
    dict(n=40, population_size=64, objective="NegSphere", initial_value=2.0, initial_stddev=1.0, seed=9, mirrored_sampling=1),
    dict(n=40, population_size=64, objective="NegEllipsoid", initial_value=2.0, initial_stddev=1.0, seed=10, diagonal_covariance=1),
    dict(n=12, population_size=24, objective="NegSphere", initial_value=1.0, initial_stddev=1.0, seed=11, lower_bound=-5.0, upper_bound=5.0),
])
def test_graph_replay_is_bit_identical_to_eager_launches(case):
    """kcma_run_generation replays one captured CUDA graph per generation from the third generation on (launch-latency-bound
    configurations, SURVEY 8d); kcma_ask / kcma_eval / kcma_tell always launch eagerly. Same kernels, same arguments except
    the generation counter (read from the device in the graph): every piece of state must be bit-identical."""
    a = _lib.Solver(**case); b = _lib.Solver(**case)
    for g in range(40):
        a.run_generation()
        b.ask(); b.eval(); b.tell()
        if g in (0, 1, 2, 3, 10, 39):
            for k in ["Current Mean", "Evolution Path", "Conjugate Evolution Path", "Covariance Matrix", "Covariance Eigenvector Matrix",
                      "Axis Lengths", "Value Vector", "Best Ever Variables"]:
                assert np.array_equal(a.get(k), b.get(k)), (g, k)
            for k in ["Sigma", "Best Ever Value", "Current Best Value", "Conjugate Evolution Path L2 Norm", "Current Generation",
                      "Model Evaluation Count", "Infeasible Sample Count"]:
                assert a.scalar(k) == b.scalar(k), (g, k)
    # state changes through the API drop the graph; the next generation is captured again and still agrees
    a.set_scalar("Sigma", 0.5); b.set_scalar("Sigma", 0.5)
    for g in range(5):
        a.run_generation()
        b.ask(); b.eval(); b.tell()
    assert np.array_equal(a.get("Covariance Matrix"), b.get("Covariance Matrix")) and a.scalar("Sigma") == b.scalar("Sigma")
    a.close(); b.close()


@pytest.mark.parametrize("mode", ["ask_tell", "timing"])
def test_graph_then_eager_then_graph_keeps_the_generation_counter(mode):
    """The graph replay reads the generation (Philox counter, hsig exponent :658) from DevScalars::gen; eager generations in
    between (kcma_ask/eval/tell, or kcma_timing_enable(1) as bench.py does) advance only the host counter. The device copy must
    be re-seeded before the next replay, otherwise earlier generations' z draws are reused."""
    case = dict(n=20, population_size=64, objective="NegRosenbrock", initial_value=0.1, initial_stddev=0.6, seed=21)
    a = _lib.Solver(**case); b = _lib.Solver(**case)
    def eager(s, k):
        for _ in range(k):
            s.ask(); s.eval(); s.tell()
    eager(b, 22)
    for _ in range(6):
        a.run_generation()                      # 1-2 eager, 3-6 graph
    if mode == "ask_tell":
        eager(a, 5)                             # 7-11 eager; the graph stays alive
    else:
        a.timing_enable(True)
        for _ in range(5):
            a.run_generation()
        a.timing_enable(False)
    for _ in range(4):
        a.run_generation()                      # 12-15 graph again
    eager(a, 3)
    for _ in range(4):
        a.run_generation()                      # 19-22
    assert a.scalar("Current Generation") == b.scalar("Current Generation") == 22
    for k in ["Current Mean", "Evolution Path", "Conjugate Evolution Path", "Covariance Matrix", "Value Vector", "Best Ever Variables"]:
        assert np.array_equal(a.get(k), b.get(k)), k
    assert a.scalar("Sigma") == b.scalar("Sigma") and a.scalar("Best Ever Value") == b.scalar("Best Ever Value")
    a.close(); b.close()


# ---------------------------------------------------------------- Use Gradient Information ------------------
@pytest.mark.parametrize("case", [
    dict(n=10, population_size=32, objective="NegSphere", initial_value=2.0, initial_stddev=1.5, gradient_step_size=0.01),
    dict(n=24, population_size=48, objective="NegRosenbrock", initial_value=0.2, initial_stddev=0.4, gradient_step_size=2e-6),
    dict(n=30, population_size=64, objective="NegEllipsoid", initial_value=1.0, initial_stddev=1.0, gradient_step_size=1e-8, mirrored_sampling=1),
    dict(n=16, population_size=40, objective="NegAckley", initial_value=1.0, initial_stddev=2.0, gradient_step_size=0.05),
    dict(n=12, population_size=24, objective="NegSphereSin2", initial_value=1.0, initial_stddev=1.0, gradient_step_size=0.02, mu_type="Linear"),
], ids=lambda c: c["objective"])
def test_gradient_information_lockstep_against_oracle(case):
    """"Use Gradient Information" (CMAES.cpp.base:611-621): device gradients of the built-in objectives and the gradient step
    of the mean against the oracle, in lockstep (same B, D, y, X injected)."""
    o = O.Oracle(seed=21, use_gradient_information=1, **case)
    s = _lib.Solver(seed=21, keep_population=1, use_gradient_information=1, **case)
    o.set_scalar("Oracle/RNG Kind", 1)
    n, lam = case["n"], case["population_size"]
    for g in range(12):
        o.ask()
        s.inject(INJ_BD, np.concatenate([o.get("Covariance Eigenvector Matrix"), o.get("Axis Lengths")]))
        s.inject(INJ_BDZ, o.get("BDZ Matrix"))
        s.ask()
        s.inject(INJ_X, o.get("Sample Population"))
        o.eval(); s.eval()
        go, gs = o.get("Gradients").reshape(lam, n), s.get("Gradients").reshape(lam, n)
        assert np.abs(gs - go).max() <= 1e-12 * np.abs(go).max(), g
        s.inject(INJ_F, o.get("Value Vector")); s.inject(INJ_GRAD, go)   # keep ranking and gradients in lockstep
        s.set_scalar("Model Evaluation Count", s.scalar("Model Evaluation Count") - lam)
        s.eval()
        o.tell(); s.tell()
        assert np.array_equal(s.get_index("Sorting Index"), o.get_index("Sorting Index")), g
        for k in ["Current Mean", "Mean Update", "Evolution Path", "Conjugate Evolution Path", "Covariance Matrix"]:
            assert relerr(s.get(k), o.get(k)) < 1e-11, (g, k, relerr(s.get(k), o.get(k)))
        assert abs(s.scalar("Sigma") - o.scalar("Sigma")) <= 1e-11 * o.scalar("Sigma")


def test_gradient_information_host_callback_injection_and_errors():
    case = dict(n=8, population_size=16, objective="External", initial_value=1.0, initial_stddev=0.7, seed=4, keep_population=1,
                use_gradient_information=1, gradient_step_size=0.01)
    a = _lib.Solver(**case)
    a.set_host_objective_grad(lambda x: (-0.5 * (x**2).sum(1), -x))
    b = _lib.Solver(**{**case, "objective": "NegSphere"})
    for g in range(20):
        a.run_generation(); b.run_generation()
    assert relerr(a.get("Current Mean"), b.get("Current Mean")) < 1e-10 and abs(a.scalar("Sigma") - b.scalar("Sigma")) < 1e-10 * b.scalar("Sigma")
    c = _lib.Solver(**case)
    c.ask()
    x = c.get("Sample Population").reshape(16, 8)
    c.inject(INJ_F, -0.5 * (x**2).sum(1))
    with pytest.raises(KcmaError, match="inject the gradients"):
        c.eval()
    with pytest.raises(KcmaError, match="Gradient Step Size must be larger than 0.0"):
        _lib.Solver(**{**case, "gradient_step_size": 0.0})
    with pytest.raises(KcmaError, match="Use Gradient Information is off"):
        d = _lib.Solver(n=4, population_size=8, objective="NegSphere", initial_value=1.0, initial_stddev=1.0)
        d.ask(); d.inject(INJ_GRAD, np.zeros(32))


# ---------------------------------------------------------------- discrete variables (Granularity) ----------
@pytest.mark.parametrize("case", [
    dict(n=6, population_size=16, objective="NegSphere", initial_value=3.3, initial_stddev=2.0, lower_bound=-20.0, upper_bound=20.0,
         granularity=np.array([1.0, 1.0, 0.0, 0.0, 0.5, 0.0])),
    dict(n=10, population_size=8, objective="NegEllipsoid", initial_value=1.0, lower_bound=-19.0, upper_bound=21.0,
         granularity=np.array([1.0, 1.0, 0.0, 1.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0])),          # examples/optimization/discrete/run-cmaes.py
    dict(n=12, population_size=24, objective="NegSumSq", initial_value=2.7, initial_stddev=1.5, mirrored_sampling=1,
         granularity=np.array([2.0, 0.0, 0.25] * 4)),
], ids=["sphere6", "discrete-example", "mirrored"])
def test_discrete_variables_lockstep_against_oracle(case):
    """Mixed-integer CMA-ES (Granularity): the device's discrete mutations (own Philox uniform stream), discretize, masking
    matrices and masked step-size update against the oracle, in lockstep on the eigensystem and the normal draws."""
    o = O.Oracle(seed=31, **case)
    s = _lib.Solver(seed=31, **case)
    o.set_scalar("Oracle/RNG Kind", 1)
    n, lam = case["n"], case["population_size"]
    saw_mutation = False
    for g in range(60):
        o.ask()
        s.inject(INJ_BD, np.concatenate([o.get("Covariance Eigenvector Matrix"), o.get("Axis Lengths")]))
        s.inject(INJ_BDZ, o.get("BDZ Matrix"))
        s.ask()
        xo, xs = o.get("Sample Population").reshape(lam, n), s.get("Sample Population").reshape(lam, n)
        disc = case["granularity"] > 0
        assert np.array_equal(xs[:, disc], xo[:, disc]), g                      # grid values: bit-identical
        assert np.abs(xs - xo).max() <= 1e-12 * max(np.abs(xo).max(), 1.0), g
        assert np.array_equal(s.get("Discrete Mutations").reshape(lam, n)[:, disc] != 0, o.get("Discrete Mutations").reshape(lam, n)[:, disc] != 0), g
        saw_mutation |= bool(o.get("Discrete Mutations").any())
        s.inject(INJ_X, xo.ravel())
        o.eval(); s.eval()
        s.inject(INJ_F, o.get("Value Vector"))
        s.set_scalar("Model Evaluation Count", s.scalar("Model Evaluation Count") - lam)
        s.eval()
        o.tell(); s.tell()
        assert np.array_equal(s.get_index("Sorting Index"), o.get_index("Sorting Index")), g
        for k in ["Masking Matrix", "Masking Matrix Sigma"]:
            assert np.array_equal(s.get(k), o.get(k)), (g, k)
        for k in ["Number Of Discrete Mutations", "Number Masking Matrix Entries", "Infeasible Sample Count"]:
            assert s.scalar(k) == o.scalar(k), (g, k)
        assert abs(s.scalar("Chi Square Number Discrete Mutations") - o.scalar("Chi Square Number Discrete Mutations")) < 1e-14
        for k in ["Current Mean", "Evolution Path", "Conjugate Evolution Path", "Covariance Matrix"]:
            assert relerr(s.get(k), o.get(k)) < 1e-11, (g, k, relerr(s.get(k), o.get(k)))
        assert abs(s.scalar("Sigma") - o.scalar("Sigma")) <= 1e-11 * o.scalar("Sigma"), g
    assert saw_mutation


def test_discrete_variables_free_running_reaches_the_grid_optimum():
    gran = np.array([1.0, 1.0, 0.0, 1.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0])
    s = _lib.Solver(n=10, population_size=8, objective="NegEllipsoid", initial_value=1.0, lower_bound=-19.0, upper_bound=21.0, granularity=gran, seed=5)
    s.set_scalar("Termination Criteria/Max Value", -1e-9)
    done = s.run(3000)
    xb = s.get("Best Ever Variables")
    assert np.all(xb[gran > 0] == 0.0) and abs(s.scalar("Best Ever Value")) < 1e-8, (done, xb)
    with pytest.raises(KcmaError, match="Negative granularity"):
        _lib.Solver(n=2, population_size=8, objective="NegSphere", initial_value=1.0, initial_stddev=1.0, granularity=np.array([1.0, -1.0]))


def _constrained_problem(n):
    """4 half-space constraints g_c(x) = -(x_c - shift_c) <= 0 after helpers.py activeMax*: x_0, x_1 >= 1 (active at the
    optimum), x_2, x_3 >= -1 (violated by the initial mean -> viability regime, inactive at the optimum)."""
    iv = np.zeros(n); iv[0] = iv[1] = 4.0; iv[2] = iv[3] = -2.0
    return dict(objective="NegSphereSin2", constraint_family="HalfSpace", n_constraints=4,
                constraint_shift=np.array([1.0, 1.0, -1.0, -1.0]), lower_bound=-10.0, upper_bound=10.0, initial_value=iv,
                initial_stddev=1.0, is_sigma_bounded=1)


def test_constraint_path_viability_regime_against_oracle():
    """config 5 (reduced): 4 half-space constraints, infeasible initial mean -> viability regime -> regime switch.
    Counters must agree exactly, state within tolerance (sequential EMA restated in parallel, SURVEY 7)."""
    case = dict(n=20, population_size=64, viability_population_size=64, seed=1337, **_constrained_problem(20))
    s = _lib.Solver(**case); o = O.Oracle(**case); o.set_scalar("Oracle/RNG Kind", 1)
    ints = ["Is Viability Regime", "Current Population Size", "Covariance Matrix Adaptation Count", "Resampled Parameter Count",
            "Constraint Evaluation Count", "Max Constraint Violation Count", "Infeasible Sample Count", "Best Valid Sample"]
    saw_regime_switch = False
    for g in range(40):
        s.run_generation(); o.run_generation()
        for k in ints:
            assert s.scalar(k) == o.scalar(k), (g, k, s.scalar(k), o.scalar(k))
        saw_regime_switch |= (s.scalar("Is Viability Regime") == 0)
        assert np.array_equal(s.get_index("Sorting Index"), o.get_index("Sorting Index")), g
        assert np.array_equal(s.get_index("Sample Constraint Violation Counts"), o.get_index("Sample Constraint Violation Counts")), g
        for k in ["Current Mean", "Evolution Path", "Conjugate Evolution Path", "Covariance Matrix", "Viability Boundaries",
                  "Normal Constraint Approximation", "Best Ever Variables"]:
            e = relerr(s.get(k), o.get(k))
            assert e < 1e-8, (g, k, e)
        assert abs(s.scalar("Sigma") - o.scalar("Sigma")) < 1e-8 * o.scalar("Sigma"), g
    assert saw_regime_switch
    assert o.scalar("Covariance Matrix Adaptation Count") > 0


def test_constrained_optimum_config5():
    """config 5: N=100, lambda=8192 (both population sizes), 4 synthetic constraints, infeasible initial mean. Optimum of
    -sum(x^2+sin^2 x) on the feasible set: x_0 = x_1 = 1, all else 0: F* = -2 (1 + sin(1)^2)."""
    case = dict(n=100, population_size=8192, viability_population_size=8192, seed=1337, **_constrained_problem(100))
    s = _lib.Solver(**case)
    s.set_scalar("Termination Criteria/Max Generations", 400)
    s.set_scalar("Termination Criteria/Max Model Evaluations", 1e15)
    done = s.run(401)
    fstar = -2 * (1 + np.sin(1.0) ** 2)
    best = s.scalar("Best Ever Value")
    xb = s.get("Best Ever Variables")
    print("config5: best %.10f (F* %.10f) after %d generations, corrections %d" % (best, fstar, done, s.scalar("Covariance Matrix Adaptation Count")))
    assert s.scalar("Is Viability Regime") == 0
    assert np.all(xb[:2] >= 1.0 - 1e-9) and np.all(xb[2:4] >= -1.0)
    assert abs(best - fstar) < 1e-6 and best <= fstar + 1e-9


def test_warm_started_eigensolver_does_not_drift():
    """The eigenvector basis is carried from generation to generation (warm start). After 1500 generations it must
    still be orthonormal and reproduce C (no accumulation of rotation round-off)."""
    n = 48
    s = _lib.Solver(n=n, population_size=96, objective="NegRosenbrock", seed=4, initial_value=0.0, initial_stddev=0.5)
    s.set_scalar("Termination Criteria/Max Model Evaluations", 1e15)
    s.run(1500)
    c = s.get("Covariance Matrix").reshape(n, n)
    s.ask()
    b = s.get("Covariance Eigenvector Matrix").reshape(n, n)
    d = s.get("Axis Lengths")
    orth = np.abs(b.T @ b - np.eye(n)).max()
    res = np.abs((b * d**2) @ b.T - c).max() / np.abs(c).max()
    print("after 1500 generations: |B^T B - I| = %.2e, |B D^2 B^T - C|/|C| = %.2e, cond = %.2e" % (orth, res, (d.max() / d.min())**2))
    assert orth < 1e-12 and res < 1e-12


# ---------------------------------------------------------------- edge cases ---------------------------------
@pytest.mark.parametrize("kw", [
    dict(n=1, population_size=2, objective="NegSphere", initial_value=1.0, initial_stddev=1.0),
    dict(n=1, population_size=8, objective="NegSumSq", mirrored_sampling=1, initial_value=2.0, initial_stddev=1.0),
    dict(n=3, population_size=5, mu_value=2, objective="NegRosenbrock", initial_value=0.0, initial_stddev=0.3),   # mu = 1 would make C = aI + b y y^T degenerate: eigenbasis arbitrary
    dict(n=17, population_size=34, objective="NegEllipsoid", mirrored_sampling=1, initial_value=1.0, initial_stddev=1.0),
    dict(n=25, population_size=26, objective="NegSphere", initial_value=1.0, initial_stddev=1.0),      # smallest N on the Gram eigen path
    dict(n=129, population_size=130, objective="NegSphere", diagonal_covariance=1, initial_value=1.0, initial_stddev=1.0),
    dict(n=130, population_size=64, mu_type="Proportional", objective="NegSumSq", initial_value=1.0, initial_stddev=0.5),
], ids=lambda k: "N%d-l%d" % (k["n"], k["population_size"]))
def test_ragged_and_minimal_shapes_free_running(kw):
    """Smallest / odd / ragged shapes through the whole generation loop against the oracle. When mu >= N the spectrum of C
    is non-degenerate and both sides run free on the Philox stream; otherwise C = aI + (rank < N) has a degenerate
    eigenspace whose basis is arbitrary, so the oracle's (B, D, y) are injected and the rest of the loop is compared."""
    n, lam = kw["n"], kw["population_size"]
    mu = kw.get("mu_value", lam // 2)
    free = (mu >= n) and not kw.get("mirrored_sampling") or kw.get("diagonal_covariance")
    s = _lib.Solver(seed=7, keep_population=1, **kw); o = O.Oracle(seed=7, **kw); o.set_scalar("Oracle/RNG Kind", 1)
    for g in range(6):
        if free:
            s.run_generation(); o.run_generation()
        else:
            o.ask()
            s.inject(INJ_BD, np.concatenate([o.get("Covariance Eigenvector Matrix"), o.get("Axis Lengths")]))
            s.inject(INJ_BDZ, o.get("BDZ Matrix"))
            s.ask()
            assert relerr(s.get("Sample Population"), o.get("Sample Population")) < 1e-12
            s.inject(INJ_X, o.get("Sample Population"))
            s.eval(); o.eval(); s.tell(); o.tell()
        assert np.array_equal(s.get_index("Sorting Index"), o.get_index("Sorting Index")), g
        for k in ["Current Mean", "Evolution Path", "Conjugate Evolution Path", "Covariance Matrix"]:
            assert relerr(s.get(k), o.get(k)) < 1e-9, (g, k)
        assert abs(s.scalar("Sigma") - o.scalar("Sigma")) < 1e-9 * o.scalar("Sigma")
    # the device's own eigensolver + sampler on this shape: B D^2 B^T == C, finite samples
    c = s.get("Covariance Matrix").reshape(n, n)
    s.ask()
    b = s.get("Covariance Eigenvector Matrix").reshape(n, n); d = s.get("Axis Lengths")
    if not kw.get("diagonal_covariance"):
        assert np.abs((b * d**2) @ b.T - c).max() < 1e-12 * np.abs(c).max()
        assert np.abs(b.T @ b - np.eye(n)).max() < 1e-12
    assert np.isfinite(s.get("Sample Population")).all()


def test_invalid_configurations_raise():
    """setInitialConfiguration range checks (CMAES.cpp.base:26, 89-93, 111-126, 131-136)."""
    base = dict(n=4, population_size=8, objective="NegSphere", initial_value=0.0, initial_stddev=1.0)
    for bad, match in [(dict(population_size=1), "larger 1"), (dict(population_size=7, mirrored_sampling=1), "even Sample Population"),
                       (dict(initial_value=None), "cannot be inferred"), (dict(initial_stddev=None), "cannot be inferred"),
                       (dict(mirrored_sampling=1, constraint_family="HalfSpace", n_constraints=1), "not applicable to problems with constraints"),
                       (dict(constraint_family="HalfSpace", n_constraints=2, target_success_rate=1.5), "Invalid Target Success Rate"),
                       (dict(objective=77), None)]:
        kw = dict(base); kw.update(bad)
        if bad.get("objective") == 77:
            s = _lib.Solver(**kw)
            with pytest.raises(KcmaError, match="unknown objective"):
                s.run_generation()
            continue
        with pytest.raises(KcmaError, match=match):
            _lib.Solver(**kw)
    # defaults inferred from the bounds: mid-domain start, 0.3 * width (:111-126)
    s = _lib.Solver(n=2, population_size=4, objective="NegSphere", lower_bound=[-2.0, 0.0], upper_bound=[4.0, 10.0])
    assert np.array_equal(s.get("Current Mean"), [1.0, 5.0])
    assert abs(s.scalar("Sigma") - np.sqrt((1.8**2 + 3.0**2) / 2)) < 1e-14


def test_bound_violations_counted_and_resampled_like_the_oracle():
    """isSampleFeasible + the rejection loop of prepareGeneration (:446-459). Default (Max Infeasible Resamplings = 0, SURVEY Q2):
    violations are counted, never resampled. With a finite limit every infeasible sample is redrawn (Philox attempt counter)."""
    kw = dict(n=6, population_size=64, objective="NegSphere", lower_bound=-1.0, upper_bound=1.0, initial_value=0.5, initial_stddev=1.0, seed=3)
    s = _lib.Solver(keep_population=1, **kw); o = O.Oracle(**kw); o.set_scalar("Oracle/RNG Kind", 1)
    s.ask(); o.ask()
    assert s.scalar("Infeasible Sample Count") == o.scalar("Infeasible Sample Count") > 0
    assert relerr(s.get("Sample Population"), o.get("Sample Population")) < 1e-13
    kw["max_infeasible_resamplings"] = 100000
    s = _lib.Solver(keep_population=1, **kw); o = O.Oracle(**kw); o.set_scalar("Oracle/RNG Kind", 1)
    for g in range(3):
        s.ask(); o.ask()
        x = s.get("Sample Population")
        assert np.all(np.abs(x) <= 1.0)                              # every sample feasible after resampling
        assert s.scalar("Infeasible Sample Count") == o.scalar("Infeasible Sample Count")
        assert relerr(x, o.get("Sample Population")) < 1e-12          # same (sample, attempt) Philox counters
        s.eval(); o.eval(); s.tell(); o.tell()


@pytest.mark.parametrize("mirrored", [0, 1])
@pytest.mark.parametrize("maxres", [1, 7, 40, 41, 200])
def test_resampling_budget_exhausted_mid_population_like_the_reference(mirrored, maxres):
    """'Max Infeasible Resamplings' bounds the rejection loop by the CUMULATIVE counter (:459, :490), so when the budget runs out
    the reference's sample-by-sample order decides which draws are kept: samples before that point are resampled to the end, the
    one that exhausts the budget keeps an infeasible draw, every later sample keeps its first draw. The device redraws in rounds
    and settles the budget afterwards (settle_resampling_budget): counter and population must equal the oracle's sequential loop."""
    kw = dict(n=5, population_size=48, objective="NegSphere", lower_bound=-1.0, upper_bound=1.0, initial_value=0.6, initial_stddev=1.2, seed=17,
              mirrored_sampling=mirrored, max_infeasible_resamplings=maxres)
    s = _lib.Solver(keep_population=1, **kw); o = O.Oracle(**kw); o.set_scalar("Oracle/RNG Kind", 1)
    for g in range(3):
        s.ask(); o.ask()
        assert s.scalar("Infeasible Sample Count") == o.scalar("Infeasible Sample Count"), (g, s.scalar("Infeasible Sample Count"), o.scalar("Infeasible Sample Count"))
        assert relerr(s.get("Sample Population"), o.get("Sample Population")) < 1e-12, g
        s.eval(); o.eval(); s.tell(); o.tell()
        assert np.array_equal(s.get_index("Sorting Index"), o.get_index("Sorting Index")), g
    assert s.scalar("Infeasible Sample Count") >= maxres
    fin_s, why_s = s.check_termination(); fin_o, why_o = o.check_termination()
    assert fin_s and fin_o and "Max Infeasible Resamplings" in why_s and why_s == why_o


def test_nonfinite_objective_is_an_error():
    """Optimization::evaluate throws on a non-finite F(x) (optimization.cpp.base:32-33)."""
    s = _lib.Solver(n=4, population_size=8, objective="NegEllipsoid", objective_coef=[1.0, 1.0, np.inf, 1.0], initial_value=1.0, initial_stddev=1.0)
    with pytest.raises(KcmaError, match="Non finite value of function evaluation"):
        s.run_generation()
    s = _lib.Solver(n=4, population_size=8, objective="External", initial_value=1.0, initial_stddev=1.0)
    s.ask()
    with pytest.raises(KcmaError, match="Non finite"):
        s.inject(INJ_F, [1.0, 2.0, np.nan, 0, 0, 0, 0, 0])
