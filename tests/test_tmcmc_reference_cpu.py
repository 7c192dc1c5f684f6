"""Bayesian/Reference on the CPU: the oracle's per-point likelihood terms (oracle/otmcmc.c) against scipy, its TMCMC evidence against
independently computed evidences over 10 seeds, and the configuration errors of the Korali surface (raised before any device is
needed)."""
import ctypes as C
import numpy as np
import pytest
from scipy import integrate, special, stats
import korali_b200 as korali
from korali_b200._tmcmc import LIKELIHOODS
import tmcmc_reference_oracle as otmcmc
from tmcmc_reference_oracle import OracleTMCMC

SEEDS = range(1, 11)


def _f(name, *argtypes):
    f = getattr(otmcmc.lib(), name)
    f.restype, f.argtypes = C.c_double, list(argtypes)
    return np.vectorize(f, otypes=[np.float64])


TERM = _f("otmcmc_reference_term", C.c_int32, C.c_double, C.c_double, C.c_double)
LOG_NDTR = _f("otmcmc_log_ndtr", C.c_double)
ERFCX = _f("otmcmc_erfcx", C.c_double)


def close(a, b, rtol, atol=0.0):
    a, b = np.asarray(a), np.asarray(b)
    same_inf = np.isinf(a) & (a == b)
    with np.errstate(invalid="ignore"):
        return bool(np.all(same_inf | (np.abs(a - b) <= rtol * np.abs(b) + atol)))


# ---- the terms against scipy (1e-13 relative per term)

def test_normal_term():
    r = np.random.default_rng(1)
    d, g, s = r.normal(0, 5, 2000), r.normal(0, 5, 2000), np.exp(r.uniform(-8, 8, 2000))
    assert close(TERM(LIKELIHOODS["Normal"], d, g, s), stats.norm.logpdf(d, loc=g, scale=s), 1e-13)


def test_log_ndtr_is_finite_where_the_naive_form_is_not():
    """log Phi(u) over [-1e4, 40]. Above u = -1 it is log(erfc(-u / sqrt 2) / 2), whose absolute error is one rounding of a value near
    1 (log Phi -> 0 from below there), hence the absolute floor of 2.3e-16."""
    u = np.concatenate([-np.logspace(4, -3, 3000), np.linspace(0, 40, 1000)])
    with np.errstate(divide="ignore"):
        assert np.isinf(np.log(special.ndtr(-40.0)))      # the naive form
    got = LOG_NDTR(u)
    assert np.isfinite(got[u < 38]).all()
    assert close(got, special.log_ndtr(u), 1e-13, 2.3e-16)


def test_positive_normal_term():
    """The Normal term minus log Phi(g / sigma), down to g / sigma = -1e4. The two parts cancel for very negative g / sigma, so the
    tolerance is relative to their magnitudes."""
    r = np.random.default_rng(2)
    s = np.exp(r.uniform(-4, 4, 3000))
    u = np.concatenate([-np.logspace(4, -2, 1500), r.uniform(-3, 40, 1500)])
    g, d = u * s, r.uniform(0, 10, 3000)
    n, c = stats.norm.logpdf(d, loc=g, scale=s), special.log_ndtr(g / s)
    got = TERM(LIKELIHOODS["Positive Normal"], d, g, s)
    assert np.isfinite(got).all()
    assert np.all(np.abs(got - (n - c)) <= 1e-13 * (np.abs(n) + np.abs(c)) + 2.3e-16)


def test_student_t_term():
    """Against scipy below nu = 100; above, scipy's log(poch(nu / 2, 1 / 2)) loses up to 5e-13 (nu ~ 800) and 1e-11 (nu ~ 1e4), so
    the reference there is the same formula in 40-digit arithmetic (mpmath)."""
    import mpmath
    r = np.random.default_rng(3)
    nu = np.concatenate([np.logspace(np.log10(0.5), 6, 2000), [49.999999, 50.0, 50.000001]])
    d, g = r.normal(0, 3, nu.size), r.normal(0, 3, nu.size)
    got = TERM(LIKELIHOODS["StudentT"], d, g, nu)
    lo = nu < 100
    assert close(got[lo], stats.t.logpdf(d[lo] - g[lo], nu[lo]), 1e-13)
    mpmath.mp.dps = 40
    def exact(x, n):
        x, n = mpmath.mpf(x), mpmath.mpf(n)
        return float(mpmath.loggamma((n + 1) / 2) - mpmath.loggamma(n / 2) - mpmath.log(n * mpmath.pi) / 2 - (n + 1) / 2 * mpmath.log1p(x * x / n))
    assert close(got[~lo], [exact(a - b, n) for a, b, n in zip(d[~lo], g[~lo], nu[~lo])], 1e-13)


def test_poisson_term():
    r = np.random.default_rng(4)
    d = np.concatenate([r.integers(0, 200, 2000), [0, 0, 3]]).astype(np.float64)
    g = np.concatenate([np.exp(r.uniform(-5, 6, 2000)), [0.0, 2.5, 0.0]])
    got, ref = TERM(LIKELIHOODS["Poisson"], d, g, 0.0), stats.poisson.logpmf(d, g)
    assert got[-3] == 0.0 and got[-2] == -2.5 and got[-1] == -np.inf
    assert close(got, ref, 1e-13)


def test_erfcx_against_scipy():
    x = np.concatenate([np.linspace(-20, 10, 3001), np.logspace(1, 5, 2000), [49.999999, 50.0, 50.000001]])
    assert close(ERFCX(x), special.erfcx(x), 1e-13)


# ---- the oracle's TMCMC against independent evidences (4 standard errors over 10 seeds)

def evidence_runs(kw, model):
    z = []
    for s in SEEDS:
        o = OracleTMCMC(seed=s, **kw)
        o.set_host_reference(model)
        o.run(1000)
        assert o.scalar("Annealing Exponent") == 1.0
        z.append(o.scalar("LogEvidence"))
    return np.array(z)


def within(z, log_z):
    assert abs(z.mean() - log_z) <= 4 * z.std(ddof=1) / np.sqrt(len(z)), (z.mean(), z.std(ddof=1), log_z)


def quad_log_evidence(loglik, lo, hi):
    """log of (1 / (hi - lo)) * integral of exp(loglik) over [lo, hi] (one variable, Uniform prior)."""
    grid = np.linspace(lo, hi, 2001)
    shift = max(loglik(x) for x in grid)
    val, _ = integrate.quad(lambda x: np.exp(loglik(x) - shift), lo, hi, points=[grid[np.argmax([loglik(x) for x in grid])]], limit=200,
                            epsabs=0, epsrel=1e-10)
    return np.log(val / (hi - lo)) + shift


def test_normal_linear_model_meets_the_gaussian_evidence():
    """g_j = a + b t_j, known sigma, Normal priors: log Z = log N(d; Phi mu0, sigma^2 I + Phi Sigma0 Phi^T)."""
    t = np.linspace(-1.0, 1.0, 8)
    sigma, mu0, s0 = 0.5, np.array([0.3, -0.2]), np.array([1.0, 1.5])
    d = 0.7 + 1.3 * t + sigma * np.random.default_rng(5).normal(size=t.size)
    Phi = np.stack([np.ones_like(t), t], 1)
    exact = stats.multivariate_normal.logpdf(d, Phi @ mu0, sigma**2 * np.eye(t.size) + Phi @ np.diag(s0**2) @ Phi.T)
    kw = dict(n=2, population_size=2000, priors=[("Normal", mu0[0], s0[0]), ("Normal", mu0[1], s0[1])], reference=("Normal", d))
    within(evidence_runs(kw, lambda X: (X[:, :1] + X[:, 1:2] * t, sigma)), exact)


def test_positive_normal_evidence():
    d, sigma = np.array([0.2, 1.1, 0.6, 0.05, 1.7]), 0.8
    def loglik(th):
        return np.sum(stats.norm.logpdf(d, th, sigma)) - d.size * special.log_ndtr(th / sigma)
    kw = dict(n=1, population_size=2000, priors=[("Uniform", -3.0, 3.0)], reference=("Positive Normal", d))
    within(evidence_runs(kw, lambda X: (X[:, :1], sigma)), quad_log_evidence(loglik, -3.0, 3.0))


def test_student_t_evidence():
    d, nu = np.array([1.2, -0.4, 2.9, 0.8, 1.5, 0.1]), 3.0
    def loglik(th):
        return np.sum(stats.t.logpdf(d - th, nu))
    kw = dict(n=1, population_size=2000, priors=[("Uniform", -5.0, 5.0)], reference=("StudentT", d))
    within(evidence_runs(kw, lambda X: (X[:, :1], nu)), quad_log_evidence(loglik, -5.0, 5.0))


def test_poisson_evidence():
    d = np.array([3.0, 5.0, 2.0, 4.0, 0.0, 6.0])
    def loglik(th):
        return np.sum(stats.poisson.logpmf(d, th))
    kw = dict(n=1, population_size=2000, priors=[("Uniform", 0.0, 12.0)], reference=("Poisson", d))
    within(evidence_runs(kw, lambda X: X[:, :1]), quad_log_evidence(loglik, 0.0, 12.0))


# ---- configuration errors of the Korali surface

def base(likelihood="Normal", data=(0.5, 1.0, 1.5)):
    e = korali.Experiment()
    e["Problem"]["Type"] = "Bayesian/Reference"
    e["Problem"]["Likelihood Model"] = likelihood
    e["Problem"]["Reference Data"] = list(data)
    e["Problem"]["Computational Model"] = lambda s: None
    e["Distributions"][0]["Name"] = "P"
    e["Distributions"][0]["Type"] = "Univariate/Uniform"
    e["Distributions"][0]["Minimum"] = -10.0
    e["Distributions"][0]["Maximum"] = 10.0
    e["Variables"][0]["Name"] = "X0"
    e["Variables"][0]["Prior Distribution"] = "P"
    e["Solver"]["Type"] = "Sampler/TMCMC"
    e["Solver"]["Population Size"] = 100
    e["Console Output"]["Verbosity"] = "Silent"
    e["File Output"]["Enabled"] = False
    return e


def without(key):
    e = korali.Experiment()
    e["Problem"]["Type"] = "Bayesian/Reference"
    for k, v in (("Likelihood Model", "Normal"), ("Reference Data", [1.0]), ("Computational Model", lambda s: None)):
        if k != key:
            e["Problem"][k] = v
    e["Distributions"][0]["Name"] = "P"
    e["Distributions"][0]["Type"] = "Univariate/Uniform"
    e["Distributions"][0]["Minimum"] = -1.0
    e["Distributions"][0]["Maximum"] = 1.0
    e["Variables"][0]["Prior Distribution"] = "P"
    e["Solver"]["Type"] = "Sampler/TMCMC"
    e["Solver"]["Population Size"] = 100
    return e


@pytest.mark.parametrize("key", ["Likelihood Model", "Reference Data", "Computational Model"])
def test_mandatory_keys(key):
    with pytest.raises(RuntimeError, match=r"Bayesian/Reference \] \n \+ Key:    \['%s'\]\n \+ Reason: mandatory setting missing" % key):
        korali.Engine().run(without(key))


@pytest.mark.parametrize("make,match", [
    (lambda: base("Banana"), r"\['Likelihood Model'\]\n \+ Reason: unknown value 'Banana'"),
    (lambda: base("Positive StudentT"), "'Positive StudentT' is not built on the B200 path"),
    (lambda: base("geometric"), "'geometric' is not built on the B200 path"),
    (lambda: base("Negative Binomial"), "Normal, Positive Normal, StudentT and Poisson are"),
    (lambda: base(data=()), r"\['Reference Data'\]\n \+ Reason: a non-empty array"),
    (lambda: base(data=(1.0, float("nan"))), "entry 1 is not a finite number"),
    (lambda: base(data=(float("inf"),)), "entry 0 is not a finite number"),
    (lambda: base("Poisson", (1.0, -2.0)), "entry 1 .* must be a non-negative integer for the Poisson likelihood"),
    (lambda: base("Poisson", (1.5,)), "entry 0 .* must be a non-negative integer for the Poisson likelihood"),
    (lambda: base("Positive Normal", (0.0, -0.1)), r"entry 1 \(-0.1\) must be >= 0 for the Positive Normal likelihood"),
])
def test_configuration_errors(make, match):
    with pytest.raises(RuntimeError, match=match):
        korali.Engine().run(make())


def test_string_computational_model():
    e = base()
    e["Problem"]["Computational Model"] = "Sphere"
    with pytest.raises(RuntimeError, match="there is no built-in device computational model"):
        korali.Engine().run(e)


def test_unrecognised_problem_key():
    e = base()
    e["Problem"]["Bogus Key"] = 1
    with pytest.raises(RuntimeError, match="Unrecognized settings for Korali module: Bayesian/Reference"):
        korali.Engine().run(e)


def test_likelihood_names_are_case_insensitive():
    """A valid configuration gets past the parsing: without a GPU it stops at the device, not at a setting."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("CPU-only behaviour")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        korali.Engine().run(base("positive normal"))
