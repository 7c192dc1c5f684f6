"""The TMCMC oracle (oracle/otmcmc.c) against closed forms, the invariants of the algorithm stated in include/ktmcmc.h, and the
configuration errors of the Bayesian/Custom + Sampler/TMCMC surface (raised before any device is needed). CPU only."""
import numpy as np
import pytest
import korali_b200 as korali
from oracle.otmcmc import OracleTMCMC

SEEDS = range(1, 11)


def runs(kw):
    z, m, v = [], [], []
    for s in SEEDS:
        o = OracleTMCMC(seed=s, **kw)
        o.run(1000)
        assert o.scalar("Annealing Exponent") == 1.0
        X = o.get("Sample Database").reshape(kw["population_size"], kw["n"])
        z.append(o.scalar("LogEvidence")); m.append(X.mean(0)); v.append(X.var(0))
    return np.array(z), np.array(m), np.array(v)


def check(z, m, v, log_z, mean, var):
    """Every estimate within 4 standard errors of the 10 seeds' mean."""
    k = len(z)
    assert abs(z.mean() - log_z) <= 4 * z.std(ddof=1) / np.sqrt(k), (z.mean(), log_z)
    assert np.all(np.abs(m.mean(0) - mean) <= 4 * m.std(0, ddof=1) / np.sqrt(k)), (m.mean(0), mean)
    assert np.all(np.abs(v.mean(0) - var) <= 4 * v.std(0, ddof=1) / np.sqrt(k)), (v.mean(0), var)


def test_sphere_uniform_prior():
    """-x.x/2 with Uniform[-a, a]^N priors: log Z = N (log(2 pi)/2 - log 2a). lambda = 2000, N = 2, a = 10, seeds 1..10: log Z
    -4.220 +- 0.123 (exact -4.154)."""
    a, n = 10.0, 2
    z, m, v = runs(dict(n=n, population_size=2000, priors=[("Uniform", -a, a)] * n, loglik="NegSphere"))
    check(z, m, v, n * (0.5 * np.log(2 * np.pi) - np.log(2 * a)), np.zeros(n), np.ones(n))


def test_ellipsoid_uniform_prior():
    """-sum c_i x_i^2 with c = (0.5, 2) and Uniform[-8, 8]^2: a product of Gaussians of variance 1 / (2 c_i),
    log Z = sum_i (log(pi / c_i)/2 - log 16). Seeds 1..10: -4.463 +- 0.132 (exact -4.400)."""
    c = np.array([0.5, 2.0])
    z, m, v = runs(dict(n=2, population_size=2000, priors=[("Uniform", -8.0, 8.0)] * 2, loglik="NegEllipsoid", loglik_coef=c))
    check(z, m, v, np.sum(0.5 * np.log(np.pi / c) - np.log(16.0)), np.zeros(2), 1.0 / (2 * c))


def test_normal_prior_conjugate():
    """Normal(mu0 = 0.5, s0 = 2) prior x exp(-x^2/2) likelihood, per dimension: posterior N(mu0 / (1 + s0^2), s0^2 / (1 + s0^2)),
    log Z = -log(1 + s0^2)/2 - mu0^2 / (2 (1 + s0^2)). Seeds 1..10, N = 2: -1.657 +- 0.039 (exact -1.659)."""
    mu0, s0, n = 0.5, 2.0, 2
    z, m, v = runs(dict(n=n, population_size=2000, priors=[("Normal", mu0, s0)] * n, loglik="NegSphere"))
    q = 1 + s0 * s0
    check(z, m, v, n * (-0.5 * np.log(q) - mu0 * mu0 / (2 * q)), np.full(n, mu0 / q), np.full(n, s0 * s0 / q))


@pytest.mark.parametrize("L,burn", [(1, 0), (3, 0), (2, 2)])
def test_invariants(L, burn):
    lam, n = 500, 3
    o = OracleTMCMC(n=n, population_size=lam, max_chain_length=L, default_burn_in=burn, priors=[("Uniform", -2.0, 2.0)] * n,
                      loglik="NegEllipsoid", seed=4)
    o.run_generation()
    assert o.scalar("Model Evaluation Count") == lam
    while o.scalar("Annealing Exponent") < 1.0:
        evals = o.scalar("Model Evaluation Count")
        o.anneal()
        if o.scalar("Annealing Exponent") < 1.0 and o.scalar("Annealing Exponent Update") > 1e-5:
            assert abs(o.scalar("Coefficient Of Variation") - 1.0) <= 1e-8
        elif o.scalar("Annealing Exponent") < 1.0:     # clamped to "Min Annealing Exponent Update"
            assert o.scalar("Coefficient Of Variation") > 1.0
        o.resample()
        counts, lens = o.get("Selection Counts"), o.get("Chain Lengths")
        assert counts.sum() == lam and lens.sum() == lam and lens.max() <= L
        assert (o.get("Chain Leaders") == np.repeat(np.nonzero(counts)[0], np.ceil(counts[counts > 0] / L).astype(int))).all()
        assert o.scalar("Max Chain Steps") == burn + lens.max()
        for _ in range(int(o.scalar("Max Chain Steps"))):
            o.propose()
            evals += (o.get("Proposal Support") == 1).sum()
            o.eval(); o.accept()
        assert o.scalar("Model Evaluation Count") == evals      # out-of-support proposals are not evaluated
        assert o.get("Sample Database").size == lam * n and np.isfinite(o.get("Sample LogPrior Database")).all()


def base():
    e = korali.Experiment()
    e["Problem"]["Type"] = "Bayesian/Custom"
    e["Problem"]["Likelihood Model"] = "Sphere"
    e["Distributions"][0]["Name"] = "P"
    e["Distributions"][0]["Type"] = "Univariate/Uniform"
    e["Distributions"][0]["Minimum"] = -10.0
    e["Distributions"][0]["Maximum"] = 10.0
    for i in range(2):
        e["Variables"][i]["Name"] = "X%d" % i
        e["Variables"][i]["Prior Distribution"] = "P"
    e["Solver"]["Type"] = "Sampler/TMCMC"
    e["Solver"]["Population Size"] = 100
    e["Console Output"]["Verbosity"] = "Silent"
    e["File Output"]["Enabled"] = False
    return e


def without_likelihood_model():
    e2 = korali.Experiment()
    e2["Problem"]["Type"] = "Bayesian/Custom"
    e2["Distributions"][0]["Name"] = "P"
    e2["Distributions"][0]["Type"] = "Univariate/Uniform"
    e2["Distributions"][0]["Minimum"] = -1.0
    e2["Distributions"][0]["Maximum"] = 1.0
    e2["Variables"][0]["Prior Distribution"] = "P"
    e2["Solver"]["Type"] = "Sampler/TMCMC"
    e2["Solver"]["Population Size"] = 100
    return e2


@pytest.mark.parametrize("mod,match", [
    (lambda e: e["Distributions"][0].__setitem__("Type", "Univariate/Gamma"), "prior distribution type 'Univariate/Gamma'"),
    (lambda e: e["Variables"][2].__setitem__("Name", "X2"), "has no 'Prior Distribution'"),
    (lambda e: e["Variables"][1].__setitem__("Prior Distribution", "Q"), "'Q' is not defined"),
    (lambda e: e["Solver"].__setitem__("Version", "mTMCMC"), "mTMCMC is not built"),
    (lambda e: e["Problem"].__setitem__("Type", "Optimization"), "only Problem Type 'Bayesian/Custom'"),
    (lambda e: e["Solver"].__setitem__("Bogus Key", 1), "Unrecognized settings for Korali module: TMCMC"),
    (lambda e: e["Problem"].__setitem__("Likelihood Model", "Banana"), "Unknown device likelihood model"),
    (lambda e: e["Solver"].__setitem__("Termination Criteria", 5), r"TMCMC \] \n \+ Key:    \['Termination Criteria'\]\n \+ Reason: not an object"),
])
def test_configuration_errors(mod, match):
    e = base()
    mod(e)
    e["Solver"]["Type"]     # reset the cursor after the chained access above
    with pytest.raises(RuntimeError, match=match):
        korali.Engine().run(e)


def test_missing_likelihood_model():
    with pytest.raises(RuntimeError, match="Likelihood Model"):
        korali.Engine().run(without_likelihood_model())


def test_runs_on_one_device():
    k = korali.Engine()
    k["Conduit"]["Devices"] = 2
    with pytest.raises(RuntimeError, match="Sampler/TMCMC runs on one device"):
        k.run(base())

