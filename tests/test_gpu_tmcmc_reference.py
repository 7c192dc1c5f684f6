"""Sampler/TMCMC for Bayesian/Reference problems on the B200: the likelihood kernel (tm_reference_loglik_kernel) against the CPU oracle
(oracle/otmcmc.c) and scipy, the device stepped in lockstep with the oracle for every likelihood, the three computational-model
kinds of the Korali surface, a full-size run against the closed form, the runtime errors and the README example."""
import os
import numpy as np
import pytest
import torch
from scipy import special, stats
import korali_b200 as korali
from korali_b200 import _tmcmc
from tmcmc_reference_oracle import OracleTMCMC

pytestmark = pytest.mark.gpu

LIKS = ["Normal", "Positive Normal", "StudentT", "Poisson"]


def rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


# ---- the kernel against the oracle and scipy

def pending_eval(make, rows, lik, data):
    """A handle (one variable, Normal prior) with `rows` evaluation rows waiting. One row: generation 1 with a single sample of finite
    log-likelihood, so that every draw picks it, Max Chain Length = lambda makes one chain, and a zero proposal factor keeps it."""
    kw = dict(n=1, priors=[("Normal", 0.0, 1.0)], reference=(lik, data), seed=5)
    if rows > 1:
        h = make(population_size=rows, **kw)
        h.propose()
        return h
    h = make(population_size=64, max_chain_length=64, **kw)
    h.propose(); h.inject_loglik([0.0] + [-np.inf] * 63); h.eval(); h.accept()
    h.anneal(); h.inject_factor([0.0]); h.resample(); h.propose()
    return h


def outputs(lik, rows, m, seed=1):
    """Data and model outputs with the edge values of each likelihood: sigma down to 1e-8, g / sigma down to -1e3, nu from 0.5 to
    1e6, Poisson zeros (d = 0, and g = 0 where d = 0)."""
    r = np.random.default_rng(seed)
    G, P = np.empty((rows, m)), np.empty((rows, m))
    if lik == "Poisson":
        d = r.integers(0, 50, m).astype(np.float64)
        d[::3] = 0.0
    elif lik == "Positive Normal":
        d = r.uniform(0.0, 3.0, m)
    else:
        d = r.normal(0.0, 1.0, m)
    for i0 in range(0, rows, 4096):
        k = min(rows, i0 + 4096) - i0
        if lik == "Normal":
            P[i0:i0 + k] = np.exp(r.uniform(np.log(1e-3), np.log(1e3), (k, m)))
            P[i0:i0 + k, ::97] = 1e-8
            G[i0:i0 + k] = d + r.normal(0.0, 1.0, (k, m))
        elif lik == "Positive Normal":
            P[i0:i0 + k] = np.exp(r.uniform(np.log(1e-2), np.log(1e2), (k, m)))
            u = np.where(r.random((k, m)) < 0.3, r.uniform(-1e3, -1.0, (k, m)), r.uniform(-3.0, 5.0, (k, m)))
            G[i0:i0 + k] = u * P[i0:i0 + k]
        elif lik == "StudentT":
            P[i0:i0 + k] = 10.0 ** r.uniform(np.log10(0.5), 6.0, (k, m))
            G[i0:i0 + k] = d + r.normal(0.0, 2.0, (k, m))
        else:
            G[i0:i0 + k] = np.exp(r.uniform(-3.0, 4.0, (k, m)))
            G[i0:i0 + k, ::6] = 0.0
    return d, G, (None if lik == "Poisson" else P)


def scipy_terms(lik, d, G, P):
    """(sum_j t_j, sum_j |parts of t_j|) per row from scipy, in row chunks."""
    s, a = np.empty(G.shape[0]), np.empty(G.shape[0])
    for i0 in range(0, G.shape[0], 4096):
        g = G[i0:i0 + 4096]
        p = None if P is None else P[i0:i0 + 4096]
        if lik == "Normal":
            t = stats.norm.logpdf(d, g, p); mag = np.abs(t)
        elif lik == "Positive Normal":
            n, c = stats.norm.logpdf(d, g, p), special.log_ndtr(g / p)
            t, mag = n - c, np.abs(n) + np.abs(c)
        elif lik == "StudentT":
            t = stats.t.logpdf(d - g, p); mag = np.abs(t)
        else:
            t = stats.poisson.logpmf(d, g); mag = np.abs(t)
        s[i0:i0 + 4096], a[i0:i0 + 4096] = t.sum(1), mag.sum(1)
    return s, a


@pytest.mark.parametrize("lik", LIKS)
@pytest.mark.parametrize("m", [1, 31, 32, 33, 1000, 4097])
@pytest.mark.parametrize("rows", [1, 63, 65536])
def test_kernel_matches_the_oracle(lik, rows, m):
    """|l_device - l_oracle| <= 1e-12 sum_j |t_j| (CUDA's lgamma / log / erfcx and libm differ in the last bits); scipy's row sums
    agree to 1e-10 of the same scale (its t.logpdf loses up to 1e-11 at large nu)."""
    d, G, P = outputs(lik, rows, m)
    s, o = pending_eval(_tmcmc.Solver, rows, lik, d), pending_eval(OracleTMCMC, rows, lik, d)
    assert s.get("Evaluation Rows").size == rows and o.get("Evaluation Rows").size == rows
    for h in (s, o):
        h.inject_reference(G, P)
        h.eval()
    ls, lo = s.get("Evaluation LogLikelihoods"), o.get("Evaluation LogLikelihoods")
    ref, scale = scipy_terms(lik, d, G, P)
    assert ls.size == rows and np.isfinite(ls).all() and np.isfinite(lo).all()
    assert np.all(np.abs(ls - lo) <= 1e-12 * scale), np.max(np.abs(ls - lo) / scale)
    assert np.all(np.abs(ls - ref) <= 1e-10 * scale), np.max(np.abs(ls - ref) / scale)


def test_poisson_zero_mean_gives_minus_infinity():
    d = np.array([0.0, 2.0, 1.0])
    s = pending_eval(_tmcmc.Solver, 63, "Poisson", d)
    G = np.ones((63, 3))
    G[5, 1] = 0.0           # g = 0 < d: -inf (weight 0); g = 0 = d elsewhere would be 0
    G[7, 0] = 0.0
    s.inject_reference(G)
    s.eval()
    l = s.get("Evaluation LogLikelihoods")
    assert l[5] == -np.inf and np.isfinite(np.delete(l, 5)).all()
    assert l[7] == pytest.approx(l[6] + 1.0, rel=1e-13)


# ---- the device in lockstep with the oracle, host reference models on both sides

T = np.linspace(0.0, 1.0, 37)


def problem(lik):
    r = np.random.default_rng(9)
    if lik == "Poisson":
        return r.poisson(np.exp(0.5 + 1.0 * T)).astype(np.float64), lambda X: np.exp(X[:, :1] + X[:, 1:2] * T)
    d = 1.0 + 2.0 * T + 0.3 * r.normal(size=T.size)
    if lik == "Positive Normal":
        d = np.abs(d)
    p = 4.0 if lik == "StudentT" else 0.3
    return d, lambda X: (X[:, :1] + X[:, 1:2] * T, p)


@pytest.mark.parametrize("lik", LIKS)
def test_lockstep_with_oracle(lik):
    d, model = problem(lik)
    kw = dict(n=2, population_size=512, max_chain_length=2, default_burn_in=1, priors=[("Normal", 0.0, 2.0)] * 2, reference=(lik, d), seed=11)
    s, o = _tmcmc.Solver(**kw), OracleTMCMC(**kw)
    s.set_host_reference(model); o.set_host_reference(model)
    s.run_generation(); o.run_generation()
    assert rel(s.get("Sample LogLikelihood Database"), o.get("Sample LogLikelihood Database")) <= 1e-12
    for g in range(40):
        if o.scalar("Annealing Exponent") >= 1.0:
            break
        s.anneal(); o.anneal()
        assert abs(s.scalar("LogEvidence") - o.scalar("LogEvidence")) <= 1e-9 * max(1.0, abs(o.scalar("LogEvidence")))
        s.inject_factor(o.get("Proposal Factor"))
        s.resample(); o.resample()
        for k in ("Selection Counts", "Chain Leaders", "Chain Lengths"):
            assert np.array_equal(s.get(k), o.get(k)), k
        for t in range(int(o.scalar("Max Chain Steps"))):
            s.propose(); o.propose()
            assert np.array_equal(s.get("Proposal Support"), o.get("Proposal Support"))
            s.eval(); o.eval()
            le, lo = s.get("Evaluation LogLikelihoods"), o.get("Evaluation LogLikelihoods")
            assert le.size == lo.size and (le.size == 0 or rel(le, lo) <= 1e-9)
            s.accept(); o.accept()
            assert np.array_equal(s.get("Accept Flags"), o.get("Accept Flags"))
        assert s.scalar("Model Evaluation Count") == o.scalar("Model Evaluation Count")
        assert rel(s.get("Sample Database"), o.get("Sample Database")) <= 1e-9
        assert rel(s.get("Sample LogLikelihood Database"), o.get("Sample LogLikelihood Database")) <= 1e-9
    assert o.scalar("Annealing Exponent") == 1.0
    assert abs(s.scalar("LogEvidence") - o.scalar("LogEvidence")) <= 1e-9 * max(1.0, abs(o.scalar("LogEvidence")))


# ---- the Korali surface

def experiment(model, lik="Normal", data=None, lam=512, seed=7, priors=(("Normal", 0.0, 2.0), ("Normal", 0.0, 2.0), ("Uniform", 0.2, 2.0))):
    e = korali.Experiment()
    e["Problem"]["Type"] = "Bayesian/Reference"
    e["Problem"]["Likelihood Model"] = lik
    e["Problem"]["Reference Data"] = list(problem("Normal")[0] if data is None else data)
    e["Problem"]["Computational Model"] = model
    for i, (ty, a, b) in enumerate(priors):
        e["Distributions"][i]["Name"] = "P%d" % i
        e["Distributions"][i]["Type"] = "Univariate/" + ty
        e["Distributions"][i]["Minimum" if ty == "Uniform" else "Mean"] = a
        e["Distributions"][i]["Maximum" if ty == "Uniform" else "Standard Deviation"] = b
        e["Variables"][i]["Name"] = "X%d" % i
        e["Variables"][i]["Prior Distribution"] = "P%d" % i
    e["Solver"]["Type"] = "Sampler/TMCMC"
    e["Solver"]["Population Size"] = lam
    e["Console Output"]["Verbosity"] = "Silent"
    e["File Output"]["Enabled"] = False
    e["Random Seed"] = seed
    return e


def per_sample(s):
    a, b, sig = s["Parameters"]
    s["Reference Evaluations"] = [a + b * t for t in T]
    s["Standard Deviation"] = [sig] * len(T)


def test_model_kinds_agree():
    """The per-sample callable, korali.batched and korali.batched_device give the same run; sigma is the third variable, returned as
    a (rows, 1) column that is broadcast over the data points."""
    Td = torch.tensor(T, dtype=torch.float64, device="cuda")
    runs = []
    for model in (per_sample,
                  korali.batched(lambda X: {"Reference Evaluations": X[:, :1] + X[:, 1:2] * T, "Standard Deviation": X[:, 2:3]}),
                  korali.batched_device(lambda X: {"Reference Evaluations": X[:, :1] + X[:, 1:2] * Td, "Standard Deviation": X[:, 2:3]})):
        e = experiment(model)
        korali.Engine().run(e)
        runs.append((e["Results"]["Log Evidence"], np.array(e["Results"]["Posterior Sample Database"])))
    z0, d0 = runs[0]
    assert np.isfinite(z0) and d0.shape == (512, 3)
    for z, db in runs[1:]:
        assert abs(z - z0) <= 1e-12 * abs(z0)
        assert rel(db, d0) <= 1e-12


def test_full_size_linear_gaussian_meets_the_closed_form():
    """lambda = 65536, g_j = a + b t_j (50 points), known sigma = 0.3, Normal(0, 2) priors, Burn In 5, Covariance Scaling 0.2, a
    korali.batched_device model: log Z = log N(d; 0, sigma^2 I + 4 Phi Phi^T), and the posterior N(mu, S) with
    S = (I / 4 + Phi^T Phi / sigma^2)^-1, mu = S Phi^T d / sigma^2. Measured (B200, seed 3): log Z -22.4641 (exact -22.4595), mean
    within 0.0012 posterior standard deviations, covariance entries within 0.8 %. Tolerances: 0.05 in log Z, 0.02 posterior standard
    deviations in the mean and 5 % of sqrt(S_ii S_jj) in the covariance."""
    t = np.linspace(0.0, 1.0, 50)
    sigma = 0.3
    d = 1.0 + 2.0 * t + sigma * np.random.default_rng(3).normal(size=t.size)
    Phi = np.stack([np.ones_like(t), t], 1)
    exact_z = stats.multivariate_normal.logpdf(d, np.zeros(t.size), sigma**2 * np.eye(t.size) + 4.0 * Phi @ Phi.T)
    S = np.linalg.inv(np.eye(2) / 4.0 + Phi.T @ Phi / sigma**2)
    mu = S @ Phi.T @ d / sigma**2
    td = torch.tensor(t, dtype=torch.float64, device="cuda")
    e = experiment(korali.batched_device(lambda X: {"Reference Evaluations": X[:, :1] + X[:, 1:2] * td, "Standard Deviation": sigma}),
                   data=d, lam=65536, seed=3, priors=(("Normal", 0.0, 2.0), ("Normal", 0.0, 2.0)))
    e["Solver"]["Default Burn In"] = 5
    e["Solver"]["Covariance Scaling"] = 0.2
    korali.Engine().run(e)
    z = e["Results"]["Log Evidence"]
    X = np.array(e["Results"]["Posterior Sample Database"])
    m, C = X.mean(0), np.cov(X.T)
    sd = np.sqrt(np.diag(S))
    print("lambda=65536 linear-Gaussian: log Z %.4f (exact %.4f); mean %s (exact %s); cov %s (exact %s)"
          % (z, exact_z, m, mu, C.ravel(), S.ravel()))
    assert abs(z - exact_z) <= 0.05
    assert np.all(np.abs(m - mu) <= 0.02 * sd)
    assert np.all(np.abs(C - S) <= 0.05 * np.sqrt(np.outer(np.diag(S), np.diag(S))))


M3 = [0.5, 1.0, 1.5]


@pytest.mark.parametrize("lik,model,match", [
    ("Normal", korali.batched(lambda X: {"Reference Evaluations": X[:, :1] + 0 * np.array(M3), "Standard Deviation": np.where(X[:, :1] > 0, -1.0, 1.0)}),
     r"'Standard Deviation' of sample \d+ contains a value that is not positive and finite"),
    ("StudentT", korali.batched(lambda X: {"Reference Evaluations": X[:, :1], "Degrees Of Freedom": 0.0}),
     r"'Degrees Of Freedom' of sample 0 contains a value that is not positive and finite"),
    ("Poisson", korali.batched(lambda X: X[:, :1]), r"'Reference Evaluations' of sample \d+ contains a negative Poisson mean"),
    ("Normal", korali.batched(lambda X: {"Reference Evaluations": np.full((X.shape[0], 3), np.inf), "Standard Deviation": 1.0}),
     r"'Reference Evaluations' of sample 0 contains a non-finite value"),
    ("Normal", korali.batched(lambda X: {"Reference Evaluations": np.zeros((X.shape[0], 4)), "Standard Deviation": 1.0}),
     r"'Reference Evaluations' has shape \(\d+, 4\), which does not broadcast to \d+ samples x 3 reference points"),
    ("Normal", korali.batched(lambda X: {"Reference Evaluations": X[:, :1]}), "did not return 'Standard Deviation'"),
    ("Normal", korali.batched(lambda X: X[:, :1]), "a bare array is accepted for Poisson only"),
    ("Normal", korali.batched_device(lambda X: {"Reference Evaluations": X[:, :1]}), "did not return 'Standard Deviation'"),
    ("Normal", korali.batched_device(lambda X: {"Reference Evaluations": X[:, :1].repeat(1, 2), "Standard Deviation": 1.0}),
     r"'Reference Evaluations' has shape \(\d+, 2\), which does not broadcast"),
    ("Normal", lambda s: s.__setitem__("Reference Evaluations", [0.0] * 3), "did not set 'Standard Deviation' for sample 0"),
    ("Normal", lambda s: (s.__setitem__("Reference Evaluations", [0.0] * 2), s.__setitem__("Standard Deviation", [1.0] * 3)),
     "'Reference Evaluations' of sample 0 must be a list of 3 values"),
])
def test_runtime_errors(lik, model, match):
    e = experiment(model, lik=lik, data=[1.0, 2.0, 3.0] if lik == "Poisson" else M3, lam=64,
                   priors=(("Uniform", -1.0, 1.0),))
    with pytest.raises(RuntimeError, match=match):
        korali.Engine().run(e)


def test_readme_example_runs(capsys):
    """The Bayesian/Reference block of README.md runs unchanged and prints a log evidence near the exact one."""
    readme = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "README.md")).read()
    blocks = [b.split("```", 1)[0] for b in readme.split("```python")[1:]]
    code = next(b for b in blocks if "Bayesian/Reference" in b)
    g = {"__name__": "__readme__"}
    exec(compile(code, "README.md", "exec"), g)
    logz = float(capsys.readouterr().out.strip().splitlines()[-1].split()[-1])
    t, d, sigma = g["t"], np.asarray(g["d"]), 0.1
    Phi = np.stack([np.ones_like(t), t], 1)
    exact = stats.multivariate_normal.logpdf(d, np.zeros(t.size), sigma**2 * np.eye(t.size) + 25.0 * Phi @ Phi.T)
    print("README Bayesian/Reference: log Z %.4f, exact %.4f" % (logz, exact))
    assert abs(logz - exact) <= 0.1
