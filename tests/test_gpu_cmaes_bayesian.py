"""Optimizer/CMAES on Bayesian/Custom and Bayesian/Reference problems on the B200: F(x) = the log-posterior (include/kcma.h) against
numpy / scipy, the closed-form maximum a posteriori estimates through korali.Engine().run(e), the same run as an equivalent Optimization,
the prior's support, graph replay, several devices and resume."""
import os
import numpy as np
import pytest
import torch
import korali_b200 as korali
from korali_b200 import _lib
from korali_b200._abi import KcmaError
from test_gpu_tmcmc_reference import outputs, scipy_terms

pytestmark = pytest.mark.gpu

HALF_LOG_2PI = 0.5 * np.log(2.0 * np.pi)


def prior_terms(X, priors):
    """Per-element log-prior terms (rows x n)."""
    T = np.empty_like(X)
    for d, (t, a, b) in enumerate(priors):
        x = X[:, d]
        if t == "Uniform":
            T[:, d] = np.where((x >= a) & (x <= b), -np.log(b - a), -np.inf)
        else:
            T[:, d] = -0.5 * ((x - a) / b) ** 2 - np.log(b) - HALF_LOG_2PI
    return T


def loglik_terms(name, X):
    """(l, sum |terms|) of the built-in log-likelihoods."""
    n = X.shape[1]
    if name == "NegSphere":
        t = 0.5 * X * X
        return -t.sum(1), t.sum(1)
    if name == "NegSumSq":
        t = X * X
        return -t.sum(1), t.sum(1)
    if name == "NegEllipsoid":
        t = 10.0 ** (6.0 * np.arange(n) / max(n - 1, 1)) * X * X
        return -t.sum(1), t.sum(1)
    if name == "NegRosenbrock":
        t = 100.0 * (X[:, 1:] - X[:, :-1] ** 2) ** 2 + (1.0 - X[:, :-1]) ** 2
        return -t.sum(1), t.sum(1)
    if name == "NegSphereSin2":
        t = X * X + np.sin(X) ** 2
        return -t.sum(1), t.sum(1)
    s1, s2 = np.sqrt((X * X).sum(1) / n), np.cos(2.0 * np.pi * X).sum(1) / n   # NegAckley
    return 20.0 * np.exp(-0.2 * s1) + np.exp(s2) - 20.0 - np.e, 50.0 + (X * X).sum(1)


PRIORS = {
    "uniform": lambda n: [("Uniform", -1.5, 2.0)] * n,
    "normal": lambda n: [("Normal", 0.3, 0.7)] * n,
    "mixed": lambda n: [("Uniform", -1.0, 1.5) if d % 3 == 0 else ("Normal", -0.2 * d, 1.0 + 0.1 * d) for d in range(n)],
}


def check_posterior(F, X, priors, l, lscale):
    T = prior_terms(X, priors)
    p = T.sum(1)
    out = ~np.isfinite(p)
    assert np.all(F[out] == -np.inf)
    scale = np.abs(T[~out]).sum(1) + lscale[~out]
    assert np.all(np.abs(F[~out] - (p[~out] + l[~out])) <= 1e-12 * scale), np.max(np.abs(F[~out] - (p[~out] + l[~out])) / scale)
    return out


@pytest.mark.parametrize("objective", ["NegSphere", "NegRosenbrock", "NegAckley", "NegEllipsoid", "NegSumSq", "NegSphereSin2"])
@pytest.mark.parametrize("prior", ["uniform", "normal", "mixed"])
@pytest.mark.parametrize("mirrored", [0, 1])
def test_builtin_log_posterior_matches_numpy(objective, prior, mirrored):
    n, lam = 300, 1024
    priors = PRIORS[prior](n)
    s = _lib.Solver(n=n, population_size=lam, objective=objective, priors=priors, keep_population=1, mirrored_sampling=mirrored,
                    initial_value=0.1, initial_stddev=0.05 if prior != "mixed" else 0.2, seed=11)
    for _ in range(2):
        s.ask(); s.eval()
        X, F = s.get("Sample Population").reshape(lam, n), s.get("Value Vector")
        l, ls = loglik_terms(objective, X)
        check_posterior(F, X, priors, l, ls)
        s.tell()


@pytest.mark.parametrize("lik", ["Normal", "Positive Normal", "StudentT", "Poisson"])
@pytest.mark.parametrize("m", [1, 33, 1000])
@pytest.mark.parametrize("rows", [63, 65536])
def test_reference_log_posterior_matches_scipy(lik, rows, m):
    """The edge-value model outputs of the TMCMC tests; rows outside the Uniform prior's support get NaN outputs, which are ignored."""
    d, G, P = outputs(lik, rows, m)
    priors = [("Uniform", -1.0, 1.0), ("Normal", 0.5, 2.0)]
    s = _lib.Solver(n=2, population_size=rows, objective="External", keep_population=1, priors=priors, reference=(lik, d),
                    initial_value=0.0, initial_stddev=1.0, seed=2)
    seen = {}

    def model(X):
        out = ~np.isfinite(prior_terms(X, priors).sum(1))
        seen["out"] = out
        g = G.copy(); g[out] = np.nan
        return g if P is None else (g, P)
    s.set_host_reference(model)
    s.ask(); s.eval()
    X, F = s.get("Sample Population").reshape(rows, 2), s.get("Value Vector")
    l, ls = scipy_terms(lik, d, G, P)
    # |dF| <= 1e-12 (|p| + sum |t_j|) holds against exact terms; scipy's own logpdf / log_ndtr / t.logpdf are accurate to 1e-10 of
    # sum |t_j| only (test_gpu_tmcmc_reference: its t.logpdf loses up to 1e-11 at large nu), so the likelihood part is allowed 1e-10
    out = check_posterior(F, X, priors, l, ls * 1e2)
    assert out.any() and not out.all() and np.array_equal(out, seen["out"])


def test_custom_models_output_outside_the_support_is_ignored():
    """A Bayesian/Custom host model (numpy) and device model (torch) that return NaN on the rows outside a Uniform prior's support: those
    rows get F = -inf and no error; the others get p + l."""
    n, lam = 5, 256
    priors = [("Uniform", -1.0, 1.0)] * 2 + [("Normal", 0.5, 2.0)] * 3

    def loglik(X, lib):
        out = (X[:, :2] < -1.0).any(1) | (X[:, :2] > 1.0).any(1)
        return lib.where(out, lib.full_like(X[:, 0], float("nan")), -0.5 * (X * X).sum(1))
    s = _lib.Solver(n=n, population_size=lam, objective="External", keep_population=1, priors=priors, initial_value=0.0,
                    initial_stddev=1.0, seed=6)
    s.set_host_objective(lambda X: loglik(X, np))
    for _ in range(3):
        s.ask(); s.eval()
        X, F = s.get("Sample Population").reshape(lam, n), s.get("Value Vector")
        out = check_posterior(F, X, priors, -0.5 * (X * X).sum(1), 0.5 * (X * X).sum(1))
        assert out.any() and not out.all()
        s.tell()
    e = sphere_experiment(np.zeros(n), np.ones(n), n, korali.batched_device(lambda X: loglik(X, torch)), gens=20, pop=lam)
    for i in range(2):
        e["Distributions"][i + n]["Name"] = "U%d" % i
        e["Distributions"][i + n]["Type"] = "Univariate/Uniform"
        e["Distributions"][i + n]["Minimum"] = -1.0
        e["Distributions"][i + n]["Maximum"] = 1.0
        e["Variables"][i]["Prior Distribution"] = "U%d" % i
    korali.Engine().run(e)
    F = np.array(e["Solver"]["Value Vector"])
    assert np.isfinite(e["Results"]["Best Sample"]["F(x)"]) and not np.isnan(F).any()


def test_nan_log_likelihood_inside_the_support_names_the_sample():
    priors = [("Uniform", -10.0, 10.0)] * 3
    s = _lib.Solver(n=3, population_size=16, objective="External", keep_population=1, priors=priors, initial_value=0.0,
                    initial_stddev=1.0, seed=1)

    def model(X):
        f = -0.5 * (X * X).sum(1)
        f[5] = np.nan
        return f
    s.set_host_objective(model)
    s.ask()
    with pytest.raises(KcmaError, match="log-likelihood of sample 5 is nan"):
        s.eval()


def test_bad_reference_parameter_names_the_sample():
    priors = [("Normal", 0.0, 1.0)]
    s = _lib.Solver(n=1, population_size=8, objective="External", keep_population=1, priors=priors, reference=("Normal", [1.0, 2.0]),
                    initial_value=0.0, initial_stddev=1.0, seed=1)
    P = np.ones((8, 2)); P[3, 1] = -1.0
    s.set_host_reference(lambda X: (np.zeros((8, 2)), P))
    s.ask()
    with pytest.raises(KcmaError, match="'Standard Deviation' of sample 3 contains a value that is not positive"):
        s.eval()


def test_every_sample_outside_the_support_completes_a_generation():
    priors = [("Uniform", 10.0, 11.0)] * 4
    s = _lib.Solver(n=4, population_size=32, objective="NegSphere", priors=priors, initial_value=0.0, initial_stddev=0.1, seed=3)
    s.ask(); s.eval()
    assert np.all(s.get("Value Vector") == -np.inf)
    s.tell()
    assert list(s.get_index("Sorting Index")) == list(range(32))   # ties by ascending index
    s.run_generation()
    assert s.scalar("Best Ever Value") == -np.inf


def test_out_of_support_rows_rank_last_and_the_run_reaches_the_map():
    """Uniform(-0.5, 2) priors without bounds and a mean whose samples partly leave the support; Sphere log-likelihood: MAP at 0."""
    n, lam = 6, 32
    priors = [("Uniform", -0.5, 2.0)] * n
    s = _lib.Solver(n=n, population_size=lam, objective="NegSphere", priors=priors, initial_value=1.5, initial_stddev=1.0, seed=8)
    seen_finite = False
    for g in range(400):
        s.run_generation()
        F, idx = s.get("Value Vector"), s.get_index("Sorting Index").astype(np.int64)
        fin = np.isfinite(F[idx])
        assert fin[:fin.sum()].all()    # the -inf rows form the tail of the ranking
        seen_finite |= fin.any()
        if seen_finite:
            assert np.isfinite(s.scalar("Best Ever Value"))
    x = s.get("Best Ever Variables")
    assert np.abs(x).max() < 1e-6
    assert abs(s.scalar("Best Ever Value") - n * -np.log(2.5)) < 1e-9


def sphere_experiment(mu0, sd, n, model, gens=600, pop=16):
    e = korali.Experiment()
    e["Problem"]["Type"] = "Bayesian/Custom"
    e["Problem"]["Likelihood Model"] = model
    for i in range(n):
        e["Distributions"][i]["Name"] = "P%d" % i
        e["Distributions"][i]["Type"] = "Univariate/Normal"
        e["Distributions"][i]["Mean"] = float(mu0[i])
        e["Distributions"][i]["Standard Deviation"] = float(sd[i])
        e["Variables"][i]["Name"] = "X%d" % i
        e["Variables"][i]["Prior Distribution"] = "P%d" % i
        e["Variables"][i]["Initial Value"] = 0.0
        e["Variables"][i]["Initial Standard Deviation"] = 1.0
    e["Solver"]["Type"] = "Optimizer/CMAES"
    e["Solver"]["Population Size"] = pop
    e["Solver"]["Termination Criteria"]["Max Generations"] = gens
    e["Console Output"]["Verbosity"] = "Silent"
    e["File Output"]["Enabled"] = False
    e["Random Seed"] = 77
    return e


# The Sphere log-likelihood -x.x/2 summed in variable order by each model kind, so that all three produce the same bits: the three runs
# must then be the same run (the conduit does not change the result). The built-in model sums in the device's butterfly order.
def per_sample_sphere(s):
    f = 0.0
    for v in s["Parameters"]:
        f = f + v * v
    s["logLikelihood"] = -0.5 * f


def in_order_sphere(X):
    f = X[:, 0] * X[:, 0]
    for d in range(1, X.shape[1]):
        f = f + X[:, d] * X[:, d]
    return -0.5 * f


RUN_STATE = ["Current Mean", "Covariance Matrix", "Evolution Path", "Best Ever Value", "Sigma", "Value Vector"]


def run_state(e):
    return {k: e["Solver"][k] for k in RUN_STATE} | {"x": e["Results"]["Best Sample"]["Parameters"], "f": e["Results"]["Best Sample"]["F(x)"]}


def test_sphere_with_normal_priors_reaches_the_closed_form_map():
    n = 4
    mu0, sd = np.array([1.0, -2.0, 0.5, 3.0]), np.array([0.5, 1.0, 2.0, 1.5])
    xmap = mu0 / (1.0 + sd ** 2)
    fmap = -0.5 * xmap @ xmap + np.sum(-0.5 * ((xmap - mu0) / sd) ** 2 - np.log(sd) - HALF_LOG_2PI)
    runs = {}
    for kind, model in [("per-sample", per_sample_sphere), ("numpy", korali.batched(in_order_sphere)),
                        ("device", korali.batched_device(in_order_sphere)), ("built-in", "Sphere")]:
        e = sphere_experiment(mu0, sd, n, model)
        korali.Engine().run(e)
        x, f = np.array(e["Results"]["Best Sample"]["Parameters"]), e["Results"]["Best Sample"]["F(x)"]
        assert np.abs(x - xmap).max() < 1e-6, kind
        assert abs(f - fmap) < 1e-9, kind
        runs[kind] = run_state(e)
    assert runs["numpy"] == runs["per-sample"] and runs["device"] == runs["per-sample"]


T20 = np.linspace(0.0, 1.0, 20)
D20 = [1.0 + 2.0 * x + 0.1 * np.sin(40.0 * x) for x in T20]


def readme_model(s):
    a, b = s["Parameters"]
    s["Reference Evaluations"] = [a + b * x for x in T20]
    s["Standard Deviation"] = [0.1] * len(T20)


def reference_experiment(model):
    e = korali.Experiment()
    e["Problem"]["Type"] = "Bayesian/Reference"
    e["Problem"]["Likelihood Model"] = "Normal"
    e["Problem"]["Reference Data"] = D20
    e["Problem"]["Computational Model"] = model
    e["Distributions"][0]["Name"] = "Prior"
    e["Distributions"][0]["Type"] = "Univariate/Normal"
    e["Distributions"][0]["Mean"] = 0.0
    e["Distributions"][0]["Standard Deviation"] = 5.0
    for i, name in enumerate(["Intercept", "Slope"]):
        e["Variables"][i]["Name"] = name
        e["Variables"][i]["Prior Distribution"] = "Prior"
        e["Variables"][i]["Initial Value"] = 0.0
        e["Variables"][i]["Initial Standard Deviation"] = 1.0
    e["Solver"]["Type"] = "Optimizer/CMAES"
    e["Solver"]["Population Size"] = 16
    e["Solver"]["Termination Criteria"]["Max Generations"] = 400
    e["Console Output"]["Verbosity"] = "Silent"
    e["File Output"]["Enabled"] = False
    e["Random Seed"] = 5
    return e


def test_readme_linear_model_reaches_the_ridge_solution():
    phi = np.stack([np.ones_like(T20), T20], 1)
    sig, s0, d = 0.1, 5.0, np.array(D20)
    xmap = np.linalg.solve(phi.T @ phi / sig ** 2 + np.eye(2) / s0 ** 2, phi.T @ d / sig ** 2)
    r = d - phi @ xmap
    fmap = (np.sum(-0.5 * (r / sig) ** 2 - np.log(sig) - HALF_LOG_2PI) + np.sum(-0.5 * (xmap / s0) ** 2 - np.log(s0) - HALF_LOG_2PI))
    Tt = torch.tensor(T20, dtype=torch.float64, device="cuda")
    models = [("per-sample", readme_model),
              ("numpy", korali.batched(lambda X: {"Reference Evaluations": X[:, :1] + X[:, 1:2] * T20, "Standard Deviation": 0.1})),
              ("device", korali.batched_device(lambda X: {"Reference Evaluations": X[:, :1] + X[:, 1:2] * Tt, "Standard Deviation": 0.1}))]
    runs = {}
    for kind, model in models:   # the three models compute the same predictions with the same operations: the same run
        e = reference_experiment(model)
        korali.Engine().run(e)
        x, f = np.array(e["Results"]["Best Sample"]["Parameters"]), e["Results"]["Best Sample"]["F(x)"]
        assert np.abs(x - xmap).max() < 1e-6, kind
        assert abs(f - fmap) < 1e-9, kind
        runs[kind] = run_state(e)
    assert runs["numpy"] == runs["per-sample"] and runs["device"] == runs["per-sample"]


def test_readme_map_example_runs():
    """The Optimizer/CMAES block of README.md runs as printed and reaches the ridge solution it states."""
    readme = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "README.md")).read()
    blocks = [b.split("```", 1)[0] for b in readme.split("```python")[1:]]
    code = next(b for b in blocks if "Bayesian/Reference" in b and "Optimizer/CMAES" in b)
    g = {"__name__": "__readme__"}
    exec(compile(code, "README.md", "exec"), g)
    x = np.array(g["e"]["Results"]["Best Sample"]["Parameters"])
    assert np.abs(x - g["ridge"]).max() < 1e-6


def test_same_run_as_the_equivalent_optimization():
    """Built-in Ellipsoid log-likelihood + priors against an Optimization whose host objective computes the same log-posterior (the
    samples stay inside the Uniform priors' support: an Optimization rejects -inf)."""
    n, lam = 10, 64
    priors = [("Uniform", -30.0, 30.0) if d % 4 == 0 else ("Normal", 0.2 * d, 1.0 + 0.1 * d) for d in range(n)]
    kw = dict(n=n, population_size=lam, initial_value=0.5, initial_stddev=1.0, seed=19, keep_population=1)
    b = _lib.Solver(objective="NegEllipsoid", priors=priors, **kw)
    o = _lib.Solver(objective="External", **kw)

    def logpost(X):
        return prior_terms(X, priors).sum(1) + loglik_terms("NegEllipsoid", X)[0]
    o.set_host_objective(logpost)
    for g in range(30):
        b.run_generation(); o.run_generation()
        assert np.array_equal(b.get_index("Sorting Index"), o.get_index("Sorting Index")), g
    assert np.abs(b.get("Current Mean") - o.get("Current Mean")).max() <= 1e-9
    C1, C2 = b.get("Covariance Matrix"), o.get("Covariance Matrix")
    assert np.abs(C1 - C2).max() <= 1e-9 * np.abs(C2).max()
    assert abs(b.scalar("Sigma") - o.scalar("Sigma")) <= 1e-9 * o.scalar("Sigma")


STATE = ["Current Mean", "Covariance Matrix", "Evolution Path", "Conjugate Evolution Path", "Best Ever Variables", "Value Vector"]


def test_graph_replay_is_bitwise_the_eager_run():
    """Phase timers keep every generation eager; without them generations 3.. replay one captured CUDA graph."""
    n, lam = 50, 256
    priors = [("Normal", 0.5, 1.0), ("Uniform", -2.0, 2.0)] * (n // 2)
    runs = []
    for eager in (True, False):
        s = _lib.Solver(n=n, population_size=lam, objective="NegEllipsoid", priors=priors, initial_value=1.0, initial_stddev=0.5, seed=4)
        s.timing_enable(eager)
        for _ in range(12):
            s.run_generation()
        runs.append({k: s.get(k) for k in STATE} | {"Sigma": s.scalar("Sigma")})
    for k in runs[0]:
        assert np.array_equal(runs[0][k], runs[1][k]), k


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_devices_are_bitwise_one_device():
    mu0, sd = np.linspace(-1.0, 1.0, 8), np.full(8, 0.7)
    res = []
    for devices in (1, 2):
        e = sphere_experiment(mu0, sd, 8, "Ellipsoid", gens=40, pop=64)
        k = korali.Engine()
        k["Conduit"]["Devices"] = devices
        k.run(e)
        res.append({key: e["Solver"][key] for key in ["Current Mean", "Covariance Matrix", "Best Ever Value", "Sigma"]})
    assert res[0] == res[1]


def test_resume_is_bitwise(tmp_path):
    mu0, sd = np.linspace(-1.0, 2.0, 12), np.full(12, 0.8)

    def make(gens, path):
        e = sphere_experiment(mu0, sd, 12, "Ellipsoid", gens=gens, pop=32)
        e["File Output"]["Enabled"] = True
        e["File Output"]["Path"] = str(tmp_path / path)
        e["File Output"]["Frequency"] = 5
        return e
    k = korali.Engine()
    full = make(10, "full"); k.run(full)
    part = make(5, "part"); k.run(part)
    r = korali.Experiment()
    r["Problem"]["Likelihood Model"] = "Ellipsoid"
    r.loadState(str(tmp_path / "part" / "latest"))
    r["Solver"]["Termination Criteria"]["Max Generations"] = 10
    r["File Output"]["Enabled"] = False
    k.run(r)
    assert r["Current Generation"] == 10
    for key in ["Sigma", "Best Ever Value", "Current Best Value", "Current Mean", "Covariance Matrix", "Evolution Path",
                "Conjugate Evolution Path", "Best Ever Variables"]:
        assert r["Solver"][key] == full["Solver"][key], key
