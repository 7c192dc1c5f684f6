"""The reference's own CMA-ES test scripts, ported to pytest with `import korali_b200 as korali`: same experiment definitions,
same seeds, same asserted thresholds — with these stated deviations: console output is "Silent" instead of "Detailed"; the CCMAES
cases assert the reference's thresholds with 1e-6 relative slack (TestCCMAES: a different eigensolver and RNG stream move the
converged optimum in its last digits); the two `checkInfeasible` corner cases of run-cmaes.py:219-272 run with the reference's
settings ("Max Infeasible Resamplings" left at its default, which the release build reads as 0 — SURVEY Q2 — and set to 50).
  tests/statistical/optimizers/correctness/run-cmaes.py          -> TestCorrectness
  tests/statistical/optimizers/detailed/ccmaes/run-ccmaes.py      -> TestCCMAES
  tests/statistical/optimizers/termination/cmaes_termination.py   -> TestTermination
  tests/statistical/optimizers/detailed/cmaes/run-{min,max}cmaes* -> TestDetailed
CPU part: the KoraliJson cursor semantics and the strict configuration errors (no GPU needed)."""
import json
import os
import numpy as np
import pytest
import torch
import korali_b200 as korali
from korali_models.models import *  # noqa: F401,F403

gpu = pytest.mark.gpu
HAS_GPU = torch.cuda.is_available()


def checkMin(k, expectedMinimum, tol):           # correctness/helpers/helpers.py:5-8
    minimum = k["Solver"]["Best Ever Value"]
    assert np.isclose(expectedMinimum, minimum, atol=tol), (minimum, expectedMinimum, tol)


def checkInfeasible(k, expectedMinimum):         # :10-13
    assert np.less(expectedMinimum, k["Solver"]["Infeasible Sample Count"])


def base_1d(pop=8, gens=100):
    e = korali.Experiment()
    e["Problem"]["Type"] = "Optimization"
    e["Problem"]["Objective Function"] = evalmodel
    e["Variables"][0]["Name"] = "X"
    e["Variables"][0]["Lower Bound"] = -10.0
    e["Variables"][0]["Upper Bound"] = +10.0
    e["Solver"]["Type"] = "Optimizer/CMAES"
    e["Solver"]["Population Size"] = pop
    e["Solver"]["Termination Criteria"]["Max Generations"] = gens
    e["Console Output"]["Frequency"] = 10
    e["Console Output"]["Verbosity"] = "Silent"
    e["File Output"]["Enabled"] = False
    e["Random Seed"] = 1337
    return e


def base_mo():
    """examples/optimization/multiobjective/run-mocmaes.py:16-37"""
    e = korali.Experiment()
    e["Problem"]["Type"] = "Optimization"
    e["Problem"]["Objective Function"] = "RosenbrockAndSphere"
    e["Problem"]["Num Objectives"] = 2
    for i in range(4):
        e["Variables"][i]["Name"] = "X" + str(i)
        e["Variables"][i]["Lower Bound"] = -25.0
        e["Variables"][i]["Upper Bound"] = +25.0
        e["Variables"][i]["Initial Standard Deviation"] = 3.0
    e["Solver"]["Type"] = "Optimizer/MOCMAES"
    e["Solver"]["Population Size"] = 32
    e["Solver"]["Mu Value"] = 16
    e["Console Output"]["Verbosity"] = "Silent"
    e["File Output"]["Enabled"] = False
    return e


@pytest.mark.parametrize("mod,match", [
    (lambda e: e["Solver"].__setitem__("Bogus Key", 3), "Unrecognized settings for Korali module: MOCMAES"),
    (lambda e: e["Solver"]["Termination Criteria"].__setitem__("Max Fun", 1), "Unrecognized settings"),
    (lambda e: e["Solver"].__setitem__("Mu Value", 33), "must be smaller or equal with population size"),       # MOCMAES.cpp.base:26-27
    (lambda e: e["Solver"].__setitem__("Success Learning Rate", 1.5), "Invalid Global Success Learning Rate"),   # :136-137
    (lambda e: e["Solver"].__setitem__("Target Success Rate", 0.0), "Invalid Target Success Rate"),             # :138-139
    (lambda e: e["Problem"].__setitem__("Num Objectives", 1), "Problem requires multiple objectives"),           # :20-21
    (lambda e: e["Problem"].__setitem__("Objective Function", "Ellipsoid"), "Unknown multi-objective device model"),
    (lambda e: e["Problem"].__setitem__("Num Objectives", 3), "the built-in objective has 2 objectives"),
    (lambda e: e["Variables"][0].__setitem__("Upper Bound", float("inf")), "cannot be inferred"),                # :70-82
    (lambda e: e["Solver"].__setitem__("Termination Criteria", 5), r"MOCMAES \] \n \+ Key:    \['Termination Criteria'\]\n \+ Reason: not an object"),
])
def test_mocmaes_configuration_errors(mod, match):
    """The configuration checks of MOCMAES::setInitialConfiguration (tests/unit/modules/solver/optimizers.cpp:2112-2180) are raised
    before any device work."""
    e = base_mo()
    mod(e)
    e["Solver"]["Type"]
    with pytest.raises(RuntimeError, match=match):
        korali.Engine().run(e)


@pytest.mark.parametrize("mod,match", [
    (lambda e: e["Solver"].__setitem__("Bogus Key", 3), "Unrecognized settings for Korali module: DEA"),
    (lambda e: e["Solver"]["Termination Criteria"].__setitem__("Max Fun", 1), r"Unrecognized settings for Korali module: DEA\['Termination Criteria'\]"),
    (lambda e: e["Solver"].__setitem__("Termination Criteria", 5), r"DEA \] \n \+ Key:    \['Termination Criteria'\]\n \+ Reason: not an object"),
    (lambda e: e["Solver"].__setitem__("Accept Rule", "Sideways"), r"Accept Rule \(Sideways\) not recognized"),
    (lambda e: e["Solver"].__setitem__("Parent Selection Rule", "Worst"), r"Invalid setting of Parent Selection Rule \(Worst\)"),
    (lambda e: e["Solver"].__setitem__("Mutation Rule", "Self Adaptive"), "Mutation Rule 'Self Adaptive' is not built"),
    (lambda e: e["Problem"].__setitem__("Objective Function", "Banana"), "Unknown device objective 'banana'"),
    (lambda e: e["Problem"].__setitem__("Constraints", [evalmodel]), "Optimizer/DEA does not take constraints"),
    (lambda e: e["Problem"].__setitem__("Objective Function", korali.batched_device(lambda X: X.sum(1))),
     r"Optimizer/DEA takes per-sample models and korali.batched\(fn\) models"),
])
def test_dea_configuration_errors(mod, match):
    """DEA's strict configuration (termination criteria, rules, objective, constraints) is checked before any device work."""
    e = base_1d()
    e["Solver"]["Type"] = "Optimizer/DEA"
    mod(e)
    e["Solver"]["Type"]     # reset the cursor after the chained access above
    with pytest.raises(RuntimeError, match=match):
        korali.Engine().run(e)


def test_sibling_solvers_run_on_one_device():
    """k["Conduit"]["Devices"] > 1 shards the population of Optimizer/CMAES; the sibling solvers say so instead of ignoring the key."""
    e = base_mo()
    k = korali.Engine()
    k["Conduit"]["Type"] = "Device"
    k["Conduit"]["Devices"] = 2
    with pytest.raises(RuntimeError, match="Optimizer/MOCMAES runs on one device"):
        k.run(e)
    e = base_1d()
    e["Solver"]["Type"] = "Optimizer/DEA"
    k = korali.Engine()
    k["Conduit"]["Devices"] = [0, 1]
    with pytest.raises(RuntimeError, match="Optimizer/DEA runs on one device"):
        k.run(e)


# ---------------------------------------------------------------- CPU: JSON tree + strict configuration --------
def test_koralijson_cursor_semantics():
    e = korali.Experiment()
    e["Variables"][0]["Name"] = "X"
    e["Variables"][1]["Lower Bound"] = -1
    e["Solver"]["Termination Criteria"]["Max Generations"] = 100
    e["Solver"]["List"] = (1, 2.5, "a")
    e["Solver"]["Flag"] = True
    assert e["Variables"][0]["Name"] == "X"                    # elemental -> python value
    assert e["Variables"][1]["Lower Bound"] == -1
    v = e["Solver"]["Termination Criteria"]["Max Generations"]
    assert v == 100 and isinstance(v, int)
    e["Solver"]["Sigma"] = 2.0
    assert isinstance(e["Solver"]["Sigma"], int)                # whole-valued doubles come back as int (py2json.hpp:100-111)
    assert e["Solver"]["List"] == [1, 2.5, "a"]                 # tuple -> array of elementals
    node = e["Solver"]                                          # non-elemental -> the same object, cursor advanced
    assert node is e
    assert node["Termination Criteria"]["Max Generations"] == 100   # continues from the cursor, then resets
    assert e["Solver"]["Flag"] is e                             # booleans are not "elemental" (jsonInterface.cpp:42-64)
    with pytest.raises(RuntimeError):                           # the cursor still points at the boolean node
        e["Solver"]
    e["Random Seed"] = np.int64(7)
    assert e["Random Seed"] == 7


@pytest.mark.parametrize("mod,match", [
    (lambda e: e["Solver"].__setitem__("Bogus Key", 3), "Unrecognized settings for Korali module: CMAES"),
    (lambda e: e["Solver"].__setitem__("Population Size", "eight"), "Population Size"),
    (lambda e: e["Solver"].__setitem__("Mu Type", "Quadratic"), "Invalid setting of Mu Type"),
    (lambda e: e["Variables"][0].__setitem__("Granularity", -1.0), "Negative granularity"),
    (lambda e: e["Variables"][0].__setitem__("Granularity", "coarse"), "Granularity"),
    (lambda e: e["Solver"].__setitem__("Use Gradient Information", "yes"), "Use Gradient Information"),
    (lambda e: e["Solver"].__setitem__("Gradient Step Size", "big"), "Gradient Step Size"),
    (lambda e: e["Variables"][0].__setitem__("Colour", "red"), "Unrecognized settings"),
    (lambda e: e["Solver"]["Termination Criteria"].__setitem__("Max Fun", 1), "Unrecognized settings"),
    (lambda e: e["Solver"].__setitem__("Type", "Optimizer/Adam"), "is not served by korali_b200"),
    (lambda e: e["Solver"].__setitem__("Type", "Optimizer/MOCMAES"), "Problem requires multiple objectives"),   # MOCMAES.cpp.base:20-21
    (lambda e: e["Problem"].__setitem__("Type", "Bayesian/Custom"), "Problem Type"),
    (lambda e: e.__setitem__("Nonsense", 1), "Unrecognized settings for Korali module: Experiment"),
    (lambda e: e["Console Output"].__setitem__("Verbosity", "Loud"), "Verbosity"),
])
def test_strict_configuration_errors(mod, match):
    """Generated setConfiguration semantics: every wrong type / unknown key is a RuntimeError (optimizers.cpp:696-1771)."""
    e = base_1d()
    mod(e)
    e["Solver"]["Type"]     # reset the cursor after the chained access above
    with pytest.raises(RuntimeError, match=match):
        korali.Engine().run(e)


@pytest.mark.skipif(HAS_GPU, reason="CPU-only behaviour")
def test_engine_fails_loudly_without_gpu():
    with pytest.raises(RuntimeError, match="no CPU fallback|CUDA device"):
        korali.Engine().run(base_1d())


# ---------------------------------------------------------------- correctness/run-cmaes.py -------------------
@gpu
class TestCorrectness:
    def test_default(self):
        e = base_1d(); korali.Engine().run(e); checkMin(e, 0.23246, 1e-4)

    def test_diagonal_covariance(self):
        e = base_1d(); e["Solver"]["Diagonal Covariance"] = True
        korali.Engine().run(e); checkMin(e, 0.23246, 1e-4)

    def test_mirrored_sampling(self):
        e = base_1d(); e["Solver"]["Mirrored Sampling"] = True
        korali.Engine().run(e); checkMin(e, 0.23246, 1e-4)

    @pytest.mark.parametrize("mu_type,pop,tol", [("Linear", 8, 1e-4), ("Logarithmic", 8, 1e-4), ("Proportional", 64, 1e-3), ("Equal", 64, 1e-3)])
    def test_mu_types(self, mu_type, pop, tol):
        e = base_1d(pop); e["Solver"]["Mu Type"] = mu_type
        korali.Engine().run(e); checkMin(e, 0.23246, tol)

    def test_unsatisfiable_constraint(self):
        e = base_1d(16, 10)
        e["Problem"]["Constraints"] = [constraint1]
        e["Variables"][0]["Initial Value"] = 1.0
        e["Solver"]["Viability Population Size"] = 2
        korali.Engine().run(e)
        # run-cmaes.py:243. The constraint is never met: the solver stays in the viability regime, sigma doubles every generation
        # (updateSigma :722-726) and the samples leave [-10, 10]; each is counted once (default Max Infeasible Resamplings = 0, Q2)
        checkInfeasible(e, 10)
        assert e["Solver"]["Is Viability Regime"] == 1
        assert e["Current Generation"] == 10

    def test_terminates_on_max_infeasible_resamplings(self):
        """run-cmaes.py:245-272: Max Infeasible Resamplings = 50 bounds the resampling loop by the CUMULATIVE count (:459) and ends
        the run through the termination criterion (CMAES.config:114)."""
        e = base_1d(16, 100)
        e["Problem"]["Constraints"] = [constraint1]
        e["Variables"][0]["Initial Value"] = 1.0
        e["Solver"]["Viability Population Size"] = 2
        e["Solver"]["Termination Criteria"]["Max Infeasible Resamplings"] = 50
        korali.Engine().run(e)
        checkInfeasible(e, 50)
        assert e["Current Generation"] < 100

    def test_resample_until_feasible_when_the_limit_is_large(self):
        """The other reading of the default (SURVEY Q2: 2^64-1 with -march=native): every out-of-bounds draw is redrawn, so the final
        population is feasible and every rejected draw is counted."""
        e = base_1d(64, 20)
        e["Variables"][0]["Initial Value"] = 9.0
        e["Variables"][0]["Initial Standard Deviation"] = 6.0
        e["Solver"]["Termination Criteria"]["Max Infeasible Resamplings"] = 10**9
        korali.Engine().run(e)
        assert e["Solver"]["Infeasible Sample Count"] > 0
        assert all(-10.0 <= x[0] <= 10.0 for x in e["Solver"]["Sample Population"])

    def test_min_stddev_update_warning_path(self):
        e = base_1d(64, 10)
        e["Variables"][0]["Initial Value"] = 1.0
        e["Variables"][0]["Minimum Standard Deviation Update"] = 1000.0
        korali.Engine().run(e)
        assert e["Solver"]["Sigma"] * np.sqrt(e["Solver"]["Covariance Matrix"][0]) >= 1000.0

    def test_g09_with_zero_max_corrections_runs(self):
        e = korali.Experiment()
        e["Problem"]["Type"] = "Optimization"
        e["Problem"]["Objective Function"] = g09
        e["Problem"]["Constraints"] = [g1, g2, g3, g4]
        for i in range(7):
            e["Variables"][i]["Name"] = "X" + str(i)
            e["Variables"][i]["Lower Bound"] = -10.0
            e["Variables"][i]["Upper Bound"] = +10.0
        e["Solver"]["Type"] = "Optimizer/CMAES"
        e["Solver"]["Is Sigma Bounded"] = True
        e["Solver"]["Population Size"] = 32
        e["Solver"]["Viability Population Size"] = 4
        e["Solver"]["Max Covariance Matrix Corrections"] = 0
        e["Solver"]["Termination Criteria"]["Max Value"] = -680.630057374402 - 1e-4
        e["Solver"]["Termination Criteria"]["Max Generations"] = 500
        e["Console Output"]["Verbosity"] = "Silent"
        e["File Output"]["Enabled"] = False
        e["Random Seed"] = 1337
        korali.Engine().run(e)
        assert e["Current Generation"] >= 1


# ---------------------------------------------------------------- detailed/ccmaes/run-ccmaes.py --------------
CCMAES = {
    "None": ([], -6 * 1e-10),
    "Inactive": ([inactive1, inactive2], -1.8 * 1e-10),
    "Active at Max 1": ([activeMax1, activeMax2], -4.826824e+00),
    "Active at Max 2": ([activeMax1, activeMax2, activeMax3, activeMax4], -9.653645e+00),
    "Inactive at Max 1": ([inactiveMax1, inactiveMax2], -2.19963e-10),
    "Inactive at Max 2": ([inactiveMax1, inactiveMax2, inactiveMax3, inactiveMax4], -4.626392e-10),
    "Mixed": ([activeMax1, activeMax2, activeMax3, activeMax4, inactiveMax1, inactiveMax2, inactiveMax3, inactiveMax4], -7.895685e+01),
    "Stress": ([activeMax1, activeMax2, activeMax3, activeMax4, inactiveMax1, inactiveMax2, inactiveMax3, inactiveMax4, stress1, stress2,
                stress3, stress4, stress5, stress6, stress7, stress8], -7.895685e+01),
}


@gpu
class TestCCMAES:
    @pytest.mark.parametrize("name", list(CCMAES))
    def test_constraint_set(self, name, tmp_path):
        cons, threshold = CCMAES[name]
        e = korali.Experiment()
        e["Problem"]["Type"] = "Optimization"
        e["Problem"]["Objective Function"] = evaluateModel
        e["Variables"][0]["Name"] = "X"
        e["Variables"][0]["Lower Bound"] = -10.0
        e["Variables"][0]["Upper Bound"] = +10.0
        e["Variables"][1]["Name"] = "Y"
        e["Variables"][1]["Lower Bound"] = -10.0
        e["Variables"][1]["Upper Bound"] = +10.0
        e["Solver"]["Type"] = "Optimizer/CMAES"
        e["Solver"]["Population Size"] = 8
        e["Solver"]["Viability Population Size"] = 2
        e["Solver"]["Termination Criteria"]["Max Generations"] = 100
        e["Solver"]["Is Sigma Bounded"] = 1
        e["Console Output"]["Verbosity"] = "Silent"
        e["File Output"]["Path"] = str(tmp_path / "_korali_result")
        e["Random Seed"] = 1337
        if cons:
            e["Problem"]["Constraints"] = cons
        korali.Engine().run(e)
        best = e["Solver"]["Best Ever Value"]
        print(name, best, threshold)
        # the thresholds were calibrated on the reference's MT19937 stream; the Philox stream reaches the same optimum,
        # allow the last digits of a 100-generation, lambda=8 run to differ
        assert best >= threshold - max(1e-6 * abs(threshold), 1e-8), (name, best, threshold)


# ---------------------------------------------------------------- termination/cmaes_termination.py -----------
@gpu
class TestTermination:
    @pytest.mark.parametrize("criterion,value", [("Max Generations", 1), ("Max Generations", 3), ("Max Infeasible Resamplings", 1),
                                                 ("Min Value Difference Threshold", 0.1), ("Min Standard Deviation", 0.1),
                                                 ("Max Standard Deviation", 0.9), ("Max Condition Covariance Matrix", 1.0),
                                                 ("Max Value", -1.5), ("Max Model Evaluations", 64)])
    def test_criterion_fires(self, criterion, value):
        e = korali.Experiment()
        e["Problem"]["Type"] = "Optimization"
        e["Problem"]["Objective Function"] = parabola
        e["Variables"][0]["Name"] = "X"
        e["Variables"][0]["Lower Bound"] = +1.0
        e["Variables"][0]["Upper Bound"] = +10.0
        e["Solver"]["Type"] = "Optimizer/CMAES"
        e["Solver"]["Population Size"] = 8
        e["Solver"]["Termination Criteria"][criterion] = value
        e["Console Output"]["Verbosity"] = "Silent"
        e["File Output"]["Enabled"] = False
        e["Random Seed"] = 1337
        if criterion != "Max Generations":
            e["Solver"]["Termination Criteria"]["Max Generations"] = 2000
        korali.Engine().run(e)
        if criterion == "Max Generations":
            assert e["Current Generation"] == value
        elif criterion == "Max Infeasible Resamplings":
            assert e["Solver"]["Infeasible Sample Count"] >= value
        elif criterion == "Max Condition Covariance Matrix":
            assert e["Solver"]["Maximum Covariance Eigenvalue"] / e["Solver"]["Minimum Covariance Eigenvalue"] >= value
        elif criterion == "Max Value":
            assert e["Solver"]["Best Ever Value"] >= value
        elif criterion == "Min Value Difference Threshold":
            assert e["Current Generation"] < 2000
        elif criterion == "Min Standard Deviation":
            assert e["Solver"]["Current Min Standard Deviation"] <= value
        elif criterion == "Max Standard Deviation":
            assert e["Solver"]["Current Max Standard Deviation"] >= value
        elif criterion == "Max Model Evaluations":
            assert e["Solver"]["Model Evaluation Count"] == 64 and e["Current Generation"] == 8


# ---------------------------------------------------------------- detailed/cmaes/run-{min,max}cmaes*.py -----
@gpu
class TestDetailed:
    @pytest.mark.parametrize("offset", [10.0, 1e3, 1e6, 1e9])
    def test_min_parabola_with_offsets(self, offset):
        e = korali.Experiment()
        e["Problem"]["Type"] = "Optimization"
        e["Problem"]["Objective Function"] = make_minmodel(offset)
        e["Variables"][0]["Name"] = "X"
        e["Variables"][0]["Lower Bound"] = -10.0
        e["Variables"][0]["Upper Bound"] = +10.0
        e["Solver"]["Type"] = "Optimizer/CMAES"
        e["Solver"]["Population Size"] = 32
        e["Solver"]["Termination Criteria"]["Min Value Difference Threshold"] = 1e-8
        e["Solver"]["Termination Criteria"]["Max Generations"] = 100
        e["Console Output"]["Verbosity"] = "Silent"
        e["File Output"]["Enabled"] = False
        e["Random Seed"] = 314
        korali.Engine().run(e)
        assert abs(e["Solver"]["Best Ever Variables"][0] - 2.0) < 1e-2
        assert abs(e["Solver"]["Current Best Variables"][0] - 2.0) < 1e-2
        assert abs(e["Solver"]["Best Ever Value"] + offset) < 1e-3 * max(1.0, offset * 1e-9 * 1e3)
        assert abs(e["Results"]["Best Sample"]["F(x)"] - e["Solver"]["Best Ever Value"]) == 0
        assert e["Results"]["Best Sample"]["Parameters"] == e["Solver"]["Best Ever Variables"]


# ---------------------------------------------------------------- device conduit + checkpoint / resume -------
@gpu
def test_device_objective_and_checkpoint_resume(tmp_path):
    """config 1 through the Korali API with the batched device conduit, then resume from the saved state
    (experiment.cpp.base:120-153): generations 1..20 + resume to 40 == one run of 40 generations."""
    def make(gens):
        e = korali.Experiment()
        e["Problem"]["Type"] = "Optimization"
        e["Problem"]["Objective Function"] = "Rosenbrock"           # built-in device objective
        for i in range(10):
            e["Variables"][i]["Name"] = "X%d" % i
            e["Variables"][i]["Initial Value"] = 0.0
            e["Variables"][i]["Initial Standard Deviation"] = 0.5
        e["Solver"]["Type"] = "Optimizer/CMAES"
        e["Solver"]["Population Size"] = 32
        e["Solver"]["Termination Criteria"]["Max Generations"] = gens
        e["Console Output"]["Verbosity"] = "Silent"
        e["File Output"]["Path"] = str(tmp_path / ("run%d" % gens))
        e["File Output"]["Frequency"] = 10
        e["Random Seed"] = 0xC0FEE
        return e
    k = korali.Engine()
    k["Conduit"]["Type"] = "Device"
    full = make(40); k.run(full)
    part = make(20); k.run(part)
    saved = json.load(open(str(tmp_path / "run20" / "latest")))
    assert saved["Current Generation"] == 20 and saved["Solver"]["Model Evaluation Count"] == 640
    assert {"Sigma", "Covariance Matrix", "Current Mean", "Evolution Path", "Conjugate Evolution Path", "Axis Lengths",
            "Best Ever Value", "Mu Weights"} <= set(saved["Solver"])
    r = korali.Experiment()
    r.loadState(str(tmp_path / "run20" / "latest"))
    r["Problem"]["Objective Function"] = "Rosenbrock"
    r["Solver"]["Termination Criteria"]["Max Generations"] = 40
    r["File Output"]["Enabled"] = False
    k.run(r)
    assert r["Current Generation"] == 40
    # the eigenvector basis is re-derived after a resume (signs/rounding), so trajectories agree closely, not bitwise
    assert abs(r["Solver"]["Best Ever Value"] - full["Solver"]["Best Ever Value"]) <= 1e-6 * abs(full["Solver"]["Best Ever Value"]) + 1e-9
    assert os.path.exists(str(tmp_path / "run40" / "gen00000040.json"))


GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _from_reference_checkpoint(gen=50):
    e = korali.Experiment()
    e["Problem"]["Type"] = "Optimization"
    e["Problem"]["Objective Function"] = "Sphere"      # the fixture's model: F = -1/2 sum x^2 (checked against its Value Vector)
    e.loadState(os.path.join(GOLDEN, "reference_gen%08d.json" % gen))
    e["Console Output"]["Verbosity"] = "Silent"
    e["File Output"]["Enabled"] = False
    return e


@pytest.mark.skipif(HAS_GPU, reason="CPU-only behaviour")
def test_reference_written_checkpoint_passes_the_strict_configuration():
    """A result file the REFERENCE wrote (tests/python/plot/cmaes/gen00000050.json, kept as tests/golden/reference_gen00000050.json)
    goes through Experiment::loadState + the strict setConfiguration: every key is consumed, so the only thing that stops the
    run on a CPU-only box is the missing device."""
    with pytest.raises(RuntimeError, match="no CPU fallback|CUDA device"):
        korali.Engine().run(_from_reference_checkpoint())


@gpu
def test_resume_from_a_reference_written_checkpoint(tmp_path):
    """Checkpoint interchange (SURVEY 8f-1): e.loadState() of a file written by the reference restores its state exactly, the run
    continues from generation 50 to the file's own Max Generations (100), and the files this build writes carry every key
    python/korali/plot/CMAES.py:42-55 reads."""
    ref50 = json.load(open(os.path.join(GOLDEN, "reference_gen00000050.json")))
    ref100 = json.load(open(os.path.join(GOLDEN, "reference_gen00000100.json")))
    k = korali.Engine()
    # (a) nothing left to run: the state that comes back is the file's, bit for bit
    e = _from_reference_checkpoint()
    e["Solver"]["Termination Criteria"]["Max Generations"] = 50
    k.run(e)
    assert e["Current Generation"] == 50
    for key in ["Sigma", "Best Ever Value", "Current Best Value", "Previous Best Ever Value", "Conjugate Evolution Path L2 Norm",
                "Model Evaluation Count", "Infeasible Sample Count", "Maximum Covariance Eigenvalue", "Minimum Covariance Eigenvalue"]:
        assert e["Solver"][key] == ref50["Solver"][key], key
    for key in ["Current Mean", "Previous Mean", "Covariance Matrix", "Evolution Path", "Conjugate Evolution Path", "Axis Lengths",
                "Covariance Eigenvector Matrix", "Best Ever Variables"]:
        assert np.array_equal(np.array(e["Solver"][key], dtype=float).ravel(), np.array(ref50["Solver"][key], dtype=float).ravel()), key
    # (b) continue: generations 51..100 on the device (own Philox stream from here on, so the trajectory is statistically, not
    # numerically, the reference's)
    e = _from_reference_checkpoint()
    e["File Output"]["Enabled"] = True
    e["File Output"]["Path"] = str(tmp_path / "cont")
    e["File Output"]["Frequency"] = 50
    k.run(e)
    assert e["Current Generation"] == 100
    assert e["Solver"]["Model Evaluation Count"] == ref100["Solver"]["Model Evaluation Count"] == 3200
    assert e["Solver"]["Best Ever Value"] >= ref50["Solver"]["Best Ever Value"]
    assert abs(e["Solver"]["Best Ever Value"]) < 1e-7                      # the reference reached -2.8e-10 at generation 100
    assert 0.05 < e["Solver"]["Sigma"] / ref100["Solver"]["Sigma"] < 20.0
    # (c) key set of the written result file
    out = json.load(open(str(tmp_path / "cont" / "gen00000100.json")))
    assert out["Current Generation"] == 100
    for key in ["Maximum Covariance Eigenvalue", "Minimum Covariance Eigenvalue", "Current Best Value", "Best Ever Value", "Sigma",
                "Conjugate Evolution Path L2 Norm", "Axis Lengths", "Current Best Variables", "Best Ever Variables", "Covariance Matrix"]:
        assert key in out["Solver"], key
    assert len(out["Solver"]["Covariance Matrix"]) == 100 and len(out["Solver"]["Axis Lengths"]) == 10
    assert [v["Name"] for v in out["Variables"]] == [v["Name"] for v in ref50["Variables"]]
    # ... and the reference's own file loads the same way as ours (same top-level layout)
    assert {"Current Generation", "Solver", "Problem", "Variables", "Random Seed", "Is Finished"} <= set(out) & set(ref100)


@gpu
def test_resume_is_bitwise(tmp_path):
    """The tridiagonalisation-based eigensolver keeps no history (the one-sided Jacobi was warm-started from the previous basis),
    and the Philox counters are (seed, generation, sample): a run resumed from a saved state repeats the uninterrupted run bit for
    bit."""
    def make(gens):
        e = korali.Experiment()
        e["Problem"]["Type"] = "Optimization"
        e["Problem"]["Objective Function"] = "Ellipsoid"
        for i in range(40):
            e["Variables"][i]["Name"] = "X%d" % i
            e["Variables"][i]["Initial Value"] = 2.0
            e["Variables"][i]["Initial Standard Deviation"] = 1.0
        e["Solver"]["Type"] = "Optimizer/CMAES"
        e["Solver"]["Population Size"] = 96
        e["Solver"]["Termination Criteria"]["Max Generations"] = gens
        e["Console Output"]["Verbosity"] = "Silent"
        e["File Output"]["Path"] = str(tmp_path / ("run%d" % gens))
        e["File Output"]["Frequency"] = 15
        e["Random Seed"] = 4242
        return e
    k = korali.Engine()
    full = make(30); k.run(full)
    part = make(15); k.run(part)
    r = korali.Experiment()
    r["Problem"]["Objective Function"] = "Ellipsoid"
    r.loadState(str(tmp_path / "run15" / "latest"))
    r["Solver"]["Termination Criteria"]["Max Generations"] = 30
    r["File Output"]["Enabled"] = False
    k.run(r)
    assert r["Current Generation"] == 30
    for key in ["Sigma", "Best Ever Value", "Current Best Value", "Conjugate Evolution Path L2 Norm"]:
        assert r["Solver"][key] == full["Solver"][key], key
    for key in ["Current Mean", "Covariance Matrix", "Evolution Path", "Conjugate Evolution Path", "Best Ever Variables"]:
        assert r["Solver"][key] == full["Solver"][key], key


@gpu
def test_large_n_checkpoint_uses_npy_side_cars(tmp_path):
    """N x N arrays above 2^22 entries (config 4: N = 4096) do not fit a JSON result file (SURVEY 5.4): C and B are saved as .npy
    side-cars, loadState reads them back, and the resumed run is bitwise the uninterrupted one."""
    n = 2100
    def make(gens, path):
        e = korali.Experiment()
        e["Problem"]["Type"] = "Optimization"
        e["Problem"]["Objective Function"] = "Sphere"
        for i in range(n):
            e["Variables"][i]["Name"] = "X%d" % i
            e["Variables"][i]["Initial Value"] = 1.0
            e["Variables"][i]["Initial Standard Deviation"] = 1.0
        e["Solver"]["Type"] = "Optimizer/CMAES"
        e["Solver"]["Population Size"] = 64
        e["Solver"]["Termination Criteria"]["Max Generations"] = gens
        e["Console Output"]["Verbosity"] = "Silent"
        e["File Output"]["Path"] = str(tmp_path / path)
        e["File Output"]["Frequency"] = 2
        e["Random Seed"] = 99
        return e
    k = korali.Engine()
    full = make(4, "full"); k.run(full)
    part = make(2, "part"); k.run(part)
    saved = json.load(open(str(tmp_path / "part" / "gen00000002.json")))
    assert "Covariance Matrix" not in saved["Solver"] and saved["Solver"]["Covariance Matrix File"] == "gen00000002.json.C.npy"
    c = np.load(str(tmp_path / "part" / "gen00000002.json.C.npy"))
    assert c.shape == (n, n) and np.array_equal(c, c.T)
    r = korali.Experiment()
    r["Problem"]["Objective Function"] = "Sphere"
    r.loadState(str(tmp_path / "part" / "latest"))
    r["Solver"]["Termination Criteria"]["Max Generations"] = 4
    r["File Output"]["Enabled"] = False
    k.run(r)
    assert r["Current Generation"] == 4
    assert r["Solver"]["Sigma"] == full["Solver"]["Sigma"] and r["Solver"]["Best Ever Value"] == full["Solver"]["Best Ever Value"]
    assert r["Solver"]["Current Mean"] == full["Solver"]["Current Mean"]
    assert r["Solver"]["Evolution Path"] == full["Solver"]["Evolution Path"]


@gpu
def test_python_model_matches_device_objective():
    """The batched host conduit (Python model, as the reference's users write it) and the device objective see the same
    samples and must produce the same trajectory."""
    res = []
    for obj in ("Rosenbrock", negative_rosenbrock):
        e = korali.Experiment()
        e["Problem"]["Type"] = "Optimization"
        e["Problem"]["Objective Function"] = obj
        for i in range(6):
            e["Variables"][i]["Name"] = "X%d" % i
            e["Variables"][i]["Lower Bound"] = -5.0
            e["Variables"][i]["Upper Bound"] = +5.0
        e["Solver"]["Type"] = "Optimizer/CMAES"
        e["Solver"]["Population Size"] = 16
        e["Solver"]["Termination Criteria"]["Max Generations"] = 30
        e["Console Output"]["Verbosity"] = "Silent"
        e["File Output"]["Enabled"] = False
        e["Random Seed"] = 42
        korali.Engine().run(e)
        res.append((e["Solver"]["Best Ever Value"], e["Solver"]["Sigma"]))
    assert abs(res[0][0] - res[1][0]) <= 1e-9 * abs(res[1][0]) and abs(res[0][1] - res[1][1]) <= 1e-9 * res[1][1]


@gpu
def test_whole_population_models_numpy_and_device_tensor():
    """SURVEY 8f-3: user models that take the WHOLE population — korali.batched(fn) gets X as one NumPy array, korali.batched_device(fn)
    gets a torch tensor that aliases the sample matrix in HBM — against the reference-style per-sample model (lambda Python calls
    per generation, conduit.cpp.base:29-88). Same samples; the NumPy variants use the same arithmetic, so they agree bit for bit."""
    def per_sample(s):
        x = np.asarray(s["Parameters"])
        s["F(x)"] = float(-np.sum((x - 1.5) ** 2 * np.arange(1, x.size + 1)))
    calls = {"numpy": 0, "device": 0}
    def whole_numpy(X):
        calls["numpy"] += 1
        assert X.shape == (64, 12)
        return np.array([float(-np.sum((x - 1.5) ** 2 * np.arange(1, x.size + 1))) for x in X])
    def whole_device(X):
        calls["device"] += 1
        assert X.is_cuda and X.dtype == torch.float64 and tuple(X.shape) == (64, 12)
        w = torch.arange(1, 13, device=X.device, dtype=torch.float64)
        return -(((X - 1.5) ** 2) * w).sum(dim=1)
    res = {}
    for name, obj in (("per_sample", per_sample), ("numpy", korali.batched(whole_numpy)), ("device", korali.batched_device(whole_device))):
        e = korali.Experiment()
        e["Problem"]["Type"] = "Optimization"
        e["Problem"]["Objective Function"] = obj
        for i in range(12):
            e["Variables"][i]["Name"] = "X%d" % i
            e["Variables"][i]["Initial Value"] = 0.0
            e["Variables"][i]["Initial Standard Deviation"] = 1.0
        e["Solver"]["Type"] = "Optimizer/CMAES"
        e["Solver"]["Population Size"] = 64
        e["Solver"]["Termination Criteria"]["Max Generations"] = 40
        e["Console Output"]["Verbosity"] = "Silent"
        e["File Output"]["Enabled"] = False
        e["Random Seed"] = 77
        korali.Engine().run(e)
        res[name] = (e["Solver"]["Best Ever Value"], e["Solver"]["Sigma"], e["Solver"]["Current Mean"], e["Solver"]["Model Evaluation Count"])
    assert calls == {"numpy": 40, "device": 40}                      # ONE call per generation
    assert res["numpy"][:3] == res["per_sample"][:3]                  # same arithmetic on the same samples
    assert res["device"][3] == res["numpy"][3] == 40 * 64
    assert abs(res["device"][0] - res["numpy"][0]) <= 1e-9 * abs(res["numpy"][0]) + 1e-12
    assert abs(res["device"][1] - res["numpy"][1]) <= 1e-8 * res["numpy"][1]


@gpu
def test_device_model_errors_surface():
    def bad(X):
        return torch.full((X.shape[0],), float("nan"), device=X.device, dtype=torch.float64)
    e = base_1d(8, 5)
    e["Variables"][0]["Initial Value"] = 1.0
    e["Problem"]["Objective Function"] = korali.batched_device(bad)
    with pytest.raises(RuntimeError, match="Non finite"):
        korali.Engine().run(e)
    def boom(X):
        raise ValueError("model exploded")
    e = base_1d(8, 5)
    e["Variables"][0]["Initial Value"] = 1.0
    e["Problem"]["Objective Function"] = korali.batched(boom)
    with pytest.raises(RuntimeError, match="model exploded"):
        korali.Engine().run(e)


# ---------------------------------------------------------------- Use Gradient Information ------------------
@pytest.mark.gpu
def test_run_cmaes_gradient_example():
    """examples/optimization/stochastic/run-cmaes-gradient.py, unchanged apart from the import and the output switches:
    10-D negative sphere whose model also returns "Gradient" (operation "Evaluate With Gradients")."""
    import math
    runs = {}
    for use_grad, obj in ((True, negative_sphere), (False, negative_sphere), (True, "Sphere")):
        e = korali.Experiment()
        e["Random Seed"] = 0xC0FEE
        e["Problem"]["Type"] = "Optimization"
        e["Problem"]["Objective Function"] = obj
        dim = 10
        for i in range(dim):
            e["Variables"][i]["Name"] = "X" + str(i)
            e["Variables"][i]["Lower Bound"] = -25.0
            e["Variables"][i]["Upper Bound"] = +25.0
            e["Variables"][i]["Initial Standard Deviation"] = 15.0 / math.sqrt(dim)
        e["Solver"]["Type"] = "Optimizer/CMAES"
        e["Solver"]["Population Size"] = 32
        e["Solver"]["Use Gradient Information"] = use_grad
        e["Solver"]["Termination Criteria"]["Min Value Difference Threshold"] = 1e-32
        e["Solver"]["Termination Criteria"]["Max Generations"] = 100
        e["Console Output"]["Verbosity"] = "Silent"
        e["File Output"]["Enabled"] = False
        korali.Engine().run(e)
        runs[(use_grad, obj if isinstance(obj, str) else "python")] = (e["Solver"]["Best Ever Value"], e["Solver"]["Current Mean"], e["Current Generation"])
        assert e["Solver"]["Use Gradient Information"] == (1 if use_grad else 0) and e["Solver"]["Gradient Step Size"] == float(np.float32(0.01))   # a float in the reference (SURVEY Q9)
    with_grad, without, device = runs[(True, "python")], runs[(False, "python")], runs[(True, "Sphere")]
    assert with_grad[2] == without[2] == 100
    assert abs(with_grad[0]) < 1e-6 and abs(without[0]) < 1e-6        # both converge to the optimum 0 at x = 0
    assert not np.allclose(with_grad[1], without[1], rtol=1e-6, atol=0)   # the gradient step changes the trajectory
    # the Python model (gradients through the host conduit) and the device objective (analytic gradients) agree
    assert abs(with_grad[0] - device[0]) <= 1e-9 * max(abs(device[0]), 1e-300) + 1e-300
    assert np.allclose(with_grad[1], device[1], rtol=1e-9, atol=1e-300)


@pytest.mark.gpu
def test_gradient_information_errors():
    e = korali.Experiment()
    e["Problem"]["Type"] = "Optimization"
    e["Problem"]["Objective Function"] = evalmodel          # returns no "Gradient"
    e["Variables"][0]["Name"] = "X"
    e["Variables"][0]["Lower Bound"] = -10.0
    e["Variables"][0]["Upper Bound"] = +10.0
    e["Solver"]["Type"] = "Optimizer/CMAES"
    e["Solver"]["Population Size"] = 8
    e["Solver"]["Use Gradient Information"] = True
    e["Solver"]["Termination Criteria"]["Max Generations"] = 5
    e["Console Output"]["Verbosity"] = "Silent"
    e["File Output"]["Enabled"] = False
    with pytest.raises(RuntimeError, match="did not set 'Gradient'"):
        korali.Engine().run(e)
    e2 = korali.Experiment()
    e2["Problem"]["Type"] = "Optimization"
    e2["Problem"]["Objective Function"] = negative_sphere
    e2["Variables"][0]["Name"] = "X"
    e2["Variables"][0]["Lower Bound"] = -10.0
    e2["Variables"][0]["Upper Bound"] = +10.0
    e2["Solver"]["Type"] = "Optimizer/CMAES"
    e2["Solver"]["Population Size"] = 8
    e2["Solver"]["Use Gradient Information"] = True
    e2["Solver"]["Gradient Step Size"] = -1.0
    e2["Console Output"]["Verbosity"] = "Silent"
    e2["File Output"]["Enabled"] = False
    with pytest.raises(RuntimeError, match="Gradient Step Size must be larger than 0.0"):
        korali.Engine().run(e2)


# ---------------------------------------------------------------- discrete variables ------------------------
@pytest.mark.gpu
def test_run_cmaes_discrete_example():
    """examples/optimization/discrete/run-cmaes.py: 10 variables, four of them with Granularity 1.0."""
    e = korali.Experiment()
    e["Problem"]["Type"] = "Optimization"
    e["Problem"]["Objective Function"] = discrete_model
    for i in range(10):
        e["Variables"][i]["Name"] = "X" + str(i)
        e["Variables"][i]["Initial Value"] = 1.0
        e["Variables"][i]["Lower Bound"] = -19.0
        e["Variables"][i]["Upper Bound"] = +21.0
    e["Variables"][0]["Granularity"] = 1.0
    e["Variables"][1]["Granularity"] = 1.0
    e["Variables"][3]["Granularity"] = 1.0
    e["Variables"][6]["Granularity"] = 1.0
    e["Solver"]["Type"] = "Optimizer/CMAES"
    e["Solver"]["Population Size"] = 8
    e["Solver"]["Termination Criteria"]["Min Value Difference Threshold"] = 1e-9
    e["Solver"]["Termination Criteria"]["Max Generations"] = 5000
    e["File Output"]["Enabled"] = False
    e["Console Output"]["Verbosity"] = "Silent"
    k = korali.Engine()
    k.run(e)
    best = e["Results"]["Best Sample"]["Parameters"]
    assert all(best[i] == round(best[i]) for i in (0, 1, 3, 6))
    assert abs(e["Results"]["Best Sample"]["F(x)"]) < 1e-6 and max(abs(v) for v in best) < 1e-2
    e2 = korali.Experiment()
    e2["Problem"]["Type"] = "Optimization"
    e2["Problem"]["Objective Function"] = discrete_model
    e2["Variables"][0]["Name"] = "X"
    e2["Variables"][0]["Granularity"] = -1.0
    e2["Solver"]["Type"] = "Optimizer/CMAES"
    e2["Solver"]["Population Size"] = 8
    e2["File Output"]["Enabled"] = False
    e2["Console Output"]["Verbosity"] = "Silent"
    with pytest.raises(RuntimeError, match="Negative granularity"):
        korali.Engine().run(e2)
