"""Optimizer/CMAES on Bayesian/Custom and Bayesian/Reference problems: the configuration errors of the Korali surface, raised before any
device is touched."""
import numpy as np
import pytest
import korali_b200 as korali


def bayes_custom():
    e = korali.Experiment()
    e["Problem"]["Type"] = "Bayesian/Custom"
    e["Problem"]["Likelihood Model"] = "Sphere"
    e["Distributions"][0]["Name"] = "P"
    e["Distributions"][0]["Type"] = "Univariate/Normal"
    e["Distributions"][0]["Mean"] = 1.0
    e["Distributions"][0]["Standard Deviation"] = 2.0
    for i in range(2):
        e["Variables"][i]["Name"] = "X%d" % i
        e["Variables"][i]["Prior Distribution"] = "P"
        e["Variables"][i]["Initial Value"] = 0.0
        e["Variables"][i]["Initial Standard Deviation"] = 1.0
    e["Solver"]["Type"] = "Optimizer/CMAES"
    e["Solver"]["Population Size"] = 8
    e["Solver"]["Termination Criteria"]["Max Generations"] = 5
    e["Console Output"]["Verbosity"] = "Silent"
    e["File Output"]["Enabled"] = False
    e["Random Seed"] = 3
    return e


def bayes_reference():
    e = bayes_custom()
    e["Problem"]["Type"] = "Bayesian/Reference"
    e["Problem"]["Likelihood Model"] = "Normal"
    e["Problem"]["Reference Data"] = [1.0, 2.0]
    e["Problem"]["Computational Model"] = lambda s: None
    return e


@pytest.mark.parametrize("make,mod,match", [
    (bayes_custom, lambda e: e["Solver"].__setitem__("Mu Type", "Proportional"), "'Mu Type' Proportional is not defined on Bayesian problems"),
    (bayes_custom, lambda e: e["Solver"].__setitem__("Use Gradient Information", True), "'Use Gradient Information' is not built for Bayesian"),
    (bayes_custom, lambda e: e["Problem"].__setitem__("Constraints", [lambda s: None]), "'Constraints' are not defined on Bayesian problems"),
    (bayes_reference, lambda e: e["Solver"].__setitem__("Mu Type", "Proportional"), "'Mu Type' Proportional"),
    (bayes_custom, lambda e: e["Distributions"][0].__setitem__("Type", "Univariate/Gamma"),
     "Optimizer/CMAES: prior distribution type 'Univariate/Gamma' of 'P' is not built"),
    (bayes_custom, lambda e: e["Variables"][1].__setitem__("Prior Distribution", "Q"), "prior distribution 'Q' is not defined in e\\['Distributions'\\]"),
    (bayes_custom, lambda e: e["Problem"].__setitem__("Likelihood Model", "Banana"), "Unknown device likelihood model"),
    (bayes_custom, lambda e: e["Problem"].__setitem__("Likelihood Model", 3.0), "neither a callable nor the name of a device model"),
    (bayes_reference, lambda e: e["Problem"].__setitem__("Likelihood Model", "Gaussian"), "unknown value 'Gaussian'"),
    (bayes_reference, lambda e: e["Problem"].__setitem__("Likelihood Model", "Geometric"), "is not built on the B200 path"),
    (bayes_reference, lambda e: e["Problem"].__setitem__("Reference Data", [1.0, np.inf]), "entry 1 is not a finite number"),
    (bayes_reference, lambda e: e["Problem"].__setitem__("Computational Model", "Linear"), "a callable was expected"),
    (bayes_custom, lambda e: e["Problem"].__setitem__("Objective Function", "Sphere"), "Unrecognized settings"),
])
def test_configuration_errors(make, mod, match):
    e = make()
    mod(e)
    e["Solver"]["Type"]     # reset the cursor after the chained access above
    with pytest.raises(RuntimeError, match=match):
        korali.Engine().run(e)


def test_missing_prior_distribution():
    e = bayes_custom()
    e["Variables"][2]["Name"] = "Y"
    e["Variables"][2]["Initial Value"] = 0.0
    with pytest.raises(RuntimeError, match="Variable 2 \\('Y'\\) has no 'Prior Distribution'"):
        korali.Engine().run(e)


@pytest.mark.parametrize("ptype", ["Bayesian/Custom", "Bayesian/Reference"])
def test_an_optimization_experiment_keyed_as_bayesian_names_the_problem_type(ptype):
    """An experiment written for Optimization ("Objective Function", no likelihood, no priors) under a Bayesian Problem Type: the first
    error names the Problem Type."""
    e = korali.Experiment()
    e["Problem"]["Type"] = ptype
    e["Problem"]["Objective Function"] = lambda s: None
    e["Variables"][0]["Name"] = "X"
    e["Variables"][0]["Lower Bound"] = -1.0
    e["Variables"][0]["Upper Bound"] = 1.0
    e["Solver"]["Type"] = "Optimizer/CMAES"
    e["Solver"]["Population Size"] = 8
    e["Console Output"]["Verbosity"] = "Silent"
    e["File Output"]["Enabled"] = False
    with pytest.raises(RuntimeError, match="Problem Type '%s' needs a 'Likelihood Model'" % ptype):
        korali.Engine().run(e)

