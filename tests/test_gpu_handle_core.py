"""The state access and run loop the four solver ABIs share (korali_b200/csrc/handle.cuh), checked per solver on a small handle:
every get_scalar / get_array key with its element count, host-scalar round trips, the error messages, device selection and
<prefix>run's *done after a failing generation."""
import ctypes as C
import numpy as np
import pytest
import torch
from korali_b200 import _dea, _lib, _mocma, _tmcmc
from korali_b200._abi import KcmaError, _dp

pytestmark = pytest.mark.gpu

TC = "Termination Criteria/"
N = 4
CMA = dict(n=N, population_size=8, objective="NegSphere", initial_value=0.0, initial_stddev=1.0, keep_population=1, seed=1)
DEA = dict(n=N, population_size=16, objective="NegSphere", lower_bound=-5.0, upper_bound=5.0, seed=1)
MOCMA = dict(n=N, num_objectives=2, population_size=8, mu_value=4, objective="NegRosenbrockAndSphere", lower_bound=-2.0, upper_bound=2.0,
             seed=1)
TMCMC = dict(n=3, population_size=64, priors=[("Uniform", -1.0, 1.0)] * 3, loglik="NegSphere", seed=1)

# (make, keyword arguments, External variant, array keys -> count, scalar keys, writable host scalars, scalars set_scalar rejects,
#  "Current Generation" of a new handle, message for a too small buffer)
SOLVERS = {
    "kcma_": (_lib.Solver, CMA, dict(CMA, objective="External"),
              {"Covariance Matrix": N * N, "Covariance Eigenvector Matrix": N * N, "Axis Lengths": N, "Current Mean": N, "Previous Mean": N,
               "Mean Update": N, "Evolution Path": N, "Conjugate Evolution Path": N, "Auxiliar BDZ Matrix": N, "Mu Weights": 4,
               "Value Vector": 8, "Best Ever Variables": N, "Current Best Variables": N, "Objective Coefficients": N, "BDZ Matrix": 8 * N,
               "Sample Population": 8 * N},
              ["Sigma", "Conjugate Evolution Path L2 Norm", "Best Ever Value", "Previous Best Ever Value", "Previous Best Value",
               "Current Best Value", "Maximum Diagonal Covariance Matrix Element", "Minimum Diagonal Covariance Matrix Element",
               "Maximum Covariance Eigenvalue", "Minimum Covariance Eigenvalue", "Current Min Standard Deviation",
               "Current Max Standard Deviation", "Global Success Rate", "Chi Square Number Discrete Mutations", "Current Generation",
               "Model Evaluation Count", "Variable Count", "Current Population Size", "Current Mu Value", "Infeasible Sample Count",
               "Number Of Discrete Mutations", "Number Masking Matrix Entries", "Resampled Parameter Count",
               "Covariance Matrix Adaptation Count", "Max Constraint Violation Count", "Constraint Evaluation Count",
               "Covariance Matrix Adaption Factor", "Normal Vector Learning Rate", "Is Viability Regime", "Has Constraints",
               "Best Valid Sample", TC + "Max Infeasible Resamplings", "Shard Begin", "Shard End"],
              ["Trace", "Effective Mu", "Sigma Cumulation Factor", "Damp Factor", "Cumulative Covariance", "Chi Square Number",
               TC + "Max Condition Covariance Matrix", TC + "Min Standard Deviation", TC + "Max Standard Deviation", TC + "Max Value",
               TC + "Min Value Difference Threshold", TC + "Max Model Evaluations", TC + "Max Generations"],
              ["Variable Count", "Current Population Size", "Shard Begin"], 0, "buffer too small for '%s' (%d < %d)"),
    "kdea_": (_dea.Solver, DEA, dict(DEA, objective="External"),
              {"Sample Population": 16 * N, "Candidate Population": 16 * N, "Value Vector": 16, "Previous Value Vector": 16,
               "Current Mean": N, "Previous Mean": N, "Best Ever Variables": N, "Current Best Variables": N, "Max Distances": N},
              ["Best Ever Value", "Current Best Value", "Previous Best Value", "Previous Best Ever Value", "Current Minimum Step Size",
               "Best Sample Index", "Infeasible Sample Count", "Current Generation", "Model Evaluation Count", "Variable Count"],
              [TC + "Max Infeasible Resamplings", TC + "Min Value", TC + "Min Step Size", TC + "Max Value",
               TC + "Min Value Difference Threshold", TC + "Max Generations", TC + "Max Model Evaluations"],
              ["Variable Count"], 0, "buffer too small for '%s' (%d < %d)"),
    "kmocma_": (_mocma.Solver, MOCMA, dict(MOCMA, objective="External"),
                {**{p + " Sample Population": r * N for p, r in [("Current", 8), ("Previous", 8), ("Parent", 4)]},
                 **{p + " Sigma": r for p, r in [("Current", 8), ("Previous", 8), ("Parent", 4)]},
                 **{p + " Covariance Matrix": r * N * N for p, r in [("Current", 8), ("Previous", 8), ("Parent", 4)]},
                 **{p + " Evolution Paths": r * N for p, r in [("Current", 8), ("Previous", 8), ("Parent", 4)]},
                 **{p + " Success Probabilities": r for p, r in [("Current", 8), ("Previous", 8), ("Parent", 4)]},
                 "Current Values": 16, "Previous Values": 16, "Parent Index": 8, "Best Ever Values": 2, "Current Best Values": 2,
                 "Previous Best Values": 2, "Best Ever Variables Vector": 2 * N, "Current Best Variables Vector": 2 * N,
                 "Current Best Value Differences": 2, "Current Best Variable Differences": 2, "Current Min Standard Deviations": 8,
                 "Current Max Standard Deviations": 8, "Sample Collection": 0, "Sample Value Collection": 0, "Sorted Indices": 16},
                ["Current Non Dominated Sample Count", "Infeasible Sample Count", "Model Evaluation Count", "Current Generation",
                 "Sample Collection Size", "Population Size", "Mu Value", "Evolution Path Adaption Strength", "Covariance Learning Rate"],
                [TC + "Min Value Difference Threshold", TC + "Min Variable Difference Threshold", TC + "Min Standard Deviation",
                 TC + "Max Standard Deviation", TC + "Max Generations", TC + "Max Model Evaluations"],
                ["Evolution Path Adaption Strength", "Covariance Learning Rate", "Population Size", "Mu Value", "Current Generation"], 1,
                "get_array(%s): capacity %d < %d"),
    "ktmcmc_": (_tmcmc.Solver, TMCMC, {k: v for k, v in TMCMC.items() if k != "loglik"},
                {"Sample Database": 64 * 3, "Sample LogLikelihood Database": 64, "Sample LogPrior Database": 64, "Covariance Matrix": 9,
                 "Proposal Factor": 9, "Mean Theta": 3, "Weights": 64, "Selection Counts": 64, "Chain Leaders": 0, "Chain Lengths": 0,
                 "Proposal Support": 0, "Accept Flags": 0, "Evaluation Rows": 0, "Evaluation LogLikelihoods": 0},
                ["Annealing Exponent", "Previous Annealing Exponent", "Annealing Exponent Update", "Coefficient Of Variation", "LogEvidence",
                 "Max Loglikelihood", "Chain Count", "Max Chain Steps", "Current Step", "Proposals Acceptance Rate",
                 "Selection Acceptance Rate", "Model Evaluation Count", "Current Generation", "Population Size", "Burn In"],
                [TC + "Target Annealing Exponent", TC + "Max Generations", TC + "Max Model Evaluations"],
                ["Annealing Exponent", "Population Size", "Current Generation"], 1, "get_array(%s): capacity %d < %d"),
}


def _get_array(s, key, cap):
    f = s._fn("get_array", C.c_int, [C.c_void_p, C.c_char_p, _dp, C.c_size_t, C.POINTER(C.c_size_t)])
    out, cnt = np.zeros(max(cap, 1)), C.c_size_t(0)
    s._check(f(s._live(), key.encode(), out.ctypes.data_as(_dp), cap, C.byref(cnt)))
    return out[:cnt.value]


@pytest.mark.parametrize("prefix", list(SOLVERS))
def test_state_keys_counts_and_messages(prefix):
    make, kw, _, arrays, scalars, writable, read_only, gen0, too_small = SOLVERS[prefix]
    s = make(**kw)
    for key, n in arrays.items():
        assert s.get(key).size == n, key
    for key in scalars + writable:
        s.scalar(key)
    assert s.scalar("Current Generation") == gen0
    for key in writable:
        s.set_scalar(key, 123.5)
        assert s.scalar(key) == 123.5, key
    for key in read_only:
        with pytest.raises(KcmaError, match="unknown scalar key '%s'" % key):
            s.set_scalar(key, 1.0)
    with pytest.raises(KcmaError, match="unknown scalar key 'No Such Key'"):
        s.scalar("No Such Key")
    with pytest.raises(KcmaError, match="unknown array key 'No Such Key'"):
        s.get("No Such Key")
    key, n = next((k, n) for k, n in arrays.items() if n > 1)
    with pytest.raises(KcmaError) as e:
        _get_array(s, key, n - 1)
    assert str(e.value) == too_small % (key, n - 1, n)
    assert np.array_equal(_get_array(s, key, n), s.get(key))
    s.close()


@pytest.mark.parametrize("prefix", list(SOLVERS))
def test_create_rejects_a_device_out_of_range(prefix):
    make, kw = SOLVERS[prefix][:2]
    with pytest.raises(KcmaError, match="invalid CUDA device %d" % torch.cuda.device_count()):
        make(device=torch.cuda.device_count(), **kw)


@pytest.mark.parametrize("prefix", list(SOLVERS))
def test_run_writes_done_when_a_generation_fails(prefix):
    make, external = SOLVERS[prefix][0], SOLVERS[prefix][2]
    s = make(**external)   # External model with nothing set or injected: the first evaluation fails
    done = C.c_uint64(12345)
    rc = s._fn("run", C.c_int, [C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)])(s._live(), 5, C.byref(done))
    assert rc != 0 and done.value == 0
    s.close()
