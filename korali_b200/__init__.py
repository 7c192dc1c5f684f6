"""korali_b200 — a B200-native CMA-ES generation loop behind Korali's own API.

    import korali_b200 as korali
    e = korali.Experiment(); e["Solver"]["Type"] = "Optimizer/CMAES"; ...; korali.Engine().run(e)

Served: `"Solver": {"Type": "Optimizer/CMAES"}` (the hot path) and its sibling population solvers `Optimizer/DEA`, `Optimizer/MOCMAES`
of `"Problem": {"Type": "Optimization"}`, the transitional MCMC sampler `Sampler/TMCMC` of `"Problem": {"Type": "Bayesian/Custom"}`
and `"Bayesian/Reference"` (priors from `e["Distributions"]`; Reference: "Reference Data", a "Computational Model" that sets
`sample["Reference Evaluations"]`, and the Normal, Positive Normal, StudentT or Poisson "Likelihood Model", reduced on the device) —
the same Bayesian problems also run with `Optimizer/CMAES`, which maximises the log-posterior and returns the MAP estimate,
plus the float ask/tell class `fCMAES` (SURVEY.md scope).
Layers: korali_b200._host (pybind11, C++: Engine / Experiment, mirrors python/korali/__init__.py:9-20 + source/engine.cpp:201-254)
 -> include/kcma.h (C ABI) -> korali_b200/libkcma.so (hand-written sm_100a CUDA). There is no CPU fallback.
"""
import os as _os

_HERE = _os.path.dirname(_os.path.abspath(__file__))


def _load_host():
    import importlib
    from . import _lib
    _lib.lib()   # fail loudly when libkcma.so is missing
    try:
        return importlib.import_module("korali_b200._host")
    except ImportError as exc:   # pragma: no cover
        raise ImportError("korali_b200/_host*.so is missing: run `python -m korali_b200.build`") from exc


def Engine():
    """korali.Engine() (python/korali/__init__.py:9-11)."""
    return _load_host().Engine()


def Experiment():
    """korali.Experiment() (python/korali/__init__.py:14-16)."""
    return _load_host().Experiment()


def batched(fn):
    """Marks a model that evaluates the WHOLE population in one call (SURVEY 8f-3): ``fn(X)`` with ``X`` a read-only NumPy view
    ``[samples, variables]`` of the population, returning ``samples`` values F(x). The reference hands its models one ``Sample``
    at a time (conduit.cpp.base:29-88); per-sample models still work, this is the fast path for Python models.

        e["Problem"]["Objective Function"] = korali.batched(lambda X: -np.sum(X * X, axis=1))

    As a Bayesian/Reference "Computational Model", ``fn(X)`` returns a dict keyed like the sample, each value broadcast to
    ``samples x M`` (a bare array of predictions is accepted for Poisson):

        e["Problem"]["Computational Model"] = korali.batched(lambda X: {"Reference Evaluations": X[:, :1] + X[:, 1:2] * t,
                                                                         "Standard Deviation": X[:, 2:3]})
    """
    def model(X):
        return fn(X)
    model._korali_batched = "numpy"
    return model


class _DeviceArray:
    """Zero-copy view of device memory for ``torch.as_tensor`` (CUDA array interface, version 3)."""

    def __init__(self, ptr, shape, strides):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "strides": tuple(strides), "typestr": "<f8", "data": (int(ptr), False), "version": 3}


def batched_device(fn):
    """Marks a model that runs ON THE GPU: ``fn(X)`` with ``X`` a ``torch.float64`` CUDA tensor ``[samples, variables]`` that aliases
    the solver's sample matrix in HBM (no copy; do not write to it), returning a CUDA tensor of ``samples`` values F(x). The
    population never leaves the device.

        e["Problem"]["Objective Function"] = korali.batched_device(lambda X: -(X * X).sum(dim=1))

    As a Bayesian/Reference "Computational Model", ``fn(X)`` returns a dict of CUDA tensors keyed like the sample ("Reference
    Evaluations" and the likelihood's per-point parameter; a bare tensor for Poisson), each broadcast to ``samples x M`` by ``copy_``
    straight into the solver's buffers on its stream.
    """
    def model(x_ptr, rows, n, ldx, f_ptr, stream):
        import torch
        X = torch.as_tensor(_DeviceArray(x_ptr, (rows, n), (ldx * 8, 8)), device="cuda")
        F = torch.as_tensor(_DeviceArray(f_ptr, (rows,), (8,)), device="cuda")
        if stream:
            with torch.cuda.stream(torch.cuda.ExternalStream(stream)):
                F.copy_(fn(X).to(torch.float64).reshape(rows))
        else:       # the solver runs on the legacy default stream, which is also torch's default stream
            F.copy_(fn(X).to(torch.float64).reshape(rows))

    def reference(x_ptr, rows, n, ldx, g_ptr, p_ptr, m, ldm, stream, g_key, p_key):
        import contextlib
        import torch
        X = torch.as_tensor(_DeviceArray(x_ptr, (rows, n), (ldx * 8, 8)), device="cuda")
        with torch.cuda.stream(torch.cuda.ExternalStream(stream)) if stream else contextlib.nullcontext():
            r = fn(X)
            if not isinstance(r, dict):
                if p_key is not None:
                    raise ValueError("The batched computational model must return a dict with '%s' and '%s' (a bare tensor is accepted "
                                     "for Poisson only)" % (g_key, p_key))
                r = {g_key: r}
            for key, ptr in ((g_key, g_ptr), (p_key, p_ptr)):
                if key is None:
                    continue
                if key not in r:
                    raise KeyError("The batched computational model did not return '%s'" % key)
                v = torch.as_tensor(r[key], dtype=torch.float64, device="cuda")
                dst = torch.as_tensor(_DeviceArray(ptr, (rows, m), (ldm * 8, 8)), device="cuda")
                try:
                    dst.copy_(v)
                except RuntimeError:
                    raise ValueError("The batched computational model's '%s' has shape %s, which does not broadcast to %d samples x %d "
                                     "reference points" % (key, tuple(v.shape), rows, m)) from None
    model._korali_batched = "device"
    model._korali_reference = reference     # Bayesian/Reference: the outputs go to the solver's prediction / parameter buffers
    return model



def fCMAES(nVars, populationSize=0, muSize=0, device=0):
    """The ask/tell surface of the reference's float CMA-ES (deepSupervisor/optimizers/fCMAES.{hpp,cpp}) on the device generation loop:
    ``prepareGeneration()`` / ``_samplePopulation`` / ``updateDistribution(evaluations)`` / ``checkTermination()`` (korali_b200/_fcmaes.py)."""
    from ._fcmaes import fCMAES as _F
    return _F(nVars, populationSize, muSize, device)
