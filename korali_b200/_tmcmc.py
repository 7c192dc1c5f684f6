"""ctypes mirror of include/ktmcmc.h (transitional MCMC on libkcma.so). Generic over the symbol prefix so that the CPU oracle
(oracle/libokcma.so, prefix ``otmcmc_``; test infrastructure only) can be driven with the same vocabulary. Nothing here loads the oracle."""
import ctypes as C
import numpy as np
from ._abi import HandleBase, OBJECTIVES, _dp

KTMCMC_ABI_VERSION = 1
KCMA_OBJ_EXTERNAL = 100
PRIORS = {"Uniform": 0, "Normal": 1}
HOST_CB = C.CFUNCTYPE(None, C.c_void_p, _dp, C.c_uint64, C.c_uint64, _dp)

# every symbol include/ktmcmc.h declares
EXPORTS = [
    "ktmcmc_cfg_defaults", "ktmcmc_create", "ktmcmc_destroy", "ktmcmc_last_error", "ktmcmc_run_generation", "ktmcmc_anneal",
    "ktmcmc_resample", "ktmcmc_propose", "ktmcmc_eval", "ktmcmc_accept", "ktmcmc_inject_loglik", "ktmcmc_inject_factor",
    "ktmcmc_set_host_loglik", "ktmcmc_set_device_loglik", "ktmcmc_check_termination", "ktmcmc_run", "ktmcmc_get_array",
    "ktmcmc_get_scalar", "ktmcmc_set_scalar", "ktmcmc_launch_count",
]


class KtmcmcCfg(C.Structure):
    """struct ktmcmc_cfg (include/ktmcmc.h)."""
    _fields_ = [
        ("abi_version", C.c_uint32), ("reserved0", C.c_uint32),
        ("n", C.c_uint64), ("population_size", C.c_uint64), ("max_chain_length", C.c_uint64), ("default_burn_in", C.c_uint64),
        ("burn_in_count", C.c_uint64), ("per_generation_burn_in", C.POINTER(C.c_uint64)),
        ("target_cov", C.c_double), ("covariance_scaling", C.c_double), ("min_annealing_update", C.c_double),
        ("max_annealing_update", C.c_double), ("seed", C.c_uint64), ("loglik", C.c_int32), ("device", C.c_int32),
        ("prior_type", C.POINTER(C.c_int32)), ("prior_a", _dp), ("prior_b", _dp), ("loglik_coef", _dp),
    ]


class TmcmcHandle(HandleBase):
    """kw: n, population_size, priors = [(type, a, b)] * n (type "Uniform" | "Normal"), loglik (a KCMA_OBJ name such as "NegSphere",
    or "External"), per_generation_burn_in (list), loglik_coef, and the scalar fields of ktmcmc_cfg."""
    CFG = KtmcmcCfg
    ARRAYS = ("loglik_coef",)
    ENUMS = {"loglik": OBJECTIVES}

    def _field(self, cfg, k, v, kw):
        if k == "priors":
            cfg.prior_type = self._array([PRIORS[p[0]] for p in v], len(v), np.int32)
            cfg.prior_a, cfg.prior_b = self._array([p[1] for p in v], len(v)), self._array([p[2] for p in v], len(v))
        elif k == "per_generation_burn_in":
            cfg.per_generation_burn_in, cfg.burn_in_count = self._array(v, len(v), np.uint64), len(v)
        else:
            return False
        return True

    def _created(self, cfg):
        self.population_size = int(cfg.population_size)

    def anneal(self): self._call("anneal")
    def resample(self): self._call("resample")
    def propose(self): self._call("propose")
    def accept(self): self._call("accept")
    def inject_loglik(self, l): self._inject("inject_loglik", l)
    def inject_factor(self, a): self._inject("inject_factor", a)

    def set_host_loglik(self, fn):
        """fn(X: ndarray[rows, n]) -> ndarray[rows] of log-likelihoods."""
        self._set_callback("set_host_loglik", HOST_CB, fn, lambda rows, n: (rows,))


def Solver(**kw):
    """One TMCMC state resident on one B200 (a handle of libkcma.so)."""
    from . import _lib
    return TmcmcHandle(_lib.lib(), "ktmcmc_", **kw)
