"""ctypes mirror of include/kmocma.h (multi-objective CMA-ES on libkcma.so). Generic over the symbol prefix so that the CPU oracle
(oracle/libokcma.so, prefix ``omocma_``; test infrastructure only) can be driven with the same vocabulary. Nothing here loads the oracle."""
import ctypes as C
from ._abi import HandleBase, _dp

KMOCMA_ABI_VERSION = 1
OBJECTIVES = {"External": 0, "NegRosenbrockAndSphere": 1, "NegRosenbrockAndTwoSpheres": 2}
HOST_CB = C.CFUNCTYPE(None, C.c_void_p, _dp, C.c_uint64, C.c_uint64, _dp, C.c_uint64)


class KmocmaCfg(C.Structure):
    """struct kmocma_cfg (include/kmocma.h)."""
    _fields_ = [
        ("abi_version", C.c_uint32), ("reserved0", C.c_uint32),
        ("n", C.c_uint64), ("num_objectives", C.c_uint64), ("population_size", C.c_uint64), ("mu_value", C.c_uint64),
        ("evolution_path_adaption_strength", C.c_double), ("covariance_learning_rate", C.c_double),
        ("target_success_rate", C.c_double), ("threshold_probability", C.c_double), ("success_learning_rate", C.c_double),
        ("seed", C.c_uint64), ("objective", C.c_int32), ("device", C.c_int32),
        ("lower_bound", _dp), ("upper_bound", _dp), ("initial_value", _dp), ("initial_stddev", _dp),
    ]


class MocmaHandle(HandleBase):
    CFG = KmocmaCfg
    ARRAYS = ("lower_bound", "upper_bound", "initial_value", "initial_stddev")
    ENUMS = {"objective": OBJECTIVES}

    def _created(self, cfg):
        self.num_objectives = int(cfg.num_objectives)
        self.population_size, self.mu_value = int(self.scalar("Population Size")), int(self.scalar("Mu Value"))

    def inject_f(self, f):
        self._inject("inject_f", f)

    def set_host_objective(self, fn):
        """fn(X: ndarray[rows, n]) -> ndarray[rows, num_objectives]."""
        self._set_callback("set_host_objective", HOST_CB, fn, lambda rows, n, k: (rows, k))


def Solver(**kw):
    """One MOCMAES state resident on one B200 (a handle of libkcma.so)."""
    from . import _lib
    return MocmaHandle(_lib.lib(), "kmocma_", **kw)
