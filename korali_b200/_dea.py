"""ctypes mirror of include/kdea.h (Differential Evolution on libkcma.so). Generic over the symbol prefix so that the CPU oracle
(oracle/libokcma.so, prefix ``odea_``; test infrastructure only) can be driven with the same vocabulary. Nothing here loads the oracle."""
import ctypes as C
from ._abi import HandleBase, OBJECTIVES, _dp

KDEA_ABI_VERSION = 1
PARENT_RULES = {"Random": 0, "Best": 1}
ACCEPT_RULES = {"Best": 0, "Greedy": 1, "Improved": 2, "Iterative": 3}
MUTATION_RULES = {"Fixed": 0}


class KdeaCfg(C.Structure):
    """struct kdea_cfg (include/kdea.h)."""
    _fields_ = [
        ("abi_version", C.c_uint32), ("reserved0", C.c_uint32),
        ("n", C.c_uint64), ("population_size", C.c_uint64),
        ("crossover_rate", C.c_double), ("mutation_rate", C.c_double),
        ("mutation_rule", C.c_int32), ("parent_selection_rule", C.c_int32), ("accept_rule", C.c_int32), ("fix_infeasible", C.c_int32),
        ("seed", C.c_uint64), ("objective", C.c_int32), ("device", C.c_int32),
        ("lower_bound", _dp), ("upper_bound", _dp), ("objective_coef", _dp),
    ]


class DeaHandle(HandleBase):
    CFG = KdeaCfg
    ARRAYS = ("lower_bound", "upper_bound", "objective_coef")
    ENUMS = {"objective": OBJECTIVES, "parent_selection_rule": PARENT_RULES, "accept_rule": ACCEPT_RULES, "mutation_rule": MUTATION_RULES}

    def _created(self, cfg):
        self.population_size = int(cfg.population_size)

    def inject_f(self, f):
        self._inject("inject_f", f)


class Solver(DeaHandle):
    """One Differential Evolution solver state resident on one B200 (a kdea handle of libkcma.so)."""

    def __init__(self, **kw):
        from . import _lib
        super().__init__(_lib.lib(), "kdea_", **kw)

    def set_host_objective(self, fn):
        """fn(X: ndarray[rows, n]) -> ndarray[rows]; the batched host conduit."""
        self._set_callback("set_host_objective", C.CFUNCTYPE(None, C.c_void_p, _dp, C.c_uint64, C.c_uint64, _dp), fn,
                           lambda rows, n: (rows,))
