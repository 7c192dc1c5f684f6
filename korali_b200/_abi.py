"""ctypes mirror of include/kcma.h (the C ABI of libkcma.so).

The binder is generic over the symbol prefix so that the CPU oracle (oracle/libokcma.so, prefix
``okcma_``; test infrastructure only) can be driven through the same vocabulary by the tests.
Nothing in this module loads the oracle.
"""
import ctypes as C
import math
import numpy as np

KCMA_ABI_VERSION = 1
MU_TYPES = {"Linear": 0, "Equal": 1, "Logarithmic": 2, "Proportional": 3}
OBJECTIVES = {"NegSphere": 0, "NegRosenbrock": 1, "NegAckley": 2, "NegEllipsoid": 3, "NegSumSq": 4,
              "NegSphereSin2": 5, "External": 100}
CONSTRAINTS = {"None": 0, "HalfSpace": 1, "External": 100}
INJ_Z, INJ_BDZ, INJ_X, INJ_F, INJ_BD, INJ_GRAD = 0, 1, 2, 3, 4, 5

_dp = C.POINTER(C.c_double)


class KcmaCfg(C.Structure):
    """struct kcma_cfg (include/kcma.h)."""
    _fields_ = [
        ("abi_version", C.c_uint32), ("reserved0", C.c_uint32),
        ("n", C.c_uint64), ("population_size", C.c_uint64), ("mu_value", C.c_uint64),
        ("mu_type", C.c_int32), ("diagonal_covariance", C.c_int32), ("mirrored_sampling", C.c_int32),
        ("is_sigma_bounded", C.c_int32),
        ("initial_sigma_cumulation_factor", C.c_double), ("initial_damp_factor", C.c_double),
        ("initial_cumulative_covariance", C.c_double),
        ("viability_population_size", C.c_uint64), ("viability_mu_value", C.c_uint64),
        ("max_covariance_matrix_corrections", C.c_uint64),
        ("target_success_rate", C.c_double), ("covariance_matrix_adaption_strength", C.c_double),
        ("normal_vector_learning_rate", C.c_double), ("global_success_learning_rate", C.c_double),
        ("max_infeasible_resamplings", C.c_uint64), ("seed", C.c_uint64),
        ("objective", C.c_int32), ("constraint_family", C.c_int32), ("n_constraints", C.c_uint64),
        ("objective_coef", _dp), ("constraint_shift", _dp),
        ("lower_bound", _dp), ("upper_bound", _dp), ("initial_value", _dp), ("initial_stddev", _dp),
        ("min_stddev_update", _dp),
        ("device", C.c_int32), ("rank", C.c_int32), ("nranks", C.c_int32), ("keep_population", C.c_int32),
        ("use_gradient_information", C.c_int32), ("reserved1", C.c_int32), ("gradient_step_size", C.c_double),
        ("granularity", _dp),
    ]


class KcmaError(RuntimeError):
    """Raised for every non-zero return code; carries the KORALI_LOG_ERROR-style message."""


def _as_dp(a):
    return a.ctypes.data_as(_dp)


class HandleBase:
    """A solver handle of one of the C ABIs of libkcma.so (kcma_, kdea_, kmocma_, ktmcmc_), or of a CPU oracle behind the same
    vocabulary in tests (okcma_, odea_, omocma_, otmcmc_). The ABIs share the shape of their entry points; a subclass names its cfg
    struct and how keyword arguments fill it:
      CFG     the ctypes mirror of <prefix>cfg
      ARRAYS  the double-array fields, broadcast to n values (None leaves the field NULL)
      ENUMS   {field: {name: value}} for fields that also take a name
    Any other keyword goes to _field, and then to the cfg field of its name."""
    CFG = None
    ARRAYS = ()
    ENUMS = {}

    def __init__(self, lib, prefix, **kw):
        self._lib, self._p, self._keep = lib, prefix, []
        cfg = self.CFG()
        self._fn("cfg_defaults", None, [C.POINTER(self.CFG)])(C.byref(cfg))
        self.n = n = int(kw["n"])
        for k, v in kw.items():
            if k in self.ARRAYS:
                if v is not None:
                    setattr(cfg, k, self._array(v, n))
            elif k in self.ENUMS:
                setattr(cfg, k, self.ENUMS[k][v] if isinstance(v, str) else int(v))
            elif not self._field(cfg, k, v, kw):
                setattr(cfg, k, v)
        self._h = C.c_void_p()
        if self._fn("create", C.c_int, [C.POINTER(self.CFG), C.POINTER(C.c_void_p)])(C.byref(cfg), C.byref(self._h)) != 0:
            raise KcmaError(self._fn("last_error", C.c_char_p, [C.c_void_p])(None).decode())
        self._created(cfg)

    def _array(self, v, count, dtype=np.float64):
        """A pointer to a contiguous copy of v broadcast to count values, kept alive with the handle."""
        arr = np.ascontiguousarray(np.broadcast_to(np.asarray(v, dtype=dtype), (count,)))
        self._keep.append(arr)
        return arr.ctypes.data_as(C.POINTER(np.ctypeslib.as_ctypes_type(dtype)))

    def _field(self, cfg, k, v, kw):
        """Fills a cfg field that needs more than a plain assignment; returns whether it did."""
        return False

    def _created(self, cfg):
        """Runs once the handle exists."""

    def _fn(self, name, restype, argtypes):
        f = getattr(self._lib, self._p + name)
        f.restype, f.argtypes = restype, argtypes
        return f

    def _live(self):
        """The handle, or an error instead of a NULL pointer into the library once close() was called."""
        if not getattr(self, "_h", None):
            raise KcmaError("the solver handle is closed")
        return self._h

    def _check(self, rc):
        if rc != 0:
            raise KcmaError(self._fn("last_error", C.c_char_p, [C.c_void_p])(self._live()).decode())

    def close(self):
        if getattr(self, "_h", None):
            self._fn("destroy", None, [C.c_void_p])(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # --- generation loop
    def _call(self, name):
        self._check(self._fn(name, C.c_int, [C.c_void_p])(self._live()))

    def ask(self): self._call("ask")
    def eval(self): self._call("eval")
    def tell(self): self._call("tell")
    def run_generation(self): self._call("run_generation")

    def run(self, max_generations):
        done = C.c_uint64(0)
        self._check(self._fn("run", C.c_int, [C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)])(
            self._live(), int(max_generations), C.byref(done)))
        return done.value

    def check_termination(self):
        fin, reason = C.c_int(0), C.c_char_p()
        self._check(self._fn("check_termination", C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_char_p)])(
            self._live(), C.byref(fin), C.byref(reason)))
        return bool(fin.value), (reason.value or b"").decode()

    def _inject(self, name, data):
        a = np.ascontiguousarray(data, dtype=np.float64).ravel()
        self._check(self._fn(name, C.c_int, [C.c_void_p, _dp, C.c_size_t])(self._live(), _as_dp(a), a.size))

    def _set_callback(self, name, cb_t, fn, shape):
        """Registers fn(X: ndarray[rows, n]) with <prefix><name> as the host callback cb_t(user, x, rows, n, out, *extra); fn's result
        is written to out as an array of shape(rows, n, *extra)."""
        def tramp(_u, x, rows, n, out, *extra):
            s = shape(rows, n, *extra)
            np.ctypeslib.as_array(out, shape=s)[:] = np.asarray(fn(np.ctypeslib.as_array(x, shape=(rows, n))), dtype=np.float64).reshape(s)
        cb = cb_t(tramp)
        self._keep.append(cb)
        self._check(self._fn(name, C.c_int, [C.c_void_p, cb_t, C.c_void_p])(self._live(), cb, None))

    # --- state
    def get(self, key):
        """Array by Korali key (1-D float64)."""
        f = self._fn("get_array", C.c_int, [C.c_void_p, C.c_char_p, _dp, C.c_size_t, C.POINTER(C.c_size_t)])
        cnt = C.c_size_t(0)
        self._check(f(self._live(), key.encode(), None, 0, C.byref(cnt)))
        out = np.empty(cnt.value, dtype=np.float64)
        if cnt.value:
            self._check(f(self._live(), key.encode(), _as_dp(out), out.size, C.byref(cnt)))
        return out

    def set(self, key, data):
        a = np.ascontiguousarray(data, dtype=np.float64).ravel()
        self._check(self._fn("set_array", C.c_int, [C.c_void_p, C.c_char_p, _dp, C.c_size_t])(self._live(), key.encode(), _as_dp(a), a.size))

    def scalar(self, key):
        v = C.c_double(math.nan)
        self._check(self._fn("get_scalar", C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_double)])(self._live(), key.encode(), C.byref(v)))
        return v.value

    def set_scalar(self, key, value):
        self._check(self._fn("set_scalar", C.c_int, [C.c_void_p, C.c_char_p, C.c_double])(self._live(), key.encode(), float(value)))

    def launch_count(self):
        return self._fn("launch_count", C.c_uint64, [C.c_void_p])(self._live())


class Handle(HandleBase):
    """A CMA-ES solver handle of libkcma.so (prefix 'kcma_') — or of the oracle (prefix 'okcma_') in tests."""
    CFG = KcmaCfg
    ARRAYS = ("lower_bound", "upper_bound", "initial_value", "initial_stddev", "min_stddev_update", "objective_coef", "granularity")
    ENUMS = {"mu_type": MU_TYPES, "objective": OBJECTIVES, "constraint_family": CONSTRAINTS}

    def _field(self, cfg, k, v, kw):
        if k != "constraint_shift":
            return False
        if v is not None:
            cfg.constraint_shift = self._array(v, int(kw.get("n_constraints", 0)))
        return True

    def take_warnings(self):
        return self._fn("take_warnings", C.c_char_p, [C.c_void_p])(self._live()).decode()

    def inject(self, kind, data):
        a = np.ascontiguousarray(data, dtype=np.float64).ravel()
        self._check(self._fn("inject", C.c_int, [C.c_void_p, C.c_int, _dp, C.c_size_t])(self._live(), kind, _as_dp(a), a.size))

    def get_index(self, key):
        f = self._fn("get_index_array", C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_uint64), C.c_size_t, C.POINTER(C.c_size_t)])
        cnt = C.c_size_t(0)
        self._check(f(self._live(), key.encode(), None, 0, C.byref(cnt)))
        out = np.empty(cnt.value, dtype=np.uint64)
        self._check(f(self._live(), key.encode(), out.ctypes.data_as(C.POINTER(C.c_uint64)), out.size, C.byref(cnt)))
        return out
