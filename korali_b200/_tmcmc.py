"""ctypes mirror of include/ktmcmc.h (transitional MCMC on libkcma.so). Generic over the symbol prefix so that the CPU oracle
(oracle/libokcma.so, prefix ``otmcmc_``; test infrastructure only) can be driven with the same vocabulary. Nothing here loads the oracle."""
import ctypes as C
import numpy as np
from ._abi import KcmaError, OBJECTIVES, _as_dp, _dp

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


class TmcmcHandle:
    """kw: n, population_size, priors = [(type, a, b)] * n (type "Uniform" | "Normal"), loglik (a KCMA_OBJ name such as "NegSphere",
    or "External"), per_generation_burn_in (list), loglik_coef, and the scalar fields of ktmcmc_cfg."""

    def __init__(self, lib, prefix, **kw):
        self._lib, self._p, self._keep = lib, prefix, []
        cfg = KtmcmcCfg()
        self._fn("cfg_defaults", None, [C.POINTER(KtmcmcCfg)])(C.byref(cfg))
        n = int(kw["n"])
        for k, v in kw.items():
            if k == "priors":
                t = np.ascontiguousarray([PRIORS[p[0]] for p in v], dtype=np.int32)
                a = np.ascontiguousarray([p[1] for p in v], dtype=np.float64)
                b = np.ascontiguousarray([p[2] for p in v], dtype=np.float64)
                self._keep += [t, a, b]
                cfg.prior_type = t.ctypes.data_as(C.POINTER(C.c_int32))
                cfg.prior_a, cfg.prior_b = _as_dp(a), _as_dp(b)
            elif k == "per_generation_burn_in":
                arr = np.ascontiguousarray(v, dtype=np.uint64)
                self._keep.append(arr)
                cfg.per_generation_burn_in = arr.ctypes.data_as(C.POINTER(C.c_uint64))
                cfg.burn_in_count = arr.size
            elif k == "loglik_coef":
                arr = np.ascontiguousarray(np.broadcast_to(np.asarray(v, dtype=np.float64), (n,)))
                self._keep.append(arr)
                cfg.loglik_coef = _as_dp(arr)
            elif k == "loglik":
                cfg.loglik = KCMA_OBJ_EXTERNAL if v == "External" else (OBJECTIVES[v] if isinstance(v, str) else int(v))
            else:
                setattr(cfg, k, v)
        self._h = C.c_void_p()
        if self._fn("create", C.c_int, [C.POINTER(KtmcmcCfg), C.POINTER(C.c_void_p)])(C.byref(cfg), C.byref(self._h)) != 0:
            raise KcmaError(self._fn("last_error", C.c_char_p, [C.c_void_p])(None).decode())
        self.n, self.population_size = n, int(cfg.population_size)

    def _fn(self, name, restype, argtypes):
        f = getattr(self._lib, self._p + name)
        f.restype, f.argtypes = restype, argtypes
        return f

    def _live(self):
        if not getattr(self, "_h", None):
            raise KcmaError("the solver handle was closed")
        return self._h

    def _check(self, rc):
        if rc != 0:
            raise KcmaError(self._fn("last_error", C.c_char_p, [C.c_void_p])(self._h).decode())

    def close(self):
        if getattr(self, "_h", None):
            self._fn("destroy", None, [C.c_void_p])(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _call(self, name):
        self._check(self._fn(name, C.c_int, [C.c_void_p])(self._live()))

    def run_generation(self): self._call("run_generation")
    def anneal(self): self._call("anneal")
    def resample(self): self._call("resample")
    def propose(self): self._call("propose")
    def eval(self): self._call("eval")
    def accept(self): self._call("accept")

    def run(self, max_generations):
        done = C.c_uint64(0)
        self._check(self._fn("run", C.c_int, [C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)])(self._live(), int(max_generations), C.byref(done)))
        return done.value

    def check_termination(self):
        fin, why = C.c_int(0), C.c_char_p()
        self._check(self._fn("check_termination", C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_char_p)])(self._live(), C.byref(fin), C.byref(why)))
        return bool(fin.value), (why.value or b"").decode()

    def _inject(self, what, v):
        v = np.ascontiguousarray(v, dtype=np.float64).reshape(-1)
        self._check(self._fn(what, C.c_int, [C.c_void_p, _dp, C.c_size_t])(self._live(), _as_dp(v), v.size))

    def inject_loglik(self, l): self._inject("inject_loglik", l)
    def inject_factor(self, a): self._inject("inject_factor", a)

    def set_host_loglik(self, fn):
        """fn(X: ndarray[rows, n]) -> ndarray[rows] of log-likelihoods."""
        def tramp(_u, x, rows, n, out):
            xs = np.ctypeslib.as_array(x, shape=(rows, n))
            np.ctypeslib.as_array(out, shape=(rows,))[:] = np.asarray(fn(xs), dtype=np.float64).reshape(rows)
        self._cb = HOST_CB(tramp)
        self._check(self._fn("set_host_loglik", C.c_int, [C.c_void_p, HOST_CB, C.c_void_p])(self._live(), self._cb, None))

    def get(self, key):
        cnt = C.c_size_t(0)
        f = self._fn("get_array", C.c_int, [C.c_void_p, C.c_char_p, _dp, C.c_size_t, C.POINTER(C.c_size_t)])
        self._check(f(self._live(), key.encode(), None, 0, C.byref(cnt)))
        out = np.empty(cnt.value, dtype=np.float64)
        if cnt.value:
            self._check(f(self._h, key.encode(), _as_dp(out), out.size, C.byref(cnt)))
        return out

    def scalar(self, key):
        v = C.c_double(0)
        self._check(self._fn("get_scalar", C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_double)])(self._live(), key.encode(), C.byref(v)))
        return v.value

    def set_scalar(self, key, value):
        self._check(self._fn("set_scalar", C.c_int, [C.c_void_p, C.c_char_p, C.c_double])(self._live(), key.encode(), float(value)))

    def launch_count(self):
        return self._fn("launch_count", C.c_uint64, [C.c_void_p])(self._live())


def Solver(**kw):
    """One TMCMC state resident on one B200 (a handle of libkcma.so)."""
    from . import _lib
    return TmcmcHandle(_lib.lib(), "ktmcmc_", **kw)
