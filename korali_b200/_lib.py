"""Loader of korali_b200/libkcma.so (CUDA kernels + C ABI, include/kcma.h).

There is no CPU fallback: if the shared library is missing this raises, and kcma_create itself fails
when no CUDA device is visible."""
import ctypes as C
import os
import numpy as np
from ._abi import Handle, KcmaError, OBJECTIVES, _as_dp, _dp

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libkcma.so")
_LIB = None

# every symbol include/kcma.h declares
EXPORTS = [
    "kcma_cfg_defaults", "kcma_create", "kcma_destroy", "kcma_last_error", "kcma_take_warnings",
    "kcma_comm_unique_id", "kcma_comm_init", "kcma_comm_init_all", "kcma_shard_range",
    "kcma_run_generation", "kcma_ask", "kcma_eval", "kcma_tell", "kcma_check_termination", "kcma_run",
    "kcma_set_host_objective", "kcma_set_host_objective_grad", "kcma_set_device_objective", "kcma_set_host_constraints", "kcma_set_priors", "kcma_set_reference",
    "kcma_set_host_reference_model", "kcma_set_device_reference_model", "kcma_inject", "kcma_get_array", "kcma_set_array", "kcma_get_index_array", "kcma_get_scalar", "kcma_set_scalar",
    "kcma_timing_enable", "kcma_timing_get", "kcma_timing_reset", "kcma_launch_count", "kcma_flush_l2",
    "kcma_k_sort_index", "kcma_k_eigen", "kcma_k_tridiag_stage", "kcma_k_sample", "kcma_k_rank_mu", "kcma_k_philox_normal",
    "kcma_k_philox_raw", "kcma_k_objective",
    # include/kdea.h
    "kdea_cfg_defaults", "kdea_create", "kdea_destroy", "kdea_last_error", "kdea_run_generation", "kdea_ask", "kdea_eval", "kdea_tell",
    "kdea_set_host_objective", "kdea_inject_f", "kdea_check_termination", "kdea_run", "kdea_get_array", "kdea_set_array",
    "kdea_get_scalar", "kdea_set_scalar", "kdea_launch_count",
    # include/kmocma.h
    "kmocma_cfg_defaults", "kmocma_create", "kmocma_destroy", "kmocma_last_error", "kmocma_run_generation", "kmocma_ask", "kmocma_eval",
    "kmocma_tell", "kmocma_set_host_objective", "kmocma_inject_f", "kmocma_check_termination", "kmocma_run", "kmocma_get_array",
    "kmocma_get_scalar", "kmocma_set_scalar", "kmocma_launch_count",
]


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "korali_b200/libkcma.so is missing: build it with `python -m korali_b200.build` "
                "(nvcc, sm_100a). korali_b200 has no CPU fallback.")
        _LIB = C.CDLL(LIB_PATH)
    return _LIB


def _kerr():
    f = lib().kcma_last_error
    f.restype, f.argtypes = C.c_char_p, [C.c_void_p]
    return KcmaError(f(None).decode())


class Solver(Handle):
    """One CMA-ES solver state resident on one B200 (a handle of libkcma.so)."""

    def __init__(self, **kw):
        super().__init__(lib(), "kcma_", **kw)

    def comm_init(self, unique_id):
        buf = (C.c_uint8 * 128).from_buffer_copy(bytes(unique_id))
        self._check(self._fn("comm_init", C.c_int, [C.c_void_p, C.POINTER(C.c_uint8)])(self._live(), buf))

    def timing_enable(self, on=True):
        self._fn("timing_enable", C.c_int, [C.c_void_p, C.c_int])(self._live(), int(on))

    def timing_reset(self):
        self._fn("timing_reset", C.c_int, [C.c_void_p])(self._live())

    def timing(self, phase):
        ms, calls = C.c_double(0), C.c_uint64(0)
        self._fn("timing_get", C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_double), C.POINTER(C.c_uint64)])(
            self._h, phase.encode(), C.byref(ms), C.byref(calls))
        return ms.value, calls.value

    def set_host_objective(self, fn):
        """fn(X: ndarray[rows, n]) -> ndarray[rows]; the batched host conduit (needs keep_population=1)."""
        self._set_callback("set_host_objective", C.CFUNCTYPE(None, C.c_void_p, _dp, C.c_uint64, C.c_uint64, _dp), fn,
                           lambda rows, n: (rows,))

    def set_host_objective_grad(self, fn):
        """fn(X: ndarray[rows, n]) -> (F: ndarray[rows], dF/dX: ndarray[rows, n]); needs use_gradient_information=1."""
        cb_t = C.CFUNCTYPE(None, C.c_void_p, _dp, C.c_uint64, C.c_uint64, _dp, _dp)

        def tramp(_u, x, rows, n, out, gout):
            xs = np.ctypeslib.as_array(x, shape=(rows, n))
            f, g = fn(xs)
            np.ctypeslib.as_array(out, shape=(rows,))[:] = np.asarray(f, dtype=np.float64)
            np.ctypeslib.as_array(gout, shape=(rows, n))[:] = np.asarray(g, dtype=np.float64).reshape(rows, n)
        self._host_obj_grad = cb_t(tramp)
        self._check(self._fn("set_host_objective_grad", C.c_int, [C.c_void_p, cb_t, C.c_void_p])(self._live(), self._host_obj_grad, None))

    def set_host_constraints(self, fn):
        """fn(X: ndarray[rows, n]) -> ndarray[n_constraints, rows]."""
        self._set_callback("set_host_constraints", C.CFUNCTYPE(None, C.c_void_p, _dp, C.c_uint64, C.c_uint64, _dp, C.c_uint64), fn,
                           lambda rows, n, nc: (nc, rows))

    def flush_l2(self):
        self._check(self._fn("flush_l2", C.c_int, [C.c_void_p])(self._live()))


def comm_unique_id():
    out = (C.c_uint8 * 128)()
    f = lib().kcma_comm_unique_id
    f.restype, f.argtypes = C.c_int, [C.POINTER(C.c_uint8)]
    if f(out) != 0:
        raise _kerr()
    return bytes(out)


def shard_range(population, mirrored, rank, nranks):
    b, e = C.c_uint64(0), C.c_uint64(0)
    f = lib().kcma_shard_range
    f.restype, f.argtypes = None, [C.c_uint64, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    f(population, int(mirrored), rank, nranks, C.byref(b), C.byref(e))
    return b.value, e.value


# ---- single kernels on host buffers --------------------------------------------------------------------
def k_sort_index(f, device=0):
    f = np.ascontiguousarray(f, dtype=np.float64)
    out = np.empty(f.size, dtype=np.uint64)
    fn = lib().kcma_k_sort_index
    fn.restype, fn.argtypes = C.c_int, [C.c_int, _dp, C.c_uint64, C.POINTER(C.c_uint64)]
    if fn(device, _as_dp(f), f.size, out.ctypes.data_as(C.POINTER(C.c_uint64))) != 0:
        raise _kerr()
    return out


def k_eigen(c, device=0):
    c = np.ascontiguousarray(c, dtype=np.float64)
    n = c.shape[0]
    w, q = np.empty(n), np.empty((n, n))
    fn = lib().kcma_k_eigen
    fn.restype, fn.argtypes = C.c_int, [C.c_int, C.c_uint64, _dp, _dp, _dp]
    if fn(device, n, _as_dp(c), _as_dp(w), _as_dp(q)) != 0:
        raise _kerr()
    return w, q


def k_sytrd(c, device=0):
    """Householder tridiagonalisation on the device: returns (d, e, tau, vr) with vr[i] = reflector i."""
    c = np.ascontiguousarray(c, dtype=np.float64)
    n = c.shape[0]
    d, e, tau, vr = np.zeros(n), np.zeros(n), np.zeros(n), np.zeros((n, n))
    fn = lib().kcma_k_tridiag_stage
    fn.restype, fn.argtypes = C.c_int, [C.c_int, C.c_int, C.c_uint64] + [_dp] * 7
    if fn(device, 0, n, _as_dp(c), _as_dp(d), _as_dp(e), _as_dp(tau), _as_dp(vr), None, None) != 0:
        raise _kerr()
    return d, e[:n - 1], tau, vr


def k_stedc(d, e, device=0):
    """Divide & conquer on the tridiagonal (d, e): returns (lam ascending, zt with eigenvectors as rows)."""
    d = np.ascontiguousarray(d, dtype=np.float64)
    n = d.size
    ee = np.zeros(n); ee[:n - 1] = e
    lam, zt = np.zeros(n), np.zeros((n, n))
    fn = lib().kcma_k_tridiag_stage
    fn.restype, fn.argtypes = C.c_int, [C.c_int, C.c_int, C.c_uint64] + [_dp] * 7
    if fn(device, 1, n, None, _as_dp(d), _as_dp(ee), None, None, _as_dp(lam), _as_dp(zt)) != 0:
        raise _kerr()
    return lam, zt


def k_sample(z, b, d, mean, sigma, device=0):
    z = np.ascontiguousarray(z, dtype=np.float64); b = np.ascontiguousarray(b, dtype=np.float64)
    d = np.ascontiguousarray(d, dtype=np.float64); mean = np.ascontiguousarray(mean, dtype=np.float64)
    rows, n = z.shape
    y, x = np.empty((rows, n)), np.empty((rows, n))
    fn = lib().kcma_k_sample
    fn.restype, fn.argtypes = C.c_int, [C.c_int, C.c_uint64, C.c_uint64, _dp, _dp, _dp, _dp, C.c_double, _dp, _dp]
    if fn(device, n, rows, _as_dp(z), _as_dp(b), _as_dp(d), _as_dp(mean), float(sigma), _as_dp(y), _as_dp(x)) != 0:
        raise _kerr()
    return y, x


def k_rank_mu(t, w, device=0):
    t = np.ascontiguousarray(t, dtype=np.float64); w = np.ascontiguousarray(w, dtype=np.float64)
    rows, n = t.shape
    p = np.empty((n, n))
    fn = lib().kcma_k_rank_mu
    fn.restype, fn.argtypes = C.c_int, [C.c_int, C.c_uint64, C.c_uint64, _dp, _dp, _dp]
    if fn(device, n, rows, _as_dp(t), _as_dp(w), _as_dp(p)) != 0:
        raise _kerr()
    return p


def k_philox_normal(seed, generation, row_begin, rows, n, device=0):
    out = np.empty((rows, n))
    fn = lib().kcma_k_philox_normal
    fn.restype, fn.argtypes = C.c_int, [C.c_int] + [C.c_uint64] * 5 + [_dp]
    if fn(device, seed, generation, row_begin, rows, n, _as_dp(out)) != 0:
        raise _kerr()
    return out


def k_philox_raw(ctr, key, device=0):
    c = (C.c_uint32 * 4)(*ctr); k = (C.c_uint32 * 2)(*key); o = (C.c_uint32 * 4)()
    fn = lib().kcma_k_philox_raw
    fn.restype, fn.argtypes = C.c_int, [C.c_int, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
    if fn(device, c, k, o) != 0:
        raise _kerr()
    return list(o)


def k_objective(obj, x, coef=None, device=0):
    x = np.ascontiguousarray(x, dtype=np.float64)
    rows, n = x.shape
    f = np.empty(rows)
    cp = None
    if coef is not None:
        coef = np.ascontiguousarray(coef, dtype=np.float64); cp = _as_dp(coef)
    fn = lib().kcma_k_objective
    fn.restype, fn.argtypes = C.c_int, [C.c_int, C.c_int, C.c_uint64, C.c_uint64, _dp, _dp, _dp]
    if fn(device, OBJECTIVES[obj] if isinstance(obj, str) else obj, n, rows, _as_dp(x), cp, _as_dp(f)) != 0:
        raise _kerr()
    return f
