"""ctypes loader of the TMCMC oracle (oracle/otmcmc.c). TEST INFRASTRUCTURE ONLY: imported by the TMCMC tests.

otmcmc.c reuses the Philox generator, the built-in objectives and the eigensolver of okcma.c, so its library is linked from both
sources. It is compiled on first use, next to the sources, or in a temporary directory when the tree cannot be written."""
import ctypes as C
import os
import subprocess
import tempfile

_HERE = os.path.dirname(os.path.abspath(__file__))
_SOURCES = ["otmcmc.c", "okcma.c"]
_DEPS = _SOURCES + ["okcma.h", os.path.join("..", "include", "kcma.h"), os.path.join("..", "include", "ktmcmc.h")]
# the flags of oracle/Makefile: no contraction into fused multiply-adds
CFLAGS = ["-O2", "-ffp-contract=off", "-fPIC", "-Wall", "-Wextra", "-Wno-unused-parameter", "-std=gnu11"]
_LIB = None


def _stale(path):
    return not os.path.exists(path) or os.path.getmtime(path) < max(os.path.getmtime(os.path.join(_HERE, f)) for f in _DEPS)


def build():
    """Compiles libotmcmc.so if it is missing or older than its sources; returns its path."""
    out = os.path.join(_HERE, "libotmcmc.so")
    if not os.access(_HERE, os.W_OK):
        out = os.path.join(tempfile.gettempdir(), "korali_b200_otmcmc_%d" % os.getuid(), "libotmcmc.so")
        os.makedirs(os.path.dirname(out), exist_ok=True)
    if _stale(out):
        tmp = out + ".%d.tmp" % os.getpid()
        subprocess.check_call([os.environ.get("CC", "gcc")] + CFLAGS + ["-shared", "-o", tmp] +
                              [os.path.join(_HERE, f) for f in _SOURCES] + ["-lm"])
        os.replace(tmp, out)
    return out


def lib():
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(build())
    return _LIB


def OracleTMCMC(**kw):
    """The TMCMC oracle behind the vocabulary of korali_b200._tmcmc.TmcmcHandle."""
    from korali_b200._tmcmc import TmcmcHandle
    kw.pop("device", None)
    return TmcmcHandle(lib(), "otmcmc_", **kw)
