"""ctypes loader of the Bayesian/Reference TMCMC oracle (tests/helpers/otmcmc_reference.c, which includes oracle/otmcmc.c unchanged).
TEST INFRASTRUCTURE ONLY. Linked with oracle/okcma.c (Philox, built-in objectives, eigensolver) into its own library on first use, in
a temporary directory (the tree may be read-only), under the flags of oracle/otmcmc.py; driven through korali_b200._tmcmc.TmcmcHandle
with the prefix "otmcmc_"."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

from oracle import otmcmc

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
_SOURCES = [os.path.join(_HERE, "helpers", "otmcmc_reference.c"), os.path.join(_ROOT, "oracle", "okcma.c")]
_DEPS = _SOURCES + [os.path.join(_ROOT, "oracle", f) for f in ("otmcmc.c", "okcma.h")] + \
    [os.path.join(_ROOT, "include", f) for f in ("kcma.h", "ktmcmc.h")]
_LIB = None


def build():
    """Compiles the library once per content of its sources; returns its path."""
    digest = hashlib.sha256(b"".join(open(f, "rb").read() for f in _DEPS) + " ".join(otmcmc.CFLAGS).encode()).hexdigest()[:16]
    out = os.path.join(tempfile.gettempdir(), "korali_b200_otmcmc_reference_%d" % os.getuid(), digest, "libotmcmc_reference.so")
    if not os.path.exists(out):
        os.makedirs(os.path.dirname(out), exist_ok=True)
        tmp = out + ".%d.tmp" % os.getpid()
        subprocess.check_call([os.environ.get("CC", "gcc")] + otmcmc.CFLAGS + ["-shared", "-o", tmp] + _SOURCES + ["-lm"])
        os.replace(tmp, out)
    return out


def lib():
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(build())
    return _LIB


def OracleTMCMC(**kw):
    """The TMCMC oracle with Bayesian/Reference, behind the vocabulary of korali_b200._tmcmc.TmcmcHandle."""
    from korali_b200._tmcmc import TmcmcHandle
    kw.pop("device", None)
    return TmcmcHandle(lib(), "otmcmc_", **kw)
