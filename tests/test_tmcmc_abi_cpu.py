"""CPU-side checks of the ktmcmc ABI: the ctypes mirror of ktmcmc_cfg matches the C struct, libkcma.so exports every symbol
include/ktmcmc.h declares, the defaults are the documented ones, and creation fails loudly without a GPU."""
import ctypes as C
import os
import re
import subprocess
import tempfile
import pytest
import torch
from korali_b200 import _lib, _tmcmc
from korali_b200._abi import KcmaError

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ["n", "population_size", "max_chain_length", "default_burn_in", "burn_in_count", "per_generation_burn_in", "target_cov",
          "covariance_scaling", "min_annealing_update", "max_annealing_update", "seed", "loglik", "device", "prior_type", "prior_a",
          "prior_b", "loglik_coef"]


def test_cfg_struct_layout_matches_c():
    src = '#include <stdio.h>\n#include <stddef.h>\n#include "ktmcmc.h"\nint main(){ printf("%zu", sizeof(ktmcmc_cfg));'
    src += "".join(' printf(" %%zu", offsetof(ktmcmc_cfg, %s));' % f for f in FIELDS) + ' printf("\\n"); return 0; }'
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "t.c"), "w").write(src)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), os.path.join(d, "t.c"), "-o", os.path.join(d, "t")])
        out = [int(x) for x in subprocess.check_output([os.path.join(d, "t")]).decode().split()]
    assert out == [C.sizeof(_tmcmc.KtmcmcCfg)] + [getattr(_tmcmc.KtmcmcCfg, f).offset for f in FIELDS]


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "ktmcmc.h")).read()
    declared = set(re.findall(r"\b(ktmcmc_[a-z0-9_]+)\s*\(", hdr)) - {"ktmcmc_host_loglik_fn"}
    lib = _lib.lib()
    for name in sorted(declared):
        assert hasattr(lib, name), name
    assert set(_tmcmc.EXPORTS) == declared


def test_defaults():
    cfg = _tmcmc.KtmcmcCfg()
    f = _lib.lib().ktmcmc_cfg_defaults
    f.restype, f.argtypes = None, [C.POINTER(_tmcmc.KtmcmcCfg)]
    f(C.byref(cfg))
    assert cfg.abi_version == _tmcmc.KTMCMC_ABI_VERSION
    assert (cfg.max_chain_length, cfg.default_burn_in, cfg.target_cov, cfg.covariance_scaling) == (1, 0, 1.0, 0.04)
    assert (cfg.min_annealing_update, cfg.max_annealing_update, cfg.loglik) == (1e-5, 1.0, _tmcmc.KCMA_OBJ_EXTERNAL)


@pytest.mark.parametrize("kw,match", [
    (dict(population_size=1), "at least 2"),
    (dict(priors=[("Uniform", 1.0, -1.0)] * 2), "Minimum < Maximum"),
    (dict(priors=[("Normal", 0.0, 0.0)] * 2), "positive Standard Deviation"),
    (dict(covariance_scaling=0.0), "Covariance Scaling"),
])
def test_create_checks_the_configuration_first(kw, match):
    base = dict(n=2, population_size=64, priors=[("Uniform", -1.0, 1.0)] * 2, loglik="NegSphere")
    base.update(kw)
    with pytest.raises(KcmaError, match=match):
        _tmcmc.Solver(**base)


@pytest.mark.skipif(torch.cuda.is_available(), reason="CPU-only behaviour")
def test_create_fails_loudly_without_gpu():
    with pytest.raises(KcmaError, match="no CPU fallback"):
        _tmcmc.Solver(n=2, population_size=64, priors=[("Uniform", -1.0, 1.0)] * 2, loglik="NegSphere")
