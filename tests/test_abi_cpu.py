"""CPU-side checks of the drop-in boundary: libkcma.so loads and exports every symbol include/kcma.h declares,
the ctypes struct mirrors the C struct, host-only entry points behave, and compute entry points fail loudly
without a GPU (no CPU fallback)."""
import ctypes as C
import os
import re
import subprocess
import sys
import tempfile
import numpy as np
import pytest
import torch
from korali_b200 import _lib
from korali_b200._abi import KcmaCfg, KcmaError

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "kcma.h")).read()
    declared = set(re.findall(r"\b(kcma_[a-z0-9_]+)\s*\(", hdr))
    declared |= set(re.findall(r"\b(kdea_[a-z0-9_]+)\s*\(", open(os.path.join(ROOT, "include", "kdea.h")).read()))
    declared |= set(re.findall(r"\b(kmocma_[a-z0-9_]+)\s*\(", open(os.path.join(ROOT, "include", "kmocma.h")).read())) - {"kmocma_host_objective_fn"}
    lib = _lib.lib()
    for name in sorted(declared):
        assert hasattr(lib, name), name
    assert set(_lib.EXPORTS) == declared


def test_cfg_struct_layout_matches_c():
    src = r'''
    #include <stdio.h>
    #include <stddef.h>
    #include "kcma.h"
    int main(){ printf("%zu %zu %zu %zu %zu %zu\n", sizeof(kcma_cfg), offsetof(kcma_cfg, mu_type), offsetof(kcma_cfg, seed),
      offsetof(kcma_cfg, objective_coef), offsetof(kcma_cfg, lower_bound), offsetof(kcma_cfg, device)); return 0; }'''
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "t.c"), "w").write(src)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), os.path.join(d, "t.c"), "-o", os.path.join(d, "t")])
        out = subprocess.check_output([os.path.join(d, "t")]).decode().split()
    got = [C.sizeof(KcmaCfg), KcmaCfg.mu_type.offset, KcmaCfg.seed.offset, KcmaCfg.objective_coef.offset,
           KcmaCfg.lower_bound.offset, KcmaCfg.device.offset]
    assert [int(x) for x in out] == got


def test_defaults_match_reference_config():
    """kcma_cfg_defaults == "Module Defaults" of CMAES.config:485-538."""
    cfg = KcmaCfg()
    f = _lib.lib().kcma_cfg_defaults
    f.restype, f.argtypes = None, [C.POINTER(KcmaCfg)]
    f(C.byref(cfg))
    assert cfg.mu_type == 2 and cfg.viability_population_size == 2 and cfg.max_covariance_matrix_corrections == 1000000
    assert cfg.target_success_rate == 0.1818 and cfg.covariance_matrix_adaption_strength == 0.1
    assert cfg.global_success_learning_rate == 0.2 and cfg.initial_damp_factor == -1.0
    assert cfg.max_infeasible_resamplings == 0 and cfg.nranks == 1


def test_shard_ranges_partition_population():
    for lam, mirrored, g in [(65536, 0, 8), (1 << 20, 1, 8), (32, 0, 1), (4096, 0, 2), (10, 0, 4), (12, 1, 4)]:
        spans = [_lib.shard_range(lam, mirrored, r, g) for r in range(g)]
        assert spans[0][0] == 0 and spans[-1][1] == lam
        for a, b in zip(spans, spans[1:]):
            assert a[1] == b[0]
        if mirrored:
            assert all(s[0] % 2 == 0 and s[1] % 2 == 0 for s in spans)
        sizes = [s[1] - s[0] for s in spans]
        assert max(sizes) - min(sizes) <= (2 if mirrored else 1)


@pytest.mark.skipif(torch.cuda.is_available(), reason="CPU-only behaviour")
def test_no_cpu_fallback():
    with pytest.raises(KcmaError, match="CUDA device"):
        _lib.Solver(n=4, population_size=8, initial_value=np.zeros(4), initial_stddev=np.ones(4))
    with pytest.raises(KcmaError):
        _lib.k_sort_index(np.arange(4.0))


ABIS = [("kcma_", "kcma.h"), ("kdea_", "kdea.h"), ("kmocma_", "kmocma.h"), ("ktmcmc_", "ktmcmc.h")]


def _handle_entry_points(prefix, header):
    """(name, ctypes argument types) of every int-returning entry point of include/<header> whose first argument is the handle."""
    src = open(os.path.join(ROOT, "include", header)).read()
    found = []
    for name, args in re.findall(r"\bint (%s[a-z0-9_]+)\(%st\* h,?([^)]*)\);" % (prefix, prefix), src):
        types = [C.c_void_p]
        for a in filter(None, (x.strip() for x in args.split(","))):
            types.append(C.c_double if a.startswith("double ") else C.c_void_p if ("*" in a or "[" in a or "_fn " in a) else C.c_uint64)
        found.append((name, types))
    return found


def test_null_handle_is_an_error_not_a_crash():
    """In each of the four ABIs, every entry point that takes a handle returns non-zero for NULL and <prefix>last_error(NULL)
    explains; <prefix>launch_count(NULL) is 0 (run in a subprocess: it used to dereference NULL in kcma_)."""
    lib = _lib.lib()
    for prefix, header in ABIS:
        last_error = getattr(lib, prefix + "last_error")
        last_error.restype, last_error.argtypes = C.c_char_p, [C.c_void_p]
        create = getattr(lib, prefix + "create")
        create.restype, create.argtypes = C.c_int, [C.c_void_p, C.c_void_p]
        entry_points = _handle_entry_points(prefix, header)
        assert len(entry_points) >= 10, prefix
        for name, types in entry_points:
            assert create(None, C.byref(C.c_void_p())) != 0                      # leaves a different message behind
            assert b"null solver handle" not in last_error(None)
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = C.c_int, types
            assert fn(*[t(0) if t in (C.c_double, C.c_uint64) else None for t in types]) != 0, name
            assert b"null solver handle" in last_error(None), name
    code = ("import ctypes, sys; sys.path.insert(0, %r); from korali_b200 import _lib\n"
            "for p in %r:\n"
            "    f = getattr(_lib.lib(), p + 'launch_count'); f.restype, f.argtypes = ctypes.c_uint64, [ctypes.c_void_p]; print(p, f(None))"
            % (ROOT, [p for p, _ in ABIS]))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.split() == [w for p, _ in ABIS for w in (p, "0")], (r.returncode, r.stdout, r.stderr)
