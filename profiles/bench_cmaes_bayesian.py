"""Optimizer/CMAES on Bayesian problems (F = the log-posterior, include/kcma.h), on one GPU.

    python profiles/bench_cmaes_bayesian.py [--reps 3] [--gens 20] [--warmup 5]

1. bench.py's workload (N = 1000, lambda = 65536, Ellipsoid, initial value 3, standard deviation 1) as an Optimization and as a
   Bayesian/Custom problem whose log-likelihood is the same Ellipsoid with Normal(0, 10) priors on every variable, alternating the two
   handles rep by rep in one process. Generations/s from a host clock around `gens` graph-replayed generations that end in a device
   synchronise; then the "objective" phase (kcma_timing_get: CUDA events around the one objective kernel, eager generations). The fused
   kernel adds the log-prior of the same reconstructed x to a kernel that streams lambda N 8 bytes of Y.
2. Bayesian/Reference, Normal likelihood, the linear model g_j = a + b t_j as a korali.batched_device torch model writing the
   predictions and a standard deviation of 0.5, M in {16, 1024}, lambda = 65536, N = 2: generations/s (host clock, eager: a Python
   model is never graph-replayed) and the "posterior" phase (the log-posterior kernel: log-prior + M terms per row) and the
   "reference_model" phase (the torch model).
The card's name, power limit and max SM clock are read with nvidia-smi --query-gpu in the same run. Writes nothing into the tree."""
import argparse
import ctypes as C
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOAD = dict(n=1000, population_size=65536, objective="NegEllipsoid", initial_value=3.0, initial_stddev=1.0, seed=1337)
DEVICE_REFERENCE_CB = C.CFUNCTYPE(None, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64,
                                  C.c_uint64, C.c_void_p)


def card():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                       text=True).strip().splitlines()[0]
    except Exception as exc:   # pragma: no cover
        return "unknown (%s)" % exc


def rate(s, gens):
    s.scalar("Sigma")                       # synchronises
    t0 = time.perf_counter()
    for _ in range(gens):
        s.run_generation()
    s.scalar("Sigma")
    return gens / (time.perf_counter() - t0)


def phase(s, name, gens):
    s.timing_enable(True); s.timing_reset()
    for _ in range(gens):
        s.run_generation()
    ms, calls = s.timing(name)
    s.timing_enable(False)
    return ms / max(calls, 1)


def builtin(reps, gens, warmup):
    from korali_b200 import _lib
    n = WORKLOAD["n"]
    hs = {"Optimization": _lib.Solver(**WORKLOAD),
          "Bayesian/Custom": _lib.Solver(priors=[("Normal", 0.0, 10.0)] * n, **WORKLOAD)}
    for s in hs.values():
        for _ in range(warmup):
            s.run_generation()
    res = {k: [] for k in hs}
    obj = {k: [] for k in hs}
    for r in range(reps):
        for k, s in hs.items():
            res[k].append(rate(s, gens))
            obj[k].append(phase(s, "objective", 5))
            print("rep %d %-16s %.2f generations/s, objective kernel %.4f ms" % (r, k, res[k][-1], obj[k][-1]), flush=True)
    for k in hs:
        print("%-16s median %.2f generations/s (%s), objective %.4f ms (median)"
              % (k, np.median(res[k]), " ".join("%.2f" % v for v in res[k]), np.median(obj[k])), flush=True)
    a, b = np.median(res["Optimization"]), np.median(res["Bayesian/Custom"])
    print("Bayesian/Custom vs Optimization: %+.2f%% generations/s, objective %+.4f ms"
          % (100 * (b / a - 1), np.median(obj["Bayesian/Custom"]) - np.median(obj["Optimization"])), flush=True)


def reference(m, gens, warmup):
    import torch
    import korali_b200 as korali
    from korali_b200 import _lib
    t = np.linspace(0.0, 1.0, m)
    d = 1.0 + 2.0 * t + 0.5 * np.random.default_rng(1).normal(size=m)
    td = torch.tensor(t, dtype=torch.float64, device="cuda")
    wrapped = korali.batched_device(lambda X: {"Reference Evaluations": X[:, :1] + X[:, 1:2] * td, "Standard Deviation": 0.5})

    def call(_u, x, rows, n, ldx, g, p, mm, ldm, stream):
        wrapped._korali_reference(x, rows, n, ldx, g, p, mm, ldm, stream or 0, "Reference Evaluations", "Standard Deviation")
    s = _lib.Solver(n=2, population_size=65536, objective="External", keep_population=1, priors=[("Normal", 0.0, 5.0)] * 2,
                    reference=("Normal", d), initial_value=0.0, initial_stddev=1.0, seed=1)
    cb = DEVICE_REFERENCE_CB(call)
    s._check(s._fn("set_device_reference_model", C.c_int, [C.c_void_p, DEVICE_REFERENCE_CB, C.c_void_p])(s._live(), cb, None))
    for _ in range(warmup):
        s.run_generation()
    g = rate(s, gens)
    post, model = 0.0, 0.0
    s.timing_enable(True); s.timing_reset()
    for _ in range(5):
        s.run_generation()
    post = s.timing("posterior")[0] / 5
    model = s.timing("reference_model")[0] / 5
    print("Bayesian/Reference M=%5d: %.2f generations/s, posterior kernel %.4f ms (reads 65536 x %d x 2 x 8 bytes of G and P), "
          "torch model %.4f ms, best log-posterior %.6f" % (m, g, post, m, model, s.scalar("Best Ever Value")), flush=True)
    s.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--gens", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_cmaes_bayesian.py needs a CUDA device (there is no CPU fallback)")
    print("card: %s (name, power limit, max SM clock)" % card(), flush=True)
    builtin(a.reps, a.gens, a.warmup)
    for m in (16, 1024):
        reference(m, a.gens, a.warmup)


if __name__ == "__main__":
    main()
