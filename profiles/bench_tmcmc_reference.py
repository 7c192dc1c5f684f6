"""Sampler/TMCMC on a Bayesian/Reference problem: the likelihood kernel alone and whole generations, on one GPU.

    python profiles/bench_tmcmc_reference.py [--reps 5] [--gens 10] [--warmup 2]

Workload: lambda = 65536, N = 3 (a, b, sigma), the linear model g_j = a + b t_j with a per-sample sigma, Normal likelihood,
M in {16, 1024, 8192} data points; Normal(1, 1), Normal(2, 1) and Uniform(0.5, 2) priors (Normal(1, 0.1) for sigma in the kernel
timing, so that every proposal is in the support and each evaluation has lambda rows).

Kernel: after ktmcmc_inject_reference (lambda x M predictions and standard deviations copied in before the timed window), CUDA
events around ktmcmc_eval, which then launches only tm_reference_loglik_kernel<Normal>. A ~1 ms device sleep is queued before the
first event so that the host's enqueue time is not counted. It must read lambda M 8 bytes per array (G and P) plus M 8 bytes of data;
that over the kernel time is its achieved bandwidth, quoted against the data-sheet 7.7 TB/s of HBM3e (the bound of a stream like this).
The 2 x 8 KiB of data at M = 16 is not a bandwidth measurement: a kernel of a few microseconds is bounded by its launch.

Whole generation: the same problem with the linear model as a korali.batched_device torch model (its second entry point, the one a
Bayesian/Reference experiment uses), timed with CUDA events as profiles/bench_tmcmc.py: "anneal" (steps 1-3), "resample" (step 4),
"mcmc" (propose / evaluate / accept), and inside "mcmc" the model callback (the torch model writing G and P). The card's name, power
limit and max SM clock are read with nvidia-smi --query-gpu in the same run. Writes nothing into the tree."""
import argparse
import ctypes as C
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

LAM = 65536
PEAK = 7.7e12
PRIORS = [("Normal", 1.0, 1.0), ("Normal", 2.0, 1.0), ("Uniform", 0.5, 2.0)]
KERNEL_PRIORS = [("Normal", 1.0, 1.0), ("Normal", 2.0, 1.0), ("Normal", 1.0, 0.1)]   # every proposal in the support: lambda rows
DEVICE_REFERENCE_CB = C.CFUNCTYPE(None, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64,
                                  C.c_uint64, C.c_void_p)


def card():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                       text=True).strip().splitlines()[0]
    except Exception as exc:   # pragma: no cover
        return "unknown (%s)" % exc


def data(m):
    t = np.linspace(0.0, 1.0, m)
    return t, 1.0 + 2.0 * t + 0.5 * np.random.default_rng(1).normal(size=m)


def kernel(m, reps):
    import torch
    from korali_b200 import _tmcmc
    t, d = data(m)
    s = _tmcmc.Solver(n=3, population_size=LAM, priors=KERNEL_PRIORS, reference=("Normal", d), seed=1)
    r = np.random.default_rng(2)
    G = d + 0.5 * r.normal(size=(LAM, m))
    P = np.full((LAM, m), 0.5)
    times = []
    s.propose()                                   # generation 1: lambda rows
    for rep in range(reps + 1):
        if rep:
            s.anneal(); s.resample(); s.propose()   # Max Chain Length 1: lambda chains, all in the support
        rows = s.get("Evaluation Rows").size // 3
        assert rows == LAM, rows
        s.inject_reference(G[:rows], P[:rows])
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda._sleep(2_000_000)
        e0.record(); s.eval(); e1.record()
        torch.cuda.synchronize()
        if rep:                                   # the first launch warms the module up
            times.append(e0.elapsed_time(e1) * 1e-3)
        s.accept()
    rows = LAM
    nbytes = 2 * rows * m * 8 + m * 8
    tk = float(np.median(times))
    line = ("kernel M=%5d: rows %d, reads %.4g GB, time %.4f ms (median of %d; min %.4f, max %.4f)"
            % (m, rows, nbytes / 1e9, tk * 1e3, len(times), min(times) * 1e3, max(times) * 1e3))
    if m >= 1024:
        line += ", %.3f TB/s = %.1f%% of 7.7 TB/s (bandwidth-bound)" % (nbytes / tk / 1e12, 100 * nbytes / tk / PEAK)
    else:
        line += ", launch-bound (%.3g MB read; no bandwidth quoted)" % (nbytes / 1e6)
    print(line, flush=True)
    s.close()


def generations(m, gens, warmup):
    import torch
    import korali_b200 as korali
    from korali_b200 import _tmcmc
    t, d = data(m)
    td = torch.tensor(t, dtype=torch.float64, device="cuda")
    wrapped = korali.batched_device(lambda X: {"Reference Evaluations": X[:, :1] + X[:, 1:2] * td, "Standard Deviation": X[:, 2:3]})
    cb_ms = [0.0]

    def call(_u, x, rows, n, ldx, g, p, mm, ldm, stream):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        wrapped._korali_reference(x, rows, n, ldx, g, p, mm, ldm, stream or 0, "Reference Evaluations", "Standard Deviation")
        b.record()
        b.synchronize()
        cb_ms[0] += a.elapsed_time(b)
    s = _tmcmc.Solver(n=3, population_size=LAM, priors=PRIORS, reference=("Normal", d), seed=1)
    cb = DEVICE_REFERENCE_CB(call)
    f = s._fn("set_device_reference_model", C.c_int, [C.c_void_p, DEVICE_REFERENCE_CB, C.c_void_p])
    s._check(f(s._live(), cb, None))
    s.run_generation()
    for _ in range(warmup):
        s.run_generation()
    ev = lambda: torch.cuda.Event(enable_timing=True)   # noqa: E731
    tot = {"anneal": 0.0, "resample": 0.0, "mcmc": 0.0}
    cb_ms[0] = 0.0
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(gens):
        e = [ev() for _ in range(4)]
        e[0].record(); s.anneal(); e[1].record(); s.resample(); e[2].record()
        for _t in range(int(s.scalar("Max Chain Steps"))):
            s.propose(); s.eval(); s.accept()
        e[3].record()
        torch.cuda.synchronize()
        tot["anneal"] += e[0].elapsed_time(e[1]); tot["resample"] += e[1].elapsed_time(e[2]); tot["mcmc"] += e[2].elapsed_time(e[3])
    wall = time.perf_counter() - t0
    ms = sum(tot.values()) / gens
    print("generations M=%5d: %.2f generations/s (%.3f ms per generation, host wall %.3f ms); anneal+cov+eigen %.3f ms, resample %.3f ms, "
          "mcmc %.3f ms of which model callback %.3f ms; rho %.4g, log Z %.4f, %d launches"
          % (m, 1e3 / ms, ms, 1e3 * wall / gens, tot["anneal"] / gens, tot["resample"] / gens, tot["mcmc"] / gens, cb_ms[0] / gens,
             s.scalar("Annealing Exponent"), s.scalar("LogEvidence"), s.launch_count()), flush=True)
    s.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--gens", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--m", type=int, nargs="*", default=[16, 1024, 8192])
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_tmcmc_reference.py needs a CUDA device (there is no CPU fallback)")
    print("card: %s (name, power limit, max SM clock)" % card(), flush=True)
    for m in a.m:
        kernel(m, a.reps)
    for m in a.m:
        generations(m, a.gens, a.warmup)


if __name__ == "__main__":
    main()
