"""Sampler/TMCMC throughput on one GPU: generations/s, samples/s and the phase split of a generation, for the built-in "Sphere"
log-likelihood (-x.x/2) with Uniform[-10, 10] priors.

    python profiles/bench_tmcmc.py [--gens 20] [--warmup 3]

Workloads: N = 100, lambda = 65536 (Max Chain Length 1, Burn In 0), and N = 1000, lambda = 65536 with Burn In 0 and 3 (one and
four MCMC steps per generation). Every phase is timed with CUDA events on the stream the library launches on (the legacy default
stream) after warm-up generations; phases: "anneal" = annealing + weights + weighted covariance + eigendecomposition (steps 1-3),
"resample" (step 4, ends with the one host read of the chain count), "mcmc" = every propose / evaluate / accept step. The card's
name and power limit are read with nvidia-smi --query-gpu and printed with the numbers. Writes nothing into the tree."""
import argparse
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                       text=True).strip().splitlines()[0]
    except Exception as exc:   # pragma: no cover
        return "unknown (%s)" % exc


def bench(n, lam, burn, gens, warmup):
    import torch
    from korali_b200 import _tmcmc
    s = _tmcmc.Solver(n=n, population_size=lam, default_burn_in=burn, priors=[("Uniform", -10.0, 10.0)] * n, loglik="NegSphere", seed=1)
    s.run_generation()                 # generation 1: prior draws + one evaluation of the population
    for _ in range(warmup):
        s.run_generation()
    ev = lambda: torch.cuda.Event(enable_timing=True)   # noqa: E731
    tot = {"anneal": 0.0, "resample": 0.0, "mcmc": 0.0}
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
    print("N=%4d lambda=%d burn-in %d: %.2f generations/s (%.3f ms per generation, host wall %.3f ms), %.3g samples/s; "
          "anneal+cov+eigen %.3f ms, resample %.3f ms, mcmc %.3f ms (%d steps); rho %.4g, log Z %.4f, %d launches"
          % (n, lam, burn, 1e3 / ms, ms, 1e3 * wall / gens, lam * 1e3 / ms, tot["anneal"] / gens, tot["resample"] / gens,
             tot["mcmc"] / gens, 1 + burn, s.scalar("Annealing Exponent"), s.scalar("LogEvidence"), s.launch_count()), flush=True)
    s.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gens", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_tmcmc.py needs a CUDA device (there is no CPU fallback)")
    print("card: %s (name, power limit, max SM clock)" % card(), flush=True)
    bench(100, 65536, 0, a.gens, a.warmup)
    bench(1000, 65536, 0, a.gens, a.warmup)
    bench(1000, 65536, 3, a.gens, a.warmup)


if __name__ == "__main__":
    main()
