#!/usr/bin/env python
"""bench.py — CMA-ES generations/s (and samples/s) on the configuration BASELINE.json quotes its metric on:
N = 1000, lambda = 65536, mu = lambda/2, ill-conditioned ellipsoid (SURVEY.md 8d "config 3"), population sharded
over --gpus N B200s of one box (strong scaling: the population is fixed, each rank owns lambda/N samples).

A "step" is one full generation of the hot path: eigendecomposition, Philox sampling, sampling GEMM, batched
objective, ranking, mean/path updates, rank-mu covariance update (+ all-gather(F) and all-reduce(C partial) for N > 1).
Legs (DESIGN.md section 8): `value` = the shipped path (CUDA-graph replay on one GPU), the same generations again with eager launches
and phase timers (roofline, phases), `e2e` through korali_b200.Engine().run(e) (k["Conduit"]["Devices"] = N), `parity_vs_n1` for N > 1,
`cpu_baseline` on a bounded sample; `--impl reference` times REAL full-size generations of the reference algorithm on the host.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
Under torchrun (N > 1) every rank runs this file; rank 0 prints ONE JSON line.
--dump-outputs DIR writes the solver state after the last timed generation as DIR/<name>.npy (float64), so that two builds can be
compared output for output on the same seeded workload.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = dict(n=1000, population_size=65536, objective="NegEllipsoid", initial_value=3.0, initial_stddev=1.0, seed=1337)
WORKLOAD_NAME = "config3: CMA-ES 1000-D ill-conditioned ellipsoid, lambda=65536, mu=32768 (Logarithmic weights), seed 1337"
METRIC, UNIT = "cmaes_generations_per_sec_N1000_lambda65536", "generations/s"


def flops_per_generation(n, lam, mu):
    """Algorithmic flops (BASELINE.md section 3): sampling 2 N^2 lambda, rank-mu N (N+1) mu."""
    return 2.0 * n * n * lam, float(n) * (n + 1) * mu


def load_peaks():
    out = {}
    for name in ("MEASURED_PEAKS.json", "MEASURED_FP64.json"):
        p = os.path.join(ROOT, name)
        if os.path.exists(p):
            out.update(json.load(open(p)))
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.proc, self.path = device, None, "/tmp/kcma_clocks_%d.csv" % os.getpid()

    def start(self):
        try:
            self.fh = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=self.fh, stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate(); self.proc.wait(); self.fh.close()
        sm, mx, reasons = [], [], set()
        for line in open(self.path):
            p = [x.strip() for x in line.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1])); mx.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


DUMP_ARRAYS = ["Covariance Matrix", "Covariance Eigenvector Matrix", "Axis Lengths", "Current Mean", "Evolution Path",
               "Conjugate Evolution Path", "Best Ever Variables", "Value Vector"]
DUMP_SCALARS = ["Sigma", "Best Ever Value", "Current Best Value", "Conjugate Evolution Path L2 Norm", "Current Generation"]
DUMP_SAMPLE_ROWS = 2048        # the 65536 x 1000 population is 524 MB: a fixed, seeded sample of its rows is written instead


def dump_outputs(s, out_dir):
    """What a caller of the generation loop reads back after the last timed generation, as out_dir/<name>.npy (float64, about 34 MB
    at config 3). The population ('BDZ Matrix', this rank's rows) is sampled at DUMP_SAMPLE_ROWS rows drawn with a fixed seed;
    the drawn row numbers are written beside it."""
    os.makedirs(out_dir, exist_ok=True)

    def save(key, a):
        np.save(os.path.join(out_dir, key.lower().replace(" ", "_") + ".npy"), np.asarray(a, dtype=np.float64))
    for k in DUMP_ARRAYS:
        a = s.get(k)
        save(k, a.reshape(s.n, s.n) if k.endswith("Matrix") else a)
    save("Sorting Index", s.get_index("Sorting Index"))
    for k in DUMP_SCALARS:
        save(k, [s.scalar(k)])
    y = s.get("BDZ Matrix").reshape(-1, s.n)
    rows = np.sort(np.random.default_rng(0).choice(y.shape[0], min(DUMP_SAMPLE_ROWS, y.shape[0]), replace=False))
    save("BDZ Matrix Sample", y[rows])
    save("BDZ Matrix Sample Rows", rows)


# ---------------------------------------------------------------------------------------------------------
def cpu_bounded_sample(steps, warmup, sample_lambda=1024):
    """cpu_baseline leg of the default run (about 10-20 s of host work): the C restatement in oracle/ (the reference itself needs
    GSL/Eigen/meson and cannot be built here — DESIGN.md), one thread (CMAES.cpp.base has no OpenMP and its conduits only
    parallelise the user model, SURVEY F2), on a BOUNDED SAMPLE of the population: sample_lambda of the 65536 samples with all
    N = 1000 dimensions per step, plus ONE full 1000 x 1000 eigendecomposition; extrapolated linearly in lambda. The extrapolation
    FLATTERS the CPU: at the full population adaptC's double-indirect gather (CMAES.cpp.base:703-704) no longer fits the caches
    (measured: `--impl reference`, which runs real full-size generations)."""
    from oracle import oracle as O
    from korali_b200._abi import INJ_BD
    n, lam = WORKLOAD["n"], WORKLOAD["population_size"]
    kw = dict(WORKLOAD); kw["population_size"] = sample_lambda
    o = O.Oracle(**kw)
    o.set_scalar("Oracle/RNG Kind", 1)
    ident = np.concatenate([np.eye(n).ravel(), np.ones(n)])
    times = []
    for it in range(warmup + steps):
        o.inject(INJ_BD, ident)              # eigen timed separately below
        t0 = time.perf_counter()
        o.run_generation()
        t1 = time.perf_counter()
        if it >= warmup:
            times.append(t1 - t0)
    c = o.get("Covariance Matrix").reshape(n, n)
    t0 = time.perf_counter(); O.eigen(c); t_eig = time.perf_counter() - t0
    t_pop = float(np.mean(times))
    t_full = t_eig + t_pop * (lam / sample_lambda)
    return {"gens_per_sec": 1.0 / t_full, "t_eigen_s": t_eig, "t_population_sample_s": t_pop, "sample_lambda": sample_lambda,
            "ms_per_step": 1e3 * t_full}


REF_MAX_GENERATIONS = 3        # real full-size generations timed by --impl reference at --gpus 1 (one at --gpus N > 1: the CPU figure does not depend on N) ...
REF_TIME_BUDGET_S = 900.0      # ... as long as the next one is expected to end inside this budget (at least one is always run)


def reference_arm(args, rank):
    """--impl reference: REAL config-3 generations (N = 1000, lambda = 65536, own eigendecomposition, the reference's own RNG:
    MT19937 + polar Box-Muller) of the reference algorithm on the host — oracle/okcma.c, the loop-for-loop C restatement of
    CMAES.cpp.base (the reference itself cannot be built in this image: GSL, Eigen and meson-generated sources are absent,
    DESIGN.md section 5). One thread, because the reference solver is single-threaded (SURVEY F2: no OpenMP in CMAES.cpp.base; the
    Concurrent / Distributed conduits only parallelise the user model, which is 0.1 % of a generation here). A generation costs
    minutes on a host core, so at most REF_MAX_GENERATIONS are timed inside REF_TIME_BUDGET_S, without warm-up generations
    (nothing to warm on the CPU); `steps` in the line is the number actually timed."""
    if rank != 0:
        return
    from oracle import oracle as O
    lam = WORKLOAD["population_size"]
    o = O.Oracle(**WORKLOAD)
    o.set_scalar("Termination Criteria/Max Model Evaluations", 1e18)
    times, phases = [], []
    t_begin = time.perf_counter()
    for g in range(max(1, min(args.steps, REF_MAX_GENERATIONS if args.gpus <= 1 else 1))):
        t0 = time.perf_counter(); o.ask(); t1 = time.perf_counter(); o.eval(); t2 = time.perf_counter(); o.tell(); t3 = time.perf_counter()
        times.append(t3 - t0); phases.append((t1 - t0, t2 - t1, t3 - t2))
        print("reference arm: generation %d  ask %.1f s  eval %.1f s  tell %.1f s" % (g + 1, t1 - t0, t2 - t1, t3 - t2), file=sys.stderr, flush=True)
        if (time.perf_counter() - t_begin) + max(times) > REF_TIME_BUDGET_S:
            break
    if args.dump_outputs:
        dump_outputs(o, args.dump_outputs)
    t_gen = float(np.mean(times))
    gps = 1.0 / t_gen
    ph = np.mean(np.array(phases), axis=0)
    sample = ("oracle/okcma.c (C restatement of CMAES.cpp.base, gcc -O2 -ffp-contract=off), 1 thread, %d REAL generation(s) at the full "
              "size N=1000 lambda=65536 incl. the eigendecomposition: prepareGeneration %.1f s, evaluation %.1f s, updateDistribution %.1f s "
              "per generation" % (len(times), ph[0], ph[1], ph[2]))
    line = {"impl": "reference", "metric": METRIC, "value": gps, "unit": UNIT, "n_gpus": args.gpus, "steps": len(times),
            "warmup": 0, "requested_steps": args.steps, "requested_warmup": args.warmup, "ms_per_step": 1e3 * t_gen,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "samples_per_sec": gps * lam,
            "config": {"workload": WORKLOAD_NAME, "n": WORKLOAD["n"], "lambda": lam, "mu": lam // 2},
            "cpu_baseline": {"value": gps, "unit": UNIT, "cores": 1, "kind": "port", "sample": sample},
            "e2e": {"value": gps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def hbm_block(phases, steps, n, lam_local, mu_local, hbm_peak):
    """Achieved GB/s of the bandwidth-side kernels (SURVEY 8d: K1 rng, K3 objective, K4 sort, K5 gather-mean)."""
    work = {"rng": ("philox_normal_kernel: Z written (FP64 Box-Muller bound)", 8.0 * n * lam_local),
            "objective": ("objective_kernel: Y read", 8.0 * n * lam_local),
            "sort": ("radix sort, 8 passes x 12 B x lambda (sort_fused_kernel: one cooperative launch, bound by its 16 grid barriers)", 8 * 12.0 * lam_local),
            "gather_mean": ("gather_mean + mean_reduce: selected rows read + S written", 2 * 8.0 * n * mu_local)}
    out = {}
    for k, (what, nbytes) in work.items():
        ms = phases[k][0] / steps
        gbps = nbytes / (ms * 1e-3) * 1e-9 if ms > 0 else 0.0
        out[k] = {"what": what, "bytes": nbytes, "ms": ms, "GBps": gbps, "frac_of_hbm_peak": (gbps / hbm_peak) if hbm_peak else None}
    return out


def gemm_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the shipped (persistent) gemm_tn_tma_kernel at config 3 on one
    GPU, from the committed `ncu --set full` summary (profiles/r02_ncu_gemm_tn_tma.json; written by profiles/ncu_summary.py)."""
    p = os.path.join(ROOT, "profiles", "r02_ncu_gemm_tn_tma.json")
    if not os.path.exists(p):
        return None, "no ncu capture committed"
    d = json.load(open(p))
    return d.get("dram_bytes_read", 0) + d.get("dram_bytes_write", 0), os.path.relpath(p, ROOT)


def korali_experiment(max_generations):
    """The user-facing call: a Korali script for config 3 (device conduit, built-in device objective)."""
    import korali_b200 as korali
    e = korali.Experiment()
    e["Random Seed"] = WORKLOAD["seed"]
    e["Problem"]["Type"] = "Optimization"
    e["Problem"]["Objective Function"] = "Ellipsoid"
    for i in range(WORKLOAD["n"]):
        e["Variables"][i]["Name"] = "X%d" % i
        e["Variables"][i]["Initial Value"] = WORKLOAD["initial_value"]
        e["Variables"][i]["Initial Standard Deviation"] = WORKLOAD["initial_stddev"]
    e["Solver"]["Type"] = "Optimizer/CMAES"
    e["Solver"]["Population Size"] = WORKLOAD["population_size"]
    e["Solver"]["Termination Criteria"]["Max Generations"] = max_generations
    e["Solver"]["Termination Criteria"]["Max Model Evaluations"] = 1e18
    e["Console Output"]["Verbosity"] = "Silent"
    e["File Output"]["Enabled"] = False
    return korali, e


def e2e_through_engine(steps, warmup, devices):
    """generations/s of generations warmup+1 .. warmup+steps through korali_b200.Engine().run(e), wall clock around the calls:
    (time of a run of warmup+steps generations) - (time of a run of warmup generations), both from a fresh Experiment with the same
    seed (same trajectory), so that experiment set-up, handle creation, communicator set-up and the first-use allocations cancel.
    A throw-away run absorbs the once-per-process costs (CUDA contexts on all devices, NCCL bootstrap); each length is run twice
    and the faster one counts (the set-up part of a run jitters by more than a generation when a communicator is built)."""
    def run(gens):
        korali, e = korali_experiment(gens)
        k = korali.Engine()
        k["Conduit"]["Type"] = "Device"
        if devices > 1:
            k["Conduit"]["Devices"] = devices
        t0 = time.perf_counter()
        k.run(e)
        best = e["Results"]["Best Sample"]["F(x)"]      # host read of the result
        dt = time.perf_counter() - t0
        assert e["Current Generation"] == gens
        return dt, best
    run(1)
    # the difference of two wall-clock runs carries the jitter of their set-up parts (tens of ms when a communicator is built):
    # at least 100 generations keep it below a few per cent of the difference
    # (the set-up part — handle creation, communicator, one context per device — jitters by ~0.1 s: 200 / 300 generations, three runs each;
    # a 100-generation difference once gave an e2e 18 % above the device-timed value)
    k_e2e = max(steps, 200 if devices == 1 else 300)
    reps = 3
    out = {"short": min(run(warmup)[0] for _ in range(reps))}
    longs = [run(warmup + k_e2e) for _ in range(reps)]
    out["long"] = min(t for t, _ in longs)
    out["best"] = longs[0][1]
    out["generations"] = k_e2e
    out["gens_per_sec"] = k_e2e / max(out["long"] - out["short"], 1e-9)
    return out


# ---------------------------------------------------------------------------------------------------------
def timed_leg(s, steps, timers, torch, barrier):
    """K generations between two CUDA events on the launching stream (libkcma uses the legacy default stream = torch's)."""
    if timers:
        s.timing_enable(True); s.timing_reset()
    barrier()
    l0 = s.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        s.run_generation()
    e1.record()
    barrier()
    return e0.elapsed_time(e1), s.launch_count() - l0


def ours_arm(args, rank, world):
    import torch
    import torch.distributed as dist
    from korali_b200 import _lib
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    n, lam = WORKLOAD["n"], WORKLOAD["population_size"]
    mu = lam // 2

    def make_solver(nranks=world, r=rank):
        s = _lib.Solver(device=local_rank, rank=r, nranks=nranks, **WORKLOAD)
        s.set_scalar("Termination Criteria/Max Model Evaluations", 1e18)
        if nranks > 1:
            uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
            if rank == 0:
                uid = torch.tensor(list(_lib.comm_unique_id()), dtype=torch.uint8, device="cuda")
            dist.broadcast(uid, 0)
            s.comm_init(bytes(uid.cpu().tolist()))
        return s

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- leg A (`value`): the product path as shipped — generations W+1 .. W+K from a fresh state, one kcma_run_generation per
    # step (N = 1: one CUDA-graph replay per generation from the third generation on), no phase timers
    s = make_solver()
    for _ in range(args.warmup):
        s.run_generation()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    ms, launches = timed_leg(s, args.steps, False, torch, barrier)
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(s, args.dump_outputs)
    best = s.scalar("Best Ever Value")
    # ---- e2e through kcma_run (termination chain on the host every generation) on the same handle, next K generations
    barrier()
    t0 = time.perf_counter()
    done = s.run(args.steps)
    s.scalar("Best Ever Value")                 # device -> host read of the step's result
    torch.cuda.synchronize()
    t_run = time.perf_counter() - t0
    s.close()
    # ---- leg B (phases, roofline): the SAME generations W+1 .. W+K from a fresh state with eager launches and a CUDA-event pair
    # around every phase (the events keep the kernels of a generation from overlapping: slightly slower than leg A)
    s = make_solver()
    for _ in range(args.warmup):
        s.run_generation()
    ms_eager, launches_eager = timed_leg(s, args.steps, True, torch, barrier)
    phase_names = ["eigen", "eigen_sytrd", "eigen_dc", "eigen_back", "rng", "sample_gemm", "objective", "sort", "gather_mean", "rank_mu",
                   "paths", "collectives", "generation"]
    phases = {p: s.timing(p) for p in phase_names}
    sweeps = s.timing("eigen_sweeps")[1] / args.steps
    s.timing_enable(False)
    # ---- N > 1: correctness of the sharded run next to its speed — 3 generations from a fresh state against a 1-rank replica
    parity = None
    if world > 1:
        sh = make_solver()
        rep = _lib.Solver(device=local_rank, **WORKLOAD) if rank == 0 else None
        parity = {}
        for g in range(3):
            sh.run_generation()
            if rep is not None:
                rep.run_generation()
                if g == 0:
                    parity["value_vector_bit_exact_g1"] = bool(np.array_equal(sh.get("Value Vector"), rep.get("Value Vector")))
                    parity["sorting_index_equal_g1"] = bool(np.array_equal(sh.get_index("Sorting Index"), rep.get_index("Sorting Index")))
                c, c1 = sh.get("Covariance Matrix"), rep.get("Covariance Matrix")
                parity["relerr_C_g%d" % (g + 1)] = float(np.abs(c - c1).max() / np.abs(c1).max())
                m, m1 = sh.get("Current Mean"), rep.get("Current Mean")
                parity["relerr_mean_g%d" % (g + 1)] = float(np.abs(m - m1).max() / np.abs(m1).max())
                parity["relerr_sigma_g%d" % (g + 1)] = abs(sh.scalar("Sigma") - rep.scalar("Sigma")) / rep.scalar("Sigma")
        sh.close()
        if rep is not None:
            rep.close()
        t = torch.tensor([ms, t_run * 1e3, ms_eager], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, t_run, ms_eager = float(t[0]), float(t[1]) * 1e-3, float(t[2])
    s.close()
    if world > 1:   # the ranks are done with one another: the user-facing leg below drives all N devices from rank 0's process
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    # ---- e2e through the user-facing API: korali_b200.Engine().run(e), k["Conduit"]["Devices"] = N (one process, one host thread and
    # one handle per device; the other torchrun ranks have exited and left their GPUs free)
    eng = e2e_through_engine(args.steps, args.warmup, world)
    peaks = load_peaks()
    ms_step = ms / args.steps
    gens = 1e3 / ms_step
    f_sample, f_rank = flops_per_generation(n, lam // world, mu // world)
    gemm_ms, gemm_calls = phases["sample_gemm"]
    gemm_avg = gemm_ms / max(gemm_calls, 1)
    achieved = f_sample / (gemm_avg * 1e-3) * 1e-12 if gemm_avg > 0 else 0.0
    peak = peaks.get("fp64_dgemm_tflops_sustained")
    rk_ms, rk_calls = phases["rank_mu"]
    rk_avg = rk_ms / max(rk_calls, 1)
    cpu = cpu_bounded_sample(8, 1) if world == 1 else None   # ~10-20 s of host work
    traffic, traffic_src = gemm_traffic() if world == 1 else (None, None)
    eig_ms = phases["eigen"][0] / args.steps
    tridiag = phases["eigen_sytrd"][1] > 0
    e2e_value = eng["gens_per_sec"] if eng else done / t_run
    line = {
        "metric": METRIC, "value": gens, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "samples_per_sec": gens * lam,
        "config": {"workload": WORKLOAD_NAME, "n": n, "lambda": lam, "mu": mu, "parallelism": "population sharded x%d" % world,
                   "l2_hygiene": "inputs larger than L2: Z and Y are %.0f MB each per rank, re-streamed every generation" % (8.0 * n * lam / world / 1e6),
                   "host_io": "the generation loop takes no per-step host input (samples are drawn on the device from Philox(seed, generation) "
                              "counters, the objective is a device kernel): h2d 0 B, d2h 288 B = sizeof(DevScalars) for the termination chain",
                   "generations_timed": "%d..%d from a fresh state (value and phases; e2e runs on from the same fresh state to generation W+Ke)" % (args.warmup + 1, args.warmup + args.steps),
                   "best_ever_value_after_run": best},
        "value_path": "kcma_run_generation x K, CUDA events on the launching stream" + (", one CUDA-graph replay per generation" if world == 1 else ", eager launches + NCCL"),
        "value_eager_with_phase_timers": 1e3 / (ms_eager / args.steps),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 288,
                "through": "korali_b200.Engine().run(e) (k['Conduit']['Type'] = 'Device'%s, Objective Function 'Ellipsoid'), wall clock; "
                           "(run of W+Ke generations) - (run of W generations), Ke = max(K, 200) on one device and max(K, 300) on several, each the fastest of three runs"
                           % (", k['Conduit']['Devices'] = %d" % world if world > 1 else ""),
                "engine_run_seconds": {"W_generations": eng["short"], "W_plus_Ke_generations": eng["long"], "Ke": eng["generations"]} if eng else None,
                "kcma_run_generations_per_sec": done / t_run,
                "note": "no per-step host input exists on this path: h2d is 0 by construction, d2h is the scalar block the termination chain reads"},
        "gpu_launches": int(launches),
        "gpu_launches_eager_leg": int(launches_eager),
        "clocks": clk,
        "roofline": {"kernel": "gemm_tn_tma_kernel (sampling GEMM Y = Z (B D)^T, TMA + mbarrier + DMMA.8x8x4)", "bound": "tensor",
                     "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": (achieved / peak) if peak else None,
                     "traffic": traffic, "traffic_unit": "bytes per launch", "traffic_source": traffic_src,
                     "peak_source": "MEASURED_FP64.json (builder-measured; the driver's MEASURED_PEAKS.json has no FP64 entry): cuBLAS DGEMM 8192^3 "
                                    "sustained 35.44 TFLOP/s on this pool's B200; raw DMMA.8x8x4 issue peak 37.1 TFLOP/s",
                     "frac_of_dmma_issue_peak": (achieved / peaks["fp64_dmma_issue_tflops"]) if peaks.get("fp64_dmma_issue_tflops") else None,
                     "algorithmic_flops_per_launch": f_sample, "avg_launch_ms": gemm_avg},
        "phases_ms_per_generation": {k: (v[0] / args.steps) for k, v in phases.items()},
        "rank_mu": {"kernel": "syrk_sk_tma_kernel (stream-K over the lower-triangular tiles, triangular warp tiling of the diagonal tiles)", "avg_ms": rk_avg, "achieved_tflops": (f_rank / (rk_avg * 1e-3) * 1e-12) if rk_avg > 0 else 0.0,
                    "algorithmic_flops_per_launch": f_rank},
        # the HBM-side kernels of a generation: algorithmic bytes / phase time against the measured copy bandwidth
        "hbm_kernels": hbm_block(phases, args.steps, n, lam // world, mu // world, peaks.get("hbm_gbs", 6547.2)),
        "gens_per_sec_excluding_eigen": 1e3 / max(ms_eager / args.steps - eig_ms, 1e-9),
    }
    if tridiag:
        line["eigen"] = {"solver": "Householder tridiagonalisation (sytrd_reg_kernel: one persistent cooperative launch, trailing matrix resident in the register "
                                   "files of all SMs, one LL all-to-all exchange through L2 per column) + divide & conquer (dc.cu) + compact-WY back-transform on "
                                   "DMMA GEMMs (Q accumulated on a side stream beside the divide & conquer stage); replicated on every rank",
                         "avg_ms": eig_ms, "sytrd_ms": phases["eigen_sytrd"][0] / args.steps, "dc_ms": phases["eigen_dc"][0] / args.steps,
                         "back_transform_ms": phases["eigen_back"][0] / args.steps,
                         "bound": "latency: N-1 dependent Householder steps, each one exchange through L2",
                         "us_per_householder_step": phases["eigen_sytrd"][0] / args.steps * 1e3 / (n - 1),
                         "nominal_flops": 4.0 / 3.0 * n ** 3 + 4.0 / 3.0 * n ** 3 + 4.0 * n ** 3,
                         "achieved_tflops": ((4.0 / 3.0 + 4.0 / 3.0 + 4.0) * n ** 3 / (eig_ms * 1e-3) * 1e-12) if eig_ms > 0 else 0.0}
    else:
        line["eigen"] = {"solver": "jacobi_pipe_kernel (KCMA_EIGEN=jacobi: persistent cooperative one-sided Jacobi; replicated on every rank)",
                         "avg_ms": eig_ms, "sweeps_per_generation": sweeps, "executed_flops_per_sweep": 12.0 * n ** 3}
    if parity is not None:
        line["parity_vs_n1"] = parity
    if cpu:
        line["cpu_baseline"] = {"value": cpu["gens_per_sec"], "unit": UNIT, "cores": 1, "kind": "port",
                                "sample": "oracle/okcma.c, 1 thread: %d of %d samples per step (%.3f s) extrapolated linearly in lambda + one "
                                          "1000x1000 eigendecomposition (%.2f s). The extrapolation flatters the CPU (adaptC's gather leaves the caches at "
                                          "the full population): `bench.py --impl reference` times real full-size generations"
                                          % (cpu["sample_lambda"], lam, cpu["t_population_sample_s"], cpu["t_eigen_s"])}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the state after the last timed generation as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        reference_arm(args, rank)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        # convenience: re-launch under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus), "--master-addr", "127.0.0.1",
               "--master-port", "29511", os.path.abspath(__file__), "--gpus", str(args.gpus), "--steps", str(args.steps), "--warmup", str(args.warmup)]
        if args.dump_outputs:
            cmd += ["--dump-outputs", args.dump_outputs]
        sys.exit(subprocess.call(cmd))
    ours_arm(args, rank, world)


if __name__ == "__main__":
    main()
